// tests/support/ragged_dev.cu -- device problems for the ragged batched solves (dogleg_gpu_optimize_dense_batched_ragged)
// and their zero-padded uniform twins, used by tests/test_gpu_batched_ragged.py and profiles/micro/batched_ragged.py.
// Not product code.
//
// Problem b has Nmeas[b] measurements. The dense kind: the first Nmeas[b] rows of k_gen_batched's problem seed + b
// (problems_dev.cu), i.e. the numbers of the host's Problem.dense(N, Nmeas[b], seed + b). The sample kind: the
// reference's sample surface on the first Nmeas[b] of its points. Data are stored ragged (row_off); the ragged
// callback writes the ragged layout, the padded one the uniform B x Mpad layout with rows >= Nmeas[b] exact zeros.
// Both evaluate a row with the same code, so the rows < Nmeas[b] of the two layouts are bit-identical.
#include <cuda_runtime.h>
#include <cstdlib>
#include <vector>
#include "problems.h"

// problems_dev.cu's counter hash and model (bit-identical)
__host__ __device__ static inline unsigned long long dev_splitmix64(unsigned long long z)
{
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__host__ __device__ static inline double dev_uniform(unsigned long long seed, unsigned long long stream, unsigned long long idx)
{
  unsigned long long h = dev_splitmix64(dev_splitmix64(seed * 0x100000001B3ull + stream) ^ idx);
  return ((double)(h >> 11) + 0.5) * (2.0 / 9007199254740992.0) - 1.0;
}
__device__ __forceinline__ double phi(double p)  { return p + 0.1 * p * p * p; }
__device__ __forceinline__ double dphi(double p) { return 1.0 + 0.3 * p * p; }

struct dlb_ragged_problem
{
  int B, N, kind;             // kind 0: dense (k_gen_batched rows), 1: the sample surface
  int Mpad;                   // the longest count: the padded layout's Nmeas
  long long rows;             // sum of the counts
  long long* d_row_off;       // B + 1
  double* d_A;                // dense: rows x N; sample: the points (x, y)
  double* d_b;                // dense: rows; sample: the measurements of the points
  int ncalls;
};

// the problem of global row i: the last b with row_off[b] <= i (empty problems share their offset with the next)
__device__ __forceinline__ long long find_problem(const long long* off, int B, long long i)
{
  int lo = 0, hi = B;                         // off[lo] <= i < off[hi]
  while(hi - lo > 1) { const int mid = (lo + hi) >> 1; if(off[mid] <= i) lo = mid; else hi = mid; }
  return lo;
}
// output row i of either layout: its problem, its row r within the problem and whether r < Nmeas[prob].
// Mpad == 0: the ragged layout (i is the global row); else the padded one (i = prob * Mpad + r).
struct RowMap { long long prob, r; bool valid; };
__device__ __forceinline__ RowMap map_row(long long i, int Mpad, const long long* off, int B)
{
  RowMap m;
  if(Mpad == 0) { m.prob = find_problem(off, B, i); m.r = i - off[m.prob]; m.valid = true; }
  else { m.prob = i / Mpad; m.r = i - m.prob * Mpad; m.valid = m.r < off[m.prob + 1] - off[m.prob]; }
  return m;
}

__global__ void k_gen_ragged(int B, int N, unsigned long long seed, const long long* off, double* A, double* b, double* p0)
{
  const long long rows = off[B];
  for(long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += (long long)gridDim.x * blockDim.x)
  {
    const long long prob = find_problem(off, B, i), r = i - off[prob];
    const unsigned long long sd = seed + (unsigned long long)prob;
    double s = 0.0;
    for(int k = 0; k < N; k++)
    {
      const double a = dev_uniform(sd, 1, (unsigned long long)(r * N + k));
      A[i * N + k] = a;
      s += a * phi(dev_uniform(sd, 2, k));
    }
    b[i] = s + 0.01 * dev_uniform(sd, 4, (unsigned long long)r);
  }
  for(long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)B * N; i += (long long)gridDim.x * blockDim.x)
  {
    const long long prob = i / N; const int k = (int)(i - prob * N);
    const unsigned long long sd = seed + (unsigned long long)prob;
    p0[i] = dev_uniform(sd, 2, k) + 0.5 * dev_uniform(sd, 3, k);
  }
}

// dense kind, as problems_dev.cu's k_model_dense: `width` lanes per row (the power of two >= N, <= 32), shuffle tree
__global__ void k_ragged_dense(long long nout, int Mpad, int B, int N, int width, const long long* __restrict__ off,
                               const double* __restrict__ A, const double* __restrict__ bv, const double* __restrict__ p,
                               const int* __restrict__ active, double* __restrict__ x, double* __restrict__ J)
{
  const int per_warp = 32 / width;
  const int lane = threadIdx.x & 31;
  const int sub = lane / width, k = lane % width;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for(long long i0 = warp * per_warp; i0 < nout; i0 += nwarps * per_warp)
  {
    const long long i = i0 + sub;
    const RowMap m = map_row(i < nout ? i : nout - 1, Mpad, off, B);
    const bool on = i < nout && (!active || active[m.prob]);
    const long long src = off[m.prob] + m.r;
    double s = 0.0;
    for(int kk = k; kk < N; kk += width)
      if(on)
      {
        const double pk = p[m.prob * N + kk];
        const double a = m.valid ? A[src * N + kk] : 0.0;
        J[i * N + kk] = m.valid ? a * dphi(pk) : 0.0;
        s += a * phi(pk);
      }
    for(int o = width >> 1; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o, width);
    if(on && k == 0) x[i] = m.valid ? s - bv[src] : 0.0;
  }
}

// sample kind, as problems_dev.cu's k_model_sample_batched; point r of problem b is point r of the surface
__global__ void k_ragged_sample(long long nout, int Mpad, int B, const long long* __restrict__ off,
                                const double* __restrict__ xy, const double* __restrict__ meas, const double* __restrict__ p,
                                const int* __restrict__ active, double* __restrict__ x, double* __restrict__ J)
{
  for(long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nout; i += (long long)gridDim.x * blockDim.x)
  {
    const RowMap m = map_row(i, Mpad, off, B);
    if(active && !active[m.prob]) continue;
    double* g = J + i * 6;
    if(!m.valid)
    {
      for(int k = 0; k < 6; k++) g[k] = 0.0;
      x[i] = 0.0;
      continue;
    }
    const double* pp = p + m.prob * 6;
    const double X = xy[2 * m.r], Y = xy[2 * m.r + 1];
    g[0] = pp[1]*X*X; g[1] = pp[0]*X*X + pp[2]*Y*Y; g[2] = pp[1]*Y*Y + X*Y; g[3] = X; g[4] = Y; g[5] = 1.0;
    x[i] = pp[0]*pp[1]*X*X + pp[1]*pp[2]*Y*Y + pp[2]*X*Y + pp[3]*X + pp[4]*Y + pp[5] - meas[m.r];
  }
}

static dlb_ragged_problem* create_layout(int B, int N, const unsigned int* Nmeas)
{
  dlb_ragged_problem* D = (dlb_ragged_problem*)calloc(1, sizeof(*D));
  D->B = B; D->N = N;
  std::vector<long long> off((size_t)B + 1, 0);
  for(int b = 0; b < B; b++)
  {
    off[b + 1] = off[b] + Nmeas[b];
    if((int)Nmeas[b] > D->Mpad) D->Mpad = (int)Nmeas[b];
  }
  D->rows = off[B];
  if(cudaMalloc(&D->d_row_off, sizeof(long long) * ((size_t)B + 1)) != cudaSuccess) { free(D); return NULL; }
  cudaMemcpy(D->d_row_off, off.data(), sizeof(long long) * ((size_t)B + 1), cudaMemcpyHostToDevice);
  return D;
}

extern "C" void dlb_ragged_free(dlb_ragged_problem* D)
{
  if(!D) return;
  cudaFree(D->d_row_off); cudaFree(D->d_A); cudaFree(D->d_b);
  free(D);
}

// the dense kind; p0_host: B x N start points (k_gen_batched's)
extern "C" dlb_ragged_problem* dlb_ragged_create(int B, int N, const unsigned int* Nmeas, unsigned long long seed, double* p0_host)
{
  dlb_ragged_problem* D = create_layout(B, N, Nmeas);
  if(!D) return NULL;
  double* d_p0 = 0;
  if(cudaMalloc(&D->d_A, sizeof(double) * (size_t)(D->rows ? D->rows : 1) * N) != cudaSuccess ||
     cudaMalloc(&D->d_b, sizeof(double) * (size_t)(D->rows ? D->rows : 1)) != cudaSuccess ||
     cudaMalloc(&d_p0, sizeof(double) * (size_t)B * N) != cudaSuccess) { cudaFree(d_p0); dlb_ragged_free(D); return NULL; }
  k_gen_ragged<<<1184, 256>>>(B, N, seed, D->d_row_off, D->d_A, D->d_b, d_p0);
  cudaMemcpy(p0_host, d_p0, sizeof(double) * (size_t)B * N, cudaMemcpyDeviceToHost);
  cudaFree(d_p0);
  if(cudaDeviceSynchronize() != cudaSuccess) { dlb_ragged_free(D); return NULL; }
  return D;
}

// the sample kind on prefixes of the host sample problem's points (Nmeas[b] <= its M)
extern "C" dlb_ragged_problem* dlb_ragged_create_sample(const dlb_problem* P, int B, const unsigned int* Nmeas)
{
  for(int b = 0; b < B; b++)
    if(Nmeas[b] > (unsigned int)P->M) return NULL;
  dlb_ragged_problem* D = create_layout(B, 6, Nmeas);
  if(!D) return NULL;
  D->kind = 1;
  if(cudaMalloc(&D->d_A, sizeof(double) * 2 * (size_t)P->M) != cudaSuccess ||
     cudaMalloc(&D->d_b, sizeof(double) * (size_t)P->M) != cudaSuccess) { dlb_ragged_free(D); return NULL; }
  cudaMemcpy(D->d_A, P->Ax, sizeof(double) * 2 * (size_t)P->M, cudaMemcpyHostToDevice);
  cudaMemcpy(D->d_b, P->b, sizeof(double) * (size_t)P->M, cudaMemcpyHostToDevice);
  if(cudaDeviceSynchronize() != cudaSuccess) { dlb_ragged_free(D); return NULL; }
  return D;
}

extern "C" int dlb_ragged_mpad(const dlb_ragged_problem* D) { return D->Mpad; }
extern "C" long long dlb_ragged_rows(const dlb_ragged_problem* D) { return D->rows; }
extern "C" int dlb_ragged_ncalls(const dlb_ragged_problem* D) { return D->ncalls; }
extern "C" void dlb_ragged_reset(dlb_ragged_problem* D) { D->ncalls = 0; }

static int model_width(int N) { int w = 1; while(w < N && w < 32) w <<= 1; return w; }

static void evaluate(dlb_ragged_problem* D, long long nout, int Mpad, const long long* d_row_off, const double* d_p,
                     double* d_x, double* d_J, const int* d_active, cudaStream_t st)
{
  if(nout > 0)
  {
    if(D->kind == 1)
      k_ragged_sample<<<148 * 8, 256, 0, st>>>(nout, Mpad, D->B, d_row_off, D->d_A, D->d_b, d_p, d_active, d_x, d_J);
    else
      k_ragged_dense<<<148 * 16, 256, 0, st>>>(nout, Mpad, D->B, D->N, model_width(D->N), d_row_off, D->d_A, D->d_b, d_p,
                                               d_active, d_x, d_J);
  }
  D->ncalls++;
}

// dogleg_gpu_callback_dense_ragged_t: the solve's own offsets, as a user's callback would take them
extern "C" void dlb_ragged_cb(const double* d_p, double* d_x, double* d_J, const long long* d_row_off, const int* d_active,
                              int B, void* stream, void* cookie)
{
  dlb_ragged_problem* D = (dlb_ragged_problem*)cookie;
  (void)B;
  evaluate(D, D->rows, 0, d_row_off, d_p, d_x, d_J, d_active, (cudaStream_t)stream);
}
// dogleg_gpu_callback_dense_batched_t of the same batch zero-padded to Nmeas = Mpad
extern "C" void dlb_ragged_cb_padded(const double* d_p, double* d_x, double* d_J, const int* d_active, int B,
                                     void* stream, void* cookie)
{
  dlb_ragged_problem* D = (dlb_ragged_problem*)cookie;
  evaluate(D, (long long)B * D->Mpad, D->Mpad, D->d_row_off, d_p, d_x, d_J, d_active, (cudaStream_t)stream);
}
extern "C" void* dlb_ragged_cb_ptr(void)        { return (void*)&dlb_ragged_cb; }
extern "C" void* dlb_ragged_cb_padded_ptr(void) { return (void*)&dlb_ragged_cb_padded; }
