// tests/support/products_dev.cu -- device "user callbacks" of the dense-products entry points
// (dogleg_gpu_optimize_dense_products, dogleg_gpu_optimize_dense_products_batched), used by
// tests/test_gpu_products_device.py and profiles/micro/batched_products.py. Not product code.
//
// The problems are the synthetic ones of problems.c / problems_dev.cu (same formulas, same splitmix64
// counter hash): B dense problems of k_gen_batched's family, stored in HBM or regenerated on every call
// (procedural: nothing is stored, so a batch may be far larger than its Jacobians would be in HBM), the
// reference's sample surface from B start points, or one dense host problem.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include "problems.h"

// device copy of problems.h's splitmix64 counter hash (bit-identical)
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

struct dlb_prod_problem
{
  int N, M, B, model;
  double* d_A;          // PM_DENSE: B x M x N; PM_SAMPLE: M (x, y) pairs; PM_PROCEDURAL: none
  double* d_b;          // PM_DENSE: B x M; PM_SAMPLE: M
  unsigned long long seed;
  int packed, poison_inactive;       // JtJ layout (0 full, 1 packed upper); NaN into every output of inactive problems
  float ms_total; int ncalls; int timing;
  cudaEvent_t e0, e1;
};

// ---- dense-products callbacks: |x|^2, J'x and J'J per problem, in the layout the solve asks for ----
// One block takes one problem (and, when J'J has more entries than the block's threads hold, one range
// of them: blockIdx.y). Rows go through shared memory in chunks of R: the block forms each row's gradient
// and residual (one thread per row), then every thread adds the chunk's contribution to its own outputs,
// which are the upper triangle of [J x]'[J x]: J'J, J'x (column N) and |x|^2 (entry N,N).
enum { PM_DENSE = 0, PM_PROCEDURAL = 1, PM_SAMPLE = 2 };
#define PR_NT 128
#define PR_SLOTS 5
__global__ void __launch_bounds__(PR_NT)
k_model_products(int B, int M, int N, int R, int model, unsigned long long seed, const double* __restrict__ A,
                 const double* __restrict__ bvec, const double* __restrict__ p, const int* __restrict__ active,
                 int packed, int poison, double* __restrict__ n2x, double* __restrict__ Jtx, double* __restrict__ JtJ)
{
  extern __shared__ double sh[];
  const int LG = N + 1, tid = threadIdx.x;
  double* g = sh;                          // R rows: gradient (N), residual
  double* f = g + (size_t)R * LG;          // phi(p_k), dphi(p_k), phi(p_true_k)
  const int nout = (N + 1) * (N + 2) / 2;
  int kk[PR_SLOTS], ll[PR_SLOTS];
#pragma unroll
  for(int s = 0; s < PR_SLOTS; s++)
  {
    const int o = (blockIdx.y * PR_SLOTS + s) * PR_NT + tid;
    kk[s] = -1; ll[s] = 0;
    if(o < nout)
    {
      int k = 0, start = 0;
      while(o >= start + LG - k) { start += LG - k; k++; }
      kk[s] = k; ll[s] = k + (o - start);
    }
  }
  const size_t S = packed ? (size_t)N * (N + 1) / 2 : (size_t)N * N;
  for(int prob = blockIdx.x; prob < B; prob += gridDim.x)
  {
    const bool on = !active || active[prob];
    if(!on && !poison) continue;
    double acc[PR_SLOTS];
#pragma unroll
    for(int s = 0; s < PR_SLOTS; s++) acc[s] = on ? 0.0 : __longlong_as_double(0x7ff8000000000000ll);
    const unsigned long long sd = seed + (unsigned long long)prob;
    __syncthreads();
    for(int k = tid; k < N && on; k += PR_NT)
    {
      const double pk = p[(size_t)prob * N + k];
      f[k] = phi(pk); f[N + k] = dphi(pk);
      f[2 * N + k] = model == PM_PROCEDURAL ? phi(dev_uniform(sd, 2, k)) : 0.0;
    }
    for(int r0 = 0; r0 < M && on; r0 += R)
    {
      const int nr = min(R, M - r0);
      __syncthreads();
      if(model == PM_DENSE)
        for(int e = tid; e < nr * N; e += PR_NT) g[(e / N) * LG + e % N] = A[((size_t)prob * M + r0) * N + e];
      __syncthreads();
      for(int r = tid; r < nr; r += PR_NT)
      {
        double* gr = g + (size_t)r * LG;
        const int i = r0 + r;
        if(model == PM_SAMPLE)
        { // problems.c sample_eval()
          const double* pp = p + (size_t)prob * 6;
          const double X = A[2 * i], Y = A[2 * i + 1];
          gr[0] = pp[1]*X*X; gr[1] = pp[0]*X*X + pp[2]*Y*Y; gr[2] = pp[1]*Y*Y + X*Y; gr[3] = X; gr[4] = Y; gr[5] = 1.0;
          gr[6] = pp[0]*pp[1]*X*X + pp[1]*pp[2]*Y*Y + pp[2]*X*Y + pp[3]*X + pp[4]*Y + pp[5] - bvec[i];
        }
        else
        {
          double s = 0.0, bs = 0.0;
          for(int k = 0; k < N; k++)
          { // the procedural entries are k_gen_batched's, generated where they are used
            const double a = model == PM_DENSE ? gr[k] : dev_uniform(sd, 1, (unsigned long long)i * N + k);
            gr[k] = a * f[N + k];
            s += a * f[k];
            bs += a * f[2 * N + k];
          }
          const double bi = model == PM_DENSE ? bvec[(size_t)prob * M + i] : bs + 0.01 * dev_uniform(sd, 4, (unsigned long long)i);
          gr[N] = s - bi;
        }
      }
      __syncthreads();
      for(int r = 0; r < nr; r++)
      {
        const double* gr = g + (size_t)r * LG;
#pragma unroll
        for(int s = 0; s < PR_SLOTS; s++)
          if(kk[s] >= 0) acc[s] = fma(gr[kk[s]], gr[ll[s]], acc[s]);
      }
    }
#pragma unroll
    for(int s = 0; s < PR_SLOTS; s++)
    {
      const int k = kk[s], l = ll[s];
      if(k < 0) continue;
      if(l == N) { if(k == N) n2x[prob] = acc[s]; else Jtx[(size_t)prob * N + k] = acc[s]; }
      else if(packed) JtJ[prob * S + (size_t)k * N - (size_t)k * (k - 1) / 2 + (l - k)] = acc[s];
      else { JtJ[prob * S + (size_t)k * N + l] = acc[s]; JtJ[prob * S + (size_t)l * N + k] = acc[s]; }
    }
  }
}
static void launch_products(dlb_prod_problem* D, int B, const double* d_p, const int* d_active, double* d_n2x,
                            double* d_Jtx, double* d_JtJ, cudaStream_t st)
{
  const int N = D->N;
  const int R = std::min(128, (40 * 1024 / 8 - 3 * N) / (N + 1));
  const size_t smem = sizeof(double) * ((size_t)R * (N + 1) + 3 * N);
  const int nout = (N + 1) * (N + 2) / 2;
  const dim3 grid(std::min(B, 148 * 16), (nout + PR_NT * PR_SLOTS - 1) / (PR_NT * PR_SLOTS));
  if(D->timing) cudaEventRecord(D->e0, st);
  k_model_products<<<grid, PR_NT, smem, st>>>(B, D->M, N, R, D->model, D->seed, D->d_A, D->d_b, d_p, d_active,
                                              D->packed, D->poison_inactive, d_n2x, d_Jtx, d_JtJ);
  if(D->timing) { cudaEventRecord(D->e1, st); cudaEventSynchronize(D->e1); float ms; cudaEventElapsedTime(&ms, D->e0, D->e1); D->ms_total += ms; }
  D->ncalls++;
}
extern "C" void dlb_prod_cb_batched(const double* d_p, double* d_n2x, double* d_Jtx, double* d_JtJ,
                                    const int* d_active, int B, void* stream, void* cookie)
{
  launch_products((dlb_prod_problem*)cookie, B, d_p, d_active, d_n2x, d_Jtx, d_JtJ, (cudaStream_t)stream);
}
extern "C" void dlb_prod_cb(const double* d_p, double* d_n2x, double* d_Jtx, double* d_JtJ, void* stream, void* cookie)
{
  launch_products((dlb_prod_problem*)cookie, 1, d_p, NULL, d_n2x, d_Jtx, d_JtJ, (cudaStream_t)stream);
}
extern "C" void* dlb_prod_cb_ptr(void)         { return (void*)&dlb_prod_cb; }
extern "C" void* dlb_prod_cb_batched_ptr(void) { return (void*)&dlb_prod_cb_batched; }

// A (B x M x N), b (B x M): the same code as problems_dev.cu's k_gen_batched, so a stored batch equals the
// dense-form batch dlb_dev_problem_create_batched() makes from the same seed
__global__ void k_gen_batched_products(int B, int M, int N, unsigned long long seed, double* A, double* b)
{
  const long long total = (long long)B * M;
  for(long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
  {
    const long long prob = i / M;
    const unsigned long long sd = seed + (unsigned long long)prob;
    double s = 0.0;
    for(int k = 0; k < N; k++)
    {
      const double a = dev_uniform(sd, 1, (unsigned long long)((i - prob * M) * N + k));
      A[i * N + k] = a;
      s += a * phi(dev_uniform(sd, 2, k));
    }
    b[i] = s + 0.01 * dev_uniform(sd, 4, (unsigned long long)(i - prob * M));
  }
}

static dlb_prod_problem* alloc_problem(int N, int M, int B, int model)
{
  dlb_prod_problem* D = (dlb_prod_problem*)calloc(1, sizeof(*D));
  D->N = N; D->M = M; D->B = B; D->model = model;
  cudaEventCreate(&D->e0); cudaEventCreate(&D->e1);
  return D;
}
extern "C" void dlb_prod_problem_free(dlb_prod_problem* D)
{
  if(!D) return;
  cudaFree(D->d_A); cudaFree(D->d_b);
  cudaEventDestroy(D->e0); cudaEventDestroy(D->e1);
  free(D);
}
// B problems of k_gen_batched's family (seed + b for problem b, the host's Problem.dense(N, M, seed + b)), stored
// in HBM (stored != 0) or regenerated by the callback on every call. p0_host: B x N start points.
extern "C" dlb_prod_problem* dlb_prod_problem_create_batched(int B, int M, int N, unsigned long long seed, int stored,
                                                             double* p0_host)
{
  dlb_prod_problem* D = alloc_problem(N, M, B, stored ? PM_DENSE : PM_PROCEDURAL);
  D->seed = seed;
  for(long long prob = 0; prob < B; prob++)
    for(int k = 0; k < N; k++)
      p0_host[prob * N + k] = dev_uniform(seed + prob, 2, k) + 0.5 * dev_uniform(seed + prob, 3, k);
  if(stored)
  {
    if(cudaMalloc(&D->d_A, sizeof(double) * (size_t)B * M * N) != cudaSuccess ||
       cudaMalloc(&D->d_b, sizeof(double) * (size_t)B * M) != cudaSuccess) { dlb_prod_problem_free(D); return NULL; }
    k_gen_batched_products<<<1184, 256>>>(B, M, N, seed, D->d_A, D->d_b);
    if(cudaDeviceSynchronize() != cudaSuccess) { dlb_prod_problem_free(D); return NULL; }
  }
  return D;
}
// from a host problem of problems.c: the sample surface (B copies, each solved from its own start point) or
// one dense problem (B = 1)
extern "C" dlb_prod_problem* dlb_prod_problem_from_host(const dlb_problem* P, int B)
{
  const bool sample = P->kind == 1;
  if(!sample && (!P->Adense || B != 1)) return NULL;
  dlb_prod_problem* D = alloc_problem(P->N, P->M, B, sample ? PM_SAMPLE : PM_DENSE);
  const size_t na = sample ? 2 * (size_t)P->M : (size_t)P->M * P->N;
  if(cudaMalloc(&D->d_A, sizeof(double) * na) != cudaSuccess ||
     cudaMalloc(&D->d_b, sizeof(double) * (size_t)P->M) != cudaSuccess) { dlb_prod_problem_free(D); return NULL; }
  cudaMemcpy(D->d_A, sample ? P->Ax : P->Adense, sizeof(double) * na, cudaMemcpyHostToDevice);
  cudaMemcpy(D->d_b, P->b, sizeof(double) * (size_t)P->M, cudaMemcpyHostToDevice);
  if(cudaDeviceSynchronize() != cudaSuccess) { dlb_prod_problem_free(D); return NULL; }
  return D;
}
extern "C" void dlb_prod_problem_layout(dlb_prod_problem* D, int packed_upper, int poison_inactive)
{
  D->packed = packed_upper; D->poison_inactive = poison_inactive;
}
extern "C" void dlb_prod_problem_timing(dlb_prod_problem* D, int on) { D->timing = on; D->ms_total = 0; D->ncalls = 0; }
extern "C" double dlb_prod_problem_ms(dlb_prod_problem* D) { return D->ms_total; }
extern "C" int dlb_prod_problem_ncalls(dlb_prod_problem* D) { return D->ncalls; }
