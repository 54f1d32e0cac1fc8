// tests/support/f32jac_dev.cu -- float-Jacobian callbacks for the batched f32jac solves
// (dogleg_gpu_optimize_dense_batched_f32jac, _ragged_f32jac), used by tests/test_gpu_batched_f32jac.py and
// profiles/micro/batched_f32jac.py. Not product code.
//
// The problems are ragged_dev.cu's, built into this library from that file unchanged: the dense kind (problem b = the
// first Nmeas[b] rows of k_gen_batched's problem seed + b; every count equal gives problems_dev.cu's uniform batch) and
// the sample surface on prefixes of its points. A problem is stored ragged (row_off); the uniform callbacks write the
// B x Mpad layout with rows >= Nmeas[b] exact zeros, as dlb_ragged_cb_padded does.
//
// Every callback computes x exactly as ragged_dev.cu's callbacks do (same code, same order), and each entry of J as
// the same double value, then rounds it to float. The float callbacks store that float; their widened twins store it
// widened back to double, (double)(float)J. A solve with the float callback must equal the double solve with the twin,
// bit for bit. ragged_dev.cu's own callbacks (dlb_ragged_cb, dlb_ragged_cb_padded) give the unrounded double J.
#include "ragged_dev.cu"

// the float and the widened twin store the same rounded value
__device__ __forceinline__ void put(float* J, long long i, double v)  { J[i] = (float)v; }
__device__ __forceinline__ void put(double* J, long long i, double v) { J[i] = (double)(float)v; }

// dense kind, as k_ragged_dense
template<typename JT>
__global__ void k_f32_dense(long long nout, int Mpad, int B, int N, int width, const long long* __restrict__ off,
                            const double* __restrict__ A, const double* __restrict__ bv, const double* __restrict__ p,
                            const int* __restrict__ active, double* __restrict__ x, JT* __restrict__ J)
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
        put(J, i * N + kk, m.valid ? a * dphi(pk) : 0.0);
        s += a * phi(pk);
      }
    for(int o = width >> 1; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o, width);
    if(on && k == 0) x[i] = m.valid ? s - bv[src] : 0.0;
  }
}

// sample kind, as k_ragged_sample
template<typename JT>
__global__ void k_f32_sample(long long nout, int Mpad, int B, const long long* __restrict__ off,
                             const double* __restrict__ xy, const double* __restrict__ meas, const double* __restrict__ p,
                             const int* __restrict__ active, double* __restrict__ x, JT* __restrict__ J)
{
  for(long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nout; i += (long long)gridDim.x * blockDim.x)
  {
    const RowMap m = map_row(i, Mpad, off, B);
    if(active && !active[m.prob]) continue;
    const long long g = i * 6;
    if(!m.valid)
    {
      for(int k = 0; k < 6; k++) put(J, g + k, 0.0);
      x[i] = 0.0;
      continue;
    }
    const double* pp = p + m.prob * 6;
    const double X = xy[2 * m.r], Y = xy[2 * m.r + 1];
    put(J, g + 0, pp[1]*X*X); put(J, g + 1, pp[0]*X*X + pp[2]*Y*Y); put(J, g + 2, pp[1]*Y*Y + X*Y);
    put(J, g + 3, X); put(J, g + 4, Y); put(J, g + 5, 1.0);
    x[i] = pp[0]*pp[1]*X*X + pp[1]*pp[2]*Y*Y + pp[2]*X*Y + pp[3]*X + pp[4]*Y + pp[5] - meas[m.r];
  }
}

template<typename JT>
static void evaluate_f32(dlb_ragged_problem* D, long long nout, int Mpad, const long long* d_row_off, const double* d_p,
                         double* d_x, JT* d_J, const int* d_active, cudaStream_t st)
{
  if(nout > 0)
  {
    if(D->kind == 1)
      k_f32_sample<JT><<<148 * 8, 256, 0, st>>>(nout, Mpad, D->B, d_row_off, D->d_A, D->d_b, d_p, d_active, d_x, d_J);
    else
      k_f32_dense<JT><<<148 * 16, 256, 0, st>>>(nout, Mpad, D->B, D->N, model_width(D->N), d_row_off, D->d_A, D->d_b,
                                                d_p, d_active, d_x, d_J);
  }
  D->ncalls++;
}

// dogleg_gpu_callback_dense_ragged_f32jac_t and its widened twin (a dogleg_gpu_callback_dense_ragged_t)
extern "C" void dlb_f32_cb_ragged(const double* d_p, double* d_x, float* d_J, const long long* d_row_off,
                                  const int* d_active, int B, void* stream, void* cookie)
{
  dlb_ragged_problem* D = (dlb_ragged_problem*)cookie;
  (void)B;
  evaluate_f32(D, D->rows, 0, d_row_off, d_p, d_x, d_J, d_active, (cudaStream_t)stream);
}
extern "C" void dlb_f32_cb_ragged_twin(const double* d_p, double* d_x, double* d_J, const long long* d_row_off,
                                       const int* d_active, int B, void* stream, void* cookie)
{
  dlb_ragged_problem* D = (dlb_ragged_problem*)cookie;
  (void)B;
  evaluate_f32(D, D->rows, 0, d_row_off, d_p, d_x, d_J, d_active, (cudaStream_t)stream);
}
// dogleg_gpu_callback_dense_batched_f32jac_t of the batch zero-padded to Nmeas = Mpad, and its widened twin (a
// dogleg_gpu_callback_dense_batched_t)
extern "C" void dlb_f32_cb_uniform(const double* d_p, double* d_x, float* d_J, const int* d_active, int B, void* stream,
                                   void* cookie)
{
  dlb_ragged_problem* D = (dlb_ragged_problem*)cookie;
  evaluate_f32(D, (long long)B * D->Mpad, D->Mpad, D->d_row_off, d_p, d_x, d_J, d_active, (cudaStream_t)stream);
}
extern "C" void dlb_f32_cb_uniform_twin(const double* d_p, double* d_x, double* d_J, const int* d_active, int B,
                                        void* stream, void* cookie)
{
  dlb_ragged_problem* D = (dlb_ragged_problem*)cookie;
  evaluate_f32(D, (long long)B * D->Mpad, D->Mpad, D->d_row_off, d_p, d_x, d_J, d_active, (cudaStream_t)stream);
}
extern "C" void* dlb_f32_cb_ragged_ptr(void)       { return (void*)&dlb_f32_cb_ragged; }
extern "C" void* dlb_f32_cb_ragged_twin_ptr(void)  { return (void*)&dlb_f32_cb_ragged_twin; }
extern "C" void* dlb_f32_cb_uniform_ptr(void)      { return (void*)&dlb_f32_cb_uniform; }
extern "C" void* dlb_f32_cb_uniform_twin_ptr(void) { return (void*)&dlb_f32_cb_uniform_twin; }
