// dlb_common.cuh -- shared device helpers (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>

#define DLB_NT 256                   // default CTA size of the streaming kernels
#define DLB_SM_COUNT_FALLBACK 148    // B200

// cudaFuncSetAttribute is per device: a process that solves on several GPUs (dogleg_gpu_set_device)
// has to opt every kernel into its dynamic shared memory on each of them. first() is true once per
// device; two threads racing through it both set the same attribute, which is harmless.
struct DlbPerDeviceOnce
{
  unsigned char done[64] = {};
  bool first()
  {
    int d = 0;
    if(cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return true;
    if(done[d]) return false;
    done[d] = 1;
    return true;
  }
};

// device-side mirror of dlb_scalars_t (include/dogleg_gpu.h); same member order
struct DlbScalars
{
  double norm2_x, norm2_Jtx, maxabs_Jtx;
  double norm2_JJtx, k_cauchy, norm2_cauchy;
  double norm2_gn;
  double norm2_step, k_interp, Jtx_dot_step, maxabs_step, norm2_Jstep, discriminant;
  double step_type, trial_flags;     // dlb_engine_trial(): the step taken (DLB_STEP_*), 1 = a factorization + GN solve ran
  long long minor;
};

// ---- deterministic reductions: fixed shuffle tree, fixed smem tree ----
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
  for(int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;      // lane 0
}
__device__ __forceinline__ double warp_sum_all(double v)
{
#pragma unroll
  for(int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;      // every lane, same value (xor butterfly is order-symmetric)
}
__device__ __forceinline__ double warp_max(double v)
{
#pragma unroll
  for(int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_down_sync(0xffffffffu, v, o));
  return v;
}

// result valid in thread 0; sh must hold 32 doubles; all threads must call
__device__ __forceinline__ double block_sum(double v, double* sh)
{
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if(lane == 0) sh[w] = v;
  __syncthreads();
  if(w == 0)
  {
    v = (lane < (int)((blockDim.x + 31) >> 5)) ? sh[lane] : 0.0;
    v = warp_sum(v);
  }
  return v;
}
__device__ __forceinline__ double block_max(double v, double* sh)
{
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_max(v);
  __syncthreads();
  if(lane == 0) sh[w] = v;
  __syncthreads();
  if(w == 0)
  {
    v = (lane < (int)((blockDim.x + 31) >> 5)) ? sh[lane] : 0.0;
    v = warp_max(v);
  }
  return v;
}

// Grid-wide reduction of up to 4 sums and 1 max with a fixed evaluation order:
// every CTA leaves its partials in 'part' (5 doubles per CTA), the last CTA to
// arrive (ticket counter) folds them in CTA order. Returns true in thread 0 of
// that last CTA, with the totals in out[0..4]. The counter resets itself.
__device__ __forceinline__ bool grid_reduce5(double s0, double s1, double s2, double s3, double mx,
                                             double* part, unsigned int* counter, double out[5])
{
  __shared__ double sh[32];
  __shared__ bool is_last;
  s0 = block_sum(s0, sh); s1 = block_sum(s1, sh); s2 = block_sum(s2, sh); s3 = block_sum(s3, sh);
  mx = block_max(mx, sh);
  if(threadIdx.x == 0)
  {
    double* mine = part + 5 * (size_t)blockIdx.x;
    mine[0] = s0; mine[1] = s1; mine[2] = s2; mine[3] = s3; mine[4] = mx;
    __threadfence();
    const unsigned int ticket = atomicAdd(counter, 1u);
    is_last = (ticket == gridDim.x - 1);
  }
  __syncthreads();
  if(!is_last) return false;
  __threadfence();
  double a0 = 0, a1 = 0, a2 = 0, a3 = 0, am = 0;
  for(unsigned int b = threadIdx.x; b < gridDim.x; b += blockDim.x)
  {
    const volatile double* q = part + 5 * (size_t)b;
    a0 += q[0]; a1 += q[1]; a2 += q[2]; a3 += q[3]; am = fmax(am, q[4]);
  }
  a0 = block_sum(a0, sh); a1 = block_sum(a1, sh); a2 = block_sum(a2, sh); a3 = block_sum(a3, sh);
  am = block_max(am, sh);
  if(threadIdx.x == 0)
  {
    out[0] = a0; out[1] = a1; out[2] = a2; out[3] = a3; out[4] = am;
    *counter = 0;
    return true;
  }
  return false;
}

// streaming loads that should not pollute L1 (values are read exactly once per pass)
__device__ __forceinline__ double ldg_stream(const double* p)
{
  double v;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float ldg_stream(const float* p)
{
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
