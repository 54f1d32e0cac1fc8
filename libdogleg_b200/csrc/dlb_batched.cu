// dlb_batched.cu -- B independent small dense problems (config C3: Nstate=16, Nmeas=256,
// B=100k), the whole dog-leg automaton device-resident. Additive entry point
// dogleg_gpu_optimize_dense_batched() (include/dogleg_gpu.h); per problem it follows the
// reference's dense path step for step:
//   evaluation           dogleg.c:1034-1053, 1073-1081   (J'x, |x|^2, inf-norm test)
//   trust-region update  dogleg.c:1303-1356
//   loop / termination   dogleg.c:1359-1476
//   Cauchy               dogleg.c:529-617
//   JtJ + lambda, dpptrf dogleg.c:699-816,  dpptrs :867-898
//   step / interpolation dogleg.c:927-998, 1172-1297, expected improvement :1085-1165
//
// One WARP per problem and per trial. The Jacobian the callback just produced is streamed from
// HBM exactly once (the algorithmic minimum 8(MN+M) bytes per trial, SURVEY.md 8d): groups of 4
// rows go straight from global loads into FP64 tensor-core fragments (mma.sync m8n8k4, SASS
// DMMA) that accumulate JtJ = J'J and -- with x as an extra B column -- J'x in the same pass.
// Everything after that works on the 16x16 JtJ in a per-warp shared-memory scratch with
// lane == state index: |J v|^2 is evaluated as v'(JtJ)v, exactly what the reference's own
// DENSE_PRODUCTS path does (dogleg.c:582-596, 1131-1155), so a rejected step needs only the
// 2 KB JtJ of the current point (kept in HBM), never its 32 KB Jacobian. All reductions have a
// fixed order; there are no block-wide barriers.
//
// Dense-products form (dogleg_gpu_optimize_dense_products_batched): the callback hands over |x|^2,
// J'x and J'J itself (full, or the packed upper triangle), the reference's DOGLEG_DENSE_PRODUCTS
// inputs (dogleg.c:1004-1083). The same kernel, instantiated with PRODUCTS, replaces the pass over J by a
// coalesced load of those ~8(N^2 + N + 1) bytes per problem; everything from accept / reject on is
// shared code. No J is ever stored, so the batch size no longer depends on Nmeas.
//
// Final state (the `2` entry points with a dogleg_gpu_batch_t): the trial kernel also keeps the final point's
// JtJ and writes why each problem stopped; k_batched_factor factors every problem's JtJ + lambda I with the
// same ladder and solves with it (dogleg_gpu_batch_solve, dogleg_gpu_batch_covariance); k_batched_outlierness
// computes every problem's outlierness factors on the same matrix (dogleg_gpu_batch_outlierness).
//
// Ragged form (dogleg_gpu_optimize_dense_batched_ragged): problem b has its own number of measurements, its rows
// at row_off[b] of x and J. The RAGGED instantiations of the same two kernels take each warp's M and row pointers
// from the offsets and its problem from a longest-first order; everything else is the uniform code.
//
// Float-Jacobian forms (dogleg_gpu_optimize_dense_batched_f32jac, _ragged_f32jac): the callback writes J in float,
// which halves the bytes of the stream. The float instantiations load it as float and widen every value to double
// before it is used, so they compute exactly what the double kernel computes on the widened J.
#include "dlb_common.cuh"
#include "dogleg_gpu.h"
#include "dlb_outlier_math.h"
#include <vector>
#include <cstring>
#include <string>
#include <algorithm>
#include <climits>
#include <cstdint>
#include <type_traits>

extern "C" void dlb_set_error(const char* msg);

#define BT_NT 256
#define BT_WARPS (BT_NT / 32)
#define BT_NMAX 32
#define BT_RING 4

struct BatchState
{
  int B, N, M, max_iterations;
  double tr0, dec_factor, dec_thr, inc_factor, inc_thr, Jtx_thr, upd_thr, tr_thr;
  // per problem
  double *tr, *n2x_before, *n2c, *n2gn, *expected, *lambda;
  int *steps, *flags, *active;
  double *p_before, *ptrial, *Jtx, *cauchy, *gn, *JtJ;
  // callback buffers
  double *x;            // B x M
  double *J;            // B x M x N
  int *n_active;
  // dense-products callback buffers (appended: the dense instantiations keep their parameter offsets)
  double *norm2x_in;    // B
  double *Jtx_in;       // B x N
  double *JtJ_in;       // B x N*N, or B x N(N+1)/2 packed upper row-first
  int packed;
  // a dogleg_gpu_batch_t was asked for (appended likewise): B termination codes (DOGLEG_GPU_BATCH_*), and the
  // final point's JtJ is kept in JtJ. NULL: neither.
  int *status;
  // ragged form (appended likewise, read by the RAGGED instantiations only): problem b's rows are
  // [row_off[b], row_off[b + 1]) of x and J; warp slot s takes problem order[s], longest first
  const long long *row_off;
  const int *order;
  // the f32jac forms' Jacobian (appended likewise, read by the float instantiations only): J in float, in J's layout
  float *Jf;
};
enum { FL_CAUCHY = 1, FL_GN = 2, FL_EDGE = 4, FL_PENDING = 8 };

__device__ __forceinline__ void bt_dmma(double& d0, double& d1, double a, double b)
{
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// v' A v for the symmetric N x N matrix A (row stride LD) in shared memory; lane == row
__device__ __forceinline__ double bt_quadform(const double* A, int LD, const double* v, int N, int lane)
{
  double r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0;           // four chains: the row sum is latency, not work
  if(lane < N)
  {
    const double* Ar = A + lane * LD;
    int c = 0;
    for(; c + 4 <= N; c += 4)
    { r0 = fma(Ar[c], v[c], r0); r1 = fma(Ar[c + 1], v[c + 1], r1); r2 = fma(Ar[c + 2], v[c + 2], r2); r3 = fma(Ar[c + 3], v[c + 3], r3); }
    for(; c < N; c++) r0 = fma(Ar[c], v[c], r0);
    r0 = ((r0 + r1) + (r2 + r3)) * v[lane];
  }
  return warp_sum_all(r0);
}

__device__ __forceinline__ double bt_warp_max_all(double v)
{
#pragma unroll
  for(int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// two sums folded by one interleaved shuffle tree (fixed order)
__device__ __forceinline__ void bt_warp_sum2_all(double& a, double& b)
{
#pragma unroll
  for(int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
}

// Cholesky of A + lambda I with the lambda ladder (dogleg.c:699-816), lane == row; A and the factor are
// N x N, row stride 8 * NT8 + 1, in the warp's shared memory. The lane keeps ITS ROW of L in Lr; per pivot:
// the diagonal comes by one shuffle, every lane forms rsqrt(d) itself (no sqrt -> division chain, DESIGN.md
// divergence 7), the scaled column goes through shared memory once and the row updates are independent
// multiply-adds. On return sL holds L (lower triangle, zeros above), Lr this lane's row of it, rsv the
// reciprocal pivots (the same in every lane) and lam the lambda it took; lam is not finite if no lambda
// of the ladder gave a positive definite matrix.
template<int NT8>
__device__ __forceinline__ void bt_cholesky_ladder(const double* sA, double* sL, int N, int lane, double& lam,
                                                   double (&Lr)[8 * NT8], double (&rsv)[8 * NT8])
{
  constexpr int NMAX = 8 * NT8, LD = NMAX + 1;
  for(;;)
  {
#pragma unroll
    for(int c = 0; c < NMAX; c++)
    {
      const bool in = lane < N && c <= lane;
      const double val = sA[(in ? lane : 0) * LD + (in ? c : 0)];
      Lr[c] = in ? val + (c == lane ? lam : 0.0) : 0.0;
    }
    bool ok = true;
#pragma unroll
    for(int j = 0; j < NMAX; j++)
    {
      if(j >= N || !ok) continue;                    // (uniform)
      const double d = __shfl_sync(0xffffffffu, Lr[j], j);
      if(!(d > 0.0) || isinf(d)) { ok = false; continue; }
      const double rs = rsqrt(d);
      rsv[j] = rs;
      Lr[j] = lane == j ? d * rs : Lr[j] * rs;       // (zero for the lanes above the pivot)
      if(lane < N) sL[lane * LD + j] = Lr[j];
      __syncwarp();
#pragma unroll
      for(int c = j + 1; c < NMAX; c++)
        if(c <= lane && c < N) Lr[c] = fma(-Lr[j], sL[c * LD + j], Lr[c]);
    }
    if(ok) break;
    lam = lam == 0.0 ? 1e-10 : lam * 10.0;             // dogleg.c:811-813
    if(!isfinite(lam)) break;
    __syncwarp();
  }
}

// Blocks per SM the register budget is sized for: three for small dense problems (80 registers). The
// products form at NT8 == 2 spills at 80 registers; it gets two blocks (119 registers, no spills).
template<int NT8, bool PRODUCTS> constexpr int bt_min_blocks() { return NT8 == 1 ? 3 : NT8 == 2 ? (PRODUCTS ? 2 : 3) : 1; }

// JT: the element type of the callback's Jacobian (double, or float for the f32jac forms). Only the loads see it:
// every value is widened to double before it enters a DMMA or an FMA, and the sums run in the same order, so a
// float J gives the results of the double kernel on the widened J, bit for bit.
template<int NT8, int RING, bool PRODUCTS, bool RAGGED, typename JT = double>
__global__ void __launch_bounds__(BT_NT, bt_min_blocks<NT8, PRODUCTS>())
k_batched_trial(BatchState S)
{
  extern __shared__ double sm[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int b = blockIdx.x * BT_WARPS + w;
  if(b >= S.B) return;
  if constexpr(RAGGED) b = S.order[b];
  if(!S.active[b]) return;
  const int N = S.N, M = RAGGED ? (int)(S.row_off[b + 1] - S.row_off[b]) : S.M;
  constexpr int LD = 8 * NT8 + 1;          // padded row stride of the per-warp matrices
  constexpr int NPAIR = NT8 * (NT8 + 1) / 2;
  double* sA  = sm + (size_t)w * (2 * 8 * NT8 * LD + 6 * BT_NMAX);   // JtJ
  double* sL  = sA + 8 * NT8 * LD;                                    // Cholesky factor
  double* sg  = sL + 8 * NT8 * LD;         // Jt_x of the current point
  double* sgn = sg + BT_NMAX;              // Jt_x of the trial point
  double* sc  = sgn + BT_NMAX;             // cauchy
  double* sn  = sc + BT_NMAX;              // gauss-newton
  double* ss  = sn + BT_NMAX;              // step
  double* sp  = ss + BT_NMAX;              // scratch
  double n2x_new;
  if constexpr(PRODUCTS)
  { // ---- the callback's products of the trial point: JtJ staged in sL (both triangles), J'x in sgn ----
    if(S.packed)
    { // packed upper, row-first: row r holds columns r..N-1 from offset r0. Consecutive lanes read
      // consecutive entries; each lane walks its row index forward as its entry index grows.
      const double* gP = S.JtJ_in + (size_t)b * (N * (N + 1) / 2);
      int r = 0, r0 = 0;
      for(int e = lane; e < N * (N + 1) / 2; e += 32)
      {
        while(e >= r0 + N - r) { r0 += N - r; r++; }
        const int c = r + (e - r0);
        const double val = ldg_stream(gP + e);
        sL[r * LD + c] = val; sL[c * LD + r] = val;
      }
    }
    else
    {
      const double* gF = S.JtJ_in + (size_t)b * N * N;
      for(int e = lane; e < N * N; e += 32) { const int a = e / N, c = e - a * N; sL[a * LD + c] = ldg_stream(gF + e); }
    }
    if(lane < N) sgn[lane] = ldg_stream(S.Jtx_in + (size_t)b * N + lane);
    n2x_new = S.norm2x_in[b];
    (void)M;
  }
  else
  {
    const int g = lane >> 2, tt = lane & 3;

    // ---- one pass over the trial point's Jacobian: JtJ, J'x, |x|^2 ----
    const size_t row0 = RAGGED ? (size_t)S.row_off[b] : (size_t)b * M;
    const JT* gJ;
    if constexpr(std::is_same<JT, float>::value) gJ = S.Jf + row0 * N; else gJ = S.J + row0 * N;
    const double* gx = S.x + row0;
    double acc[NPAIR][2], ag[NT8][2];
#pragma unroll
    for(int i = 0; i < NPAIR; i++) { acc[i][0] = 0.0; acc[i][1] = 0.0; }
#pragma unroll
    for(int i = 0; i < NT8; i++) { ag[i][0] = 0.0; ag[i][1] = 0.0; }
    double n2 = 0.0;
    // one 4-row group: this lane's entries of the group's rows (zeros beyond the last row)
    auto load_group = [&](int r0, JT (&v)[NT8], double& xr) {
      const int row = r0 + tt;
      const bool valid = row < M;
      xr = valid ? ldg_stream(gx + row) : 0.0;
#pragma unroll
      for(int ti = 0; ti < NT8; ti++) v[ti] = (valid && 8 * ti + g < N) ? ldg_stream(gJ + (size_t)row * N + 8 * ti + g) : JT(0);
    };
    auto use_group = [&](const double (&v)[NT8], double xr) {
      // J'x by plain multiply-adds (this lane's row of the group times its x; the four lanes of a state are
      // folded after the loop): as a DMMA it cost a third of the FP64 pipe, which this kernel loads almost
      // as heavily as HBM (2.5 FMA per byte streamed against 2.9 FMA per byte of machine balance).
      // Measured in round 2 (profiles/r02_variants.txt): 1.40 -> 1.35 ms per trial launch; splitting the kernel
      // into a streaming pass and a step kernel (1.39-1.47 ms) and deeper register rings (6: 1.58 ms,
      // 8: 1.61 ms) were slower and are not kept.
      const double bx = g == 0 ? xr : 0.0;
      int idx = 0;
#pragma unroll
      for(int ti = 0; ti < NT8; ti++)
      {
#pragma unroll
        for(int tj = 0; tj <= ti; tj++, idx++) bt_dmma(acc[idx][0], acc[idx][1], v[ti], v[tj]);
        ag[ti][0] = fma(v[ti], xr, ag[ti][0]);
      }
      n2 = fma(bx, bx, n2);
    };
    if(RING > 1)
    { // register ring: the loads of group i + RING are issued before the DMMAs of group i, so RING
      // groups (3 * RING loads per lane) are in flight; groups are consumed in the same order as
      // below, hence bit-identical sums. Groups past the end are zeros. The ring holds J as loaded (a float ring
      // takes half the registers) and widens on use.
      JT vb[RING > 1 ? RING : 1][NT8];
      double xb[RING > 1 ? RING : 1];
#pragma unroll
      for(int u = 0; u < RING; u++) load_group(4 * u, vb[u], xb[u]);
      for(int r0 = 0; r0 < M; r0 += 4 * RING)
      {
#pragma unroll
        for(int u = 0; u < RING; u++)
        {
          double v[NT8];
#pragma unroll
          for(int ti = 0; ti < NT8; ti++) v[ti] = vb[u][ti];
          const double xr = xb[u];
          load_group(r0 + 4 * (u + RING), vb[u], xb[u]);
          use_group(v, xr);
        }
      }
    }
    else
    {
#pragma unroll 8
      for(int r0 = 0; r0 < M; r0 += 4)
      {
        JT vj[NT8];
        double v[NT8], xr;
        load_group(r0, vj, xr);
#pragma unroll
        for(int ti = 0; ti < NT8; ti++) v[ti] = vj[ti];
        use_group(v, xr);
      }
    }
#pragma unroll
    for(int ti = 0; ti < NT8; ti++)
    {
      ag[ti][0] += __shfl_xor_sync(0xffffffffu, ag[ti][0], 1);
      ag[ti][0] += __shfl_xor_sync(0xffffffffu, ag[ti][0], 2);
    }
    n2x_new = warp_sum_all(n2);
    {
      int idx = 0;
#pragma unroll
      for(int ti = 0; ti < NT8; ti++)
      {
#pragma unroll
        for(int tj = 0; tj <= ti; tj++, idx++)
        {
          const int a = 8 * ti + g, c0 = 8 * tj + 2 * tt;
          sL[a * LD + c0] = acc[idx][0]; sL[a * LD + c0 + 1] = acc[idx][1];       // trial-point JtJ staged in sL
          if(ti != tj) { sL[c0 * LD + a] = acc[idx][0]; sL[(c0 + 1) * LD + a] = acc[idx][1]; }
        }
        if(tt == 0) sgn[8 * ti + g] = ag[ti][0];
      }
    }
  }
  __syncwarp();

  // ---- accept / reject, trust-region update (every lane computes the same scalars) ----
  int flags = S.flags[b];
  double tr = S.tr[b];
  int steps = S.steps[b];
  const double gmax = bt_warp_max_all(lane < N ? fabs(sgn[lane]) : 0.0);
  const bool converged = !(gmax > S.Jtx_thr);
  bool done = false, accepted = false;
  if(!(flags & FL_PENDING))
  { // the initial operating point
    accepted = true;
    if(converged || S.max_iterations <= 0) done = true;
  }
  else
  {
    const double observed = S.n2x_before[b] - n2x_new;
    double rho = observed / S.expected[b];
    if(!isfinite(n2x_new)) rho = -INFINITY;              // DESIGN.md, divergence 2
    if(rho < S.dec_thr)
    {
      if(!(flags & FL_EDGE)) tr = sqrt(S.n2gn[b]);
      tr *= S.dec_factor;
    }
    else if(rho > S.inc_thr && (flags & FL_EDGE)) tr *= S.inc_factor;
    if(rho > 0.0)
    {
      accepted = true;
      steps++;
      if(converged || steps >= S.max_iterations) done = true;
    }
    else if(tr < S.tr_thr) done = true;
  }
  double* gA = S.JtJ + (size_t)b * N * N;
  if(accepted)
  { // the trial point becomes the current one: its JtJ and gradient are kept for retries
    flags &= ~(FL_CAUCHY | FL_GN | FL_EDGE);
    for(int e = lane; e < N * N; e += 32) { const int a = e / N, c = e - a * N; const double val = sL[a * LD + c]; sA[a * LD + c] = val; if(!done || S.status) gA[e] = val; }
    if(lane < N)
    {
      S.p_before[(size_t)b * N + lane] = S.ptrial[(size_t)b * N + lane];
      S.Jtx[(size_t)b * N + lane] = sgn[lane];
      sg[lane] = sgn[lane];
    }
    if(lane == 0) S.n2x_before[b] = n2x_new;
  }
  else if(!done)
  { // rejected: bring back the cached quantities of the current point
    for(int e = lane; e < N * N; e += 32) { const int a = e / N, c = e - a * N; sA[a * LD + c] = gA[e]; }
    if(lane < N)
    {
      sg[lane] = S.Jtx[(size_t)b * N + lane];
      sc[lane] = S.cauchy[(size_t)b * N + lane];
      sn[lane] = S.gn[(size_t)b * N + lane];
    }
  }
  if(lane == 0) { S.tr[b] = tr; S.steps[b] = steps; }
  if(done)
  {
    if(lane == 0)
    {
      S.flags[b] = flags; S.active[b] = 0; atomicSub(S.n_active, 1);
      // the gradient test comes before the iteration cap (dogleg_core.c run_solver)
      if(S.status) S.status[b] = !accepted ? DOGLEG_GPU_BATCH_TRUSTREGION
                                           : converged ? DOGLEG_GPU_BATCH_GRADIENT : DOGLEG_GPU_BATCH_MAX_ITERATIONS;
    }
    return;
  }
  __syncwarp();

  // ---- Cauchy step (dogleg.c:529-617, |J g|^2 = g'JtJ g as at :582-596) ----
  double n2c;
  if(!(flags & FL_CAUCHY))
  {
    const double jg2 = bt_quadform(sA, LD, sg, N, lane);
    const double g2 = warp_sum_all(lane < N ? sg[lane] * sg[lane] : 0.0);
    const double kc = -g2 / jg2;
    n2c = kc * kc * g2;
    if(lane < N) { sc[lane] = kc * sg[lane]; S.cauchy[(size_t)b * N + lane] = sc[lane]; }
    if(lane == 0) S.n2c[b] = n2c;
    flags |= FL_CAUCHY;
    __syncwarp();
  }
  else n2c = S.n2c[b];

  // ---- choose the step (dogleg.c:1192-1255) ----
  int type;
  double n2gn = 0.0;
  if(n2c >= tr * tr) { type = 0; flags |= FL_EDGE; }
  else
  {
    if(!(flags & FL_GN))
    {
      // Cholesky of JtJ + lambda I with the lambda ladder, lane == row. The two substitutions multiply by the
      // stored reciprocals and hand each solved entry round by one shuffle.
      constexpr int NMAX = 8 * NT8;
      double lam = S.lambda[b];
      double Lr[NMAX], rsv[NMAX];
      bt_cholesky_ladder<NT8>(sA, sL, N, lane, lam, Lr, rsv);
      if(lane == 0) S.lambda[b] = lam;
      // (JtJ + lambda I) u = Jt_x, gn = -u (dogleg.c:867-898)
      double yv = lane < N ? sg[lane] : 0.0;
#pragma unroll
      for(int j = 0; j < NMAX; j++)
      {
        if(j >= N) continue;
        const double yj = __shfl_sync(0xffffffffu, yv * rsv[j], j);
        if(lane == j) yv = yj;
        else if(lane > j) yv = fma(-Lr[j], yj, yv);
      }
      __syncwarp();
#pragma unroll
      for(int j = NMAX - 1; j >= 0; j--)
      {
        if(j >= N) continue;
        const double lt = sL[j * LD + (lane < j ? lane : 0)];          // L[j][lane]
        const double xj = __shfl_sync(0xffffffffu, yv * rsv[j], j);
        if(lane == j) yv = xj;
        else if(lane < j) yv = fma(-lt, xj, yv);
      }
      if(lane < N) { sn[lane] = -yv; S.gn[(size_t)b * N + lane] = -yv; }
      __syncwarp();
      n2gn = warp_sum_all(lane < N ? yv * yv : 0.0);
      if(lane == 0) S.n2gn[b] = n2gn;
      flags |= FL_GN;
    }
    else n2gn = S.n2gn[b];
    if(n2gn <= tr * tr) { type = 1; flags &= ~FL_EDGE; }
    else                { type = 2; flags |= FL_EDGE; }
  }

  // ---- the step, p + step, expected improvement, update threshold ----
  double kk = 0.0;
  if(type == 2)
  {
    double l2 = 0.0, negc = 0.0;
    if(lane < N) { const double d = sc[lane] - sn[lane]; l2 = d * d; negc = d * sc[lane]; }
    bt_warp_sum2_all(l2, negc);
    double disc = negc * negc - l2 * (n2c - tr * tr);
    if(disc < 0.0) disc = 0.0;
    kk = (negc + sqrt(disc)) / l2;
  }
  if(lane < N)
  {
    double sv;
    if(type == 0)      sv = (tr / sqrt(n2c)) * sc[lane];
    else if(type == 1) sv = sn[lane];
    else               sv = sc[lane] + kk * (sn[lane] - sc[lane]);
    ss[lane] = sv;
    S.ptrial[(size_t)b * N + lane] = S.p_before[(size_t)b * N + lane] + sv;
  }
  __syncwarp();
  const double gd = warp_sum_all(lane < N ? sg[lane] * ss[lane] : 0.0);
  const double smax = bt_warp_max_all(lane < N ? fabs(ss[lane]) : 0.0);
  const double js2 = bt_quadform(sA, LD, ss, N, lane);
  double expected = -2.0 * gd - js2;
  const bool finished = !(smax > S.upd_thr);               // dogleg.c:1289-1296, 1403-1408
  if(finished) expected = -1.0;
  if(lane == 0)
  {
    S.expected[b] = expected;
    S.flags[b] = flags | FL_PENDING;
    if(finished)
    {
      S.active[b] = 0; atomicSub(S.n_active, 1);
      if(S.status) S.status[b] = DOGLEG_GPU_BATCH_STEP;
    }
  }
  (void)sp;
}

// ---- solves with the final state of a batched solve (dogleg_gpu_batch_t) ----
// The warp's problem JtJ (N x N row-first, global) + lambda I factored by the trial kernel's ladder, starting from
// the lambda at *glam: JtJ is staged in sY (row stride 8 * NT8 + 1), L goes to sL and the reciprocal pivots to srs.
// Returns the lambda taken (not finite: no lambda of the ladder gave a positive definite matrix).
template<int NT8>
__device__ __forceinline__ double bt_load_and_factor(const double* gA, const double* glam, double* sY, double* sL,
                                                     double* srs, int N, int lane)
{
  constexpr int NMAX = 8 * NT8, LD = NMAX + 1;
  for(int e = lane; e < N * N; e += 32) { const int a = e / N, c = e - a * N; sY[a * LD + c] = ldg_stream(gA + e); }
  double lam = *glam;
  __syncwarp();
  double Lr[NMAX], rsv[NMAX];
  bt_cholesky_ladder<NT8>(sY, sL, N, lane, lam, Lr, rsv);
#pragma unroll
  for(int j = 0; j < NMAX; j++)
    if(j < N && lane == j) srs[j] = rsv[j];
  return lam;
}

// L y = r in place for this lane's right-hand side y (entries >= N are never read); L and the reciprocal pivots
// from the warp's shared memory, every lane reading the same entry (broadcasts)
template<int NT8>
__device__ __forceinline__ void bt_forward_subst(const double* sL, const double* srs, int N, double (&y)[8 * NT8])
{
  constexpr int NMAX = 8 * NT8, LD = NMAX + 1;
#pragma unroll
  for(int j = 0; j < NMAX; j++)
  {
    if(j >= N) continue;
    double acc = y[j];
#pragma unroll
    for(int i = 0; i < j; i++) acc = fma(-sL[j * LD + i], y[i], acc);
    y[j] = acc * srs[j];
  }
}

struct BatchFactorArgs
{
  int B, N, nrhs;             // nrhs: columns of R and X
  const double* JtJ;          // B x N*N
  double* lambda;             // B; raised in place by the ladder
  const double* R;            // B x N x nrhs, column-major per problem; NULL: the identity (nrhs = N)
  double* X;                  // like R; packed: B x N(N+1)/2, the upper triangle of the row-first result
  int packed;
  int* nfail;                 // counts the problems no lambda makes positive definite (may be NULL)
};

// One warp per problem: JtJ + lambda I factored by the trial kernel's ladder, then both substitutions with
// lane == right-hand-side column, up to 32 columns at a time. L and the reciprocal pivots sit in the warp's
// shared memory and every lane reads the same entry, so the reads are broadcasts and the chain is about N^2
// multiply-adds for all 32 columns. Right-hand sides and results are staged through shared memory (column k
// at sY[k * LD]) so that each problem's global reads and writes are coalesced. The sums run in the order of
// the trial kernel's substitutions, so the solve with J'x reproduces its Gauss-Newton step bit for bit.
template<int NT8>
__global__ void __launch_bounds__(BT_NT) k_batched_factor(BatchFactorArgs A)
{
  extern __shared__ double sm[];
  constexpr int NMAX = 8 * NT8, LD = NMAX + 1;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int b = blockIdx.x * BT_WARPS + w;
  if(b >= A.B) return;
  const int N = A.N;
  double* sY  = sm + (size_t)w * (32 * LD + NMAX * LD + NMAX);   // JtJ, then right-hand sides / results
  double* sL  = sY + 32 * LD;                                     // Cholesky factor
  double* srs = sL + NMAX * LD;                                   // reciprocal pivots
  const double lam = bt_load_and_factor<NT8>(A.JtJ + (size_t)b * N * N, A.lambda + b, sY, sL, srs, N, lane);
  const bool failed = !isfinite(lam);
  if(lane == 0) { A.lambda[b] = lam; if(failed && A.nfail) atomicAdd(A.nfail, 1); }
  __syncwarp();

  const int ncols = A.R ? A.nrhs : N;
  const double* gR = A.R ? A.R + (size_t)b * N * ncols : nullptr;
  double* gX = A.X + (A.packed ? (size_t)b * (N * (N + 1) / 2) : (size_t)b * N * ncols);
  for(int c0 = 0; c0 < ncols; c0 += 32)
  {
    const int nc = min(32, ncols - c0);
    if(gR)
    {
      for(int e = lane; e < nc * N; e += 32) { const int k = e / N, i = e - k * N; sY[k * LD + i] = ldg_stream(gR + (size_t)c0 * N + e); }
      __syncwarp();
    }
    double y[NMAX];                                               // entries >= N are never read
#pragma unroll
    for(int i = 0; i < NMAX; i++) y[i] = gR ? sY[lane * LD + i] : (i == c0 + lane ? 1.0 : 0.0);
    bt_forward_subst<NT8>(sL, srs, N, y);                        // L y = r
#pragma unroll
    for(int j = NMAX - 1; j >= 0; j--)                            // L' x = y
    {
      if(j >= N) continue;
      double acc = y[j];
#pragma unroll
      for(int i = NMAX - 1; i > j; i--)
        if(i < N) acc = fma(-sL[i * LD + j], y[i], acc);
      y[j] = acc * srs[j];
    }
    __syncwarp();
#pragma unroll
    for(int i = 0; i < NMAX; i++)
      if(i < N) sY[lane * LD + i] = failed ? __longlong_as_double(0x7ff8000000000000LL) : y[i];
    __syncwarp();
    if(A.packed)
    { // (covariance: one chunk) row r of the packed upper triangle = entries r..N-1 of column r
      int r = 0, r0 = 0;
      for(int e = lane; e < N * (N + 1) / 2; e += 32)
      {
        while(e >= r0 + N - r) { r0 += N - r; r++; }
        gX[e] = sY[r * LD + r + (e - r0)];
      }
    }
    else
      for(int e = lane; e < nc * N; e += 32) { const int k = e / N, i = e - k * N; gX[(size_t)c0 * N + e] = sY[k * LD + i]; }
    __syncwarp();
  }
}

// ---- outlierness factors of every problem (dogleg_gpu_batch_outlierness) ----
struct BatchOutlierArgs
{
  int B, N, M, fsize, nfeat;  // M: measurements per problem; features are fsize consecutive ones, nfeat * fsize <= M
  const double* JtJ;          // B x N*N
  double* lambda;             // B; raised in place by the ladder
  const double* x;            // B x M
  const double* J;            // B x M x N, row-first per problem
  const int* nout;            // B NoutlierFeatures, or NULL (all 0)
  double* scale;              // B, in / out
  double* factors;            // B x nfeat
  int* nfail;
  // ragged handles (appended, read by the RAGGED instantiations only): problem b's rows are [row_off[b],
  // row_off[b + 1]) of x, J and factors; nfeat_b: B feature counts (NULL: M_b / fsize); warp slot s takes problem
  // order[s]
  const long long* row_off;
  const int* nfeat_b;
  const int* order;
};

// One warp per problem. A_ij of a feature is j_i' inv(JtJ + lambda I) j_j = (L^-1 j_i) . (L^-1 j_j), so one forward
// substitution per measurement is all it takes. J is taken 32 rows at a time: a problem's row-first M x N block has
// the layout of k_batched_factor's column-major N x M right-hand sides, and is staged through shared memory the same
// way (coalesced reads); then lane == measurement substitutes its row against the broadcast L. The next chunk's
// loads are in flight during the current chunk's substitution. |x|^2 is a fixed-order warp sum and A_01 of a pair
// takes the neighbouring lane's row by shuffles, so the factors are reproducible bit for bit.
// A ragged problem whose feature count is negative or exceeds its rows gets a NaN scale and no factors. The
// ragged instantiations ask for one block per SM: left to itself, ptxas gives the NT8 == 3 one 128 registers and
// 284 bytes of spills (0 with the bound); the uniform ones compile as without a minimum (0).
template<int NT8, bool RAGGED>
__global__ void __launch_bounds__(BT_NT, RAGGED ? 1 : 0) k_batched_outlierness(BatchOutlierArgs A)
{
  extern __shared__ double sm[];
  constexpr int NMAX = 8 * NT8, LD = NMAX + 1;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int b = blockIdx.x * BT_WARPS + w;
  if(b >= A.B) return;
  if constexpr(RAGGED) b = A.order[b];
  const int N = A.N, M = RAGGED ? (int)(A.row_off[b + 1] - A.row_off[b]) : A.M, fs = A.fsize;
  const int nfeat = RAGGED ? (A.nfeat_b ? A.nfeat_b[b] : M / fs) : A.nfeat;
  if constexpr(RAGGED)
    if(nfeat < 0 || (long long)nfeat * fs > M)
    {
      if(lane == 0) A.scale[b] = __longlong_as_double(0x7ff8000000000000LL);
      return;
    }
  double* sY  = sm + (size_t)w * (32 * LD + NMAX * LD + NMAX);   // JtJ, then rows of J
  double* sL  = sY + 32 * LD;
  double* srs = sL + NMAX * LD;
  const double lam = bt_load_and_factor<NT8>(A.JtJ + (size_t)b * N * N, A.lambda + b, sY, sL, srs, N, lane);
  const bool failed = !isfinite(lam);
  if(lane == 0) { A.lambda[b] = lam; if(failed && A.nfail) atomicAdd(A.nfail, 1); }

  const size_t row0 = RAGGED ? (size_t)A.row_off[b] : (size_t)b * M;
  const double* gx = A.x + row0;
  const double* gJ = A.J + row0 * N;
  double n2 = 0.0;
  for(int m = lane; m < M; m += 32) { const double v = ldg_stream(gx + m); n2 = fma(v, v, n2); }
  double k = A.scale[b];
  outlierness_scale(&k, M, N, A.nout ? A.nout[b] : 0, fs, warp_sum_all(n2));
  if(lane == 0) A.scale[b] = k;

  // this lane's share of the 32-row chunk at row m0: entries lane + 32 t of the chunk's min(32, M - m0) * N
  double v[NMAX];
  auto load_chunk = [&](int m0) {
    const int ne = min(32, M - m0) * N;
#pragma unroll
    for(int t = 0; t < NMAX; t++)
      if(t < N && lane + 32 * t < ne) v[t] = ldg_stream(gJ + (size_t)m0 * N + lane + 32 * t);
  };
  const int Mused = nfeat * fs;
  double* gf = A.factors + (RAGGED ? row0 : (size_t)b * A.nfeat);
  load_chunk(0);
  for(int m0 = 0; m0 < Mused; m0 += 32)
  {
    const int ne = min(32, M - m0) * N;
    __syncwarp();
#pragma unroll
    for(int t = 0; t < NMAX; t++)
      if(t < N && lane + 32 * t < ne) { const int e = lane + 32 * t, r = e / N; sY[r * LD + e - r * N] = v[t]; }
    __syncwarp();
    double y[NMAX];                                               // entries >= N are never read
#pragma unroll
    for(int i = 0; i < NMAX; i++) y[i] = sY[lane * LD + i];
    const int m = m0 + lane;
    const double xm = m < M ? ldg_stream(gx + m) : 0.0;
    if(m0 + 32 < Mused) load_chunk(m0 + 32);
    bt_forward_subst<NT8>(sL, srs, N, y);
    double a = 0.0, a01 = 0.0;
#pragma unroll
    for(int i = 0; i < NMAX; i++)
      if(i < N)
      {
        a = fma(y[i], y[i], a);
        if(fs == 2) a01 = fma(y[i], __shfl_down_sync(0xffffffffu, y[i], 1), a01);
      }
    double f;
    if(fs == 1)
    {
      outlierness_factor(&f, &xm, &a, 1, k);
      if(m < Mused) gf[m] = failed ? __longlong_as_double(0x7ff8000000000000LL) : f;
    }
    else
    {
      const double A2[3] = { a, a01, __shfl_down_sync(0xffffffffu, a, 1) };
      const double x2[2] = { xm, __shfl_down_sync(0xffffffffu, xm, 1) };
      outlierness_factor(&f, x2, A2, 2, k);
      if(!(lane & 1) && m < Mused) gf[m >> 1] = failed ? __longlong_as_double(0x7ff8000000000000LL) : f;
    }
  }
}

// statistics of the last batched solve of this thread, for bench.py:
// [0] kernel launches, [1] sum over launches of active problems, [2] ms in k_batched_trial (CUDA
// events on the launching stream), [3] ms in the user callback (same events), [4] total accepted steps
static thread_local double g_batched_stats[8];
extern "C" void dogleg_gpu_batched_stats(double out[8]) { memcpy(out, g_batched_stats, sizeof(g_batched_stats)); }

static size_t batched_smem_bytes(int N)
{
  const int nt8 = (N + 7) / 8, ld = 8 * nt8 + 1;
  return sizeof(double) * (size_t)BT_WARPS * (2 * 8 * nt8 * ld + 6 * BT_NMAX);
}
typedef void (*batched_kernel_t)(BatchState);
// what the callback hands over; the two products layouts differ in the size of the JtJ buffer
enum { BF_DENSE = 0, BF_PRODUCTS_FULL = 1, BF_PRODUCTS_PACKED = 2, BF_DENSE_RAGGED = 3, BF_DENSE_F32 = 4,
       BF_DENSE_RAGGED_F32 = 5 };
static bool bf_ragged(int form) { return form == BF_DENSE_RAGGED || form == BF_DENSE_RAGGED_F32; }
static bool bf_f32(int form) { return form == BF_DENSE_F32 || form == BF_DENSE_RAGGED_F32; }
// register-ring variant of the J'J loop (BT_RING row groups in flight; measured in round 2,
// profiles/r02_variants.txt: 1.37 -> 1.20 ms per trial launch at C3). The products form has no such loop.
template<int NT8> static batched_kernel_t batched_kernel_nt8(int form)
{
  switch(form)
  {
  case BF_DENSE: return k_batched_trial<NT8, BT_RING, false, false>;
  case BF_DENSE_RAGGED: return k_batched_trial<NT8, BT_RING, false, true>;
  case BF_DENSE_F32: return k_batched_trial<NT8, BT_RING, false, false, float>;
  case BF_DENSE_RAGGED_F32: return k_batched_trial<NT8, BT_RING, false, true, float>;
  default: return k_batched_trial<NT8, BT_RING, true, false>;
  }
}
static batched_kernel_t batched_kernel(int N, int form)
{
  switch((N + 7) / 8)
  {
  case 1: return batched_kernel_nt8<1>(form);
  case 2: return batched_kernel_nt8<2>(form);
  case 3: return batched_kernel_nt8<3>(form);
  default: return batched_kernel_nt8<4>(form);
  }
}

// The row offsets (B + 1) and the longest-first order (B) of a ragged batch: a stable counting sort of the counts,
// descending, ties by index, in two passes over 16-bit digits. -1 if a count exceeds INT_MAX.
extern "C" int dlb_batched_ragged_layout(const unsigned int* Nmeas, unsigned int B, long long* row_off, int* order)
{
  row_off[0] = 0;
  for(unsigned int b = 0; b < B; b++)
  {
    if(Nmeas[b] > (unsigned int)INT_MAX) return -1;
    row_off[b + 1] = row_off[b] + Nmeas[b];
  }
  std::vector<int> tmp(B);
  for(unsigned int b = 0; b < B; b++) order[b] = (int)b;
  int* src = order; int* dst = tmp.data();
  for(int shift = 0; shift < 32; shift += 16)
  {
    std::vector<unsigned int> pos(65537, 0);
    auto digit = [&](int b) { return (~Nmeas[b] >> shift) & 0xffffu; };        // ~count: ascending = longest first
    for(unsigned int i = 0; i < B; i++) pos[digit(src[i]) + 1]++;
    for(int d = 0; d < 65536; d++) pos[d + 1] += pos[d];
    for(unsigned int i = 0; i < B; i++) dst[pos[digit(src[i])]++] = src[i];
    std::swap(src, dst);
  }
  return 0;                                                                      // (two passes: src == order)
}

// Device workspace of the last batched solve, kept for the next one of the same shape and form (the big
// cudaMalloc/cudaFree pairs cost far more than a solve); dogleg_gpu_release_batched_cache() frees it.
struct BatchWorkspace
{
  int B = 0, N = 0, M = 0, form = -1, device = -1;
  long long rows = 0;         // the ragged form's total row count
  std::vector<void*> allocs;
  cudaStream_t st = 0;
  int* h_active = 0;
  void release()
  {
    if(device >= 0) cudaSetDevice(device);
    for(void* q : allocs) cudaFree(q);
    allocs.clear();
    if(st) cudaStreamDestroy(st);
    if(h_active) cudaFreeHost(h_active);
    st = 0; h_active = 0; B = N = M = 0; rows = 0; form = -1; device = -1;
  }
};
static thread_local BatchWorkspace g_ws;
extern "C" void dogleg_gpu_release_batched_cache(void) { g_ws.release(); }

#define CUB(call) do { cudaError_t _e = (call); if(_e != cudaSuccess) { \
  dlb_set_error((std::string(#call) + ": " + cudaGetErrorString(_e)).c_str()); goto fail; } } while(0)

// The final state of a batched solve. Its own allocations: the workspace cache never aliases them.
struct dogleg_gpu_batch
{
  int device = -1, B = 0, N = 0;
  double* JtJ = 0;            // B x N*N, the final point's
  double* lambda = 0;         // B
  int* status = 0;            // B, DOGLEG_GPU_BATCH_*
  int* nfail = 0;             // 1, for the host-pointer forms
  // a ragged solve's layout (row_off == NULL: a uniform solve): B + 1 row offsets and the longest-first order on
  // the device, the counts and their sum on the host
  long long* row_off = 0;
  int* order = 0;
  std::vector<unsigned int> Nmeas;
  long long rows = 0;
  cudaStream_t st = 0;        // the host-pointer forms run here
  cudaEvent_t ev = 0;         // the handle's last enqueued work: every call is ordered after it
};

// makes the handle's device current for the scope of a call and restores the caller's afterwards
struct DeviceScope
{
  int prev = -1;
  explicit DeviceScope(int d) { if(cudaGetDevice(&prev) != cudaSuccess) prev = -1; cudaSetDevice(d); }
  ~DeviceScope() { if(prev >= 0) cudaSetDevice(prev); }
};

static void batch_destroy(dogleg_gpu_batch_t* h)
{
  DeviceScope ds(h->device);
  if(h->ev) cudaEventSynchronize(h->ev);
  cudaFree(h->JtJ); cudaFree(h->lambda); cudaFree(h->status); cudaFree(h->nfail); cudaFree(h->row_off); cudaFree(h->order);
  if(h->st) cudaStreamDestroy(h->st);
  if(h->ev) cudaEventDestroy(h->ev);
  delete h;
}

static dogleg_gpu_batch_t* batch_create(int device, int B, int N, bool ragged)
{
  dogleg_gpu_batch_t* h = new dogleg_gpu_batch_t;
  h->device = device; h->B = B; h->N = N;
  DeviceScope ds(device);
  if((ragged && (cudaMalloc((void**)&h->row_off, ((size_t)B + 1) * sizeof(long long)) != cudaSuccess ||
                 cudaMalloc((void**)&h->order, (size_t)B * sizeof(int)) != cudaSuccess)) ||
     cudaMalloc((void**)&h->JtJ, (size_t)B * N * N * sizeof(double)) != cudaSuccess ||
     cudaMalloc((void**)&h->lambda, (size_t)B * sizeof(double)) != cudaSuccess ||
     cudaMalloc((void**)&h->status, (size_t)B * sizeof(int)) != cudaSuccess ||
     cudaMalloc((void**)&h->nfail, sizeof(int)) != cudaSuccess ||
     cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking) != cudaSuccess ||
     cudaEventCreateWithFlags(&h->ev, cudaEventDisableTiming) != cudaSuccess)
  {
    cudaGetLastError();
    batch_destroy(h);
    return 0;
  }
  return h;
}

// the solve behind the batched entry points, after their argument checks; M = 0 for the products and ragged
// forms. Ragged: Nmeas (B counts) with its host row offsets and order from dlb_batched_ragged_layout.
static int batched_solve(int form, double* p, int N, int M, unsigned int B, void* f, void* cookie,
                         const dogleg_parameters2_t* parameters, double* norm2x_out, int* iterations_out,
                         dogleg_gpu_batch_t** returnBatch, const unsigned int* Nmeas = 0,
                         const long long* h_row_off = 0, const int* h_order = 0)
{
  static const char* const name[] = { "dense_batched", "dense_products_batched", "dense_products_batched",
                                      "dogleg_gpu_optimize_dense_batched_ragged",
                                      "dogleg_gpu_optimize_dense_batched_f32jac",
                                      "dogleg_gpu_optimize_dense_batched_ragged_f32jac" };
  const bool ragged = bf_ragged(form), f32 = bf_f32(form);
  const long long rows = ragged ? h_row_off[B] : 0;
  const size_t smem = batched_smem_bytes(N);
  batched_kernel_t kern = batched_kernel(N, form);
  dogleg_parameters2_t P;
  if(parameters) P = *parameters; else dogleg_getDefaultParameters(&P);
  cudaSetDevice(dogleg_gpu_get_device());

  BatchState S;
  memset(&S, 0, sizeof(S));
  S.B = (int)B; S.N = N; S.M = M; S.max_iterations = P.max_iterations;
  S.tr0 = P.trustregion0; S.dec_factor = P.trustregion_decrease_factor; S.dec_thr = P.trustregion_decrease_threshold;
  S.inc_factor = P.trustregion_increase_factor; S.inc_thr = P.trustregion_increase_threshold;
  S.Jtx_thr = P.Jt_x_threshold; S.upd_thr = P.update_threshold; S.tr_thr = P.trustregion_threshold;
  BatchWorkspace& W = g_ws;
  int result = -1;
  dogleg_gpu_batch_t* h = 0;
  if(W.B != (int)B || W.N != N || W.M != M || W.rows != rows || W.form != form || W.device != dogleg_gpu_get_device())
  {
    W.release();
    W.device = dogleg_gpu_get_device();
    const size_t bN = (size_t)B * N * sizeof(double), bd = (size_t)B * sizeof(double), bi = (size_t)B * sizeof(int);
    std::vector<size_t> sizes = { bd, bd, bd, bd, bd, bd, bi, bi, bi, bN, bN, bN, bN, bN,
                                  (size_t)B * N * N * sizeof(double), sizeof(int) };
    const size_t jsz = f32 ? sizeof(float) : sizeof(double);          // an entry of J
    if(form == BF_DENSE || form == BF_DENSE_F32) sizes.insert(sizes.end(), { (size_t)B * M * sizeof(double), (size_t)B * M * N * jsz });
    else if(ragged)
      sizes.insert(sizes.end(), { (size_t)rows * sizeof(double), (size_t)rows * N * jsz,
                                  ((size_t)B + 1) * sizeof(long long), (size_t)B * sizeof(int) });
    else
    {
      const size_t nS = form == BF_PRODUCTS_PACKED ? (size_t)N * (N + 1) / 2 : (size_t)N * N;
      sizes.insert(sizes.end(), { bd, bN, (size_t)B * nS * sizeof(double) });
    }
    for(size_t bytes : sizes)
    {
      void* q = 0;
      if(cudaMalloc(&q, bytes ? bytes : 8) != cudaSuccess) { cudaGetLastError(); break; }
      W.allocs.push_back(q);
    }
    if(W.allocs.size() != sizes.size() ||
       cudaStreamCreateWithFlags(&W.st, cudaStreamNonBlocking) != cudaSuccess ||
       cudaHostAlloc((void**)&W.h_active, sizeof(int), cudaHostAllocDefault) != cudaSuccess)
    {
      W.release();
      dlb_set_error((std::string(name[form]) + ": out of device memory").c_str());
      return -1;
    }
    W.B = (int)B; W.N = N; W.M = M; W.rows = rows; W.form = form;
  }
  {
    void** a = W.allocs.data();
    S.tr = (double*)a[0]; S.n2x_before = (double*)a[1]; S.n2c = (double*)a[2]; S.n2gn = (double*)a[3];
    S.expected = (double*)a[4]; S.lambda = (double*)a[5];
    S.steps = (int*)a[6]; S.flags = (int*)a[7]; S.active = (int*)a[8];
    S.p_before = (double*)a[9]; S.ptrial = (double*)a[10]; S.Jtx = (double*)a[11]; S.cauchy = (double*)a[12];
    S.gn = (double*)a[13]; S.JtJ = (double*)a[14]; S.n_active = (int*)a[15];
    if(form == BF_DENSE || ragged || f32)
    {
      S.x = (double*)a[16];
      if(f32) S.Jf = (float*)a[17]; else S.J = (double*)a[17];
    }
    if(ragged) { S.row_off = (const long long*)a[18]; S.order = (const int*)a[19]; }
    else if(form != BF_DENSE && form != BF_DENSE_F32) { S.norm2x_in = (double*)a[16]; S.Jtx_in = (double*)a[17]; S.JtJ_in = (double*)a[18]; S.packed = form == BF_PRODUCTS_PACKED; }
  }
  cudaStream_t st = W.st;
  int* h_active = W.h_active;
  if(returnBatch)
  {
    h = batch_create(W.device, (int)B, N, ragged);
    if(!h)
    {
      const std::string who = form == BF_DENSE ? "dense_batched2" : ragged || f32 ? name[form] : "dense_products_batched2";
      dlb_set_error((who + ": out of device memory for the returned batch").c_str());
      return -1;
    }
    if(ragged) { h->Nmeas.assign(Nmeas, Nmeas + B); h->rows = rows; }
    S.status = h->status;
    CUB(cudaMemsetAsync(S.status, 0, (size_t)B * sizeof(int), st));
  }
  CUB(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CUB(cudaMemcpyAsync(S.ptrial, p, (size_t)B * N * sizeof(double), cudaMemcpyHostToDevice, st));
  CUB(cudaMemcpyAsync(S.p_before, p, (size_t)B * N * sizeof(double), cudaMemcpyHostToDevice, st));
  CUB(cudaMemsetAsync(S.lambda, 0, (size_t)B * sizeof(double), st));
  CUB(cudaMemsetAsync(S.steps, 0, (size_t)B * sizeof(int), st));
  CUB(cudaMemsetAsync(S.flags, 0, (size_t)B * sizeof(int), st));
  if(ragged)
  {
    CUB(cudaMemcpyAsync((void*)S.row_off, h_row_off, ((size_t)B + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
    CUB(cudaMemcpyAsync((void*)S.order, h_order, (size_t)B * sizeof(int), cudaMemcpyHostToDevice, st));
  }
  {
    std::vector<double> tr(B, S.tr0);
    std::vector<int> ones(B, 1);
    const int nb = (int)B;
    CUB(cudaMemcpyAsync(S.tr, tr.data(), (size_t)B * sizeof(double), cudaMemcpyHostToDevice, st));
    CUB(cudaMemcpyAsync(S.active, ones.data(), (size_t)B * sizeof(int), cudaMemcpyHostToDevice, st));
    CUB(cudaMemcpyAsync(S.n_active, &nb, sizeof(int), cudaMemcpyHostToDevice, st));
    CUB(cudaStreamSynchronize(st));
  }
  *h_active = (int)B;
  memset(g_batched_stats, 0, sizeof(g_batched_stats));
  {
    cudaEvent_t ev[3];
    for(int u = 0; u < 3; u++) cudaEventCreate(&ev[u]);
    // every problem needs at most (max_iterations accepted + rejected) trials; rejected trials are
    // bounded by the trust region collapsing below its threshold
    const long long trial_cap = 64LL * (long long)std::max(P.max_iterations, 1) + 4096;
    for(long long t = 0; *h_active > 0 && t < trial_cap; t++)
    {
      g_batched_stats[0] += 1; g_batched_stats[1] += *h_active;
      cudaEventRecord(ev[0], st);
      if(form == BF_DENSE)
        ((dogleg_gpu_callback_dense_batched_t*)f)(S.ptrial, S.x, S.J, S.active, (int)B, (void*)st, cookie);
      else if(form == BF_DENSE_RAGGED)
        ((dogleg_gpu_callback_dense_ragged_t*)f)(S.ptrial, S.x, S.J, S.row_off, S.active, (int)B, (void*)st, cookie);
      else if(form == BF_DENSE_F32)
        ((dogleg_gpu_callback_dense_batched_f32jac_t*)f)(S.ptrial, S.x, S.Jf, S.active, (int)B, (void*)st, cookie);
      else if(form == BF_DENSE_RAGGED_F32)
        ((dogleg_gpu_callback_dense_ragged_f32jac_t*)f)(S.ptrial, S.x, S.Jf, S.row_off, S.active, (int)B, (void*)st,
                                                         cookie);
      else
        ((dogleg_gpu_callback_dense_products_batched_t*)f)(S.ptrial, S.norm2x_in, S.Jtx_in, S.JtJ_in, S.active, (int)B,
                                                            (void*)st, cookie);
      cudaEventRecord(ev[1], st);
      kern<<<(B + BT_WARPS - 1) / BT_WARPS, BT_NT, smem, st>>>(S);
      cudaEventRecord(ev[2], st);
      CUB(cudaGetLastError());
      CUB(cudaMemcpyAsync(h_active, S.n_active, sizeof(int), cudaMemcpyDeviceToHost, st));
      CUB(cudaStreamSynchronize(st));
      float ms_cb = 0, ms_k = 0;
      cudaEventElapsedTime(&ms_cb, ev[0], ev[1]); cudaEventElapsedTime(&ms_k, ev[1], ev[2]);
      g_batched_stats[2] += ms_k; g_batched_stats[3] += ms_cb;
    }
    for(int u = 0; u < 3; u++) cudaEventDestroy(ev[u]);
  }
  CUB(cudaMemcpyAsync(p, S.p_before, (size_t)B * N * sizeof(double), cudaMemcpyDeviceToHost, st));
  if(norm2x_out) CUB(cudaMemcpyAsync(norm2x_out, S.n2x_before, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st));
  if(iterations_out) CUB(cudaMemcpyAsync(iterations_out, S.steps, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  if(h)
  {
    CUB(cudaMemcpyAsync(h->JtJ, S.JtJ, (size_t)B * N * N * sizeof(double), cudaMemcpyDeviceToDevice, st));
    CUB(cudaMemcpyAsync(h->lambda, S.lambda, (size_t)B * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if(ragged)
    {
      CUB(cudaMemcpyAsync(h->row_off, S.row_off, ((size_t)B + 1) * sizeof(long long), cudaMemcpyDeviceToDevice, st));
      CUB(cudaMemcpyAsync(h->order, S.order, (size_t)B * sizeof(int), cudaMemcpyDeviceToDevice, st));
    }
  }
  CUB(cudaStreamSynchronize(st));
  result = (int)B - *h_active;
  if(h) { *returnBatch = h; h = 0; }
fail:
  if(h) batch_destroy(h);
  return result;
}

// enqueue k_batched_factor on st, after the handle's earlier work; it becomes the handle's latest
static int batch_enqueue(dogleg_gpu_batch_t* h, const double* d_R, double* d_X, int nrhs, int packed, int* nfail,
                         cudaStream_t st)
{
  typedef void (*factor_kernel_t)(BatchFactorArgs);
  const int nt8 = (h->N + 7) / 8, ld = 8 * nt8 + 1;
  const factor_kernel_t kern = nt8 == 1 ? k_batched_factor<1> : nt8 == 2 ? k_batched_factor<2>
                             : nt8 == 3 ? k_batched_factor<3> : k_batched_factor<4>;
  const size_t smem = sizeof(double) * (size_t)BT_WARPS * (32 * ld + 8 * nt8 * ld + 8 * nt8);
  BatchFactorArgs A = { h->B, h->N, nrhs, h->JtJ, h->lambda, d_R, d_X, packed, nfail };
  CUB(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CUB(cudaStreamWaitEvent(st, h->ev, 0));
  kern<<<(h->B + BT_WARPS - 1) / BT_WARPS, BT_NT, smem, st>>>(A);
  CUB(cudaGetLastError());
  CUB(cudaEventRecord(h->ev, st));
  return 0;
fail:
  return -1;
}

// the host-pointer forms: stage through device buffers on the handle's stream; returns the failed problems
static int batch_host(dogleg_gpu_batch_t* h, const double* R, double* X, int nrhs, int packed)
{
  DeviceScope ds(h->device);
  const size_t nin = R ? (size_t)h->B * h->N * nrhs : 0;
  const size_t nout = packed ? (size_t)h->B * (h->N * (h->N + 1) / 2) : (size_t)h->B * h->N * (R ? nrhs : h->N);
  double *dR = 0, *dX = 0;
  int nfail = 0, result = -1;
  CUB(cudaMalloc((void**)&dX, nout * sizeof(double)));
  if(R)
  {
    CUB(cudaMalloc((void**)&dR, nin * sizeof(double)));
    CUB(cudaMemcpyAsync(dR, R, nin * sizeof(double), cudaMemcpyHostToDevice, h->st));
  }
  CUB(cudaStreamWaitEvent(h->st, h->ev, 0));
  CUB(cudaMemsetAsync(h->nfail, 0, sizeof(int), h->st));
  if(batch_enqueue(h, dR, dX, nrhs, packed, h->nfail, h->st)) goto fail;
  CUB(cudaMemcpyAsync(X, dX, nout * sizeof(double), cudaMemcpyDeviceToHost, h->st));
  CUB(cudaMemcpyAsync(&nfail, h->nfail, sizeof(int), cudaMemcpyDeviceToHost, h->st));
  CUB(cudaStreamSynchronize(h->st));
  result = nfail;
fail:
  cudaFree(dR); cudaFree(dX);
  return result;
}

extern "C" int dogleg_gpu_batch_status(const dogleg_gpu_batch_t* h, int* status_out, double* lambda_out)
{
  if(!h) { dlb_set_error("dogleg_gpu_batch_status: NULL handle"); return -1; }
  DeviceScope ds(h->device);
  CUB(cudaStreamWaitEvent(h->st, h->ev, 0));
  if(status_out) CUB(cudaMemcpyAsync(status_out, h->status, (size_t)h->B * sizeof(int), cudaMemcpyDeviceToHost, h->st));
  if(lambda_out) CUB(cudaMemcpyAsync(lambda_out, h->lambda, (size_t)h->B * sizeof(double), cudaMemcpyDeviceToHost, h->st));
  CUB(cudaStreamSynchronize(h->st));
  return 0;
fail:
  return -1;
}

extern "C" int dogleg_gpu_batch_solve(dogleg_gpu_batch_t* h, const double* R, double* X, int nrhs)
{
  if(!h) { dlb_set_error("dogleg_gpu_batch_solve: NULL handle"); return -1; }
  if(!R || !X || nrhs < 1) { dlb_set_error("dogleg_gpu_batch_solve: bad arguments (needs R, X and nrhs >= 1)"); return -1; }
  return batch_host(h, R, X, nrhs, 0);
}

extern "C" int dogleg_gpu_batch_solve_device(dogleg_gpu_batch_t* h, const double* d_R, double* d_X, int nrhs, void* stream)
{
  if(!h) { dlb_set_error("dogleg_gpu_batch_solve_device: NULL handle"); return -1; }
  if(!d_R || !d_X || nrhs < 1) { dlb_set_error("dogleg_gpu_batch_solve_device: bad arguments (needs d_R, d_X and nrhs >= 1)"); return -1; }
  DeviceScope ds(h->device);
  return batch_enqueue(h, d_R, d_X, nrhs, 0, 0, (cudaStream_t)stream);
}

extern "C" int dogleg_gpu_batch_covariance(dogleg_gpu_batch_t* h, double* out, int packed)
{
  if(!h) { dlb_set_error("dogleg_gpu_batch_covariance: NULL handle"); return -1; }
  if(!out) { dlb_set_error("dogleg_gpu_batch_covariance: bad arguments (needs out)"); return -1; }
  return batch_host(h, 0, out, h->N, packed != 0);
}

extern "C" int dogleg_gpu_batch_covariance_device(dogleg_gpu_batch_t* h, double* d_out, int packed, void* stream)
{
  if(!h) { dlb_set_error("dogleg_gpu_batch_covariance_device: NULL handle"); return -1; }
  if(!d_out) { dlb_set_error("dogleg_gpu_batch_covariance_device: bad arguments (needs d_out)"); return -1; }
  DeviceScope ds(h->device);
  return batch_enqueue(h, 0, d_out, h->N, packed != 0, 0, (cudaStream_t)stream);
}

// the argument checks of both outlierness calls; featureSize <= 1 means 1 (as in the reference)
static bool outlier_args_ok(const char* fn, const dogleg_gpu_batch_t* h, const void* x, const void* J, const void* scale,
                            const void* factors, unsigned int Nmeas, int& featureSize, int Nfeatures)
{
  std::string msg;
  if(featureSize <= 1) featureSize = 1;
  if(!h) msg = "NULL handle";
  else if(h->row_off) msg = "the handle is from a ragged solve: use dogleg_gpu_batch_outlierness_ragged";
  else if(!x || !J || !scale || !factors) msg = "bad arguments (needs x, J, scale and factors)";
  else if(featureSize > 2) msg = "featureSize > 2 not implemented yet. Got featureSize=" + std::to_string(featureSize);
  else if(Nfeatures < 1 || Nmeas < 1 || Nmeas > (unsigned int)INT_MAX) msg = "bad arguments (needs Nfeatures >= 1 and Nmeas >= 1)";
  else if((long long)Nfeatures * featureSize > (long long)Nmeas) msg = "Nfeatures*featureSize exceeds Nmeas";
  if(msg.empty()) return true;
  dlb_set_error((std::string(fn) + ": " + msg).c_str());
  return false;
}

// enqueue k_batched_outlierness on st, after the handle's earlier work; it becomes the handle's latest
// (a ragged handle: M and nfeat unused, d_nfeat its B feature counts or NULL)
typedef void (*outlier_kernel_t)(BatchOutlierArgs);
template<bool RAGGED> static outlier_kernel_t outlier_kernel(int nt8)
{
  return nt8 == 1 ? k_batched_outlierness<1, RAGGED> : nt8 == 2 ? k_batched_outlierness<2, RAGGED>
       : nt8 == 3 ? k_batched_outlierness<3, RAGGED> : k_batched_outlierness<4, RAGGED>;
}
static int batch_outlier_enqueue(dogleg_gpu_batch_t* h, const double* d_x, const double* d_J, int M, int fsize,
                                 int nfeat, const int* d_nfeat, const int* d_nout, double* d_scale, double* d_factors,
                                 int* nfail, cudaStream_t st)
{
  const int nt8 = (h->N + 7) / 8, ld = 8 * nt8 + 1;
  const outlier_kernel_t kern = h->row_off ? outlier_kernel<true>(nt8) : outlier_kernel<false>(nt8);
  const size_t smem = sizeof(double) * (size_t)BT_WARPS * (32 * ld + 8 * nt8 * ld + 8 * nt8);
  BatchOutlierArgs A = { h->B, h->N, M, fsize, nfeat, h->JtJ, h->lambda, d_x, d_J, d_nout, d_scale, d_factors, nfail,
                         h->row_off, d_nfeat, h->order };
  CUB(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CUB(cudaStreamWaitEvent(st, h->ev, 0));
  kern<<<(h->B + BT_WARPS - 1) / BT_WARPS, BT_NT, smem, st>>>(A);
  CUB(cudaGetLastError());
  CUB(cudaEventRecord(h->ev, st));
  return 0;
fail:
  return -1;
}

extern "C" int dogleg_gpu_batch_outlierness(dogleg_gpu_batch_t* h, const double* x, const double* J, unsigned int Nmeas,
                                            int featureSize, int Nfeatures, const int* NoutlierFeatures,
                                            double* scale, double* factors)
{
  if(!outlier_args_ok("dogleg_gpu_batch_outlierness", h, x, J, scale, factors, Nmeas, featureSize, Nfeatures)) return -1;
  DeviceScope ds(h->device);
  const size_t B = (size_t)h->B, nx = B * Nmeas, nJ = nx * h->N, nf = B * Nfeatures;
  double *dx = 0, *dJ = 0, *dscale = 0, *df = 0;
  int* dnout = 0;
  int nfail = 0, result = -1;
  CUB(cudaMalloc((void**)&dx, nx * sizeof(double)));
  CUB(cudaMalloc((void**)&dJ, nJ * sizeof(double)));
  CUB(cudaMalloc((void**)&dscale, B * sizeof(double)));
  CUB(cudaMalloc((void**)&df, nf * sizeof(double)));
  CUB(cudaMemcpyAsync(dx, x, nx * sizeof(double), cudaMemcpyHostToDevice, h->st));
  CUB(cudaMemcpyAsync(dJ, J, nJ * sizeof(double), cudaMemcpyHostToDevice, h->st));
  CUB(cudaMemcpyAsync(dscale, scale, B * sizeof(double), cudaMemcpyHostToDevice, h->st));
  if(NoutlierFeatures)
  {
    CUB(cudaMalloc((void**)&dnout, B * sizeof(int)));
    CUB(cudaMemcpyAsync(dnout, NoutlierFeatures, B * sizeof(int), cudaMemcpyHostToDevice, h->st));
  }
  CUB(cudaStreamWaitEvent(h->st, h->ev, 0));
  CUB(cudaMemsetAsync(h->nfail, 0, sizeof(int), h->st));
  if(batch_outlier_enqueue(h, dx, dJ, (int)Nmeas, featureSize, Nfeatures, 0, dnout, dscale, df, h->nfail, h->st)) goto fail;
  CUB(cudaMemcpyAsync(factors, df, nf * sizeof(double), cudaMemcpyDeviceToHost, h->st));
  CUB(cudaMemcpyAsync(scale, dscale, B * sizeof(double), cudaMemcpyDeviceToHost, h->st));
  CUB(cudaMemcpyAsync(&nfail, h->nfail, sizeof(int), cudaMemcpyDeviceToHost, h->st));
  CUB(cudaStreamSynchronize(h->st));
  result = nfail;
fail:
  cudaFree(dx); cudaFree(dJ); cudaFree(dscale); cudaFree(df); cudaFree(dnout);
  return result;
}

extern "C" int dogleg_gpu_batch_outlierness_device(dogleg_gpu_batch_t* h, const double* d_x, const double* d_J,
                                                   unsigned int Nmeas, int featureSize, int Nfeatures,
                                                   const int* d_NoutlierFeatures, double* d_scale, double* d_factors,
                                                   void* stream)
{
  if(!outlier_args_ok("dogleg_gpu_batch_outlierness_device", h, d_x, d_J, d_scale, d_factors, Nmeas, featureSize,
                      Nfeatures))
    return -1;
  DeviceScope ds(h->device);
  return batch_outlier_enqueue(h, d_x, d_J, (int)Nmeas, featureSize, Nfeatures, 0, d_NoutlierFeatures, d_scale,
                               d_factors, 0, (cudaStream_t)stream);
}

// the argument checks of both ragged outlierness calls; featureSize <= 1 means 1
static bool outlier_ragged_args_ok(const char* fn, const dogleg_gpu_batch_t* h, const void* x, const void* J,
                                   const void* scale, const void* factors, int& featureSize)
{
  std::string msg;
  if(featureSize <= 1) featureSize = 1;
  if(!h) msg = "NULL handle";
  else if(!h->row_off) msg = "the handle is from a uniform batched solve: use dogleg_gpu_batch_outlierness";
  else if(!x || !J || !scale || !factors) msg = "bad arguments (needs x, J, scale and factors)";
  else if(featureSize > 2) msg = "featureSize > 2 not implemented yet. Got featureSize=" + std::to_string(featureSize);
  if(msg.empty()) return true;
  dlb_set_error((std::string(fn) + ": " + msg).c_str());
  return false;
}

extern "C" int dogleg_gpu_batch_outlierness_ragged(dogleg_gpu_batch_t* h, const double* x, const double* J,
                                                   int featureSize, const int* Nfeatures, const int* NoutlierFeatures,
                                                   double* scale, double* factors)
{
  static const char* fn = "dogleg_gpu_batch_outlierness_ragged";
  if(!outlier_ragged_args_ok(fn, h, x, J, scale, factors, featureSize)) return -1;
  if(Nfeatures)
    for(int b = 0; b < h->B; b++)
      if(Nfeatures[b] < 0 || (long long)Nfeatures[b] * featureSize > (long long)h->Nmeas[b])
      {
        dlb_set_error((std::string(fn) + ": Nfeatures[b]*featureSize must be in 0..Nmeas[b]; b = " + std::to_string(b) +
                       ", Nfeatures[b] = " + std::to_string(Nfeatures[b]) + ", Nmeas[b] = " +
                       std::to_string(h->Nmeas[b])).c_str());
        return -1;
      }
  DeviceScope ds(h->device);
  const size_t B = (size_t)h->B, nx = (size_t)h->rows, nJ = nx * h->N;
  double *dx = 0, *dJ = 0, *dscale = 0, *df = 0;
  int *dnfeat = 0, *dnout = 0;
  int nfail = 0, result = -1;
  CUB(cudaMalloc((void**)&dx, (nx ? nx : 1) * sizeof(double)));
  CUB(cudaMalloc((void**)&dJ, (nJ ? nJ : 1) * sizeof(double)));
  CUB(cudaMalloc((void**)&dscale, B * sizeof(double)));
  CUB(cudaMalloc((void**)&df, (nx ? nx : 1) * sizeof(double)));
  CUB(cudaMemcpyAsync(dx, x, nx * sizeof(double), cudaMemcpyHostToDevice, h->st));
  CUB(cudaMemcpyAsync(dJ, J, nJ * sizeof(double), cudaMemcpyHostToDevice, h->st));
  CUB(cudaMemcpyAsync(dscale, scale, B * sizeof(double), cudaMemcpyHostToDevice, h->st));
  CUB(cudaMemcpyAsync(df, factors, nx * sizeof(double), cudaMemcpyHostToDevice, h->st));     // rows that are no feature stay
  if(Nfeatures)
  {
    CUB(cudaMalloc((void**)&dnfeat, B * sizeof(int)));
    CUB(cudaMemcpyAsync(dnfeat, Nfeatures, B * sizeof(int), cudaMemcpyHostToDevice, h->st));
  }
  if(NoutlierFeatures)
  {
    CUB(cudaMalloc((void**)&dnout, B * sizeof(int)));
    CUB(cudaMemcpyAsync(dnout, NoutlierFeatures, B * sizeof(int), cudaMemcpyHostToDevice, h->st));
  }
  CUB(cudaStreamWaitEvent(h->st, h->ev, 0));
  CUB(cudaMemsetAsync(h->nfail, 0, sizeof(int), h->st));
  if(batch_outlier_enqueue(h, dx, dJ, 0, featureSize, 0, dnfeat, dnout, dscale, df, h->nfail, h->st)) goto fail;
  CUB(cudaMemcpyAsync(factors, df, nx * sizeof(double), cudaMemcpyDeviceToHost, h->st));
  CUB(cudaMemcpyAsync(scale, dscale, B * sizeof(double), cudaMemcpyDeviceToHost, h->st));
  CUB(cudaMemcpyAsync(&nfail, h->nfail, sizeof(int), cudaMemcpyDeviceToHost, h->st));
  CUB(cudaStreamSynchronize(h->st));
  result = nfail;
fail:
  cudaFree(dx); cudaFree(dJ); cudaFree(dscale); cudaFree(df); cudaFree(dnfeat); cudaFree(dnout);
  return result;
}

extern "C" int dogleg_gpu_batch_outlierness_ragged_device(dogleg_gpu_batch_t* h, const double* d_x, const double* d_J,
                                                          int featureSize, const int* d_Nfeatures,
                                                          const int* d_NoutlierFeatures, double* d_scale,
                                                          double* d_factors, void* stream)
{
  if(!outlier_ragged_args_ok("dogleg_gpu_batch_outlierness_ragged_device", h, d_x, d_J, d_scale, d_factors, featureSize))
    return -1;
  DeviceScope ds(h->device);
  return batch_outlier_enqueue(h, d_x, d_J, 0, featureSize, 0, d_Nfeatures, d_NoutlierFeatures, d_scale, d_factors, 0,
                               (cudaStream_t)stream);
}

extern "C" void dogleg_gpu_batch_free(dogleg_gpu_batch_t** batch)
{
  if(!batch || !*batch) return;
  batch_destroy(*batch);
  *batch = 0;
}

extern "C" int dogleg_gpu_optimize_dense_batched2(double* p, unsigned int Nstate, unsigned int Nmeas,
                                                  unsigned int B, dogleg_gpu_callback_dense_batched_t* f,
                                                  void* cookie, const dogleg_parameters2_t* parameters,
                                                  double* norm2x_out, int* iterations_out,
                                                  dogleg_gpu_batch_t** returnBatch)
{
  if(returnBatch) *returnBatch = 0;
  if(dogleg_gpu_device_count() <= 0) { dlb_set_error("no CUDA device available: libdogleg-b200 has no CPU fallback"); return -1; }
  if(!f || !p || B == 0) { dlb_set_error("dense_batched: bad arguments"); return -1; }
  const int N = (int)Nstate;
  if(N > BT_NMAX || N < 1)
  {
    dlb_set_error("dense_batched: needs Nstate <= 32; use dogleg_optimize_dense2 per problem for bigger ones");
    return -1;
  }
  return batched_solve(BF_DENSE, p, N, (int)Nmeas, B, (void*)f, cookie, parameters, norm2x_out, iterations_out,
                       returnBatch);
}

extern "C" int dogleg_gpu_optimize_dense_batched(double* p, unsigned int Nstate, unsigned int Nmeas,
                                                 unsigned int B, dogleg_gpu_callback_dense_batched_t* f,
                                                 void* cookie, const dogleg_parameters2_t* parameters,
                                                 double* norm2x_out, int* iterations_out)
{
  return dogleg_gpu_optimize_dense_batched2(p, Nstate, Nmeas, B, f, cookie, parameters, norm2x_out, iterations_out, 0);
}

// The checks and the host layout of both ragged entry points (form: BF_DENSE_RAGGED or BF_DENSE_RAGGED_F32), then the
// solve. Refuses, before the first callback and naming the entry point: Nstate outside 1..32, B == 0, a NULL p, Nmeas
// or callback, a count above INT_MAX and a batch whose x and J would not fit in a size_t.
static int ragged_solve(int form, const char* entry, double* p, unsigned int Nstate, const unsigned int* Nmeas,
                        unsigned int B, void* f, void* cookie, const dogleg_parameters2_t* parameters, double* norm2x_out,
                        int* iterations_out, dogleg_gpu_batch_t** returnBatch)
{
  const std::string fn = std::string(entry) + ": ";
  if(returnBatch) *returnBatch = 0;
  if(dogleg_gpu_device_count() <= 0) { dlb_set_error((fn + "no CUDA device available: libdogleg-b200 has no CPU fallback").c_str()); return -1; }
  if(!f || !p || !Nmeas || B == 0) { dlb_set_error((fn + "bad arguments (needs p, Nmeas, a callback and B > 0)").c_str()); return -1; }
  const int N = (int)Nstate;
  if(N > BT_NMAX || N < 1)
  {
    dlb_set_error((fn + "needs 1 <= Nstate <= 32; use dogleg_optimize_dense2 per problem for bigger ones").c_str());
    return -1;
  }
  std::vector<long long> row_off((size_t)B + 1);
  std::vector<int> order(B);
  if(dlb_batched_ragged_layout(Nmeas, B, row_off.data(), order.data()) != 0)
  {
    unsigned int b = 0;
    while(Nmeas[b] <= (unsigned int)INT_MAX) b++;
    dlb_set_error((fn + "Nmeas[" + std::to_string(b) + "] = " + std::to_string(Nmeas[b]) + " exceeds INT_MAX").c_str());
    return -1;
  }
  // bytes per row: x and J
  const size_t max_rows = form == BF_DENSE_RAGGED_F32 ? SIZE_MAX / (sizeof(double) + sizeof(float) * N)
                                                      : SIZE_MAX / sizeof(double) / (N + 1);
  if(row_off[B] > (long long)max_rows)
  {
    dlb_set_error((fn + "out of device memory").c_str());
    return -1;
  }
  return batched_solve(form, p, N, 0, B, f, cookie, parameters, norm2x_out, iterations_out, returnBatch, Nmeas,
                       row_off.data(), order.data());
}

extern "C" int dogleg_gpu_optimize_dense_batched_ragged(double* p, unsigned int Nstate, const unsigned int* Nmeas,
                                                        unsigned int B, dogleg_gpu_callback_dense_ragged_t* f,
                                                        void* cookie, const dogleg_parameters2_t* parameters,
                                                        double* norm2x_out, int* iterations_out,
                                                        dogleg_gpu_batch_t** returnBatch)
{
  return ragged_solve(BF_DENSE_RAGGED, "dogleg_gpu_optimize_dense_batched_ragged", p, Nstate, Nmeas, B, (void*)f, cookie,
                      parameters, norm2x_out, iterations_out, returnBatch);
}

extern "C" int dogleg_gpu_optimize_dense_batched_ragged_f32jac(double* p, unsigned int Nstate, const unsigned int* Nmeas,
                                                               unsigned int B, dogleg_gpu_callback_dense_ragged_f32jac_t* f,
                                                               void* cookie, const dogleg_parameters2_t* parameters,
                                                               double* norm2x_out, int* iterations_out,
                                                               dogleg_gpu_batch_t** returnBatch)
{
  return ragged_solve(BF_DENSE_RAGGED_F32, "dogleg_gpu_optimize_dense_batched_ragged_f32jac", p, Nstate, Nmeas, B,
                      (void*)f, cookie, parameters, norm2x_out, iterations_out, returnBatch);
}

extern "C" int dogleg_gpu_optimize_dense_batched_f32jac(double* p, unsigned int Nstate, unsigned int Nmeas,
                                                        unsigned int B, dogleg_gpu_callback_dense_batched_f32jac_t* f,
                                                        void* cookie, const dogleg_parameters2_t* parameters,
                                                        double* norm2x_out, int* iterations_out,
                                                        dogleg_gpu_batch_t** returnBatch)
{
  static const std::string fn = "dogleg_gpu_optimize_dense_batched_f32jac: ";
  if(returnBatch) *returnBatch = 0;
  if(dogleg_gpu_device_count() <= 0) { dlb_set_error((fn + "no CUDA device available: libdogleg-b200 has no CPU fallback").c_str()); return -1; }
  if(!f || !p || B == 0) { dlb_set_error((fn + "bad arguments (needs p, a callback and B > 0)").c_str()); return -1; }
  const int N = (int)Nstate;
  if(N > BT_NMAX || N < 1)
  {
    dlb_set_error((fn + "needs 1 <= Nstate <= 32; use dogleg_optimize_dense2 per problem for bigger ones").c_str());
    return -1;
  }
  if(Nmeas > (unsigned int)INT_MAX) { dlb_set_error((fn + "Nmeas exceeds INT_MAX").c_str()); return -1; }
  return batched_solve(BF_DENSE_F32, p, N, (int)Nmeas, B, (void*)f, cookie, parameters, norm2x_out, iterations_out,
                       returnBatch);
}

extern "C" int dogleg_gpu_optimize_dense_products_batched2(double* p, unsigned int Nstate, unsigned int B,
                                                           dogleg_gpu_callback_dense_products_batched_t* f, void* cookie,
                                                           const dogleg_parameters2_t* parameters,
                                                           double* norm2x_out, int* iterations_out,
                                                           dogleg_gpu_batch_t** returnBatch)
{
  if(returnBatch) *returnBatch = 0;
  if(dogleg_gpu_device_count() <= 0) { dlb_set_error("no CUDA device available: libdogleg-b200 has no CPU fallback"); return -1; }
  if(!f || !p || B == 0) { dlb_set_error("dense_products_batched: bad arguments (needs p, a callback and B > 0)"); return -1; }
  const int N = (int)Nstate;
  if(N > BT_NMAX || N < 1)
  {
    dlb_set_error("dense_products_batched: needs 1 <= Nstate <= 32; use dogleg_gpu_optimize_dense_products per problem for bigger ones");
    return -1;
  }
  const bool packed = parameters && parameters->JtJ_packed;
  if(packed && !parameters->JtJ_upper)
  { // dogleg.c:597-601: the reference cannot form the Cauchy step from a packed lower triangle
    dlb_set_error("dense_products_batched: a packed JtJ must be the upper triangle (JtJ_upper); packed lower is not supported");
    return -1;
  }
  return batched_solve(packed ? BF_PRODUCTS_PACKED : BF_PRODUCTS_FULL, p, N, 0, B, (void*)f, cookie, parameters,
                       norm2x_out, iterations_out, returnBatch);
}

extern "C" int dogleg_gpu_optimize_dense_products_batched(double* p, unsigned int Nstate, unsigned int B,
                                                          dogleg_gpu_callback_dense_products_batched_t* f, void* cookie,
                                                          const dogleg_parameters2_t* parameters,
                                                          double* norm2x_out, int* iterations_out)
{
  return dogleg_gpu_optimize_dense_products_batched2(p, Nstate, B, f, cookie, parameters, norm2x_out, iterations_out, 0);
}
