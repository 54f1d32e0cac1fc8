// dlb_front.cu -- multifrontal numeric Cholesky and triangular solves.
//
// Replaces cholmod_factorize[_p] (reference dogleg.c:656-665) and
// cholmod_solve(CHOLMOD_A) (:853-856) -- and, for the dense solve types where
// the whole matrix is a single front, dpptrf/dpotrf + dpptrs/dpotrs
// (:779-804, :872-892).
//
// Every supernode s owns a front: an r x r column-major lower-triangular block.
// One launch handles all fronts of one elimination-tree level, one CTA per
// front:
//   1. zero the front
//   2. add the partial JtJ blocks (Gpart) of the pattern classes assigned to it
//   3. extend-add the update matrices of its children (pull, fixed child order)
//   4. add lambda on the pivot diagonal
//   5. eliminate its ncols pivot columns (right-looking, in shared memory when
//      the front fits); the trailing block is left for the parent
// All sums are performed in a fixed order: results are bit-reproducible.
// A pivot <= 0 or non-finite marks the matrix as not positive definite (the
// LAPACK dpptrf rule; CHOLMOD's simplicial LDL' only flags exact zeros --
// documented divergence, SURVEY.md 2.2): the smallest failing column is kept.
#include "dlb_common.cuh"
#include "dlb_device.h"
#include "dlb_devfn.cuh"

#define FRONT_NT 256

// mode 0: full (assemble + children + lambda + eliminate); mode 1: elements only (tests)
template<bool SMEM, int NT>
__global__ void __launch_bounds__(NT)
k_front_level(DlbFrontDev F, DlbSparseDev S, int l0, double* __restrict__ fronts,
              const double* __restrict__ Gpart, double lambda, long long* minor, int mode)
{
  extern __shared__ double sh_front[];
  const int s   = F.level_sn[l0 + blockIdx.x];
  const int c0  = F.sn_first[s], nc = F.sn_first[s+1] - c0;
  const int rp  = F.rows_ptr[s], r = F.rows_ptr[s+1] - rp;
  double* Ag = fronts + F.front_off[s];
  double* A  = SMEM ? sh_front : Ag;
  const int tid = threadIdx.x;

  // Gpart == NULL: the front arrives pre-filled (dense solve types, row-sharded sums); else start
  // from zero -- unless the children have already been gathered into it (large fronts, -2). A large
  // front of 159 or 160 rows still fits the shared-memory variant: it then loads what was gathered.
  const long long toff = F.heavy_tmp_off ? F.heavy_tmp_off[s] : -1;
  const bool gathered_in_place = toff == -2 && mode != 1;
  if(Gpart && !gathered_in_place) for(int idx = tid; idx < r * r; idx += NT) A[idx] = 0.0;
  else if(SMEM) for(int idx = tid; idx < r * r; idx += NT) A[idx] = Ag[idx];
  __syncthreads();

  // ---- elements: classes assigned to this front ----
  if(Gpart)
    for(int ci = F.fcls_ptr[s]; ci < F.fcls_ptr[s+1]; ci++)
    {
      const int c = F.fcls_list[ci];
      const int k = S.cls_ptr[c+1] - S.cls_ptr[c];
      const int* loc = S.cls_loc + S.cls_ptr[c];
      const int npairs = k * (k + 1) / 2;
      const int t0 = F.cls_task_ptr[c], t1 = F.cls_task_ptr[c+1];
      for(int q = tid; q < npairs; q += NT)
      {
        double g = 0.0;
        for(int t = t0; t < t1; t++) g += Gpart[S.task_Goff[t] + q];
        int a, b; pair_from_index(q, a, b);
        const int la = loc[a], lb = loc[b];
        const int row = la > lb ? la : lb, col = la > lb ? lb : la;
        A[row + col * r] += g;
      }
      __syncthreads();
    }

  if(mode == 0 || mode == 2)
  {
    // ---- children: extend-add their update matrices ----
    if(toff >= 0)
    { // children already summed by k_extend_gather into this front's temporary, in its indexing
      const double* T0 = F.heavy_tmp + toff;
      for(int idx = tid; idx < r * r; idx += NT) A[idx] += T0[idx];
      __syncthreads();
    }
    for(int ch = (toff != -1) ? F.child_ptr[s+1] : F.child_ptr[s]; ch < F.child_ptr[s+1]; ch++)
    {
      const int c   = F.child_list[ch];
      const int ncc = F.sn_first[c+1] - F.sn_first[c];
      const int rc  = F.rows_ptr[c+1] - F.rows_ptr[c];
      const int nb  = rc - ncc;
      const double* U = fronts + F.front_off[c];
      const int* rel = F.rel + F.rows_ptr[c] + ncc;
      for(int idx = tid; idx < nb * nb; idx += NT)
      {
        const int j = idx / nb, i = idx - j * nb;
        if(i >= j) A[rel[i] + rel[j] * r] += U[(ncc + i) + (size_t)(ncc + j) * rc];
      }
      __syncthreads();
    }
    for(int j = tid; j < nc; j += NT) A[j + j * r] += lambda;
    __syncthreads();

    // ---- eliminate the pivot columns (mode 2: left to the blocked tensor-core path) ----
    if(mode != 2)
    {
      const int fail = front_eliminate<NT>(A, r, nc, r, r, tid, (double*)0);
      if(fail >= 0 && tid == 0) atomicMin(minor, (long long)(c0 + fail));
    }
  }
  if(SMEM)
  {
    __syncthreads();
    for(int idx = tid; idx < r * r; idx += NT) Ag[idx] = A[idx];
  }
}

// one warp per receiving block (gather_targets, dlb_devfn.cuh)
__global__ void __launch_bounds__(256)
k_extend_gather(DlbGather G, long long t0, long long t1, double* pool, int accumulate)
{
  gather_targets(G, t0, t1, pool, accumulate, (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5),
                 (long long)gridDim.x * (blockDim.x >> 5), threadIdx.x & 31);
}
void dlb_launch_extend_gather(const DlbGather& G, long long t0, long long t1, double* pool, int accumulate, cudaStream_t st)
{
  if(t1 <= t0) return;
  long long g = (t1 - t0 + 7) / 8;
  if(g > 148 * 32) g = 148 * 32;
  k_extend_gather<<<(int)g, 256, 0, st>>>(G, t0, t1, pool, accumulate);
}

__global__ void __launch_bounds__(256)
k_zero_bigfronts(const DlbBigFront* __restrict__ descs, double* __restrict__ fronts)
{
  const DlbBigFront f = descs[blockIdx.y];
  const size_t n = (size_t)f.r * f.r;
  double* A = fronts + f.off;
  for(size_t idx = (size_t)blockIdx.x * 256 + threadIdx.x; idx < n; idx += (size_t)gridDim.x * 256) A[idx] = 0.0;
}
void dlb_launch_zero_bigfronts(const DlbBigFront* d_descs, int nfronts, int max_r, double* fronts, cudaStream_t st)
{
  if(nfronts <= 0) return;
  long long chunks = ((long long)max_r * max_r + 256 * 8 - 1) / (256 * 8);
  if(chunks > 1024) chunks = 1024;
  for(int f0 = 0; f0 < nfronts; f0 += 65535)                  // blockIdx.y carries the front: slices of the grid limit
    k_zero_bigfronts<<<dim3((unsigned)chunks, nfronts - f0 < 65535 ? nfronts - f0 : 65535), 256, 0, st>>>(d_descs + f0, fronts);
}

template<int NT>
static void launch_front_level_nt(const DlbFrontDev& F, const DlbSparseDev& S, int l0, int nf, double* fronts,
                                  const double* Gpart, double lambda, long long* minor, int mode, size_t smem,
                                  cudaStream_t st)
{
  if(smem <= 200 * 1024)
  {
    static DlbPerDeviceOnce attr_once;
    if(attr_once.first())
      cudaFuncSetAttribute(k_front_level<true, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    k_front_level<true, NT><<<nf, NT, smem, st>>>(F, S, l0, fronts, Gpart, lambda, minor, mode);
  }
  else k_front_level<false, NT><<<nf, NT, 0, st>>>(F, S, l0, fronts, Gpart, lambda, minor, mode);
}

void dlb_launch_front_level(const DlbFrontDev& F, const DlbSparseDev& S, int l0, int l1,
                            double* fronts, const double* Gpart, double lambda,
                            long long* minor, int max_rows, int skip_elimination, cudaStream_t st)
{
  const int nf = l1 - l0;
  if(nf <= 0) return;
  const int mode = lambda < 0.0 ? 1 : (skip_elimination ? 2 : 0);   // lambda < 0: elements only
  const size_t smem = (size_t)max_rows * max_rows * sizeof(double);
  // more threads for bigger fronts (128 registers per thread are needed: the diagonal block lives in registers)
  if(max_rows > 64)      launch_front_level_nt<512>(F, S, l0, nf, fronts, Gpart, lambda, minor, mode, smem, st);
  else if(max_rows > 40) launch_front_level_nt<256>(F, S, l0, nf, fronts, Gpart, lambda, minor, mode, smem, st);
  else                   launch_front_level_nt<128>(F, S, l0, nf, fronts, Gpart, lambda, minor, mode, smem, st);
}

// ------------------------------------------------------------------ solves
// Fronts here are small (tens to hundreds of rows), so the solves are latency bound: the
// work per front is arranged to avoid block-wide barriers.
//   forward  y = L^-1 P b, leaves to root: every warp gathers a fixed subset of the children's
//            tails into its own shared-memory vector (no conflicts), the vectors are added in
//            warp order, then ONE warp runs the substitution with __syncwarp only.
//   backward x = L^-T y, root to leaves, in place in zperm: one warp, shuffle reductions.
// Fronts too big for that (r > SOLVE_WARP_MAX or shared memory) use the block-wide variant.
#define SOLVE_WARP_MAX 12000

template<int SOLVE_NT>
__global__ void __launch_bounds__(SOLVE_NT)
k_solve_fwd_level(DlbFrontDev F, int l0, const double* __restrict__ fronts,
                  const double* __restrict__ rhs, double* __restrict__ ywork,
                  double* __restrict__ zperm, int nrhs, int gather_warps, int max_rows, size_t panel_elems)
{
  extern __shared__ double sh_y[];          // [0,max_rows): y ; gather_warps vectors of r ; the staged L panel
  __shared__ double sh_D[32][33];
  const int s  = F.level_sn[l0 + blockIdx.x];
  const int c0 = F.sn_first[s], nc = F.sn_first[s+1] - c0;
  const int rp = F.rows_ptr[s], r = F.rows_ptr[s+1] - rp;
  const double* A = fronts + F.front_off[s];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int nch = F.child_ptr[s+1] - F.child_ptr[s];
  const bool in_smem = gather_warps > 0;
  // the r x nc panel of L is staged behind the vectors when panel_elems > 0 (latency: the
  // substitution below is a serial chain of dependent loads otherwise)
  double* sh_L = sh_y + (size_t)(1 + gather_warps) * max_rows;
  const bool panel_staged = in_smem && (size_t)r * nc <= panel_elems;
  if(panel_staged) for(size_t idx = tid; idx < (size_t)r * nc; idx += SOLVE_NT) sh_L[idx] = A[idx];
  for(int rh = 0; rh < nrhs; rh++)
  {
    double* yg = ywork + (size_t)rh * F.ytot + rp;
    double* y  = in_smem ? sh_y : yg;
    const bool gathered = F.sg_flag && F.sg_flag[s];   // children already summed into yg by the solve gather
    for(int i = tid; i < r; i += SOLVE_NT)
      y[i] = (i < nc ? rhs[(size_t)rh * F.n + F.perm[c0 + i]] : 0.0) + (gathered ? yg[i] : 0.0);
    if(gathered) __syncthreads();
    else if(in_smem && nch > 0)
    {
      for(int i = tid; i < gather_warps * r; i += SOLVE_NT) sh_y[r + i] = 0.0;
      __syncthreads();
      if(w < gather_warps)
      {
        double* mine = sh_y + (size_t)(1 + w) * r;
        for(int ch = F.child_ptr[s] + w; ch < F.child_ptr[s+1]; ch += gather_warps)
        {
          const int c   = F.child_list[ch];
          const int ncc = F.sn_first[c+1] - F.sn_first[c];
          const int rc  = F.rows_ptr[c+1] - F.rows_ptr[c];
          const double* yc = ywork + (size_t)rh * F.ytot + F.rows_ptr[c];
          const int* rel = F.rel + F.rows_ptr[c];
          for(int i = ncc + lane; i < rc; i += 32) mine[rel[i]] += yc[i];
          __syncwarp();
        }
      }
      __syncthreads();
      for(int i = tid; i < r; i += SOLVE_NT)
      {
        double acc = 0.0;
        for(int g = 0; g < gather_warps; g++) acc += sh_y[(size_t)(1 + g) * r + i];
        y[i] += acc;
      }
    }
    else
    {
      __syncthreads();
      for(int ch = F.child_ptr[s]; ch < F.child_ptr[s+1]; ch++)
      {
        const int c   = F.child_list[ch];
        const int ncc = F.sn_first[c+1] - F.sn_first[c];
        const int rc  = F.rows_ptr[c+1] - F.rows_ptr[c];
        const double* yc = ywork + (size_t)rh * F.ytot + F.rows_ptr[c];
        const int* rel = F.rel + F.rows_ptr[c];
        for(int i = ncc + tid; i < rc; i += SOLVE_NT) y[rel[i]] += yc[i];
        __syncthreads();
      }
    }
    __syncthreads();
    if(in_smem)
    { // blocked substitution, 32 columns at a time: the 32x32 diagonal block is staged in shared
      // memory and solved by one warp with shuffles (lane i owns y[b0+i]), then all threads
      // update the rows below with those 32 columns. Same summation order as column-by-column.
      const double* Ap = panel_staged ? sh_L : A;
      for(int b0 = 0; b0 < nc; b0 += 32)
      {
        const int bw = nc - b0 < 32 ? nc - b0 : 32;
        for(int idx = tid; idx < bw * bw; idx += SOLVE_NT)
        {
          const int j = idx / bw, i = idx - j * bw;
          const double v = Ap[(b0 + i) + (size_t)(b0 + j) * r];
          sh_D[i][j] = i == j ? 1.0 / v : v;        // reciprocal pivots: no division in the serial chain
        }
        __syncthreads();
        if(w == 0)
        {
          double yi = lane < bw ? y[b0 + lane] : 0.0;
          for(int j = 0; j < bw; j++)
          {
            const double yj = __shfl_sync(0xffffffffu, yi, j) * sh_D[j][j];
            if(lane == j) yi = yj;
            else if(lane > j && lane < bw) yi = fma(-sh_D[lane][j], yj, yi);
          }
          if(lane < bw) y[b0 + lane] = yi;
        }
        __syncthreads();
        for(int i = b0 + bw + tid; i < r; i += SOLVE_NT)
        { // 8 panel entries in flight per thread (the panel of a large front comes from global
          // memory: one dependent load per column made this loop pure latency); same FMA order
          double acc = y[i];
          const double* Ai = Ap + i + (size_t)b0 * r;
          int c = 0;
          if(bw == 32)
          { // the common full block: all 32 panel entries of the row in flight at once
            double l[32];
#pragma unroll
            for(int u = 0; u < 32; u++) l[u] = Ai[(size_t)u * r];
#pragma unroll
            for(int u = 0; u < 32; u++) acc = fma(-l[u], y[b0 + u], acc);
            c = 32;
          }
          for(; c + 8 <= bw; c += 8)
          {
            double l[8];
#pragma unroll
            for(int u = 0; u < 8; u++) l[u] = Ai[(size_t)(c + u) * r];
#pragma unroll
            for(int u = 0; u < 8; u++) acc = fma(-l[u], y[b0 + c + u], acc);
          }
          for(; c < bw; c++) acc = fma(-Ai[(size_t)c * r], y[b0 + c], acc);
          y[i] = acc;
        }
        __syncthreads();
      }
      for(int i = tid; i < r; i += SOLVE_NT) yg[i] = y[i];
    }
    else
      for(int j = 0; j < nc; j++)
      {
        if(tid == 0) y[j] /= A[j + (size_t)j * r];
        __syncthreads();
        const double yj = y[j];
        for(int i = j + 1 + tid; i < r; i += SOLVE_NT) y[i] = fma(-A[i + (size_t)j * r], yj, y[i]);
        __syncthreads();
      }
    for(int i = tid; i < nc; i += SOLVE_NT) zperm[(size_t)rh * F.n + c0 + i] = y[i];
    __syncthreads();
  }
}

template<int SOLVE_NT>
__global__ void __launch_bounds__(SOLVE_NT)
k_solve_bwd_level(DlbFrontDev F, int l0, const double* __restrict__ fronts,
                  double* __restrict__ zperm, int nrhs, int in_smem, int max_rows, size_t panel_elems)
{
  extern __shared__ double sh_x[];          // max_rows entries: x of this front's rows ; the staged L panel
  __shared__ double sh[32];
  __shared__ double sh_D[32][33];
  const int s  = F.level_sn[l0 + blockIdx.x];
  const int c0 = F.sn_first[s], nc = F.sn_first[s+1] - c0;
  const int rp = F.rows_ptr[s], r = F.rows_ptr[s+1] - rp;
  const double* A = fronts + F.front_off[s];
  const int* rows = F.rows + rp;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  double* sh_L = sh_x + max_rows;
  const bool panel_staged = in_smem && (size_t)r * nc <= panel_elems;
  if(panel_staged) for(size_t idx = tid; idx < (size_t)r * nc; idx += SOLVE_NT) sh_L[idx] = A[idx];
  const double* Ap = panel_staged ? sh_L : A;
  for(int rh = 0; rh < nrhs; rh++)
  {
    double* z = zperm + (size_t)rh * F.n;
    if(in_smem)
    {
      for(int i = tid; i < r; i += SOLVE_NT) sh_x[i] = z[rows[i]];
      __syncthreads();
      // blocked, 32 columns at a time from the last block: the warps take the columns of the
      // block and dot them with the already known x below the block, then one warp solves the
      // 32x32 transposed triangle with shuffles (lane c owns x[b0+c])
      for(int b0 = ((nc - 1) / 32) * 32; b0 >= 0; b0 -= 32)
      {
        const int bw = nc - b0 < 32 ? nc - b0 : 32;
        for(int idx = tid; idx < bw * bw; idx += SOLVE_NT)
        {
          const int j = idx / bw, i = idx - j * bw;
          const double v = Ap[(b0 + i) + (size_t)(b0 + j) * r];
          sh_D[i][j] = i == j ? 1.0 / v : v;
        }
        for(int cc = w; cc < bw; cc += SOLVE_NT / 32)
        {
          double acc = 0.0;
          const double* Ac = Ap + (size_t)(b0 + cc) * r;
          int i = b0 + bw + lane;
          for(; i + 96 < r; i += 128)
          { // four loads in flight per lane; per-lane accumulation order unchanged
            const double l0 = Ac[i], l1 = Ac[i + 32], l2 = Ac[i + 64], l3 = Ac[i + 96];
            acc = fma(l0, sh_x[i], acc); acc = fma(l1, sh_x[i + 32], acc);
            acc = fma(l2, sh_x[i + 64], acc); acc = fma(l3, sh_x[i + 96], acc);
          }
          for(; i < r; i += 32) acc = fma(Ac[i], sh_x[i], acc);
          acc = warp_sum_all(acc);
          if(lane == 0) sh[cc] = acc;
        }
        __syncthreads();
        if(w == 0)
        {
          double v = lane < bw ? sh_x[b0 + lane] - sh[lane] : 0.0;
          for(int j = bw - 1; j >= 0; j--)
          {
            const double xj = __shfl_sync(0xffffffffu, v, j) * sh_D[j][j];
            if(lane == j) v = xj;
            else if(lane < j) v = fma(-sh_D[j][lane], xj, v);
          }
          if(lane < bw) sh_x[b0 + lane] = v;
        }
        __syncthreads();
      }
      for(int i = tid; i < nc; i += SOLVE_NT) z[c0 + i] = sh_x[i];
      __syncthreads();
    }
    else
      for(int j = nc - 1; j >= 0; j--)
      {
        double acc = 0.0;
        for(int i = j + 1 + tid; i < r; i += SOLVE_NT) acc = fma(A[i + (size_t)j * r], z[rows[i]], acc);
        acc = block_sum(acc, sh);
        if(tid == 0) z[c0 + j] = (z[c0 + j] - acc) / A[j + (size_t)j * r];
        __syncthreads();
      }
  }
}

template<int NT>
static void launch_solve_fwd_nt(const DlbFrontDev& F, int l0, int l1, const double* fronts,
                                const double* rhs, double* ywork, double* zperm, int nrhs,
                                int max_rows, int max_cols, cudaStream_t st)
{
  static DlbPerDeviceOnce attr_once;
  if(attr_once.first())
  {
    cudaFuncSetAttribute(k_solve_fwd_level<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  }
  // as many gather vectors as fit (at most one per warp); 0 selects the block-wide variant;
  // what is left of the budget holds the staged L panel. Small fronts get a small budget so that
  // many CTAs share an SM.
  const size_t budget = (max_rows <= 64 ? 12 * 1024 : 200 * 1024) / sizeof(double);
  int gw = 0;
  if(max_rows <= SOLVE_WARP_MAX)
  {
    gw = (int)(budget / (size_t)max_rows) - 1;
    if(gw > NT / 32) gw = NT / 32;
    if(gw < 1) gw = 0;
  }
  size_t vec = gw ? (size_t)(1 + gw) * max_rows : 0;
  size_t panel = 0;
  if(gw && (size_t)max_rows * max_cols <= budget - vec) panel = (size_t)max_rows * max_cols;
  const size_t smem = (vec + panel) * sizeof(double);
  k_solve_fwd_level<NT><<<l1 - l0, NT, smem, st>>>(F, l0, fronts, rhs, ywork, zperm, nrhs, gw, max_rows, panel);
}
void dlb_launch_solve_fwd_level(const DlbFrontDev& F, int l0, int l1, const double* fronts,
                                const double* rhs, double* ywork, double* zperm, int nrhs,
                                int max_rows, int max_cols, cudaStream_t st)
{
  if(l1 <= l0) return;
  if(max_rows <= 64) launch_solve_fwd_nt<128>(F, l0, l1, fronts, rhs, ywork, zperm, nrhs, max_rows, max_cols, st);
  else               launch_solve_fwd_nt<512>(F, l0, l1, fronts, rhs, ywork, zperm, nrhs, max_rows, max_cols, st);
}
template<int NT>
static void launch_solve_bwd_nt(const DlbFrontDev& F, int l0, int l1, const double* fronts,
                                double* zperm, int nrhs, int max_rows, int max_cols, cudaStream_t st)
{
  static DlbPerDeviceOnce attr_once;
  if(attr_once.first())
  {
    cudaFuncSetAttribute(k_solve_bwd_level<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  }
  const size_t budget = (max_rows <= 64 ? 12 * 1024 : 200 * 1024) / sizeof(double);
  const int in_smem = max_rows <= SOLVE_WARP_MAX ? 1 : 0;
  size_t panel = 0;
  if(in_smem && (size_t)max_rows * max_cols <= budget - max_rows) panel = (size_t)max_rows * max_cols;
  const size_t smem = in_smem ? ((size_t)max_rows + panel) * sizeof(double) : 0;
  k_solve_bwd_level<NT><<<l1 - l0, NT, smem, st>>>(F, l0, fronts, zperm, nrhs, in_smem, max_rows, panel);
}
void dlb_launch_solve_bwd_level(const DlbFrontDev& F, int l0, int l1, const double* fronts,
                                double* zperm, int nrhs, int max_rows, int max_cols, cudaStream_t st)
{
  if(l1 <= l0) return;
  if(max_rows <= 64) launch_solve_bwd_nt<128>(F, l0, l1, fronts, zperm, nrhs, max_rows, max_cols, st);
  else               launch_solve_bwd_nt<512>(F, l0, l1, fronts, zperm, nrhs, max_rows, max_cols, st);
}

// tests: scatter the assembled (elements-only) fronts into a dense n x n matrix
__global__ void k_fronts_to_dense(DlbFrontDev F, const double* __restrict__ fronts, double* out)
{
  const int s  = blockIdx.x;
  const int rp = F.rows_ptr[s], r = F.rows_ptr[s+1] - rp;
  const double* A = fronts + F.front_off[s];
  for(int idx = threadIdx.x; idx < r * r; idx += blockDim.x)
  {
    const int j = idx / r, i = idx - j * r;
    if(i < j) continue;
    const double v = A[i + (size_t)j * r];
    if(v == 0.0) continue;
    const int gi = F.perm[F.rows[rp + i]], gj = F.perm[F.rows[rp + j]];
    atomicAdd(&out[(size_t)gi * F.n + gj], v);
    if(gi != gj) atomicAdd(&out[(size_t)gj * F.n + gi], v);
  }
}
void dlb_launch_fronts_to_dense(const DlbFrontDev& F, const double* fronts, double* out, cudaStream_t st)
{
  k_fronts_to_dense<<<F.nsuper, 256, 0, st>>>(F, fronts, out);
}
