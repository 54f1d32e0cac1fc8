/* dogleg_gpu.h -- additive C-ABI of the B200-native dog-leg solver.
 *
 * dogleg.h is the unchanged libdogleg API. This header adds what the reference
 * has no surface for (SURVEY.md 8b "additive surface") and exposes the device
 * hot path one operation at a time ("engine" calls) so that tests and the
 * benchmark can drive and time exactly what dogleg_optimize*() runs per
 * iteration. Plain C: pointers and sizes only, no CUDA or torch types.
 *
 * Each engine call names the reference code it replaces. "slot" is 0 or 1: the
 * two operating points (beforeStep / afterStep, reference dogleg.h:181-182).
 * All vectors live in HBM; the engine owns pinned host mirrors for everything
 * the reference API exposes through dogleg_operatingPoint_t.
 */
#pragma once
#include <stddef.h>
#include "dogleg.h"
#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------- device control */
int         dogleg_gpu_device_count(void);          /* 0 if there is no usable GPU */
int         dogleg_gpu_set_device(int device);      /* device for contexts created afterwards (default 0) */
int         dogleg_gpu_get_device(void);
const char* dogleg_gpu_last_error(void);            /* message of the last failed call in this thread */
const char* dogleg_gpu_version(void);

/* Injected fill-reducing ordering for the NEXT sparse context created on this
 * thread (perm[k] = state eliminated k-th, the cholmod convention); NULL/0
 * returns to the built-in AMD-style ordering. postorder!=0 lets the library
 * apply an elimination-tree postorder on top (equivalent fill). */
void        dogleg_gpu_set_permutation(const int* perm, int n, int postorder);

/* --------------------------------------------------- device-resident callbacks */
/* Like dogleg_callback_t but everything is in HBM: d_p (Nstate), d_x (Nmeas),
 * d_Jt_values (NJnnz, in the order of the fixed CCS pattern given at the call).
 * 'stream' is the cudaStream_t to enqueue work on (do not synchronise). */
typedef void (dogleg_gpu_callback_sparse_t)(const double* d_p, double* d_x, double* d_Jt_values,
                                            void* stream, void* cookie);
typedef void (dogleg_gpu_callback_dense_t)(const double* d_p, double* d_x, double* d_J,
                                           void* stream, void* cookie);

/* dogleg_optimize2 with the Jacobian produced on the device (no PCIe traffic
 * per evaluation). Jp/Ji: host CCS pattern of Jt, fixed for the solve. */
double dogleg_gpu_optimize_sparse(double* p, unsigned int Nstate, unsigned int Nmeas, unsigned int NJnnz,
                                  const int* Jp, const int* Ji,
                                  dogleg_gpu_callback_sparse_t* f, void* cookie,
                                  const dogleg_parameters2_t* parameters,
                                  dogleg_solverContext_t** returnContext);
double dogleg_gpu_optimize_dense(double* p, unsigned int Nstate, unsigned int Nmeas,
                                 dogleg_gpu_callback_dense_t* f, void* cookie,
                                 const dogleg_parameters2_t* parameters,
                                 dogleg_solverContext_t** returnContext);

/* dogleg_optimize_dense_products with the products produced on the device: d_norm2x is one double,
 * d_Jtx Nstate doubles, d_JtJ the layout parameters->JtJ_packed / JtJ_upper select (Nstate*Nstate
 * row-first, or Nstate*(Nstate+1)/2 packed upper, row-first). Packed lower is rejected before the first
 * callback (the reference cannot take a Cauchy step with it, dogleg.c:597-601). */
typedef void (dogleg_gpu_callback_dense_products_t)(const double* d_p, double* d_norm2x, double* d_Jtx,
                                                     double* d_JtJ, void* stream, void* cookie);
double dogleg_gpu_optimize_dense_products(double* p, unsigned int Nstate,
                                          dogleg_gpu_callback_dense_products_t* f, void* cookie,
                                          const dogleg_parameters2_t* parameters,
                                          dogleg_solverContext_t** returnContext);

/* ----------------------------------------- using the factorization of a returned context */
/* The reference lets a returnContext caller solve with ctx->factorization through CHOLMOD
 * (dogleg.h:188-195, README.pod:105-111; dogleg.c:853-856 is how the library does it itself). Here the
 * numeric factor lives in HBM:
 *   dogleg_gpu_solve():         X = (JtJ + lambda I)^-1 B at ctx->beforeStep (factorizing first if needed);
 *                               B and X are host arrays, Nstate x nrhs column-major. Any solve type.
 *   dogleg_gpu_export_factor(): sparse solves: fills ctx->factorization->x (supernodal L L', CHOLMOD's
 *                               layout: supernode s = nsrow x nscol column-major panel at x[px[s]]; rows
 *                               s[pi[s]..], columns super[s]..super[s+1]-1, ordering Perm) for host code.
 * Both return 0 on success. */
int dogleg_gpu_solve(dogleg_solverContext_t* ctx, const double* B, double* X, int nrhs);
int dogleg_gpu_export_factor(dogleg_solverContext_t* ctx);

/* ------------------------------------------------- streaming host callbacks (optional) */
/* With host callbacks (dogleg_optimize2 / dogleg_optimize_dense2) x and the Jacobian values cross PCIe on
 * a side stream from the pinned buffers the callback writes into. A callback that fills Jt->x (or J) and
 * x FRONT TO BACK may call this from inside the callback, as often as it likes, to announce that the first
 * n_values_final Jacobian values and the first n_x_final entries of x will not change any more: those
 * pieces start their transfer at once, so the copy overlaps the rest of the callback instead of
 * following it. Calling it is optional; calling it outside a callback does nothing. */
void dogleg_gpu_host_progress(size_t n_values_final, size_t n_x_final);

/* ------------------------------------------------------ row-sharded multi-GPU */
/* One process per GPU. Rank 0 calls dogleg_gpu_nccl_get_unique_id(), the launcher hands the 128
 * bytes to every rank (torch.distributed, MPI, a file ...), every rank calls
 * dogleg_gpu_nccl_init() after dogleg_gpu_set_device(). libnccl.so.2 is loaded at run time. */
int  dogleg_gpu_nccl_get_unique_id(unsigned char id[128]);
int  dogleg_gpu_nccl_init(int rank, int world, const unsigned char id[128]);
void dogleg_gpu_nccl_finalize(void);
int  dogleg_gpu_nccl_world(void);

/* dogleg_optimize2 with the measurements split by rows of J (columns of Jt): this rank evaluates
 * the measurement columns [col_begin, col_begin + Nmeas_local) only. Jp_global/Ji_global: the CCS
 * pattern of ALL Nmeas_total columns (needed for a symbolic analysis that is identical on every
 * rank). Exactly one of f_host / f_device is non-NULL; the callback fills x[Nmeas_local] and the
 * values of this rank's columns (a host callback sees a cholmod_sparse with Nmeas_local columns).
 * Partial Jt*x, |x|^2, |J v|^2 and partial fronts are summed with ncclAllReduce; every rank
 * returns the same p and cost. All ranks must pass the same p, parameters and global pattern. */
double dogleg_gpu_optimize_sparse_sharded(double* p, unsigned int Nstate,
                                          unsigned int Nmeas_total, const int* Jp_global, const int* Ji_global,
                                          unsigned int col_begin, unsigned int Nmeas_local,
                                          dogleg_callback_t* f_host, dogleg_gpu_callback_sparse_t* f_device,
                                          void* cookie, const dogleg_parameters2_t* parameters,
                                          dogleg_solverContext_t** returnContext);

/* dogleg_optimize_dense2 with the rows of J split over the ranks: this rank's callback fills
 * x[Nmeas_local] and J[Nmeas_local][Nstate] for the rows [row_begin, row_begin + Nmeas_local).
 * Partial J'x, |x|^2, |J v|^2 and the partial N x N J'J are summed with ncclAllReduce; the Cholesky
 * runs redundantly on every rank. Exactly one of f_host / f_device is non-NULL. */
double dogleg_gpu_optimize_dense_sharded(double* p, unsigned int Nstate, unsigned int Nmeas_total,
                                         unsigned int row_begin, unsigned int Nmeas_local,
                                         dogleg_callback_dense_t* f_host, dogleg_gpu_callback_dense_t* f_device,
                                         void* cookie, const dogleg_parameters2_t* parameters,
                                         dogleg_solverContext_t** returnContext);

/* Layout this library was built with: [0]=sizeof(dogleg_solverContext_t) [1]=sizeof(cholmod_common)
 * [2]=offsetof(beforeStep) [3]=offsetof(factorization) [4]=offsetof(lambda) [5]=1 if built against the
 * bundled compat/cholmod.h, 0 if against a real SuiteSparse header. An application that keeps a returned
 * context must be compiled against the same cholmod.h: check these against its own sizeof/offsetof. */
void dogleg_gpu_context_layout(size_t out[6]);

/* Statistics of the last solve run through a context (or the thread's last
 * solve if ctx is NULL): out[0]=accepted steps, [1]=callback evaluations,
 * [2]=rejected trials, [3]=factorizations, [4]=kernel launches,
 * [5]=H2D bytes, [6]=D2H bytes, [7]=seconds inside user callbacks. */
void dogleg_gpu_get_stats(const dogleg_solverContext_t* ctx, double out[8]);
/* Row-sharded solves: out[0] = collective calls (grouped NCCL operations), out[1] = bytes this rank
 * contributed to them, both for the thread's last solve. */
void dogleg_gpu_get_comm_stats(double out[2]);
/* With DOGLEG_GPU_PHASE_TIMING=1 in the environment every engine phase of a solve is bracketed by
 * CUDA events on the solver's stream; this returns the sums (ms) for this thread's last solve:
 * [0]=h2d [1]=gradient [2]=cauchy(Jv) [3]=assemble [4]=factor [5]=solve [6]=step(Jv) [7]=d2h.
 * Engines on the fused schedule (the default for unsharded sparse solves): [1]=the fused evaluation pass
 * (gradient + |x|^2 + class blocks), [3]=its per-state reduction, [4]=the trial kernel (Cauchy,
 * factorization, solves, step, expected improvement in one launch); [2],[5],[6] stay 0. */
void dogleg_gpu_get_phase_ms(double out[8]);

/* -------------------------------------------------------- batched dense solves */
/* B independent dense problems of identical shape, the whole trust-region
 * automaton device-resident. The callback evaluates ALL problems at once:
 * d_p is B x Nstate, d_x is B x Nmeas, d_J is B x Nmeas x Nstate (row-first per
 * problem); d_active[b]==0 marks problems that are already finished (their
 * outputs are ignored). */
typedef void (dogleg_gpu_callback_dense_batched_t)(const double* d_p, double* d_x, double* d_J,
                                                   const int* d_active, int B,
                                                   void* stream, void* cookie);
/* p: host B x Nstate in/out; norm2x_out: host B (may be NULL); iterations_out:
 * host B accepted-step counts (may be NULL). Returns the number of problems
 * solved without error, or <0 on a CUDA failure. */
int dogleg_gpu_optimize_dense_batched(double* p, unsigned int Nstate, unsigned int Nmeas,
                                      unsigned int B,
                                      dogleg_gpu_callback_dense_batched_t* f, void* cookie,
                                      const dogleg_parameters2_t* parameters,
                                      double* norm2x_out, int* iterations_out);

/* B independent dense-products problems: the callback fills, for every active problem b,
 * d_norm2x[b], d_Jtx[b*Nstate ..] and its JtJ at d_JtJ + b*S, S = Nstate*Nstate (row-first, both
 * triangles) or Nstate*(Nstate+1)/2 (packed upper, row-first: parameters->JtJ_packed && JtJ_upper).
 * Packed lower is rejected (the reference cannot take a Cauchy step with it, dogleg.c:597-601).
 * No Jacobian is stored, so the batch size does not depend on the number of measurements.
 * d_active[b]==0: finished, outputs ignored. Nstate <= 32. Return value, p, norm2x_out and
 * iterations_out as dogleg_gpu_optimize_dense_batched. */
typedef void (dogleg_gpu_callback_dense_products_batched_t)(const double* d_p, double* d_norm2x, double* d_Jtx,
                                                             double* d_JtJ, const int* d_active, int B,
                                                             void* stream, void* cookie);
int dogleg_gpu_optimize_dense_products_batched(double* p, unsigned int Nstate, unsigned int B,
                                               dogleg_gpu_callback_dense_products_batched_t* f, void* cookie,
                                               const dogleg_parameters2_t* parameters,
                                               double* norm2x_out, int* iterations_out);

/* ------------------------------------------- the final state of a batched solve */
/* What a batched caller needs for per-problem uncertainties, the batched counterpart of returnContext +
 * dogleg_gpu_solve: each problem's JtJ at the p it returned, its lambda and why it stopped. */
typedef struct dogleg_gpu_batch dogleg_gpu_batch_t;

/* dogleg_gpu_optimize_dense_batched / dogleg_gpu_optimize_dense_products_batched (those two are these with
 * returnBatch == NULL). If returnBatch != NULL, *returnBatch receives a handle that holds each problem's final
 * JtJ (at the returned p), its lambda and its termination status, on the device the solve ran on;
 * *returnBatch = NULL on failure. Free it with dogleg_gpu_batch_free(). The handle owns its memory: later
 * batched solves, dogleg_gpu_release_batched_cache() and dogleg_gpu_release_cache() do not touch it. */
int dogleg_gpu_optimize_dense_batched2(double* p, unsigned int Nstate, unsigned int Nmeas, unsigned int B,
                                       dogleg_gpu_callback_dense_batched_t* f, void* cookie,
                                       const dogleg_parameters2_t* parameters,
                                       double* norm2x_out, int* iterations_out, dogleg_gpu_batch_t** returnBatch);
int dogleg_gpu_optimize_dense_products_batched2(double* p, unsigned int Nstate, unsigned int B,
                                                dogleg_gpu_callback_dense_products_batched_t* f, void* cookie,
                                                const dogleg_parameters2_t* parameters,
                                                double* norm2x_out, int* iterations_out,
                                                dogleg_gpu_batch_t** returnBatch);

/* Why a problem stopped, in the order the single-problem solver tests (dogleg_core.c run_solver): after an
 * accepted step the gradient test comes before the iteration cap; at the initial point a problem is
 * GRADIENT if it has converged, else MAX_ITERATIONS if max_iterations <= 0. */
enum { DOGLEG_GPU_BATCH_UNFINISHED = 0,      /* still running when the solve stopped (trial cap) */
       DOGLEG_GPU_BATCH_GRADIENT = 1,        /* max|J'x| <= Jt_x_threshold */
       DOGLEG_GPU_BATCH_STEP = 2,            /* max|step| <= update_threshold: the step was not taken */
       DOGLEG_GPU_BATCH_TRUSTREGION = 3,     /* rejected and trust region < trustregion_threshold */
       DOGLEG_GPU_BATCH_MAX_ITERATIONS = 4 };

/* Every call below works on JtJ_b + lambda_b I with the problem's sticky lambda at the end of its solve: the
 * matrix dogleg_gpu_solve() uses on a returned context. A problem may have stopped without a Gauss-Newton
 * step at its final point, so its JtJ can be singular; the factorization then climbs the solver's ladder
 * (0 -> 1e-10 -> x10) and stores the raised lambda in the handle, as dogleg_computeJtJfactorization() does
 * for ctx->lambda. Return 0 on success, < 0 with dogleg_gpu_last_error() set on bad arguments or a CUDA
 * failure. A problem whose matrix is not positive definite at any lambda (non-finite entries) gets NaN
 * outputs; the host-pointer forms return the number of such problems, the _device forms return 0 once the
 * work is enqueued (they do not synchronise). */

/* host arrays of B entries, either may be NULL; waits for the handle's pending work */
int  dogleg_gpu_batch_status(const dogleg_gpu_batch_t* batch, int* status_out, double* lambda_out);
/* X_b = (JtJ_b + lambda_b I)^-1 R_b for every problem. R, X: B x Nstate x nrhs, each problem's block
 * column-major as in dogleg_gpu_solve. Host pointers; the _device form takes device pointers and enqueues on
 * `stream` (a cudaStream_t, NULL = the legacy default stream) without synchronising. */
int  dogleg_gpu_batch_solve(dogleg_gpu_batch_t* batch, const double* R, double* X, int nrhs);
int  dogleg_gpu_batch_solve_device(dogleg_gpu_batch_t* batch, const double* d_R, double* d_X, int nrhs, void* stream);
/* (JtJ_b + lambda_b I)^-1 for every problem: B x Nstate^2 (column k of problem b's block is the solve with
 * e_k, so the layout reads as row-first and as column-first), or, if packed != 0, B x Nstate(Nstate+1)/2:
 * the upper triangle of that row-first matrix, packed row-first (the products layout) */
int  dogleg_gpu_batch_covariance(dogleg_gpu_batch_t* batch, double* out, int packed);
int  dogleg_gpu_batch_covariance_device(dogleg_gpu_batch_t* batch, double* d_out, int packed, void* stream);
void dogleg_gpu_batch_free(dogleg_gpu_batch_t** batch);   /* sets *batch = NULL; NULL is fine */

/* statistics of this thread's last batched solve (either form): [0] trial launches, [1] sum over launches of
 * active problems, [2] ms inside the trial kernel, [3] ms inside the callback (CUDA events) */
void dogleg_gpu_batched_stats(double out[8]);
/* the device workspace of the last batched solve is kept for the next one of the same shape and form;
 * this frees it (dogleg_gpu_release_cache() does too) */
void dogleg_gpu_release_batched_cache(void);

/* --------------------------------------------------- symbolic analysis (host) */
typedef struct dlb_symbolic dlb_symbolic_t;
dlb_symbolic_t* dlb_symbolic_create(int Nstate, int Nmeas, const int* Jp, const int* Ji,
                                    const int* perm_or_null, int postorder);
void            dlb_symbolic_free(dlb_symbolic_t* S);
/* out: [0]=ncls [1]=nsuper [2]=nlevels [3]=nnz(L) [4]=max front rows
 *      [5]=front storage (doubles) [6]=sum colcount^2 (flops) [7]=rows array length */
void            dlb_symbolic_info(const dlb_symbolic_t* S, long long out[8]);
enum { DLB_SYM_PERM = 0, DLB_SYM_PARENT = 1, DLB_SYM_COLCOUNT = 2, DLB_SYM_SN_FIRST = 3,
       DLB_SYM_ROWS_PTR = 4, DLB_SYM_ROWS = 5, DLB_SYM_SN_PARENT = 6, DLB_SYM_CLS_OF_COL = 7,
       DLB_SYM_CLS_FRONT = 8, DLB_SYM_SN_LEVEL = 9, DLB_SYM_REL = 10, DLB_SYM_CHILD_PTR = 11,
       DLB_SYM_CHILD_LIST = 12, DLB_SYM_LEVEL_PTR = 13, DLB_SYM_LEVEL_SN = 14, DLB_SYM_CLS_PTR = 15,
       DLB_SYM_CLS_ROWS = 16, DLB_SYM_CLS_LOC = 17, DLB_SYM_MEM_PTR = 18, DLB_SYM_MEM_COL = 19 };
/* copies min(cap, length) ints of the named array, returns its length */
long long       dlb_symbolic_get(const dlb_symbolic_t* S, int what, int* out, long long cap);
/* nsuper+1 offsets (doubles) of the r x r column-major fronts in the front pool */
long long       dlb_symbolic_front_off(const dlb_symbolic_t* S, long long* out, long long cap);

/* The extend-add of the multifrontal factorization (the supernodal assembly CHOLMOD performs behind
 * reference dogleg.c:666) and the forward solve's y(parent) += y(child) as precomputed block
 * gathers; host-side integer plan, exposed for the CPU tests (tests/test_gatherplan.py).
 * Parameters <= 0 (heavy < 0) select the engine's defaults. Target t of a list is an h x |w| block
 * at offset dst[t] (leading dimension ld[t]; w < 0 = lower-triangular strip) that receives the sum
 * of its sources src_base[src_ptr[t] .. src_ptr[t+1]) with leading dimensions src_ld, in list order.
 * Front offsets address the pool [fronts | temporaries | scratch], solve offsets [rows | scratch].
 * level_ptr[2l .. 2l+2]: pass 1 (overwrite scratch chunks) and pass 2 (accumulate) of level l. */
typedef struct dlb_gather_plan dlb_gather_plan_t;
dlb_gather_plan_t* dlb_gather_plan_create(const dlb_symbolic_t* S, int small_front_max, int heavy,
                                          int gsplit, int gchunk, int gtile);
void            dlb_gather_plan_free(dlb_gather_plan_t* G);
/* out: [0]=front pool doubles [1]=temporaries [2]=front scratch [3]=solve rows [4]=solve scratch
 *      [5]=front targets [6]=solve targets [7]=levels */
void            dlb_gather_plan_info(const dlb_gather_plan_t* G, long long out[8]);
enum { DLB_GP_DST = 0, DLB_GP_SRC_PTR = 1, DLB_GP_SRC_BASE = 2, DLB_GP_LD = 3, DLB_GP_H = 4, DLB_GP_W = 5,
       DLB_GP_SRC_LD = 6, DLB_GP_LEVEL_PTR = 7, DLB_GP_TMP_OFF = 8, DLB_GP_LEVEL_TMP = 9, DLB_GP_SG_FLAG = 10 };
/* list 0 = fronts, 1 = forward solve; TMP_OFF / LEVEL_TMP / SG_FLAG are per supernode / level and
 * ignore list. Copies min(cap, length) values widened to long long, returns the length. */
long long       dlb_gather_plan_get(const dlb_gather_plan_t* G, int list, int what, long long* out, long long cap);

/* The streaming passes over Jt (gradient Jt*x, |J v|^2, assembly of Jt*Jt': reference
 * dogleg.c:249-281 and the A*A' inside CHOLMOD) as a host-side integer plan: tasks = (pattern
 * class, chunk of member columns), range tasks = runs of consecutive columns with periodic classes,
 * the offsets of the partial results and the inverse map that sums them per state. Exposed for
 * the CPU tests (tests/test_taskplan.py). Jp = column pointers of the whole pattern; the plan covers
 * the columns [col_begin, col_begin + ncols) (a rank's slice when row-sharded). */
typedef struct dlb_task_plan dlb_task_plan_t;
dlb_task_plan_t* dlb_task_plan_create(const dlb_symbolic_t* S, const int* Jp, int col_begin, int ncols,
                                      int sm_count, int ranges_enabled);
void            dlb_task_plan_free(dlb_task_plan_t* T);
enum { DLB_TP_TASK_CLS = 0, DLB_TP_TASK_M0 = 1, DLB_TP_TASK_M1 = 2, DLB_TP_CLS_TASK_PTR = 3, DLB_TP_TASK_GOFF = 4,
       DLB_TP_TASK_GGOFF = 5, DLB_TP_MEM_COL = 6, DLB_TP_MEM_POS = 7, DLB_TP_BIG_TASKS = 8, DLB_TP_SMALL_TASKS = 9,
       DLB_TP_GJ_BIG_TASKS = 10, DLB_TP_RANGED = 11, DLB_TP_GP_COUNT = 12, DLB_TP_GP_FIRST = 13, DLB_TP_GINV_PTR = 14,
       DLB_TP_GINV_CLS = 15, DLB_TP_GINV_OFF = 16, DLB_TP_HEAVY = 17, DLB_TP_MEDIUM = 18,
       DLB_TP_SIZES = 19,        /* [0]=gpart doubles [1]=Gpart doubles [2]=range_kmax [3]=heavy threshold */
       DLB_TP_RANGE_TASKS = 20   /* 17 values per task: j0 ncols P Ktot pos0 | cls[4] | koff[4] | goff[4] */ };
/* copies min(cap, length) values widened to long long, returns the length */
long long       dlb_task_plan_get(const dlb_task_plan_t* T, int what, long long* out, long long cap);

/* ------------------------------------------------------------------- engine */
typedef struct dlb_engine dlb_engine_t;

typedef struct
{
  /* evaluate: reference dogleg.c:1025-1027, 1073-1081 */
  double norm2_x, norm2_Jtx, maxabs_Jtx;
  /* cauchy: dogleg.c:556-607 */
  double norm2_JJtx, k_cauchy, norm2_cauchy;
  /* gauss-newton: dogleg.c:862-865 */
  double norm2_gn;
  /* step: dogleg.c:964-987, 1107-1109, 1289-1291 */
  double norm2_step, k_interp, Jtx_dot_step, maxabs_step, norm2_Jstep, discriminant;
  /* dlb_engine_trial(): the step type it chose (DLB_STEP_*); 1.0 if it had to factorize and solve */
  double step_type, trial_flags;
  long long minor;            /* factorization: -1 = positive definite, else failing column */
} dlb_scalars_t;

enum { DLB_STEP_CAUCHY = 0, DLB_STEP_GAUSSNEWTON = 1, DLB_STEP_INTERPOLATED = 2 };

/* solve_type: dogleg_solve_type_t. packed/upper only matter for DENSE_PRODUCTS.
 * Returns NULL (see dogleg_gpu_last_error) if there is no GPU: there is no CPU
 * fallback. */
dlb_engine_t* dlb_engine_create(int solve_type, unsigned int Nstate, unsigned int Nmeas,
                                unsigned int NJnnz, int packed, int upper);
/* flags: DLB_ENGINE_NO_HOST_INPUTS = do not allocate pinned host mirrors for x / Jacobian /
 * pattern (device-callback solves whose context is not handed back to the caller) */
enum { DLB_ENGINE_NO_HOST_INPUTS = 1 };
dlb_engine_t* dlb_engine_create2(int solve_type, unsigned int Nstate, unsigned int Nmeas,
                                 unsigned int NJnnz, int packed, int upper, int flags);
/* row-sharded engine: Nmeas/NJnnz are this rank's counts, its columns are
 * [col_begin, col_begin + Nmeas) of Nmeas_total (0 = not sharded); set_pattern then takes the
 * GLOBAL pattern */
dlb_engine_t* dlb_engine_create3(int solve_type, unsigned int Nstate, unsigned int Nmeas,
                                 unsigned int NJnnz, int packed, int upper, int flags,
                                 unsigned int Nmeas_total, unsigned int col_begin);
/* [0] all-reduce calls, [1] bytes all-reduced */
void          dlb_engine_comm_stats(const dlb_engine_t* e, double out[2]);
/* Idle engines are kept (at most 2) so that repeated solves of the same shape skip allocation
 * and, if the pattern is unchanged, the symbolic analysis; DOGLEG_GPU_ENGINE_CACHE=0 turns
 * this off, dogleg_gpu_release_cache() frees them. */
void          dlb_engine_destroy(dlb_engine_t* e);
void          dogleg_gpu_release_cache(void);
/* A cached symbolic analysis is reused only if a 64-bit hash of the WHOLE pattern (Jp and Ji) matches
 * (~2 ms per 100 MB of pattern, once per solve). A caller that guarantees an unchanged pattern from
 * solve to solve may switch the hash off for this thread (a sample of both arrays is still compared);
 * DOGLEG_GPU_TRUST_PATTERN=1 does the same for the process. */
void          dogleg_gpu_assume_pattern_unchanged(int on);
/* DOGLEG_GPU_CHECK_PATTERN=1: 1 if (Jp, Ji) equals the pattern the engine was analysed for, 0 if not, -1 if no copy is kept */
int           dlb_engine_pattern_equals(const dlb_engine_t* e, const int* Jp, const int* Ji);

/* pinned host mirrors the engine owns (what dogleg_operatingPoint_t points at) */
enum { DLB_BUF_P = 0, DLB_BUF_X = 1, DLB_BUF_JTX = 2, DLB_BUF_CAUCHY = 3, DLB_BUF_GN = 4,
       DLB_BUF_STEP = 5, DLB_BUF_JVALUES = 6, DLB_BUF_JP = 7, DLB_BUF_JI = 8,
       DLB_BUF_NORM2X = 9   /* device only, DENSE_PRODUCTS: the |x|^2 a device callback writes */ };
void*         dlb_engine_host_buffer(dlb_engine_t* e, int slot, int which);
/* raw device pointers of the same (for device callbacks and for wrapping as
 * tensors in the multi-GPU reduce); DLB_BUF_JVALUES .. only */
void*         dlb_engine_device_buffer(dlb_engine_t* e, int slot, int which);
void*         dlb_engine_stream(dlb_engine_t* e);

/* sparse only: take the CCS pattern currently in host slot 'slot' (or the given
 * arrays), run the symbolic analysis and upload all index data. Once per solve
 * (reference dogleg.c:648-654). */
int  dlb_engine_set_pattern(dlb_engine_t* e, const int* Jp, const int* Ji,
                            const int* perm_or_null, int postorder);
const dlb_symbolic_t* dlb_engine_symbolic(const dlb_engine_t* e);

/* a15: H2D of x and Jacobian values from the slot's pinned mirrors (skipped if
 * from_host==0: a device callback already filled them), then Jt*x, |x|^2,
 * |Jt x|^2, max|Jt x| in one pass (dogleg.c:1025-1027, 1073-1081). For
 * DENSE_PRODUCTS norm2_x is taken from norm2x_products (from_host) or from the
 * slot's DLB_BUF_NORM2X device buffer (from_host==0). */
int  dlb_engine_evaluate(dlb_engine_t* e, int slot, int from_host, double norm2x_products);
/* called right before a host callback writes the slot's pinned buffers: arms dogleg_gpu_host_progress() */
void dlb_engine_begin_host_fill(dlb_engine_t* e, int slot);
/* a6: dogleg.c:529-617 */
int  dlb_engine_cauchy(dlb_engine_t* e, int slot);
/* a7/a17-a19: assemble JtJ + lambda I and factorize (dogleg.c:656-665, 699-805).
 * scalars.minor tells whether it was positive definite. */
int  dlb_engine_factorize(dlb_engine_t* e, int slot, double lambda);
/* a8: dogleg.c:839-898 */
int  dlb_engine_gauss_newton(dlb_engine_t* e, int slot);
/* a10-a12: build the step of the given type from slot 'from' with trust region
 * radius delta into slot 'to' (step_to_here, p), with the expected-improvement
 * ingredients; p[to] is copied to its host mirror (dogleg.c:1192-1296). */
int  dlb_engine_step(dlb_engine_t* e, int from, int to, int step_type, double delta);
/* One launch for the whole trial step (dlb_trial.cu; a6-a12 + a7/a8 when needed): available when every
 * front of the elimination tree fits in shared memory (dlb_engine_has_trial). Forms the Cauchy step of
 * slot 'from' unless cached, the Gauss-Newton step (factorization with the given lambda + solves) if the
 * Cauchy step is shorter than delta and it is not cached, chooses the step as dogleg.c:1192-1255
 * does, writes step and p into slot 'to' and leaves in the scalars: step_type, trial_flags,
 * norm2_cauchy, norm2_gn, norm2_step, k_interp, discriminant, Jtx_dot_step, maxabs_step, norm2_Jstep.
 * minor >= 0: not positive definite -- call again with a larger lambda (dogleg.c:668-677). */
int  dlb_engine_has_trial(const dlb_engine_t* e);
/* 1 if dlb_engine_evaluate() runs the fused pass (gradient partials + class blocks in one pass over Jt, phase 1)
 * followed by the per-state reduction (phase 3 of dlb_engine_phase_ms) */
int  dlb_engine_has_fused_eval(const dlb_engine_t* e);
int  dlb_engine_trial(dlb_engine_t* e, int from, int to, double delta, double lambda);
/* lazy p: dlb_engine_step() stops copying the new p to its host mirror (device-callback solves
 * do not need it between the steps); dlb_engine_download_p() fetches it on request */
void dlb_engine_set_lazy_p(dlb_engine_t* e, int on);
int  dlb_engine_download_p(dlb_engine_t* e, int slot);
/* bring every host mirror of the slot up to date (SURVEY.md 5 "checkpoint") */
int  dlb_engine_download(dlb_engine_t* e, int slot);
/* copy p from the host mirror to the device (start of a solve) */
int  dlb_engine_upload_p(dlb_engine_t* e, int slot);
const dlb_scalars_t* dlb_engine_scalars(const dlb_engine_t* e);

/* multi-RHS solve with the current factor: X = (JtJ + lambda I)^-1 B, B and X
 * host Nstate x nrhs column-major (what cholmod_solve / dpptrs do at
 * dogleg.c:1845-1852, 1914-1918) */
int  dlb_engine_solve(dlb_engine_t* e, const double* B, double* X, int nrhs);
/* test access: the assembled JtJ + lambda I (dense Nstate x Nstate row-first)
 * as the device sees it before factorization, and the dense factor */
int  dlb_engine_debug_JtJ(dlb_engine_t* e, int slot, double lambda, double* JtJ_out);
/* dense / dense-products: host copy of the factor in the reference's layout
 * (what ctx->factorization_dense holds after dpptrf/dpotrf) */
int  dlb_engine_dense_factor_to_host(dlb_engine_t* e, double* out);

/* counters: [0]=kernel launches [1]=H2D bytes [2]=D2H bytes [3]=factorizations */
void dlb_engine_counters(const dlb_engine_t* e, double out[4]);
/* per-phase device time (ms) accumulated with CUDA events when enabled:
 * [0]=h2d [1]=gradient [2]=cauchy(Jv) [3]=assemble [4]=factor [5]=solve [6]=step(Jv) [7]=d2h */
void dlb_engine_enable_timing(dlb_engine_t* e, int on);
void dlb_engine_phase_ms(const dlb_engine_t* e, double out[8]);

#ifdef __cplusplus
}
#endif
