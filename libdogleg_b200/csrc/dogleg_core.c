/* dogleg_core.c -- the public dogleg.h API and the trust-region automaton.
 *
 * Host side stays C (BASELINE.json north_star): this file holds no arithmetic
 * on vectors at all. Every O(Nstate) or O(NJnnz) operation of the reference is
 * a dlb_engine_* call (CUDA, include/dogleg_gpu.h); what is left here is the
 * control flow of Powell's dog-leg method, branching on the scalars the engine
 * hands back, with the reference's observable behaviour:
 *   parameters / globals      dogleg.c:117-181
 *   operating-point evaluation dogleg.c:1004-1083
 *   step selection             dogleg.c:1172-1297
 *   trust-region update        dogleg.c:1303-1356
 *   outer / retry loops        dogleg.c:1359-1476
 *   entry points, context      dogleg.c:1633-1818, 1613-1631
 *   vnlog / human diagnostics  dogleg.c:22-113
 * Intentional divergences are marked DIVERGENCE below and listed in DESIGN.md.
 */
#define _GNU_SOURCE
#include <stdio.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <time.h>
#include "dogleg.h"
#include "dogleg_gpu.h"
#include "dogleg_internal.h"

#define SAY(fmt, ...) fprintf(stderr, "libdogleg at %s:%d: " fmt "\n", __FILE__, __LINE__, ## __VA_ARGS__)
#define SAY_IF_VERBOSE(fmt, ...) do { if(ctx->parameters->debug && !ctx->parameters->debug_vnlog) SAY(fmt, ## __VA_ARGS__); } while(0)

#define LAMBDA_FIRST 1e-10     /* first diagonal loading after a singular JtJ; then x10 (dogleg.c:138, 670-672) */

/* ---------------------------------------------------------------- parameters */
#define DEFAULTS { .max_iterations = 100, .trustregion0 = 1.0e3,                      \
                   .trustregion_decrease_factor = 0.1,  .trustregion_decrease_threshold = 0.25, \
                   .trustregion_increase_factor = 2,    .trustregion_increase_threshold = 0.75, \
                   .Jt_x_threshold = 1e-8, .update_threshold = 1e-8, .trustregion_threshold = 1e-8 }
static const dogleg_parameters2_t factory_settings = DEFAULTS;
static       dogleg_parameters2_t global_settings  = DEFAULTS;

void dogleg_getDefaultParameters(dogleg_parameters2_t* parameters) { *parameters = factory_settings; }
void dogleg_setMaxIterations(int n) { global_settings.max_iterations = n; }
void dogleg_setInitialTrustregion(double t) { global_settings.trustregion0 = t; }
void dogleg_setTrustregionUpdateParameters(double downFactor, double downThreshold,
                                           double upFactor,   double upThreshold)
{
  global_settings.trustregion_decrease_factor    = downFactor;
  global_settings.trustregion_decrease_threshold = downThreshold;
  global_settings.trustregion_increase_factor    = upFactor;
  global_settings.trustregion_increase_threshold = upThreshold;
}
void dogleg_setThresholds(double Jt_x, double update, double trustregion)
{
  if(Jt_x        > 0.0) global_settings.Jt_x_threshold        = Jt_x;
  if(update      > 0.0) global_settings.update_threshold      = update;
  if(trustregion > 0.0) global_settings.trustregion_threshold = trustregion;
}
void dogleg_setDebug(int debug)
{
  const int vnlog = (debug & DOGLEG_DEBUG_VNLOG) != 0;
  global_settings.debug_vnlog = vnlog;
  global_settings.debug       = (debug != 0) && !vnlog;
}

/* -------------------------------------------------------------- vnlog record */
/* One record per trial step, same columns and formatting as the reference
 * (dogleg.c:42-113): unset fields print as "-", every field is followed by a
 * space. Like the reference this record is process-global (not re-entrant). */
enum { F_NORM2X_BEFORE, F_NORM2X_AFTER, F_LEN_CAUCHY, F_LEN_GN, F_LEN_INTERP, F_K, F_LEN,
       F_STEP_TYPE, F_DIRECTION_CHANGE, F_EXPECTED, F_OBSERVED, F_RHO, F_TR_BEFORE, F_TR_AFTER, F_COUNT };
static const char* const vnlog_names[F_COUNT] = {
  "norm2x_before", "norm2x_after", "step_len_cauchy", "step_len_gauss_newton", "step_len_interpolated",
  "k_cauchy_to_gn", "step_len", "step_type", "step_direction_change_deg", "expected_improvement",
  "observed_improvement", "rho", "trustregion_before", "trustregion_after" };
static const char* const step_type_names[] = { "cauchy", "gaussnewton", "interpolated", "failed" };
static double vnlog_rec[F_COUNT];
static void vnlog_clear(void) { for(int i = 0; i < F_COUNT; i++) vnlog_rec[i] = INFINITY; }
static void vnlog_legend(void)
{
  vnlog_clear();
  printf("# iteration step_accepted");
  for(int i = 0; i < F_COUNT; i++) printf(" %s", vnlog_names[i]);
  printf("\n");
}
static void vnlog_emit(int iteration, int accepted)
{
  printf("%d %d ", iteration, accepted);
  for(int i = 0; i < F_COUNT; i++)
  {
    if(vnlog_rec[i] == INFINITY) printf("- ");
    else if(i == F_STEP_TYPE)    printf("%s ", step_type_names[(int)vnlog_rec[i]]);
    else                         printf("%g ", vnlog_rec[i]);
  }
  printf("\n");
  fflush(stdout);
  vnlog_clear();
}
#define VNLOG(field, value) do { if(ctx->parameters->debug_vnlog) vnlog_rec[field] = (value); } while(0)

/* ------------------------------------------------------- private per context */
static __thread double last_stats[8];
static __thread double last_comm[2];
static __thread double last_phase_ms[8];

#ifdef DLB_CHOLMOD_IS_SHIM
static dlb_private_t* priv_of(const dogleg_solverContext_t* ctx) { return (dlb_private_t*)ctx->common.dlb_private; }
static void priv_set(dogleg_solverContext_t* ctx, dlb_private_t* pv) { ctx->common.dlb_private = pv; }
#else
/* real SuiteSparse headers: cholmod_common has no spare member, keep a side table (grows on demand) */
#include <pthread.h>
static struct side_entry { const dogleg_solverContext_t* ctx; dlb_private_t* pv; }* side_table;
static size_t side_cap;
static pthread_mutex_t side_lock = PTHREAD_MUTEX_INITIALIZER;
static dlb_private_t* priv_of(const dogleg_solverContext_t* ctx)
{
  dlb_private_t* pv = NULL;
  pthread_mutex_lock(&side_lock);
  for(size_t i = 0; i < side_cap; i++) if(side_table[i].ctx == ctx) { pv = side_table[i].pv; break; }
  pthread_mutex_unlock(&side_lock);
  return pv;
}
static void priv_set(dogleg_solverContext_t* ctx, dlb_private_t* pv)
{
  pthread_mutex_lock(&side_lock);
  size_t at = side_cap;
  for(size_t i = 0; i < side_cap; i++)
    if(side_table[i].ctx == ctx) { at = i; break; }
    else if(pv && side_table[i].ctx == NULL && at == side_cap) at = i;
  if(at == side_cap && pv)
  {
    const size_t ncap = side_cap ? 2 * side_cap : 64;
    struct side_entry* t = realloc(side_table, ncap * sizeof(*t));
    if(t) { memset(t + side_cap, 0, (ncap - side_cap) * sizeof(*t)); side_table = t; side_cap = ncap; }
  }
  if(at < side_cap) { side_table[at].ctx = pv ? ctx : NULL; side_table[at].pv = pv; }
  pthread_mutex_unlock(&side_lock);
}
#endif

dlb_private_t* dlb_private_of(const dogleg_solverContext_t* ctx) { return priv_of(ctx); }

static int slot_of(const dlb_private_t* pv, const dogleg_operatingPoint_t* point)
{
  if(point == pv->points[0]) return 0;
  if(point == pv->points[1]) return 1;
  return -1;
}

int dlb_slot_of(const dogleg_solverContext_t* ctx, const dogleg_operatingPoint_t* point)
{ const dlb_private_t* pv = priv_of(ctx); return pv ? slot_of(pv, point) : -1; }

static double wall_s(void)
{
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

/* ------------------------------------------------ operating-point evaluation */
/* reference computeCallbackOperatingPoint(), dogleg.c:1004-1083 */
static bool evaluate_point(bool* converged, dogleg_operatingPoint_t* point, dogleg_solverContext_t* ctx)
{
  dlb_private_t* pv = priv_of(ctx);
  const int s = slot_of(pv, point);
  point->norm2_x = -1.;
  memset(point->dummy_bits, 0, sizeof(point->dummy_bits));

  double norm2x_products = 0.0;
  const double t0 = wall_s();
  if(pv->device_callbacks)
  {
    double* d_p = dlb_engine_device_buffer(pv->eng, s, DLB_BUF_P);
    double* d_x = dlb_engine_device_buffer(pv->eng, s, DLB_BUF_X);
    double* d_J = dlb_engine_device_buffer(pv->eng, s, DLB_BUF_JVALUES);
    if(ctx->solve_type == DOGLEG_SPARSE)     pv->f_gpu_sparse(d_p, d_x, d_J, dlb_engine_stream(pv->eng), ctx->cookie);
    else if(ctx->solve_type == DOGLEG_DENSE) pv->f_gpu_dense (d_p, d_x, d_J, dlb_engine_stream(pv->eng), ctx->cookie);
    else /* d_J holds the slot's JtJ */      pv->f_gpu_products(d_p, dlb_engine_device_buffer(pv->eng, s, DLB_BUF_NORM2X),
                                                                dlb_engine_device_buffer(pv->eng, s, DLB_BUF_JTX), d_J,
                                                                dlb_engine_stream(pv->eng), ctx->cookie);
  }
  else if(ctx->solve_type == DOGLEG_SPARSE)   { dlb_engine_begin_host_fill(pv->eng, s); ctx->f(point->p, point->x, point->Jt, ctx->cookie); }
  else if(ctx->solve_type == DOGLEG_DENSE)    { dlb_engine_begin_host_fill(pv->eng, s); ctx->f_dense(point->p, point->x, point->J_dense, ctx->cookie); }
  else ctx->f_dense_products(point->p, &norm2x_products, point->Jt_x, point->JtJ, ctx->cookie);
  pv->stats[7] += wall_s() - t0;
  pv->stats[1] += 1;

  if(ctx->solve_type == DOGLEG_SPARSE && !pv->device_callbacks)
  {
    /* The sparsity pattern is analysed once and assumed fixed (dogleg.c:648-654) */
    if(!pv->pattern_set)
    {
      if(dlb_engine_set_pattern(pv->eng, point->Jt->p, point->Jt->i,
                                pv->have_user_perm ? pv->user_perm : NULL, pv->user_perm_postorder))
      { SAY("could not analyse the Jacobian pattern: %s", dogleg_gpu_last_error()); return false; }
      pv->pattern_set = 1;
      pv->pattern_slot = s;
    }
    else if(s != pv->pattern_slot || pv->check_pattern)
    {
      const int* p0 = pv->points[pv->pattern_slot]->Jt->p; const int* p1 = point->Jt->p;
      const int* i0 = pv->points[pv->pattern_slot]->Jt->i; const int* i1 = point->Jt->i;
      const int M = ctx->Nmeasurements;
      bool same = p0[M] == p1[M];
      if(same && pv->check_pattern)
      { /* exhaustive, against the engine's own copy of the analysed pattern: the callback may have
         * changed the very buffer the analysis was taken from */
        const int eq = dlb_engine_pattern_equals(pv->eng, p1, i1);
        same = eq < 0 ? (!memcmp(p0, p1, sizeof(int) * (M + 1)) && !memcmp(i0, i1, sizeof(int) * (size_t)p0[M])) : eq == 1;
      }
      else if(same && p0 != p1)
      {
        if(0) { }
        else
        { /* cheap spot check: both ends of both arrays */
          const size_t np = (size_t)M + 1, ni = (size_t)p0[M];
          const size_t cp = np < 64 ? np : 64, ci = ni < 64 ? ni : 64;
          same = !memcmp(p0, p1, sizeof(int) * cp) && !memcmp(p0 + np - cp, p1 + np - cp, sizeof(int) * cp) &&
                 !memcmp(i0, i1, sizeof(int) * ci) && !memcmp(i0 + ni - ci, i1 + ni - ci, sizeof(int) * ci);
        }
      }
      if(!same) { SAY("the sparsity pattern of Jt changed between evaluations; it must stay fixed"); return false; }
    }
  }

  if(dlb_engine_evaluate(pv->eng, s, !pv->device_callbacks, norm2x_products))
  { SAY("device evaluation failed: %s", dogleg_gpu_last_error()); return false; }
  const dlb_scalars_t* sc = dlb_engine_scalars(pv->eng);
  point->norm2_x = sc->norm2_x;
  if(ctx->solve_type == DOGLEG_DENSE_PRODUCTS) { point->have_Jtx = true; point->have_JtJ = true; }
  else { point->have_x = true; point->have_J = true; point->have_Jtx = true; }

  /* inf-norm of the gradient against the threshold (dogleg.c:1073-1081) */
  *converged = !(sc->maxabs_Jtx > ctx->parameters->Jt_x_threshold);
  if(*converged) SAY_IF_VERBOSE("Jt_x all below the threshold. Done iterating!");
  return true;
}

/* reference compute_updateCauchy(), dogleg.c:529-617 */
static bool cauchy_at(dogleg_operatingPoint_t* point, dogleg_solverContext_t* ctx)
{
  dlb_private_t* pv = priv_of(ctx);
  if(!point->have_updateCauchy)
  {
    if(!point->have_Jtx) { SAY("%s() needs Jtx, but it isn't available", __func__); return false; }
    if(ctx->solve_type == DOGLEG_DENSE_PRODUCTS ? !point->have_JtJ : !point->have_J)
    { SAY("%s() needs J, but it isn't available", __func__); return false; }
    if(dlb_engine_cauchy(pv->eng, slot_of(pv, point)))
    { SAY("%s", dogleg_gpu_last_error()); return false; }
    point->norm2_updateCauchy = dlb_engine_scalars(pv->eng)->norm2_cauchy;
    point->have_updateCauchy = true;
    SAY_IF_VERBOSE("cauchy step size %.6g", sqrt(point->norm2_updateCauchy));
  }
  VNLOG(F_LEN_CAUCHY, sqrt(point->norm2_updateCauchy));
  return true;
}

/* reference dogleg_computeJtJfactorization(), dogleg.c:634-820 */
bool dogleg_computeJtJfactorization(dogleg_operatingPoint_t* point, dogleg_solverContext_t* ctx)
{
  if(point->have_factorization) return true;
  dlb_private_t* pv = priv_of(ctx);
  if(!pv) { SAY("this context was not created by this library"); return false; }
  const int s = slot_of(pv, point);
  if(s < 0) { SAY("%s(): unknown operating point", __func__); return false; }
  if(ctx->solve_type == DOGLEG_DENSE_PRODUCTS ? !point->have_JtJ : !point->have_J)
  { SAY("%s() needs J, but it isn't available", __func__); return false; }

  /* the cholmod_factor descriptor (permutation, column counts, supernodes: copies of arrays of
   * the size of L's pattern) only exists for callers who can look at it, i.e. when the context is
   * handed back; building it for every solve cost 80 ms at bundle-adjustment scale */
  if(ctx->solve_type == DOGLEG_SPARSE && !ctx->factorization && pv->context_returned)
    ctx->factorization = dlb_factor_descriptor_new(dlb_engine_symbolic(pv->eng), ctx->Nstate);

  for(;;)
  {
    if(dlb_engine_factorize(pv->eng, s, ctx->lambda))
    { SAY("factorization failed: %s", dogleg_gpu_last_error()); return false; }
    pv->stats[3] += 1;
    const long long minor = dlb_engine_scalars(pv->eng)->minor;
    if(ctx->solve_type == DOGLEG_SPARSE && ctx->factorization)
      ctx->factorization->minor = minor < 0 ? (size_t)ctx->Nstate : (size_t)minor;
    if(minor < 0) break;

    /* singular JtJ: load the diagonal and go again; lambda stays for the rest of the solve */
    ctx->lambda = ctx->lambda == 0.0 ? LAMBDA_FIRST : ctx->lambda * 10.0;
    if(!isfinite(ctx->lambda)) { SAY("ASSERTION FAILED: lambda is not finite"); return false; }
    SAY_IF_VERBOSE("singular JtJ. Have rank/full rank: %lld/%d. Adding %g I from now on",
                   minor, ctx->Nstate, ctx->lambda);
  }
  point->have_factorization = true;
  return true;
}

/* SURVEY.md 8f2: what a returnContext user of the reference does with ctx->factorization
 * (cholmod_solve at dogleg.c:853-856, 1914-1918; README.pod:105-111), on the device factor.
 * X = (JtJ + lambda I)^-1 B at ctx->beforeStep; B, X: host, Nstate x nrhs column-major. */
int dogleg_gpu_solve(dogleg_solverContext_t* ctx, const double* B, double* X, int nrhs)
{
  dlb_private_t* pv = ctx ? priv_of(ctx) : NULL;
  if(!pv || !B || !X || nrhs < 1) { SAY("%s(): bad arguments or a context this library did not create", __func__); return -1; }
  if(!dogleg_computeJtJfactorization(ctx->beforeStep, ctx)) return -1;
  if(dlb_engine_solve(pv->eng, B, X, nrhs)) { SAY("%s", dogleg_gpu_last_error()); return -1; }
  return 0;
}
/* Fill ctx->factorization->x with the numeric factor (supernodal L L', CHOLMOD's layout: supernode s
 * is an nsrow x nscol column-major panel at x[px[s]], rows s[pi[s]..pi[s+1]), columns super[s]..super[s+1]-1,
 * in the ordering Perm) so that host code can run its own triangular solves. Sparse solves only: the
 * dense factor is already in ctx->factorization_dense. */
int dogleg_gpu_export_factor(dogleg_solverContext_t* ctx)
{
  dlb_private_t* pv = ctx ? priv_of(ctx) : NULL;
  if(!pv || ctx->solve_type != DOGLEG_SPARSE) { SAY("%s(): needs a sparse context created by this library", __func__); return -1; }
  if(!ctx->factorization) ctx->factorization = dlb_factor_descriptor_new(dlb_engine_symbolic(pv->eng), ctx->Nstate);
  if(!ctx->factorization) { SAY("out of memory"); return -1; }
  if(!dogleg_computeJtJfactorization(ctx->beforeStep, ctx)) return -1;
  cholmod_factor* L = ctx->factorization;
  if(!L->x) L->x = malloc(sizeof(double) * (L->xsize ? L->xsize : 1));
  if(!L->x) { SAY("out of memory"); return -1; }
  if(dlb_engine_export_factor(pv->eng, (const int*)L->px, (long long)L->xsize, (double*)L->x))
  { SAY("%s", dogleg_gpu_last_error()); return -1; }
  L->minor = (size_t)ctx->Nstate;
  return 0;
}

/* reference compute_updateGN(), dogleg.c:822-908 */
static bool gauss_newton_at(dogleg_operatingPoint_t* point, dogleg_solverContext_t* ctx)
{
  dlb_private_t* pv = priv_of(ctx);
  if(!point->have_updateGN)
  {
    if(!dogleg_computeJtJfactorization(point, ctx)) return false;
    if(!point->have_Jtx) { SAY("%s() needs Jtx, but it isn't available", __func__); return false; }
    const int s = slot_of(pv, point);
    if(dlb_engine_gauss_newton(pv->eng, s)) { SAY("%s", dogleg_gpu_last_error()); return false; }
    point->norm2_updateGN = dlb_engine_scalars(pv->eng)->norm2_gn;
    if(ctx->solve_type == DOGLEG_SPARSE) point->updateGN_cholmoddense = &pv->gn_header[s];
    SAY_IF_VERBOSE("gn step size %.6g", sqrt(point->norm2_updateGN));
    point->have_updateGN = true;
  }
  VNLOG(F_LEN_GN, sqrt(point->norm2_updateGN));
  return true;
}

/* The same decisions as take_step() below when the engine runs the whole trial step as one kernel
 * (dlb_engine_trial): Cauchy step, Gauss-Newton step if needed (with the lambda ladder of
 * dogleg.c:668-677 driven from here), step selection. Returns the chosen type or -1. */
static int trial_on_device(dogleg_operatingPoint_t* from, dogleg_operatingPoint_t* to, double trustregion,
                           dogleg_solverContext_t* ctx)
{
  dlb_private_t* pv = priv_of(ctx);
  const int s = slot_of(pv, from);
  if(!from->have_Jtx || !from->have_J) { SAY("%s() needs J and Jtx, but they aren't available", __func__); return -1; }
  if(ctx->solve_type == DOGLEG_SPARSE && !ctx->factorization && pv->context_returned)
    ctx->factorization = dlb_factor_descriptor_new(dlb_engine_symbolic(pv->eng), ctx->Nstate);
  const dlb_scalars_t* sc = dlb_engine_scalars(pv->eng);
  for(;;)
  {
    if(dlb_engine_trial(pv->eng, s, slot_of(pv, to), trustregion, ctx->lambda))
    { SAY("%s", dogleg_gpu_last_error()); return -1; }
    if(!from->have_updateCauchy)
    {
      from->norm2_updateCauchy = sc->norm2_cauchy;
      from->have_updateCauchy = true;
      SAY_IF_VERBOSE("cauchy step size %.6g", sqrt(from->norm2_updateCauchy));
    }
    if(sc->minor < 0) break;
    /* singular JtJ: load the diagonal and go again; lambda stays for the rest of the solve */
    pv->stats[3] += 1;
    if(ctx->factorization) ctx->factorization->minor = (size_t)sc->minor;
    ctx->lambda = ctx->lambda == 0.0 ? LAMBDA_FIRST : ctx->lambda * 10.0;
    if(!isfinite(ctx->lambda)) { SAY("ASSERTION FAILED: lambda is not finite"); return -1; }
    SAY_IF_VERBOSE("singular JtJ. Have rank/full rank: %lld/%d. Adding %g I from now on",
                   sc->minor, ctx->Nstate, ctx->lambda);
  }
  VNLOG(F_LEN_CAUCHY, sqrt(from->norm2_updateCauchy));
  const int type = (int)sc->step_type;
  if(type != DLB_STEP_CAUCHY)
  {
    if(!from->have_updateGN)
    {
      pv->stats[3] += 1;
      if(ctx->factorization) ctx->factorization->minor = (size_t)ctx->Nstate;
      from->have_factorization = true;
      from->norm2_updateGN = sc->norm2_gn;
      if(ctx->solve_type == DOGLEG_SPARSE) from->updateGN_cholmoddense = &pv->gn_header[s];
      SAY_IF_VERBOSE("gn step size %.6g", sqrt(from->norm2_updateGN));
      from->have_updateGN = true;
    }
    VNLOG(F_LEN_GN, sqrt(from->norm2_updateGN));
  }
  return type;
}

/* reference takeStepFrom() + computeInterpolatedUpdate() + computeExpectedImprovement(),
 * dogleg.c:1172-1297, 927-998, 1085-1165 */
static bool take_step(double* expectedImprovement, dogleg_operatingPoint_t* from,
                      dogleg_operatingPoint_t* to, double trustregion, dogleg_solverContext_t* ctx)
{
  dlb_private_t* pv = priv_of(ctx);
  SAY_IF_VERBOSE("taking step with trustregion %.6g", trustregion);
  VNLOG(F_TR_BEFORE, trustregion);
  VNLOG(F_NORM2X_BEFORE, from->norm2_x);

  const bool on_device = dlb_engine_has_trial(pv->eng);
  int type;
  if(on_device)
  {
    type = trial_on_device(from, to, trustregion, ctx);
    if(type < 0) return false;
    if(type == DLB_STEP_CAUCHY)           SAY_IF_VERBOSE("taking cauchy step");
    else if(type == DLB_STEP_GAUSSNEWTON) SAY_IF_VERBOSE("taking GN step");
    else                                  SAY_IF_VERBOSE("taking interpolated step");
    from->didStepToEdgeOfTrustRegion = type != DLB_STEP_GAUSSNEWTON;
  }
  else if(!cauchy_at(from, ctx)) return false;
  else if(from->norm2_updateCauchy >= trustregion * trustregion)
  {
    SAY_IF_VERBOSE("taking cauchy step");
    type = DLB_STEP_CAUCHY;
    from->didStepToEdgeOfTrustRegion = true;
  }
  else
  {
    if(!gauss_newton_at(from, ctx)) return false;
    if(from->norm2_updateGN <= trustregion * trustregion)
    {
      SAY_IF_VERBOSE("taking GN step");
      type = DLB_STEP_GAUSSNEWTON;
      from->didStepToEdgeOfTrustRegion = false;
    }
    else
    {
      SAY_IF_VERBOSE("taking interpolated step");
      type = DLB_STEP_INTERPOLATED;
      from->didStepToEdgeOfTrustRegion = true;
    }
  }

  if(!on_device && dlb_engine_step(pv->eng, slot_of(pv, from), slot_of(pv, to), type, trustregion))
  { SAY("%s", dogleg_gpu_last_error()); return false; }
  const dlb_scalars_t* sc = dlb_engine_scalars(pv->eng);
  to->norm2_step_to_here = sc->norm2_step;

  if(type == DLB_STEP_INTERPOLATED)
  {
    if(sc->discriminant < 0.0) SAY("negative discriminant: %.6g!", sc->discriminant);
    SAY_IF_VERBOSE("k_cauchy_to_gn %.6g, norm %.6g", sc->k_interp, sqrt(sc->norm2_step));
    VNLOG(F_LEN_INTERP, sqrt(sc->norm2_step));
    VNLOG(F_K, sc->k_interp);
  }
  VNLOG(F_STEP_TYPE, (double)type);
  /* for a clipped cauchy step this is the UNCLIPPED length, as in the reference (dogleg.c:1198) */
  VNLOG(F_LEN, sqrt(sc->norm2_step));

  /* F(0) - F(step) for the linearised x: -2 Jt_x.step - |J step|^2 */
  *expectedImprovement = -2.0 * sc->Jtx_dot_step - sc->norm2_Jstep;
  VNLOG(F_EXPECTED, *expectedImprovement);
  /* step_direction_change_deg needs from->have_step_to_here, which never survives the evaluation of
   * the point (every evaluation clears all flags): like the reference this column always prints "-" */

  if(sc->maxabs_step > ctx->parameters->update_threshold) return true;
  SAY_IF_VERBOSE("update small enough. Done iterating!");
  *expectedImprovement = -1.0;
  return true;
}

/* reference evaluateStep_adjustTrustRegion(), dogleg.c:1303-1356 */
static bool judge_step(bool* accept, double* trustregion,
                       const dogleg_operatingPoint_t* before, const dogleg_operatingPoint_t* after,
                       double expectedImprovement, dogleg_solverContext_t* ctx)
{
  const dogleg_parameters2_t* P = ctx->parameters;
  const double observed = before->norm2_x - after->norm2_x;
  double rho = observed / expectedImprovement;
  /* DIVERGENCE: a non-finite cost makes the reference retry forever with an unchanged trust region
   * (rho = NaN matches no branch). Treat it as the worst possible step instead. */
  if(!isfinite(after->norm2_x)) rho = -INFINITY;
  SAY_IF_VERBOSE("observed/expected improvement: %.6g/%.6g. rho = %.6g", observed, expectedImprovement, rho);
  VNLOG(F_OBSERVED, observed);
  VNLOG(F_RHO, rho);

  if(rho < P->trustregion_decrease_threshold)
  {
    SAY_IF_VERBOSE("rho too small. decreasing trust region");
    if(!before->didStepToEdgeOfTrustRegion)
    {
      if(!before->have_updateGN)
      { SAY("ERROR: In %s() updateGN should already have been computed. This is a bug", __func__); return false; }
      *trustregion = sqrt(before->norm2_updateGN);
    }
    *trustregion *= P->trustregion_decrease_factor;
  }
  else if(rho > P->trustregion_increase_threshold && before->didStepToEdgeOfTrustRegion)
  {
    SAY_IF_VERBOSE("rho large enough. increasing trust region");
    *trustregion *= P->trustregion_increase_factor;
  }
  VNLOG(F_TR_AFTER, *trustregion);
  *accept = rho > 0.0;
  return true;
}

/* reference runOptimizer(), dogleg.c:1359-1476. Returns accepted steps or <0 */
static int run_solver(dogleg_solverContext_t* ctx)
{
  dlb_private_t* pv = priv_of(ctx);
  double trustregion = ctx->parameters->trustregion0;
  int steps = 0;
  bool converged;
  if(!evaluate_point(&converged, ctx->beforeStep, ctx)) return -1;
  if(converged) return steps;
  SAY_IF_VERBOSE("Initial operating point has norm2_x %.6g", ctx->beforeStep->norm2_x);

  while(steps < ctx->parameters->max_iterations)
  {
    SAY_IF_VERBOSE("================= step %d", steps);
    for(;;)
    {
      SAY_IF_VERBOSE("--------");
      ctx->afterStep->have_step_to_here = false;
      double expected;
      if(!take_step(&expected, ctx->beforeStep, ctx->afterStep, trustregion, ctx)) return -1;
      ctx->afterStep->have_step_to_here = true;

      if(expected < 0.0)
      { /* the step is too small to bother: stop WITHOUT applying it (dogleg.c:1403-1408) */
        if(ctx->parameters->debug_vnlog) vnlog_emit(steps, 1);
        return steps;
      }

      bool after_converged;
      if(!evaluate_point(&after_converged, ctx->afterStep, ctx)) return -1;
      SAY_IF_VERBOSE("Evaluated operating point with norm2_x %.6g", ctx->afterStep->norm2_x);
      VNLOG(F_NORM2X_AFTER, ctx->afterStep->norm2_x);

      bool accept;
      if(!judge_step(&accept, &trustregion, ctx->beforeStep, ctx->afterStep, expected, ctx)) return -1;
      if(accept)
      {
        SAY_IF_VERBOSE("accepted step");
        if(ctx->parameters->debug_vnlog) vnlog_emit(steps, 1);
        steps++;
        dogleg_operatingPoint_t* t = ctx->afterStep; ctx->afterStep = ctx->beforeStep; ctx->beforeStep = t;
        if(after_converged)
        {
          SAY_IF_VERBOSE("Gradient low enough and we just improved. Done iterating!");
          return steps;
        }
        break;
      }
      SAY_IF_VERBOSE("rejected step");
      pv->stats[2] += 1;
      if(ctx->parameters->debug_vnlog) vnlog_emit(steps, 0);
      if(trustregion < ctx->parameters->trustregion_threshold)
      {
        SAY_IF_VERBOSE("trust region small enough. Giving up. Done iterating!");
        return steps;
      }
    }
  }
  if(steps == ctx->parameters->max_iterations) SAY_IF_VERBOSE("Exceeded max number of iterations");
  return steps;
}

/* --------------------------------------------------------- context lifecycle */
static dogleg_operatingPoint_t* make_point(dogleg_solverContext_t* ctx, dlb_private_t* pv, int s, unsigned int NJnnz)
{
  dogleg_operatingPoint_t* pt = calloc(1, sizeof(*pt));
  if(!pt) return NULL;
  dlb_engine_t* e = pv->eng;
  pt->p            = dlb_engine_host_buffer(e, s, DLB_BUF_P);
  pt->x            = ctx->solve_type == DOGLEG_DENSE_PRODUCTS ? NULL : dlb_engine_host_buffer(e, s, DLB_BUF_X);
  pt->Jt_x         = dlb_engine_host_buffer(e, s, DLB_BUF_JTX);
  pt->updateCauchy = dlb_engine_host_buffer(e, s, DLB_BUF_CAUCHY);
  pt->step_to_here = dlb_engine_host_buffer(e, s, DLB_BUF_STEP);
  if(ctx->solve_type == DOGLEG_SPARSE)
  {
    /* same shape cholmod_allocate_sparse(Nstate,Nmeas,NJnnz,sorted,packed,stype 0,REAL) gives
     * (dogleg.c:1534-1539); the arrays are the engine's pinned staging buffers */
    cholmod_sparse* Jt = calloc(1, sizeof(*Jt));
    if(!Jt) { free(pt); return NULL; }
    Jt->nrow = ctx->Nstate; Jt->ncol = ctx->Nmeasurements; Jt->nzmax = NJnnz;
    Jt->p = dlb_engine_host_buffer(e, s, DLB_BUF_JP);
    Jt->i = dlb_engine_host_buffer(e, s, DLB_BUF_JI);
    Jt->x = dlb_engine_host_buffer(e, s, DLB_BUF_JVALUES);
    Jt->stype = 0; Jt->itype = CHOLMOD_INT; Jt->xtype = CHOLMOD_REAL; Jt->dtype = CHOLMOD_DOUBLE;
    Jt->sorted = 1; Jt->packed = 1;
    pt->Jt = Jt;
    pt->updateGN_cholmoddense = NULL;     /* appears once a Gauss-Newton step exists, as in the reference */
    cholmod_dense* g = &pv->gn_header[s];
    g->nrow = ctx->Nstate; g->ncol = 1; g->nzmax = ctx->Nstate; g->d = ctx->Nstate;
    g->x = dlb_engine_host_buffer(e, s, DLB_BUF_GN); g->z = NULL;
    g->xtype = CHOLMOD_REAL; g->dtype = CHOLMOD_DOUBLE;
  }
  else
  {
    if(ctx->solve_type == DOGLEG_DENSE) pt->J_dense = dlb_engine_host_buffer(e, s, DLB_BUF_JVALUES);
    else                                pt->JtJ     = dlb_engine_host_buffer(e, s, DLB_BUF_JVALUES);
    pt->updateGN_dense = dlb_engine_host_buffer(e, s, DLB_BUF_GN);
  }
  return pt;
}

void dogleg_freeContext(dogleg_solverContext_t** pctx)
{
  if(!pctx || !*pctx) return;
  dogleg_solverContext_t* ctx = *pctx;
  dlb_private_t* pv = priv_of(ctx);
  if(pv)
  {
    for(int s = 0; s < 2; s++)
      if(pv->points[s])
      {
        if(ctx->solve_type == DOGLEG_SPARSE) free(pv->points[s]->Jt);
        free(pv->points[s]);
      }
    if(ctx->solve_type == DOGLEG_SPARSE) dlb_factor_descriptor_free(ctx->factorization);
    else                                 free(ctx->factorization_dense);
    dlb_engine_destroy(pv->eng);
    free(pv->user_perm);
    priv_set(ctx, NULL);
    free(pv);
  }
  free(ctx);
  *pctx = NULL;
}

/* pending ordering injection for the next sparse context of this thread */
static __thread int* pending_perm; static __thread int pending_perm_n, pending_perm_post;
void dogleg_gpu_set_permutation(const int* perm, int n, int postorder)
{
  free(pending_perm); pending_perm = NULL; pending_perm_n = 0; pending_perm_post = postorder;
  if(perm && n > 0)
  {
    pending_perm = malloc(sizeof(int) * n);
    memcpy(pending_perm, perm, sizeof(int) * n);
    pending_perm_n = n;
  }
}

/* What this build of the library thinks dogleg_solverContext_t looks like. A returned context is only
 * readable by an application compiled against the SAME cholmod.h (cholmod_common sits by value at the
 * head of the struct): compare with your own sizeof/offsetof before touching a returned context. */
void dogleg_gpu_context_layout(size_t out[6])
{
  out[0] = sizeof(dogleg_solverContext_t);
  out[1] = sizeof(cholmod_common);
  out[2] = offsetof(dogleg_solverContext_t, beforeStep);
  out[3] = offsetof(dogleg_solverContext_t, factorization);
  out[4] = offsetof(dogleg_solverContext_t, lambda);
  out[5] =
#ifdef DLB_CHOLMOD_IS_SHIM
    1;            /* built against compat/cholmod.h */
#else
    0;            /* built against a real SuiteSparse cholmod.h */
#endif
}

void dogleg_gpu_get_phase_ms(double out[8]) { memcpy(out, last_phase_ms, sizeof(last_phase_ms)); }

void dogleg_gpu_get_comm_stats(double out[2]) { memcpy(out, last_comm, sizeof(last_comm)); }

void dogleg_gpu_get_stats(const dogleg_solverContext_t* ctx, double out[8])
{
  const dlb_private_t* pv = ctx ? priv_of(ctx) : NULL;
  memcpy(out, pv ? pv->stats : last_stats, sizeof(last_stats));
}

/* bring the host-visible state of the final operating point up to date (SURVEY.md 5, checkpoint row) */
static bool publish_results(dogleg_solverContext_t* ctx)
{
  dlb_private_t* pv = priv_of(ctx);
  /* p of the final point is current on the host (the step kernel's D2H, or the caller's start
   * point) -- except in device-callback solves, which fetch it here; everything else is only
   * visible through a returned context */
  if(pv->device_callbacks && dlb_engine_download_p(pv->eng, slot_of(pv, ctx->beforeStep))) return false;
  if(pv->context_returned)
  {
    for(int s = 0; s < 2; s++)
      if(dlb_engine_download(pv->eng, s)) return false;
    if(pv->device_callbacks)
      for(int s = 0; s < 2; s++)
        if(dlb_engine_download_inputs(pv->eng, s)) return false;
    if(ctx->solve_type != DOGLEG_SPARSE)
    {
      if(dlb_engine_dense_factor_to_host(pv->eng, ctx->factorization_dense)) return false;
    }
  }
  dlb_engine_phase_ms(pv->eng, last_phase_ms);
  double c[4];
  dlb_engine_counters(pv->eng, c);
  pv->stats[4] = c[0]; pv->stats[5] = c[1]; pv->stats[6] = c[2];
  memcpy(last_stats, pv->stats, sizeof(last_stats));
  dlb_engine_comm_stats(pv->eng, last_comm);
  return true;
}

/* reference _dogleg_optimize(), dogleg.c:1633-1753 */
/* Nmeas / NJnnz are this process's counts; Nmeas_total > 0 declares a row-sharded solve in which
 * they cover the columns [col_begin, col_begin + Nmeas) and Jp/Ji are the global pattern */
static double optimize_common(double* p, unsigned int Nstate, unsigned int Nmeas, unsigned int NJnnz,
                              dogleg_solve_type_t type,
                              void* host_callback, void* gpu_callback, const int* Jp, const int* Ji,
                              unsigned int Nmeas_total, unsigned int col_begin,
                              void* cookie, const dogleg_parameters2_t* parameters,
                              dogleg_solverContext_t** returnContext)
{
  if(returnContext) *returnContext = NULL;
  const int verbose_t = getenv("DOGLEG_GPU_VERBOSE") && atoi(getenv("DOGLEG_GPU_VERBOSE")) > 1;
  struct timespec ts0, ts1, ts2, ts3;
  clock_gettime(CLOCK_MONOTONIC, &ts0);
  dogleg_solverContext_t* ctx = calloc(1, sizeof(*ctx));
  dlb_private_t* pv = calloc(1, sizeof(*pv));
  if(!ctx || !pv) { free(ctx); free(pv); SAY("out of memory"); return -1.0; }
  ctx->cookie = cookie; ctx->lambda = 0.0;
  ctx->Nstate = (int)Nstate; ctx->Nmeasurements = (int)Nmeas;
  ctx->parameters = parameters ? parameters : &global_settings;
  ctx->solve_type = type;
  if(type == DOGLEG_SPARSE)     ctx->f = (dogleg_callback_t*)host_callback;
  else if(type == DOGLEG_DENSE) ctx->f_dense = (dogleg_callback_dense_t*)host_callback;
  else                          ctx->f_dense_products = (dogleg_callback_dense_products_t*)host_callback;
  priv_set(ctx, pv);
  if(gpu_callback)
  {
    pv->device_callbacks = 1;
    if(type == DOGLEG_SPARSE)     pv->f_gpu_sparse   = (dogleg_gpu_callback_sparse_t*)gpu_callback;
    else if(type == DOGLEG_DENSE) pv->f_gpu_dense    = (dogleg_gpu_callback_dense_t*)gpu_callback;
    else                          pv->f_gpu_products = (dogleg_gpu_callback_dense_products_t*)gpu_callback;
  }
  { const char* env = getenv("DOGLEG_GPU_CHECK_PATTERN"); pv->check_pattern = env && atoi(env) != 0; }
  if(type == DOGLEG_SPARSE && pending_perm && pending_perm_n == (int)Nstate)
  {
    pv->user_perm = pending_perm; pending_perm = NULL; pending_perm_n = 0;
    pv->have_user_perm = 1; pv->user_perm_postorder = pending_perm_post;
  }

  if(ctx->parameters->debug_vnlog) vnlog_legend();

  /* nobody can look at the host mirrors of x / J of a device-callback solve unless the context is returned */
  pv->eng = dlb_engine_create3(type, Nstate, Nmeas, NJnnz, ctx->parameters->JtJ_packed, ctx->parameters->JtJ_upper,
                               (gpu_callback && !returnContext) ? DLB_ENGINE_NO_HOST_INPUTS : 0,
                               Nmeas_total, col_begin);
  if(!pv->eng)
  {
    SAY("ERROR: %s", dogleg_gpu_last_error());
    dogleg_freeContext(&ctx);
    return -1.0;
  }
  { const char* env = getenv("DOGLEG_GPU_PHASE_TIMING"); if(env && atoi(env) != 0) dlb_engine_enable_timing(pv->eng, 1); }
  /* device callbacks read p from HBM: no need to bring every trial p to the host */
  dlb_engine_set_lazy_p(pv->eng, pv->device_callbacks);
  if(type != DOGLEG_SPARSE)
  {
    const size_t n = Nstate;
    const size_t sz = (type == DOGLEG_DENSE || ctx->parameters->JtJ_packed) ? n * (n + 1) / 2 : n * n;
    ctx->factorization_dense = calloc(sz ? sz : 1, sizeof(double));
    if(!ctx->factorization_dense) { SAY("Couldn't malloc factorization_dense"); dogleg_freeContext(&ctx); return -1.0; }
  }
  for(int s = 0; s < 2; s++)
  {
    pv->points[s] = make_point(ctx, pv, s, NJnnz);
    if(!pv->points[s]) { SAY("out of memory"); dogleg_freeContext(&ctx); return -1.0; }
  }
  ctx->beforeStep = pv->points[0];
  ctx->afterStep  = pv->points[1];
  if(returnContext) *returnContext = ctx;
  pv->context_returned = returnContext != NULL;

  if(type == DOGLEG_SPARSE && (pv->device_callbacks || Nmeas_total > 0))
  {
    /* the pattern was given up front (device callbacks never write it; a row-sharded solve needs
     * the global one); the host copies hold this process's columns, re-based to 0 */
    for(int s = 0; s < 2 && returnContext && pv->device_callbacks; s++)
    {
      int* hp = pv->points[s]->Jt->p;
      for(unsigned int j = 0; j <= Nmeas; j++) hp[j] = Jp[col_begin + j] - Jp[col_begin];
      memcpy(pv->points[s]->Jt->i, Ji + Jp[col_begin], sizeof(int) * (size_t)NJnnz);
    }
    if(dlb_engine_set_pattern(pv->eng, Jp, Ji, pv->have_user_perm ? pv->user_perm : NULL, pv->user_perm_postorder))
    {
      SAY("could not analyse the Jacobian pattern: %s", dogleg_gpu_last_error());
      if(returnContext) *returnContext = NULL;
      dogleg_freeContext(&ctx);
      return -1.0;
    }
    pv->pattern_set = 1;
  }

  clock_gettime(CLOCK_MONOTONIC, &ts1);
  memcpy(ctx->beforeStep->p, p, Nstate * sizeof(double));
  bool ok = dlb_engine_upload_p(pv->eng, 0) == 0;

  int numsteps = ok ? run_solver(ctx) : -1;
  clock_gettime(CLOCK_MONOTONIC, &ts2);
  const double norm2_x = ctx->beforeStep->norm2_x;
  pv->stats[0] = numsteps;
  if(numsteps < 0 || !publish_results(ctx))
  {
    SAY("ERROR: %s() failed", __func__);
    /* DIVERGENCE: the reference leaks here and leaves *returnContext dangling; we clean up */
    if(returnContext) *returnContext = NULL;
    dogleg_freeContext(&ctx);
    return -1.0;
  }
  memcpy(p, ctx->beforeStep->p, Nstate * sizeof(double));
  SAY_IF_VERBOSE("success! took %d iterations", numsteps);
  if(!returnContext) dogleg_freeContext(&ctx);
  if(verbose_t)
  {
    clock_gettime(CLOCK_MONOTONIC, &ts3);
#define DLB_MS(a, b) (1e3 * (double)((b).tv_sec - (a).tv_sec) + 1e-6 * (double)((b).tv_nsec - (a).tv_nsec))
    fprintf(stderr, "libdogleg-b200: solve timing: setup %.2f ms, iterations %.2f ms, results + teardown %.2f ms\n",
            DLB_MS(ts0, ts1), DLB_MS(ts1, ts2), DLB_MS(ts2, ts3));
  }
  return norm2_x;
}

/* ------------------------------------------------------------- entry points */
double dogleg_optimize2(double* p, unsigned int Nstate, unsigned int Nmeas, unsigned int NJnnz,
                        dogleg_callback_t* f, void* cookie,
                        const dogleg_parameters2_t* parameters, dogleg_solverContext_t** returnContext)
{
  if(NJnnz == 0) { SAY("I must have NJnnz > 0, instead I have %d", NJnnz); return -1.0; }
  if(!f) { SAY("ERROR: exactly one of (f,f_dense,f_dense_products) must be non-NULL"); return -1.0; }
  return optimize_common(p, Nstate, Nmeas, NJnnz, DOGLEG_SPARSE, (void*)f, NULL, NULL, NULL, 0, 0,
                         cookie, parameters, returnContext);
}
double dogleg_optimize(double* p, unsigned int Nstate, unsigned int Nmeas, unsigned int NJnnz,
                       dogleg_callback_t* f, void* cookie, dogleg_solverContext_t** returnContext)
{
  return dogleg_optimize2(p, Nstate, Nmeas, NJnnz, f, cookie, NULL, returnContext);
}
double dogleg_optimize_dense2(double* p, unsigned int Nstate, unsigned int Nmeas,
                              dogleg_callback_dense_t* f, void* cookie,
                              const dogleg_parameters2_t* parameters, dogleg_solverContext_t** returnContext)
{
  if(!f) { SAY("ERROR: exactly one of (f,f_dense,f_dense_products) must be non-NULL"); return -1.0; }
  return optimize_common(p, Nstate, Nmeas, 0, DOGLEG_DENSE, (void*)f, NULL, NULL, NULL, 0, 0,
                         cookie, parameters, returnContext);
}
double dogleg_optimize_dense(double* p, unsigned int Nstate, unsigned int Nmeas,
                             dogleg_callback_dense_t* f, void* cookie, dogleg_solverContext_t** returnContext)
{
  return dogleg_optimize_dense2(p, Nstate, Nmeas, f, cookie, NULL, returnContext);
}
double dogleg_optimize_dense_products(double* p, unsigned int Nstate,
                                      dogleg_callback_dense_products_t* f, void* cookie,
                                      const dogleg_parameters2_t* parameters, dogleg_solverContext_t** returnContext)
{
  if(!f) { SAY("ERROR: exactly one of (f,f_dense,f_dense_products) must be non-NULL"); return -1.0; }
  return optimize_common(p, Nstate, 0, 0, DOGLEG_DENSE_PRODUCTS, (void*)f, NULL, NULL, NULL, 0, 0,
                         cookie, parameters, returnContext);
}
double dogleg_gpu_optimize_sparse(double* p, unsigned int Nstate, unsigned int Nmeas, unsigned int NJnnz,
                                  const int* Jp, const int* Ji,
                                  dogleg_gpu_callback_sparse_t* f, void* cookie,
                                  const dogleg_parameters2_t* parameters, dogleg_solverContext_t** returnContext)
{
  if(NJnnz == 0 || !f || !Jp || !Ji) { SAY("dogleg_gpu_optimize_sparse: need NJnnz>0, a callback and the CCS pattern"); return -1.0; }
  return optimize_common(p, Nstate, Nmeas, NJnnz, DOGLEG_SPARSE, NULL, (void*)f, Jp, Ji, 0, 0,
                         cookie, parameters, returnContext);
}
double dogleg_gpu_optimize_dense(double* p, unsigned int Nstate, unsigned int Nmeas,
                                 dogleg_gpu_callback_dense_t* f, void* cookie,
                                 const dogleg_parameters2_t* parameters, dogleg_solverContext_t** returnContext)
{
  if(!f) { SAY("dogleg_gpu_optimize_dense: need a callback"); return -1.0; }
  return optimize_common(p, Nstate, Nmeas, 0, DOGLEG_DENSE, NULL, (void*)f, NULL, NULL, 0, 0,
                         cookie, parameters, returnContext);
}
double dogleg_gpu_optimize_dense_products(double* p, unsigned int Nstate,
                                          dogleg_gpu_callback_dense_products_t* f, void* cookie,
                                          const dogleg_parameters2_t* parameters, dogleg_solverContext_t** returnContext)
{
  if(returnContext) *returnContext = NULL;
  const dogleg_parameters2_t* P = parameters ? parameters : &global_settings;
  const char* err = NULL;
  if(dogleg_gpu_device_count() <= 0) err = "no CUDA device available: libdogleg-b200 has no CPU fallback";
  else if(!f || !p || Nstate == 0)   err = "dogleg_gpu_optimize_dense_products: need p, Nstate > 0 and a callback";
  /* the reference accepts a packed lower JtJ and fails at the first Cauchy step (dogleg.c:597-601); refuse it
   * before any evaluation instead */
  else if(P->JtJ_packed && !P->JtJ_upper) err = "dogleg_gpu_optimize_dense_products: a packed JtJ must be the upper triangle (JtJ_upper)";
  if(err) { dlb_set_error(err); SAY("ERROR: %s", err); return -1.0; }
  return optimize_common(p, Nstate, 0, 0, DOGLEG_DENSE_PRODUCTS, NULL, (void*)f, NULL, NULL, 0, 0,
                         cookie, parameters, returnContext);
}
double dogleg_gpu_optimize_dense_sharded(double* p, unsigned int Nstate, unsigned int Nmeas_total,
                                         unsigned int row_begin, unsigned int Nmeas_local,
                                         dogleg_callback_dense_t* f_host, dogleg_gpu_callback_dense_t* f_device,
                                         void* cookie, const dogleg_parameters2_t* parameters,
                                         dogleg_solverContext_t** returnContext)
{
  if((!f_host == !f_device) || Nmeas_local == 0 || (unsigned long long)row_begin + Nmeas_local > Nmeas_total)
  { SAY("dogleg_gpu_optimize_dense_sharded: need exactly one callback and a valid, non-empty row range"); return -1.0; }
  return optimize_common(p, Nstate, Nmeas_local, 0, DOGLEG_DENSE, (void*)f_host, (void*)f_device,
                         NULL, NULL, Nmeas_total, row_begin, cookie, parameters, returnContext);
}
double dogleg_gpu_optimize_sparse_sharded(double* p, unsigned int Nstate,
                                          unsigned int Nmeas_total, const int* Jp_global, const int* Ji_global,
                                          unsigned int col_begin, unsigned int Nmeas_local,
                                          dogleg_callback_t* f_host, dogleg_gpu_callback_sparse_t* f_device,
                                          void* cookie, const dogleg_parameters2_t* parameters,
                                          dogleg_solverContext_t** returnContext)
{
  if(!Jp_global || !Ji_global || (!f_host == !f_device) || (unsigned long long)col_begin + Nmeas_local > Nmeas_total)
  { SAY("dogleg_gpu_optimize_sparse_sharded: need the global pattern, one callback and a valid column range"); return -1.0; }
  const unsigned int nnz_local = (unsigned int)(Jp_global[col_begin + Nmeas_local] - Jp_global[col_begin]);
  if(nnz_local == 0) { SAY("dogleg_gpu_optimize_sparse_sharded: this rank has no nonzeros"); return -1.0; }
  return optimize_common(p, Nstate, Nmeas_local, nnz_local, DOGLEG_SPARSE, (void*)f_host, (void*)f_device,
                         Jp_global, Ji_global, Nmeas_total, col_begin, cookie, parameters, returnContext);
}
