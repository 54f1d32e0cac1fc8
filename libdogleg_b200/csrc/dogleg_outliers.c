/* dogleg_outliers.c -- outlier / confidence helpers on the device factorization.
 *
 * Reference: dogleg.c:1826-1921 (pseudo-inverse chunks), :2294-2399 (factor and scale),
 * :2401-2791 (dogleg_getOutliernessFactors), :2793-3012 (trace for a hypothetical new feature),
 * :3016-3149 (mark / report). API: dogleg.h:333-392, "experimental" there as here.
 *
 * What is computed, per feature (a group of featureSize consecutive measurements, size 1 or 2):
 *     A = J* inv(JtJ + lambda I) J*'          (featureSize x featureSize, symmetric)
 * and from A, the feature's residuals x* and a scale k the "Cook's self+others" factor of the
 * reference. The only heavy part is inv(JtJ) J*'. Up to 16384 states: inv(JtJ) itself by Nstate
 * right-hand sides on the device factor, then every feature's A in ONE kernel
 * (dlb_engine_outlier_products: no per-chunk copies, solves or synchronisations). Beyond that:
 * multi-right-hand-side solves (dlb_engine_solve) in chunks of OUTLIER_CHUNK measurements (the
 * reference uses chunks of 4 because cholmod_solve works 4 columns at a time).
 *
 * DIVERGENCE: for DOGLEG_DENSE with featureSize == 2 the reference indexes the second row of
 * the feature as J_dense[Nstate*i_measurement + j + k] (dogleg.c:2490), i.e. shifted by one
 * element instead of one row; here the second row is used, so dense and sparse agree.
 */
#define _GNU_SOURCE
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <float.h>
#include "dogleg.h"
#include "dogleg_gpu.h"
#include "dogleg_internal.h"
#include "dlb_outlier_math.h"

#define SAY(fmt, ...) fprintf(stderr, "libdogleg at %s:%d: " fmt "\n", __FILE__, __LINE__, ## __VA_ARGS__)
#define SAY_IF_VERBOSE(fmt, ...) do { if(ctx->parameters->debug && !ctx->parameters->debug_vnlog) SAY(fmt, ## __VA_ARGS__); } while(0)
#define OUTLIER_CHUNK 64
#define OUTLIER_CONFIDENCE_DROP_THRESHOLD 0.05

bool dogleg_getOutliernessFactors(double* factors, double* scale, int featureSize, int Nfeatures,
                                  int NoutlierFeatures, dogleg_operatingPoint_t* point, dogleg_solverContext_t* ctx)
{
  if(!point->have_x) { SAY("%s() needs x, but it isn't available", __func__); return false; }
  if(!point->have_J) { SAY("%s() needs J, but it isn't available", __func__); return false; }
  if(featureSize <= 1) featureSize = 1;
  if(featureSize > 2) { SAY("featureSize > 2 not implemented yet. Got featureSize=%d", featureSize); return false; }
  if(ctx->solve_type == DOGLEG_DENSE_PRODUCTS)
  { SAY("outlierness factors need J: not available for dense-products solves (nor in the reference)"); return false; }
  dlb_private_t* pv = dlb_private_of(ctx);
  if(!pv) { SAY("this context was not created by this library"); return false; }
  if(!point->x || (ctx->solve_type == DOGLEG_SPARSE && !point->Jt->x))
  { SAY("%s() needs the host copies of x and J: keep the context (returnContext) of a host-callback solve", __func__); return false; }
  if(!dogleg_computeJtJfactorization(point, ctx)) return false;

  const int N = ctx->Nstate, M = ctx->Nmeasurements;
  if((long long)Nfeatures * featureSize > M) { SAY("%s(): Nfeatures*featureSize exceeds Nmeasurements", __func__); return false; }
  outlierness_scale(scale, M, N, NoutlierFeatures, featureSize, point->norm2_x);

  bool ok = false;
  double* rhs = NULL; double* sol = NULL;
  /* device path: inv(JtJ) once, then all features in one kernel (dlb_engine_outlier_products) */
  {
    const char* force = getenv("DOGLEG_GPU_OUTLIER_CHUNKED");      /* tests: take the chunked-solve path */
    const int slot = (force && atoi(force) != 0) ? -1 : dlb_slot_of(ctx, point);
    const int npairs = featureSize * (featureSize + 1) / 2;
    double* Aall = slot >= 0 ? malloc(sizeof(double) * (size_t)(Nfeatures > 0 ? Nfeatures : 1) * npairs) : NULL;
    if(Aall)
    {
      const int rc = dlb_engine_outlier_products(pv->eng, slot,
                                                 ctx->solve_type == DOGLEG_SPARSE ? (const int*)point->Jt->p : NULL,
                                                 ctx->solve_type == DOGLEG_SPARSE ? (const int*)point->Jt->i : NULL,
                                                 featureSize, Nfeatures, Aall);
      if(rc == 0)
      {
        ok = true;
        for(int f = 0; f < Nfeatures && ok; f++)
          ok = outlierness_factor(&factors[f], &point->x[(size_t)f * featureSize], Aall + (size_t)f * npairs, featureSize, *scale);
      }
      free(Aall);
      if(rc == 0) return ok;
      if(rc < 0) { SAY("Couldn't compute the outlierness products: %s", dogleg_gpu_last_error()); return false; }
    }
  }
  rhs = malloc(sizeof(double) * (size_t)N * OUTLIER_CHUNK);
  sol = malloc(sizeof(double) * (size_t)N * OUTLIER_CHUNK);
  if(!rhs || !sol) { SAY("out of memory"); goto done; }
  const int*    Jp = ctx->solve_type == DOGLEG_SPARSE ? (const int*)point->Jt->p : NULL;
  const int*    Ji = ctx->solve_type == DOGLEG_SPARSE ? (const int*)point->Jt->i : NULL;
  const double* Jx = ctx->solve_type == DOGLEG_SPARSE ? (const double*)point->Jt->x : NULL;

  const int Mused = Nfeatures * featureSize;
  for(int m0 = 0; m0 < Mused; m0 += OUTLIER_CHUNK)
  {
    const int nc = Mused - m0 < OUTLIER_CHUNK ? Mused - m0 : OUTLIER_CHUNK;
    /* the chunk of Jt, dense: column c = gradient of measurement m0+c */
    if(Jp)
    {
      memset(rhs, 0, sizeof(double) * (size_t)N * nc);
      for(int c = 0; c < nc; c++)
        for(int q = Jp[m0 + c]; q < Jp[m0 + c + 1]; q++) rhs[(size_t)c * N + Ji[q]] = Jx[q];
    }
    else memcpy(rhs, point->J_dense + (size_t)m0 * N, sizeof(double) * (size_t)N * nc);
    if(dlb_engine_solve(pv->eng, rhs, sol, nc)) { SAY("Couldn't compute pinv: %s", dogleg_gpu_last_error()); goto done; }

    for(int c = 0; c + featureSize <= nc; c += featureSize)
    {
      double A[3]; int iA = 0;
      for(int i = 0; i < featureSize; i++)
        for(int j = i; j < featureSize; j++, iA++)
        {
          /* A_ij = (inv(JtJ) j_i) . j_j */
          const double* w = sol + (size_t)(c + i) * N;
          double s = 0.0;
          if(Jp) for(int q = Jp[m0 + c + j]; q < Jp[m0 + c + j + 1]; q++) s += w[Ji[q]] * Jx[q];
          else   { const double* row = point->J_dense + (size_t)(m0 + c + j) * N; for(int k = 0; k < N; k++) s += w[k] * row[k]; }
          A[iA] = s;
        }
      if(!outlierness_factor(&factors[(m0 + c) / featureSize], &point->x[m0 + c], A, featureSize, *scale)) goto done;
    }
  }
  ok = true;
done:
  free(rhs); free(sol);
  return ok;
}

/* dogleg.c:3016-3100 */
bool dogleg_markOutliers(struct dogleg_outliers_t* markedOutliers, double* scale, int* Noutliers,
                         double (getConfidence)(int i_feature_exclude), int featureSize, int Nfeatures,
                         dogleg_operatingPoint_t* point, dogleg_solverContext_t* ctx)
{
  if(featureSize <= 1) featureSize = 1;
  bool markedAny = false;
  double* factors = malloc(sizeof(double) * (Nfeatures > 0 ? Nfeatures : 1));
  if(!factors) { SAY("Error allocating factors"); return false; }
  if(!dogleg_getOutliernessFactors(factors, scale, featureSize, Nfeatures, *Noutliers, point, ctx)) goto done;

  const double confidence0 = getConfidence(-1);
  if(confidence0 < 0.0) goto done;
  SAY_IF_VERBOSE("Initial confidence: %g", confidence0);

  *Noutliers = 0;
  for(int i = 0; i < Nfeatures; i++)
  {
    if(markedOutliers[i].marked) { (*Noutliers)++; continue; }
    if(factors[i] < 1.0) continue;
    const double confidence_excluded = getConfidence(i);
    if(confidence_excluded < 0.0) { free(factors); return false; }
    const double drop = 1.0 - confidence_excluded / confidence0;
    if(drop < OUTLIER_CONFIDENCE_DROP_THRESHOLD)
    {
      markedOutliers[i].marked = true;
      markedAny = true;
      (*Noutliers)++;
      SAY_IF_VERBOSE("Feature %d has outlierness factor %f. Culling produces a confidence: %g. relative loss: %g... YES an outlier; confidence drops little",
                     i, factors[i], confidence_excluded, drop);
    }
    else
      SAY_IF_VERBOSE("Feature %d has outlierness factor %f. Culling produces a confidence: %g. relative loss: %g... NOT an outlier: confidence drops too much",
                     i, factors[i], confidence_excluded, drop);
  }
done:
  free(factors);
  return markedAny;
}

/* dogleg.c:3106-3149 */
void dogleg_reportOutliers(double (getConfidence)(int i_feature_exclude), double* scale, int featureSize,
                           int Nfeatures, int Noutliers, dogleg_operatingPoint_t* point, dogleg_solverContext_t* ctx)
{
  if(featureSize <= 1) featureSize = 1;
  double* factors = malloc(sizeof(double) * (Nfeatures > 0 ? Nfeatures : 1));
  if(!factors) { SAY("Error allocating factors"); return; }
  dogleg_getOutliernessFactors(factors, scale, featureSize, Nfeatures, Noutliers, point, ctx);
  SAY("## Outlier statistics");
  SAY("# i_feature outlier_factor confidence_drop_relative_if_removed");
  const double confidence_full = getConfidence(-1);
  for(int i = 0; i < Nfeatures; i++)
  {
    const double confidence = getConfidence(i);
    SAY("%5d %9.3g %9.3g", i, factors[i], 1.0 - confidence / confidence_full);
  }
  free(factors);
}

/* dogleg.c:2793-3012: k (2 - trace(inv(I + J* inv(JtJ) J*'))) for a hypothetical new 2-measurement
 * feature whose gradients are nonzero only in states [istateActive, istateActive+NstateActive);
 * JqueryFeature is featureSize x NstateActive, row per measurement */
double dogleg_getOutliernessTrace_newFeature_sparse(const double* JqueryFeature, int istateActive, int NstateActive,
                                                    int featureSize, int NoutlierFeatures,
                                                    dogleg_operatingPoint_t* point, dogleg_solverContext_t* ctx)
{
  if(!point->have_x) { SAY("%s() needs x, but it isn't available", __func__); return -1.0; }
  if(!point->have_J) { SAY("%s() needs J, but it isn't available", __func__); return -1.0; }
  if(featureSize != 2) { SAY("%s(): only featureSize == 2 is implemented (as in the reference)", __func__); return -1.0; }
  dlb_private_t* pv = dlb_private_of(ctx);
  if(!pv) { SAY("this context was not created by this library"); return -1.0; }
  const int N = ctx->Nstate;
  if(istateActive < 0 || NstateActive < 0 || istateActive + NstateActive > N) { SAY("%s(): active states out of range", __func__); return -1.0; }
  if(!dogleg_computeJtJfactorization(point, ctx)) return -1.0;

  double* rhs = calloc((size_t)N * 2, sizeof(double));
  double* sol = malloc(sizeof(double) * (size_t)N * 2);
  double result = -1.0;
  if(!rhs || !sol) { SAY("out of memory"); goto done; }
  for(int i = 0; i < 2; i++)
    for(int j = 0; j < NstateActive; j++) rhs[(size_t)i * N + istateActive + j] = JqueryFeature[j + i * NstateActive];
  if(dlb_engine_solve(pv->eng, rhs, sol, 2)) { SAY("%s", dogleg_gpu_last_error()); goto done; }
  double a00 = 0, a01 = 0, a11 = 0;
  for(int j = 0; j < NstateActive; j++)
  {
    a00 += sol[istateActive + j]               * JqueryFeature[j];
    a01 += sol[istateActive + j]               * JqueryFeature[j + NstateActive];
    a11 += sol[(size_t)N + istateActive + j]   * JqueryFeature[j + NstateActive];
  }
  {
    const double iB00 = a00 + 1.0, iB01 = a01, iB11 = a11 + 1.0;
    const double rdet = 1.0 / (iB00 * iB11 - iB01 * iB01);
    const double traceB = iB11 * rdet + iB00 * rdet;
    double scale = -1.0;
    outlierness_scale(&scale, ctx->Nmeasurements, N, NoutlierFeatures, featureSize, point->norm2_x);
    result = scale * (2.0 - traceB);
  }
done:
  free(rhs); free(sol);
  return result;
}
