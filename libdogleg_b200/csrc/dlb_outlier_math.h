/* dlb_outlier_math.h -- the per-feature outlierness formula of dogleg_getOutliernessFactors (reference
 * dogleg.c:2294-2399), shared by the single-problem path (dogleg_outliers.c, gcc) and the batched kernel
 * (dlb_batched.cu, nvcc) so that both compute the same thing. */
#ifndef DLB_OUTLIER_MATH_H
#define DLB_OUTLIER_MATH_H

#include <math.h>
#include <float.h>
#ifndef __cplusplus
#include <stdbool.h>
#endif

#ifdef __CUDACC__
#define DLB_OUTLIER_HD __host__ __device__
#else
#define DLB_OUTLIER_HD
#endif

/* k = N_ok / (4 (Nstate+1) |x|^2 / (N_ok - Nstate - 1)), kept if already positive (dogleg.c:2381-2399). Every
 * one of the Nmeasurements counts, also those after the last feature. */
DLB_OUTLIER_HD static inline void outlierness_scale(double* scale, int Nmeasurements, int Nstate, int NoutlierFeatures,
                                                    int featureSize, double norm2_x)
{
  if(*scale > 0.0) return;
  const int Nok = Nmeasurements - NoutlierFeatures * featureSize;
  *scale = (double)Nok / (4. * ((double)(Nstate + 1) * norm2_x / (double)(Nok - Nstate - 1)));
}

/* A holds the upper triangle row-first: [a00] or [a00 a01 a11] (dogleg.c:2294-2379). false for a featureSize
 * other than 1 or 2 (the caller reports it). */
DLB_OUTLIER_HD static inline bool outlierness_factor(double* factor, const double* x, const double* A, int featureSize,
                                                     double k)
{
  if(featureSize == 1)
  {
    const double denom = 1.0 - A[0];
    if(fabs(denom) < 1e-8) { *factor = DBL_MAX; return true; }      /* certainly an outlier */
    *factor = x[0] * x[0] / denom;
  }
  else if(featureSize == 2)
  {
    const double det = (1.0 - A[0]) * (1.0 - A[2]) - A[1] * A[1];
    if(fabs(det) < 1e-8) { *factor = DBL_MAX; return true; }
    /* B = inv(A - I) scaled by det; Cook's self+others: x'Bx + |Bx|^2 */
    const double B00 = A[2] - 1.0, B11 = A[0] - 1.0, B01 = -A[1];
    const double xBx = (x[0] * x[0] * B00 + x[0] * x[1] * B01 * 2.0 + x[1] * x[1] * B11) / det;
    const double v1 = x[0] * B00 + x[1] * B01, v2 = x[0] * B01 + x[1] * B11;
    *factor = xBx + (v1 * v1 + v2 * v2) / (det * det);
  }
  else
    return false;
  /* the reference's own "hack": the threshold should be 1 but the scale is divided by 8 (dogleg.c:2373-2375) */
  *factor *= k / 8.;
  return true;
}

#endif
