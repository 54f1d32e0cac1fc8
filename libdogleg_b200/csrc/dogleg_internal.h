/* dogleg_internal.h -- private glue between the C state machine (dogleg_core.c),
 * the engine (dlb_engine.cu) and the symbolic layer. Not installed. */
#pragma once
#include "dogleg.h"
#include "dogleg_gpu.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct dlb_private
{
  dlb_engine_t* eng;
  dogleg_operatingPoint_t* points[2];     /* points[s] lives in engine slot s */
  cholmod_dense gn_header[2];             /* what point->updateGN_cholmoddense points at (sparse) */
  int device_callbacks;
  int context_returned;
  dogleg_gpu_callback_sparse_t* f_gpu_sparse;
  dogleg_gpu_callback_dense_t*  f_gpu_dense;
  dogleg_gpu_callback_dense_products_t* f_gpu_products;
  int pattern_set, pattern_slot, check_pattern;
  int have_user_perm, user_perm_postorder;
  int* user_perm;
  double stats[8];
} dlb_private_t;

dlb_private_t* dlb_private_of(const dogleg_solverContext_t* ctx);

/* dlb_engine.cu */
int  dlb_engine_download_inputs(dlb_engine_t* e, int slot);
void dlb_set_error(const char* msg);
int  dlb_engine_export_factor(dlb_engine_t* e, const int* px, long long xsize, double* x_host);
/* f1 on the device: 0 done, 1 not applicable (caller falls back to chunked solves), -1 error */
int  dlb_engine_outlier_products(dlb_engine_t* e, int slot, const int* Jp, const int* Ji, int featureSize, int nfeatures, double* A_host);
int  dlb_slot_of(const dogleg_solverContext_t* ctx, const dogleg_operatingPoint_t* point);

/* dlb_capi_symbolic.cpp: a host-side cholmod_factor describing the device factor
 * (n, minor, Perm, ColCount, supernodal integer structure; values stay in HBM) */
cholmod_factor* dlb_factor_descriptor_new(const dlb_symbolic_t* S, int n);
void            dlb_factor_descriptor_free(cholmod_factor* L);

#ifdef __cplusplus
}
#endif
