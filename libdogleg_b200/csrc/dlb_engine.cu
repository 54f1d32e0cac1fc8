// dlb_engine.cu -- the device engine behind dogleg_optimize*(): owns HBM and
// pinned host buffers for the two operating points, the symbolic data, the
// multifrontal workspace and one stream; every public dogleg.h entry point is a
// host-side state machine (dogleg_core.c) issuing the dlb_engine_* calls below.
// C-ABI declared in include/dogleg_gpu.h. There is no CPU fallback: without a
// CUDA device dlb_engine_create() fails.
#include "dlb_common.cuh"
#include "dlb_device.h"
#include "dlb_symbolic.h"
#include "dlb_gatherplan.h"
#include "dlb_taskplan.h"
#include "dogleg_gpu.h"
#include <vector>
#include <string>
#include <cstring>
#include <cstdlib>
#include <climits>
#include <algorithm>
#include <type_traits>
#include <mutex>
#include <chrono>
#include <thread>

static_assert(sizeof(DlbScalars) == sizeof(dlb_scalars_t), "scalar block mirrors must agree");
#define DLB_SMALL_FRONT_MAX 158      // r*r doubles must fit in 200 KB of shared memory

// ------------------------------------------------------------------ errors
static thread_local std::string g_last_error;
static int g_device = 0;
extern "C" const char* dogleg_gpu_last_error(void) { return g_last_error.c_str(); }
extern "C" const char* dogleg_gpu_version(void)    { return "libdogleg-b200 0.1 (sm_100a)"; }
extern "C" void dlb_set_error(const char* msg)     { g_last_error = msg ? msg : ""; }
extern "C" int dogleg_gpu_device_count(void)
{
  int n = 0;
  if(cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}
extern "C" int dogleg_gpu_set_device(int device)
{
  if(device < 0 || device >= dogleg_gpu_device_count()) { g_last_error = "no such CUDA device"; return -1; }
  g_device = device;
  return 0;
}
extern "C" int dogleg_gpu_get_device(void) { return g_device; }

#define CU(call) do { cudaError_t _e = (call); if(_e != cudaSuccess) { \
  g_last_error = std::string(#call) + ": " + cudaGetErrorString(_e); \
  fprintf(stderr, "libdogleg-b200: CUDA error at %s:%d: %s\n", __FILE__, __LINE__, g_last_error.c_str()); \
  return -1; } } while(0)

// -------------------------------------------------------------------- NCCL
// Row-sharded solves (SURVEY.md 8e): every rank holds a contiguous block of measurement columns,
// forms its partial Jt*x, |x|^2, |J v|^2 and partial (unfactored) fronts, and the partials are
// summed with ncclAllReduce over NVLink; the tiny factorization / solve / step then run
// redundantly on every rank, so no broadcast of the step is needed and all ranks walk the same
// path bit for bit (NCCL delivers identical sums to all ranks). libnccl is loaded at run time so
// that single-GPU users do not need it.
#include <dlfcn.h>
typedef struct { char internal[128]; } dlb_ncclUniqueId;
typedef void* dlb_ncclComm_t;
static struct
{
  void* lib = 0;
  int (*GetUniqueId)(dlb_ncclUniqueId*) = 0;
  int (*CommInitRank)(dlb_ncclComm_t*, int, dlb_ncclUniqueId, int) = 0;
  int (*AllReduce)(const void*, void*, size_t, int, int, dlb_ncclComm_t, cudaStream_t) = 0;
  int (*AllGather)(const void*, void*, size_t, int, dlb_ncclComm_t, cudaStream_t) = 0;
  int (*Broadcast)(const void*, void*, size_t, int, int, dlb_ncclComm_t, cudaStream_t) = 0;
  int (*GroupStart)() = 0;
  int (*GroupEnd)() = 0;
  int (*CommDestroy)(dlb_ncclComm_t) = 0;
  const char* (*GetErrorString)(int) = 0;
  dlb_ncclComm_t comm = 0;
  int rank = 0, world = 1;
} g_nccl;
static int nccl_load()
{
  if(g_nccl.lib) return 0;
  const char* names[] = { "libnccl.so.2", "libnccl.so" };
  for(const char* n : names) { g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if(g_nccl.lib) break; }
  if(!g_nccl.lib) { g_last_error = "cannot load libnccl.so.2"; return -1; }
  g_nccl.GetUniqueId  = (int (*)(dlb_ncclUniqueId*))dlsym(g_nccl.lib, "ncclGetUniqueId");
  g_nccl.CommInitRank = (int (*)(dlb_ncclComm_t*, int, dlb_ncclUniqueId, int))dlsym(g_nccl.lib, "ncclCommInitRank");
  g_nccl.AllReduce    = (int (*)(const void*, void*, size_t, int, int, dlb_ncclComm_t, cudaStream_t))dlsym(g_nccl.lib, "ncclAllReduce");
  g_nccl.AllGather    = (int (*)(const void*, void*, size_t, int, dlb_ncclComm_t, cudaStream_t))dlsym(g_nccl.lib, "ncclAllGather");
  g_nccl.Broadcast    = (int (*)(const void*, void*, size_t, int, int, dlb_ncclComm_t, cudaStream_t))dlsym(g_nccl.lib, "ncclBroadcast");
  g_nccl.GroupStart   = (int (*)())dlsym(g_nccl.lib, "ncclGroupStart");
  g_nccl.GroupEnd     = (int (*)())dlsym(g_nccl.lib, "ncclGroupEnd");
  g_nccl.CommDestroy  = (int (*)(dlb_ncclComm_t))dlsym(g_nccl.lib, "ncclCommDestroy");
  g_nccl.GetErrorString = (const char* (*)(int))dlsym(g_nccl.lib, "ncclGetErrorString");
  if(!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy ||
     !g_nccl.AllGather || !g_nccl.Broadcast || !g_nccl.GroupStart || !g_nccl.GroupEnd)
  { g_last_error = "libnccl is missing symbols"; return -1; }
  return 0;
}
extern "C" int dogleg_gpu_nccl_get_unique_id(unsigned char id[128])
{
  if(nccl_load()) return -1;
  dlb_ncclUniqueId u;
  if(g_nccl.GetUniqueId(&u) != 0) { g_last_error = "ncclGetUniqueId failed"; return -1; }
  memcpy(id, u.internal, 128);
  return 0;
}
extern "C" int dogleg_gpu_nccl_init(int rank, int world, const unsigned char id[128])
{
  if(nccl_load()) return -1;
  if(g_nccl.comm) { g_nccl.CommDestroy(g_nccl.comm); g_nccl.comm = 0; }
  if(cudaSetDevice(g_device) != cudaSuccess) { g_last_error = "cudaSetDevice failed"; return -1; }
  dlb_ncclUniqueId u;
  memcpy(u.internal, id, 128);
  const int rc = g_nccl.CommInitRank(&g_nccl.comm, world, u, rank);
  if(rc != 0) { g_last_error = std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "failed"); g_nccl.comm = 0; return -1; }
  g_nccl.rank = rank; g_nccl.world = world;
  return 0;
}
extern "C" void dogleg_gpu_nccl_finalize(void)
{
  if(g_nccl.comm) { g_nccl.CommDestroy(g_nccl.comm); g_nccl.comm = 0; }
  g_nccl.rank = 0; g_nccl.world = 1;
}
extern "C" int dogleg_gpu_nccl_world(void) { return g_nccl.comm ? g_nccl.world : 1; }

// ------------------------------------------------------------------ engine
struct Slot
{
  double *h_p = 0, *h_x = 0, *h_Jtx = 0, *h_cauchy = 0, *h_gn = 0, *h_step = 0, *h_J = 0;
  int    *h_Jp = 0, *h_Ji = 0;
  double *d_p = 0, *d_x = 0, *d_Jtx = 0, *d_cauchy = 0, *d_gn = 0, *d_step = 0, *d_J = 0;
  double norm2_x = 0;
  // sparse: the class blocks of Jt*Jt' formed from this slot's Jacobian (one buffer per operating point: the
  // fused evaluation forms them for every point, and a rejected trial must not clobber the blocks of the
  // point the next trial starts from), and what the fused trial kernel caches per point
  double* d_G = 0; bool have_G = false;
  double norm2_Jtx = 0, norm2_cauchy = 0, norm2_gn = 0; bool have_cauchy = false, have_gn = false;
};

struct dlb_engine
{
  int type = 0, N = 0, M = 0, packed = 0, upper = 0, device = 0, sm_count = DLB_SM_COUNT_FALLBACK;
  unsigned int nnz = 0;
  size_t Jcount = 0;
  cudaStream_t st = 0;
  // host-callback solves: x and the Jacobian values travel on a side stream (pinned cudaMemcpyAsync), in pieces
  // while the callback is still writing if it announces its progress (dogleg_gpu_host_progress)
  cudaStream_t st_copy = 0; cudaEvent_t ev_copy = 0, ev_idle = 0;
  Slot slot[2];
  DlbScalars* d_sc = 0;
  dlb_scalars_t* h_sc = 0;                 // = &h_pub->sc
  // mapped pinned block the fused kernels publish the scalars into (then the sequence number: the
  // host spins on it instead of a D2H copy + stream synchronisation)
  DlbPublished* h_pub = 0; DlbPublished* d_pub = 0; unsigned long long seq = 0;
  double* d_part = 0; unsigned int* d_counter = 0;
  long long* d_minor = 0; long long* h_minor = 0;
  // sparse
  DlbSymbolic* sym = 0;
  DlbSparseDev S{}; DlbFrontDev F{};
  std::vector<void*> dev_allocs;
  std::vector<int> level_ptr;
  std::vector<long long> level_gt_ptr;     // gather targets by level: [2l,2l+1) pass 1 (chunks), [2l+1,2l+2) pass 2
  std::vector<long long> level_tmp_size;   // doubles of heavy-front temporaries used by each level
  std::vector<long long> level_sg_ptr;     // the same ranges for the forward-solve gather
  bool any_solve_gather = false;
  // per level the fronts are ordered small first: [level_ptr[l], level_mid[l]) fit in shared memory,
  // [level_mid[l], level_ptr[l+1]) go through the blocked tensor-core path (dlb_bigfront.cu)
  std::vector<int> level_mid;
  std::vector<std::vector<DlbBigFront>> level_big;
  std::vector<int> level_big_ptr, level_big_max_r, level_big_max_nc;   // offsets into d_big_descs per level
  const DlbBigFront* d_big_descs = 0;
  int* d_big_cnt = 0;                      // per large front: tiles that have loaded the current diagonal block
  double* d_biginv = 0;                    // inverted diagonal blocks of the large fronts (DlbBigFront::inv_off)
  const long long* d_big_part_off = 0; double* d_big_partial = 0;   // dlb_bigsolve.cu: backward partial sums of the large fronts
  int max_small_rows = 0;
  int max_front_rows = 0, max_front_cols = 0;
  // per level: max rows of the shared-memory fronts, max rows / pivot columns of all fronts
  // (kernel shapes are chosen per level: a million 39-row leaf fronts must not be launched with
  // the shared memory of the biggest front of the tree)
  std::vector<int> level_small_rows, level_rows, level_cols;
  // the first nleaf fronts of level 0 are handled by the warp-per-front kernels of dlb_leaf.cu
  int nleaf = 0, leaf_max_rows = 0;
  bool leaf_mma = false;                   // every fused leaf has <= 4 pivots: tensor-core leaf kernel
  int leaf_max_pairs = 0;                  // most measurement columns of a fused leaf front
  double *d_gpart = 0, *d_n2part = 0, *d_jvpart = 0, *d_fronts = 0, *d_ywork = 0, *d_zperm = 0;
  bool G_shared = false;                   // both slots alias one class-block buffer (nothing reads it per point)
  bool G_global = false;                   // row-sharded + fused: the class blocks are all-reduced, everything after the evaluation is rank-local
  long long Goff_total = 0;
  // fused evaluation (gradient + class blocks in one pass over Jt) / persistent trial kernel (dlb_trial.cu)
  bool fused_eval = false, fused_trial = false;
  int trial_grid = 0;
  const int* d_level_ptr = 0; const long long *d_level_gt = 0, *d_level_sg = 0, *d_level_tmp = 0;
  double* d_trial_part = 0; unsigned int* d_bar = 0;
  unsigned int trial_parity = 0; bool minor_dirty = true;    // which of the two failure-flag slots the next trial launch uses
  const int *d_eg_ptr = 0, *d_eg_sptr = 0, *d_eg_src = 0; const unsigned int* d_eg_dst = 0;   // element lists of the fronts
  unsigned long long* d_prof = 0;          // DOGLEG_GPU_TRIAL_PROF=1: phase time stamps of the trial kernel
  double *d_rhs = 0; int rhs_cap = 0;
  // row sharding: this engine holds measurement columns [col_begin, col_begin + M) of M_total
  bool sharded = false; int M_total = 0, col_begin = 0;
  // "gather" flavour of a row-sharded solve (large sparse problems, whose fronts are far bigger
  // than their Jacobian): every rank evaluates its slice of x / Jt values into a FULL-size device
  // buffer, the slices are exchanged (one ncclBroadcast per rank and array, grouped), and
  // everything downstream runs replicated on the full problem -- bit-identical to one GPU. What
  // is shared out is the callback work and, with host callbacks, the PCIe transfer.
  bool gather = false;
  long long slice_off = 0;                 // first value of this rank's slice in the full value array
  std::vector<long long> rank_cb, rank_m, rank_off, rank_nnz;   // the slices of all ranks
  double* d_fronts_asm = 0;                // all-reduced assembled (unfactored) fronts
  double n_allreduce = 0, allreduce_bytes = 0;
  bool pattern_set = false;
  bool pattern_verified = false;           // a cached engine must re-check the pattern it was built for
  bool host_inputs = true;                 // pinned mirrors of x / Jacobian / pattern exist
  std::vector<int> pat_sample;             // strided sample of (Jp, Ji) + the injected permutation, for re-use checks
  unsigned long long pat_hash = 0;         // hash of the whole pattern the analysis was made for
  std::vector<int> pat_full_p, pat_full_i; // full copies when DOGLEG_GPU_CHECK_PATTERN=1
  std::vector<int> perm_used; int postorder_used = 0;
  // dense
  double *d_work = 0, *d_xAx = 0;
  // bookkeeping
  int factor_slot = -1; double factor_lambda = 0;
  int asm_slot = 0;                        // slot whose Jacobian the current factorization is built from
  bool jv_quad = true;                     // |Jv|^2 as v'(JtJ)v from the slot's class blocks instead of a pass over Jt
  bool lazy_p = false;                     // device callbacks: p goes to the host on request only, not after every step
  double n_launch = 0, n_h2d = 0, n_d2h = 0, n_factor = 0;
  bool timing = false; double phase_ms[8] = {0};
  cudaEvent_t ev0 = 0, ev1 = 0;
};

template<class T> static int dev_upload(dlb_engine* e, const std::vector<T>& v, const T** out)
{
  T* d = 0;
  const size_t bytes = std::max<size_t>(v.size(), 1) * sizeof(T);
  CU(cudaMalloc(&d, bytes));
  e->dev_allocs.push_back(d);
  if(!v.empty()) CU(cudaMemcpyAsync(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, e->st));
  *out = d;
  return 0;
}
template<class T> static int dev_alloc(dlb_engine* e, size_t count, T** out)
{
  T* d = 0;
  CU(cudaMalloc(&d, std::max<size_t>(count, 1) * sizeof(T)));
  e->dev_allocs.push_back(d);
  *out = d;
  return 0;
}

// descriptors of the large fronts, level after level, for the batched tensor-core kernels
static int upload_big_descs(dlb_engine* e)
{
  std::vector<DlbBigFront> all;
  const size_t nlev = e->level_big.size();
  e->level_big_ptr.assign(nlev + 1, 0); e->level_big_max_r.assign(nlev, 0); e->level_big_max_nc.assign(nlev, 0);
  for(size_t l = 0; l < nlev; l++)
  {
    for(const DlbBigFront& b : e->level_big[l])
    {
      all.push_back(b);
      e->level_big_max_r[l] = std::max(e->level_big_max_r[l], b.r);
      e->level_big_max_nc[l] = std::max(e->level_big_max_nc[l], b.nc);
    }
    e->level_big_ptr[l+1] = (int)all.size();
  }
  // scratch of the backward solve: per large front nchunk x nc partial sums, levels reuse one buffer
  std::vector<long long> part_off(all.size(), 0);
  long long need = 1;
  for(size_t l = 0; l < nlev; l++)
  {
    long long off = 0;
    for(int q = e->level_big_ptr[l]; q < e->level_big_ptr[l+1]; q++)
    {
      part_off[q] = off;
      off += dlb_bigsolve_partial_size(all[q].r, all[q].nc);
    }
    need = std::max(need, off);
  }
  // inverted 64 x 64 diagonal blocks of every large front (dlb_bigfront.cu writes them, dlb_bigsolve.cu multiplies by them)
  long long inv_total = 0;
  for(DlbBigFront& b : all) { b.inv_off = inv_total; inv_total += (long long)((b.nc + 63) / 64) * 8192; }
  int rc = dev_upload(e, all, &e->d_big_descs);
  rc |= dev_alloc(e, (size_t)std::max<long long>(inv_total, 1), &e->d_biginv);
  rc |= dev_alloc(e, all.size() + 1, &e->d_big_cnt);
  if(!rc) CU(cudaMemsetAsync(e->d_big_cnt, 0, sizeof(int) * (all.size() + 1), e->st));
  rc |= dev_upload(e, part_off, &e->d_big_part_off);
  rc |= dev_alloc(e, (size_t)need, &e->d_big_partial);
  return rc;
}

struct PhaseTimer
{
  dlb_engine* e; int phase;
  PhaseTimer(dlb_engine* e_, int ph) : e(e_), phase(ph) { if(e->timing) cudaEventRecord(e->ev0, e->st); }
  ~PhaseTimer()
  {
    if(!e->timing) return;
    cudaEventRecord(e->ev1, e->st); cudaEventSynchronize(e->ev1);
    float ms = 0; cudaEventElapsedTime(&ms, e->ev0, e->ev1);
    e->phase_ms[phase] += ms;
  }
};

static int sync_scalars(dlb_engine* e)
{
  CU(cudaMemcpyAsync(e->h_sc, e->d_sc, sizeof(DlbScalars), cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  e->n_d2h += sizeof(DlbScalars);
  return 0;
}

// wait until the fused kernels have published sequence number e->seq (mapped pinned memory)
static int wait_published(dlb_engine* e)
{
  volatile unsigned long long* q = &e->h_pub->seq;
  for(unsigned long spin = 0;; spin++)
  {
    if(*q == e->seq) break;
    if((spin & 0xfff) == 0xfff)
    { // a failed launch or a faulting kernel must not hang the host
      const cudaError_t rc = cudaStreamQuery(e->st);
      if(rc == cudaSuccess) { if(*q == e->seq) break; g_last_error = "the device finished without publishing its results"; return -1; }
      if(rc != cudaErrorNotReady) { g_last_error = std::string("device error: ") + cudaGetErrorString(rc); return -1; }
    }
  }
  __sync_synchronize();
  e->n_d2h += sizeof(DlbScalars);
  return 0;
}

// ---- idle-engine cache: repeated solves of the same shape (outlier-rejection loops,
// benchmarks) skip pinned/device allocation and, if the pattern is unchanged, the
// symbolic analysis. DOGLEG_GPU_ENGINE_CACHE=0 disables it.
extern "C" void dlb_trial_dbg_dump();
static std::mutex g_pool_mu;
static std::vector<dlb_engine*> g_pool;
static const size_t POOL_MAX = 2;
static bool cache_enabled()
{
  const char* env = getenv("DOGLEG_GPU_ENGINE_CACHE");
  return !(env && atoi(env) == 0);
}
static void engine_free(dlb_engine* e);
extern "C" void dogleg_gpu_release_batched_cache(void);
extern "C" void dogleg_gpu_release_cache(void)
{
  dogleg_gpu_release_batched_cache();
  std::vector<dlb_engine*> victims;
  { std::lock_guard<std::mutex> lk(g_pool_mu); victims.swap(g_pool); }
  for(dlb_engine* e : victims) engine_free(e);
}

// in-place sum over the ranks of a sharded solve (FP64), on the engine's stream
static int allreduce_sum(dlb_engine* e, double* d_buf, size_t count)
{
  if(!e->sharded || g_nccl.world <= 1) return 0;
  if(!g_nccl.comm) { g_last_error = "sharded engine without dogleg_gpu_nccl_init()"; return -1; }
  const int rc = g_nccl.AllReduce(d_buf, d_buf, count, /*ncclFloat64*/ 8, /*ncclSum*/ 0, g_nccl.comm, e->st);
  if(rc != 0) { g_last_error = std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "failed"); return -1; }
  e->n_allreduce += 1; e->allreduce_bytes += 8.0 * count;
  return 0;
}
extern "C" void dlb_engine_comm_stats(const dlb_engine_t* e, double out[2]) { out[0] = e->n_allreduce; out[1] = e->allreduce_bytes; }

extern "C" dlb_engine_t* dlb_engine_create(int solve_type, unsigned int Nstate, unsigned int Nmeas,
                                           unsigned int NJnnz, int packed, int upper)
{
  return dlb_engine_create2(solve_type, Nstate, Nmeas, NJnnz, packed, upper, 0);
}

extern "C" dlb_engine_t* dlb_engine_create2(int solve_type, unsigned int Nstate, unsigned int Nmeas,
                                            unsigned int NJnnz, int packed, int upper, int flags)
{
  return dlb_engine_create3(solve_type, Nstate, Nmeas, NJnnz, packed, upper, flags, 0, 0);
}

// Nmeas / NJnnz are the LOCAL counts; Nmeas_total > 0 declares a row-sharded engine holding the
// measurement columns [col_begin, col_begin + Nmeas) of Nmeas_total
static dlb_engine_t* engine_create_impl(int solve_type, unsigned int Nstate, unsigned int Nmeas,
                                        unsigned int NJnnz, int packed, int upper, int flags,
                                        unsigned int Nmeas_total, unsigned int col_begin);
extern "C" dlb_engine_t* dlb_engine_create3(int solve_type, unsigned int Nstate, unsigned int Nmeas,
                                            unsigned int NJnnz, int packed, int upper, int flags,
                                            unsigned int Nmeas_total, unsigned int col_begin)
{
  dlb_engine_t* e = engine_create_impl(solve_type, Nstate, Nmeas, NJnnz, packed, upper, flags, Nmeas_total, col_begin);
  if(!e && g_last_error.find("out of memory") != std::string::npos)
  { // idle cached engines (multi-GB at bundle-adjustment scale) must not starve a differently shaped problem
    dogleg_gpu_release_cache();
    cudaGetLastError();
    e = engine_create_impl(solve_type, Nstate, Nmeas, NJnnz, packed, upper, flags, Nmeas_total, col_begin);
  }
  return e;
}
static dlb_engine_t* engine_create_impl(int solve_type, unsigned int Nstate, unsigned int Nmeas,
                                        unsigned int NJnnz, int packed, int upper, int flags,
                                        unsigned int Nmeas_total, unsigned int col_begin)
{
  const bool want_sharded = Nmeas_total > 0;
  if(want_sharded && (solve_type == DOGLEG_DENSE_PRODUCTS || (unsigned long long)col_begin + Nmeas > Nmeas_total))
  { g_last_error = "sharded engine: bad column range or solve type"; return NULL; }
  if(dogleg_gpu_device_count() <= 0)
  {
    g_last_error = "no CUDA device available: libdogleg-b200 has no CPU fallback";
    return NULL;
  }
  if(cudaSetDevice(g_device) != cudaSuccess) { g_last_error = "cudaSetDevice failed"; return NULL; }
  const bool want_host_inputs = !(flags & DLB_ENGINE_NO_HOST_INPUTS);
  if(cache_enabled())
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    for(size_t i = 0; i < g_pool.size(); i++)
    {
      dlb_engine* c = g_pool[i];
      if(c->type == solve_type && c->N == (int)Nstate && c->M == (int)Nmeas && c->nnz == NJnnz &&
         c->packed == packed && c->upper == upper && c->device == g_device &&
         (c->host_inputs || !want_host_inputs) && (c->sharded || c->gather) == want_sharded &&
         (!want_sharded || (c->M_total == (int)Nmeas_total && c->col_begin == (int)col_begin)))
      {
        g_pool.erase(g_pool.begin() + i);
        c->factor_slot = -1; c->factor_lambda = 0; c->lazy_p = false;
        for(int sl = 0; sl < 2; sl++) { c->slot[sl].have_G = c->slot[sl].have_cauchy = c->slot[sl].have_gn = false; }
        c->n_launch = c->n_h2d = c->n_d2h = c->n_factor = 0;
        c->timing = false; memset(c->phase_ms, 0, sizeof(c->phase_ms));
        memset(c->h_sc, 0, sizeof(*c->h_sc));
        c->pattern_verified = false;
        c->n_allreduce = c->allreduce_bytes = 0;
        return c;
      }
    }
  }
  dlb_engine* e = new dlb_engine();
  e->host_inputs = want_host_inputs;
  { const char* jp = getenv("DOGLEG_GPU_JV_PASS"); e->jv_quad = !(jp && atoi(jp) != 0); }
  e->sharded = want_sharded; e->M_total = want_sharded ? (int)Nmeas_total : (int)Nmeas; e->col_begin = (int)col_begin;
  {
    // reduce (sum partial fronts) or gather (exchange Jacobian slices): gather when the state is large
    const char* sm = getenv("DOGLEG_GPU_SHARD_MODE");
    const bool want_gather = sm ? !strcmp(sm, "gather") : Nstate >= 16384;
    if(want_sharded && solve_type == DOGLEG_SPARSE && want_gather) { e->gather = true; e->sharded = false; }
  }
  e->type = solve_type; e->N = (int)Nstate; e->M = (int)Nmeas; e->nnz = NJnnz;
  e->packed = packed; e->upper = upper; e->device = g_device;
  cudaDeviceProp prop;
  if(cudaGetDeviceProperties(&prop, g_device) == cudaSuccess) e->sm_count = prop.multiProcessorCount;
  const size_t N = e->N, M = e->M;
  if(solve_type == DOGLEG_SPARSE)              e->Jcount = NJnnz;
  else if(solve_type == DOGLEG_DENSE)          e->Jcount = M * N;
  else                                         e->Jcount = packed ? N * (N + 1) / 2 : N * N;

  auto fail = [&](const char* what) { g_last_error = what; engine_free(e); return (dlb_engine_t*)NULL; };
  if(cudaStreamCreateWithFlags(&e->st, cudaStreamNonBlocking) != cudaSuccess) return fail("cudaStreamCreate failed");
  cudaEventCreate(&e->ev0); cudaEventCreate(&e->ev1);
  if(cudaStreamCreateWithFlags(&e->st_copy, cudaStreamNonBlocking) != cudaSuccess) return fail("cudaStreamCreate failed");
  cudaEventCreateWithFlags(&e->ev_copy, cudaEventDisableTiming); cudaEventCreateWithFlags(&e->ev_idle, cudaEventDisableTiming);
  bool ok = true;
  auto hostalloc = [&](size_t count, auto** out) {
    typedef typename std::remove_reference<decltype(**out)>::type T;
    void* p = 0;
    const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
    if(cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { ok = false; p = 0; }
    else memset(p, 0, bytes);
    *out = static_cast<T*>(p);
  };
  auto devalloc = [&](size_t count, auto** out) {
    typedef typename std::remove_reference<decltype(**out)>::type T;
    void* p = 0;
    if(cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T)) != cudaSuccess) { ok = false; p = 0; }
    *out = static_cast<T*>(p);
  };
  for(int s = 0; s < 2; s++)
  {
    Slot& L = e->slot[s];
    hostalloc(N, &L.h_p); hostalloc(N, &L.h_Jtx); hostalloc(N, &L.h_cauchy); hostalloc(N, &L.h_gn); hostalloc(N, &L.h_step);
    devalloc(N, &L.d_p);  devalloc(N + 1, &L.d_Jtx);  devalloc(N, &L.d_cauchy);  devalloc(N, &L.d_gn);  devalloc(N, &L.d_step);
    if(solve_type != DOGLEG_DENSE_PRODUCTS) { if(e->host_inputs) hostalloc(M, &L.h_x); if(!e->gather) devalloc(M, &L.d_x); }
    if(e->host_inputs) hostalloc(e->Jcount, &L.h_J);
    // +16 bytes: the bulk copies of the range kernels read 16-byte aligned supersets. Gather mode: the
    // full-size buffers are allocated once the global pattern is known (set_pattern)
    if(!e->gather) devalloc(e->Jcount + 2, &L.d_J);
    if(solve_type == DOGLEG_SPARSE && e->host_inputs) { hostalloc(M + 1, &L.h_Jp); hostalloc(NJnnz, &L.h_Ji); }
  }
  {
    void* hp = 0; void* dpub = 0;
    if(cudaHostAlloc(&hp, sizeof(DlbPublished), cudaHostAllocMapped) != cudaSuccess) ok = false;
    else
    {
      memset(hp, 0, sizeof(DlbPublished));
      e->h_pub = (DlbPublished*)hp; e->h_sc = (dlb_scalars_t*)&e->h_pub->sc;
      if(cudaHostGetDevicePointer(&dpub, hp, 0) != cudaSuccess) ok = false;
      e->d_pub = (DlbPublished*)dpub;
    }
  }
  devalloc(1, &e->d_sc);
  hostalloc(1, &e->h_minor); devalloc(2, &e->d_minor);
  devalloc(5 * (size_t)e->sm_count * 8 + 64, &e->d_part);
  devalloc(4, &e->d_counter);
  if(!ok) return fail("out of memory allocating operating-point buffers");
  cudaMemsetAsync(e->d_counter, 0, 4 * sizeof(unsigned int), e->st);
  cudaMemsetAsync(e->d_sc, 0, sizeof(DlbScalars), e->st);

  if(solve_type != DOGLEG_SPARSE)
  {
    // the whole matrix is one front
    std::vector<int> sn_first{0, e->N}, rows_ptr{0, e->N}, rows(N), rel(N, -1), sn_parent{-1},
                     child_ptr{0, 0}, child_list, fptr{0, 0}, flist, ctask{0}, level_sn{0}, perm(N);
    std::vector<long long> front_off{0, (long long)(N * N)};
    for(size_t i = 0; i < N; i++) { rows[i] = (int)i; perm[i] = (int)i; }
    DlbFrontDev& F = e->F;
    F.n = e->N; F.nsuper = 1; F.ytot = (long long)N;
    int rc = 0;
    rc |= dev_upload(e, sn_first, &F.sn_first);   rc |= dev_upload(e, rows_ptr, &F.rows_ptr);
    rc |= dev_upload(e, rows, &F.rows);           rc |= dev_upload(e, rel, &F.rel);
    rc |= dev_upload(e, sn_parent, &F.sn_parent); rc |= dev_upload(e, child_ptr, &F.child_ptr);
    rc |= dev_upload(e, child_list, &F.child_list); rc |= dev_upload(e, front_off, &F.front_off);
    rc |= dev_upload(e, fptr, &F.fcls_ptr);       rc |= dev_upload(e, flist, &F.fcls_list);
    rc |= dev_upload(e, ctask, &F.cls_task_ptr);  rc |= dev_upload(e, level_sn, &F.level_sn);
    rc |= dev_upload(e, perm, &F.perm);
    e->level_ptr = {0, 1};
    e->max_front_rows = e->N; e->max_front_cols = e->N;
    e->level_big.assign(1, {});
    if(e->N > DLB_SMALL_FRONT_MAX) { e->level_mid = {0}; e->level_big[0].push_back({0, e->N, e->N, 0, 0}); e->max_small_rows = 0; }
    else                           { e->level_mid = {1}; e->max_small_rows = e->N; }
    e->level_small_rows = {e->max_small_rows}; e->level_rows = {e->N}; e->level_cols = {e->N};
    rc |= upload_big_descs(e);
    const int nblk = std::max(1, std::min((e->M + 63) / 64, e->sm_count * 4));
    size_t work = (size_t)nblk * (N + 1) + 16;
    if(solve_type == DOGLEG_DENSE) work = std::max(work, dlb_dense_syrk_work_size(e->M, e->N, e->sm_count));
    rc |= dev_alloc(e, N * N + 128, &e->d_fronts);
    rc |= dev_alloc(e, work, &e->d_work);
    rc |= dev_alloc(e, (size_t)2048, &e->d_xAx);
    rc |= dev_alloc(e, N, &e->d_ywork);
    rc |= dev_alloc(e, N, &e->d_zperm);
    if(rc) return fail("out of memory allocating dense workspace");
    e->pattern_set = true;
  }
  if(cudaStreamSynchronize(e->st) != cudaSuccess) return fail("device initialisation failed");
  return e;
}

extern "C" void dlb_engine_destroy(dlb_engine_t* e)
{
  if(!e) return;
  if(cache_enabled() && e->st && e->pattern_set)
  {
    cudaSetDevice(e->device);
    // an engine whose stream is in an error state (a failed launch, a faulting kernel) is not reused
    if(cudaStreamSynchronize(e->st) != cudaSuccess || cudaGetLastError() != cudaSuccess) { engine_free(e); return; }
    dlb_engine* evicted = NULL;
    {
      std::lock_guard<std::mutex> lk(g_pool_mu);
      g_pool.push_back(e);
      if(g_pool.size() > POOL_MAX) { evicted = g_pool.front(); g_pool.erase(g_pool.begin()); }
    }
    if(evicted) engine_free(evicted);
    return;
  }
  engine_free(e);
}

static void engine_free(dlb_engine* e)
{
  if(!e) return;
  cudaSetDevice(e->device);
  if(e->st) cudaStreamSynchronize(e->st);
  for(int s = 0; s < 2; s++)
  {
    Slot& L = e->slot[s];
    void* hs[] = {L.h_p, L.h_x, L.h_Jtx, L.h_cauchy, L.h_gn, L.h_step, L.h_J, L.h_Jp, L.h_Ji};
    void* ds[] = {L.d_p, L.d_x, L.d_Jtx, L.d_cauchy, L.d_gn, L.d_step, L.d_J};
    for(void* p : hs) if(p) cudaFreeHost(p);
    for(void* p : ds) if(p) cudaFree(p);
  }
  if(e->h_pub) cudaFreeHost(e->h_pub);
  if(e->h_minor) cudaFreeHost(e->h_minor);
  void* ds[] = {e->d_sc, e->d_minor, e->d_part, e->d_counter, e->d_rhs};
  for(void* p : ds) if(p) cudaFree(p);
  for(void* p : e->dev_allocs) cudaFree(p);
  if(e->ev0) cudaEventDestroy(e->ev0);
  if(e->ev1) cudaEventDestroy(e->ev1);
  if(e->ev_copy) cudaEventDestroy(e->ev_copy);
  if(e->ev_idle) cudaEventDestroy(e->ev_idle);
  if(e->st_copy) cudaStreamDestroy(e->st_copy);
  if(e->st) cudaStreamDestroy(e->st);
  delete e->sym;
  delete e;
}

extern "C" void* dlb_engine_host_buffer(dlb_engine_t* e, int s, int which)
{
  Slot& L = e->slot[s & 1];
  switch(which)
  {
  case DLB_BUF_P: return L.h_p;       case DLB_BUF_X: return L.h_x;     case DLB_BUF_JTX: return L.h_Jtx;
  case DLB_BUF_CAUCHY: return L.h_cauchy; case DLB_BUF_GN: return L.h_gn; case DLB_BUF_STEP: return L.h_step;
  case DLB_BUF_JVALUES: return L.h_J; case DLB_BUF_JP: return L.h_Jp;   case DLB_BUF_JI: return L.h_Ji;
  }
  return NULL;
}
extern "C" void* dlb_engine_device_buffer(dlb_engine_t* e, int s, int which)
{
  Slot& L = e->slot[s & 1];
  switch(which)
  {
  case DLB_BUF_P: return L.d_p;       case DLB_BUF_JTX: return L.d_Jtx;
  case DLB_BUF_CAUCHY: return L.d_cauchy; case DLB_BUF_GN: return L.d_gn; case DLB_BUF_STEP: return L.d_step;
  // gather mode: this rank's slice inside the full-size arrays
  case DLB_BUF_X:       return L.d_x ? L.d_x + (e->gather ? e->col_begin : 0) : NULL;
  case DLB_BUF_JVALUES: return L.d_J ? L.d_J + (e->gather ? e->slice_off : 0) : NULL;
  // the entry behind the gradient (d_Jtx holds N + 1); dense-products engines are never sharded, which is
  // the only other use of it
  case DLB_BUF_NORM2X:  return e->type == DOGLEG_DENSE_PRODUCTS ? L.d_Jtx + e->N : NULL;
  }
  return NULL;
}
// exhaustive comparison of a pattern with the one this engine was analysed for (DOGLEG_GPU_CHECK_PATTERN=1
// keeps full copies); 1 = equal, 0 = different, -1 = no copy kept
extern "C" int dlb_engine_pattern_equals(const dlb_engine_t* e, const int* Jp, const int* Ji)
{
  if(e->pat_full_p.empty()) return -1;
  const size_t np = e->pat_full_p.size(), ni = e->pat_full_i.size();
  if((size_t)(unsigned int)Jp[np - 1] != ni) return 0;
  return !memcmp(e->pat_full_p.data(), Jp, sizeof(int) * np) && !memcmp(e->pat_full_i.data(), Ji, sizeof(int) * ni) ? 1 : 0;
}
extern "C" void* dlb_engine_stream(dlb_engine_t* e) { return (void*)e->st; }
extern "C" const dlb_scalars_t* dlb_engine_scalars(const dlb_engine_t* e) { return e->h_sc; }
extern "C" const dlb_symbolic_t* dlb_engine_symbolic(const dlb_engine_t* e) { return (const dlb_symbolic_t*)e->sym; }
extern "C" void dlb_engine_counters(const dlb_engine_t* e, double out[4])
{ out[0] = e->n_launch; out[1] = e->n_h2d; out[2] = e->n_d2h; out[3] = e->n_factor; }
extern "C" void dlb_engine_enable_timing(dlb_engine_t* e, int on) { e->timing = on != 0; memset(e->phase_ms, 0, sizeof(e->phase_ms)); }
extern "C" void dlb_engine_phase_ms(const dlb_engine_t* e, double out[8]) { memcpy(out, e->phase_ms, sizeof(e->phase_ms)); }

// 64-bit hash of the whole CCS pattern (column pointers, then row indices), four threads over the big
// array: the identity of what a cached symbolic analysis was computed for. A strided sample (round 1)
// lets a few re-associated observations between two solves slip through and silently reuses a stale
// analysis; hashing costs ~2 ms per 100 MB of pattern.
static inline unsigned long long hash_mix(unsigned long long h, unsigned long long v)
{
  h ^= v + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
  return h * 0xff51afd7ed558ccdull;
}
static unsigned long long hash_ints(const int* a, size_t n, unsigned long long seed)
{
  unsigned long long h0 = seed, h1 = seed ^ 0x1234567ull, h2 = seed ^ 0x89abcdefull, h3 = seed ^ 0x5555aaaaull;
  size_t i = 0;
  for(; i + 8 <= n; i += 8)
  {
    unsigned long long v[4];
    memcpy(v, a + i, 32);
    h0 = hash_mix(h0, v[0]); h1 = hash_mix(h1, v[1]); h2 = hash_mix(h2, v[2]); h3 = hash_mix(h3, v[3]);
  }
  for(; i < n; i++) h0 = hash_mix(h0, (unsigned long long)(unsigned int)a[i]);
  return hash_mix(hash_mix(h0, h1), hash_mix(h2, h3));
}
static unsigned long long pattern_hash(const int* Jp, size_t np, const int* Ji, size_t ni)
{
  const int NTH = ni > (1u << 22) ? 4 : 1;
  unsigned long long part[4] = {0, 0, 0, 0};
  std::vector<std::thread> th;
  for(int t = 1; t < NTH; t++)
    th.emplace_back([&, t]() { const size_t a = ni * t / NTH, b = ni * (t + 1) / NTH; part[t] = hash_ints(Ji + a, b - a, 0xabcdull + t); });
  part[0] = hash_ints(Ji, ni / NTH, 0xabcdull);
  for(auto& x : th) x.join();
  unsigned long long h = hash_ints(Jp, np, 0x77ull);
  for(int t = 0; t < NTH; t++) h = hash_mix(h, part[t]);
  return hash_mix(h, (unsigned long long)ni);
}
// Callers that guarantee an unchanged pattern from solve to solve (the benchmark; an outlier-rejection
// loop over one problem) can skip the hash: the cheap sample of both arrays is compared instead.
static thread_local int g_trust_pattern = -1;
extern "C" void dogleg_gpu_assume_pattern_unchanged(int on) { g_trust_pattern = on ? 1 : 0; }
static bool trust_pattern()
{
  if(g_trust_pattern >= 0) return g_trust_pattern != 0;
  const char* env = getenv("DOGLEG_GPU_TRUST_PATTERN");
  return env && atoi(env) != 0;
}

// ------------------------------------------------------------ set_pattern
extern "C" int dlb_engine_set_pattern(dlb_engine_t* e, const int* Jp, const int* Ji,
                                      const int* perm_or_null, int postorder)
{
  if(e->type != DOGLEG_SPARSE) return 0;
  if(e->pattern_set && e->pattern_verified) return 0;
  cudaSetDevice(e->device);
  if(!Jp) { Jp = e->slot[0].h_Jp; Ji = e->slot[0].h_Ji; }
  if(!Jp || !Ji) { g_last_error = "set_pattern: no pattern given"; return -1; }
  // Jp/Ji describe all M_total columns (the global pattern when row-sharded); this engine's values
  // cover the columns [col_begin, col_begin + M)
  const int Mtot = e->M_total, cb = e->col_begin;
  if((unsigned int)(Jp[cb + e->M] - Jp[cb]) > e->nnz) { g_last_error = "the pattern has more nonzeros than NJnnz"; return -1; }

  // sample of the pattern (+ ordering request) that identifies what this engine was analysed for
  const char* env = getenv("DOGLEG_GPU_CHECK_PATTERN");
  const bool full_check = env && atoi(env) != 0;
  std::vector<int> sample;
  {
    auto take = [&](const int* a, size_t len) {
      const size_t stride = std::max<size_t>(1, len / 4096);
      sample.push_back((int)len);
      for(size_t i = 0; i < len; i += stride) sample.push_back(a[i]);
      for(size_t i = 0; i < std::min<size_t>(len, 64); i++) { sample.push_back(a[i]); sample.push_back(a[len - 1 - i]); }
    };
    take(Jp, (size_t)Mtot + 1);
    take(Ji, (size_t)(unsigned int)Jp[Mtot]);
  }
  std::vector<int> perm_req;
  if(perm_or_null) perm_req.assign(perm_or_null, perm_or_null + e->N);
  if(e->pattern_set)
  {
    bool same = sample == e->pat_sample && perm_req == e->perm_used && (perm_req.empty() || postorder == e->postorder_used);
    // the whole pattern decides (hash), unless the caller vouches for it
    if(same && !trust_pattern()) same = pattern_hash(Jp, (size_t)Mtot + 1, Ji, (size_t)(unsigned int)Jp[Mtot]) == e->pat_hash;
    if(same && full_check)
      same = e->pat_full_p.size() == (size_t)Mtot + 1 && !memcmp(e->pat_full_p.data(), Jp, sizeof(int) * ((size_t)Mtot + 1)) &&
             !memcmp(e->pat_full_i.data(), Ji, sizeof(int) * e->pat_full_i.size());
    if(same) { e->pattern_verified = true; return 0; }
    // a different pattern: drop everything derived from the old one
    CU(cudaStreamSynchronize(e->st));
    for(void* q : e->dev_allocs) cudaFree(q);
    e->dev_allocs.clear();
    delete e->sym; e->sym = 0;
    e->pattern_set = false;
    e->d_gpart = e->d_n2part = e->d_jvpart = e->d_fronts = e->d_ywork = e->d_zperm = 0;
    e->slot[0].d_G = e->slot[1].d_G = 0; e->slot[0].have_G = e->slot[1].have_G = false;
    e->fused_eval = e->fused_trial = false; e->d_trial_part = 0; e->d_bar = 0; e->d_prof = 0;
  }
  e->pat_sample.swap(sample);
  e->pat_hash = pattern_hash(Jp, (size_t)Mtot + 1, Ji, (size_t)(unsigned int)Jp[Mtot]);
  e->perm_used.swap(perm_req); e->postorder_used = postorder;
  if(full_check) { e->pat_full_p.assign(Jp, Jp + Mtot + 1); e->pat_full_i.assign(Ji, Ji + (unsigned int)Jp[Mtot]); }
  else { e->pat_full_p.clear(); e->pat_full_i.clear(); }
  e->sym = new DlbSymbolic();
  const bool verbose = getenv("DOGLEG_GPU_VERBOSE") && atoi(getenv("DOGLEG_GPU_VERBOSE")) != 0;
  const auto t_begin = std::chrono::steady_clock::now();
  if(!dlb_symbolic_analyze(*e->sym, e->N, Mtot, Jp, Ji, perm_or_null, postorder != 0))
  { g_last_error = "malformed Jt pattern (indices must be ascending and in range)"; return -1; }
  const DlbSymbolic& Y = *e->sym;
  const auto t_sym = std::chrono::steady_clock::now();
  // entry offsets inside a front are 32-bit (row + col * r)
  if(Y.max_front_rows > 46340) { g_last_error = "a front has more than 46340 rows: not supported"; return -1; }

  // gather mode: the kernels see the FULL problem (all columns, values at their global positions)
  const int cbk = e->gather ? 0 : cb, Mk = e->gather ? Mtot : e->M;
  if(e->gather)
  {
    // full-size device buffers of both operating points, the slice table of all ranks
    const size_t nnz_full = (size_t)(unsigned int)Jp[Mtot];
    for(int sl = 0; sl < 2; sl++)
    {
      Slot& L = e->slot[sl];
      if(L.d_x) cudaFree(L.d_x);
      if(L.d_J) cudaFree(L.d_J);
      L.d_x = L.d_J = 0;
      CU(cudaMalloc(&L.d_x, sizeof(double) * std::max<size_t>(Mtot, 1)));
      CU(cudaMalloc(&L.d_J, sizeof(double) * (nnz_full + 2)));
    }
    e->slice_off = Jp[cb];
    const int world = g_nccl.comm ? g_nccl.world : 1, rank = g_nccl.comm ? g_nccl.rank : 0;
    std::vector<long long> mine{(long long)cb, (long long)e->M}, all(2 * (size_t)world, 0);
    if(world > 1)
    {
      long long* d_tab = 0;
      CU(cudaMalloc(&d_tab, sizeof(long long) * 2 * (size_t)(world + 1)));
      CU(cudaMemcpyAsync(d_tab, mine.data(), sizeof(long long) * 2, cudaMemcpyHostToDevice, e->st));
      if(g_nccl.AllGather(d_tab, d_tab + 2, 2, /*ncclInt64*/ 4, g_nccl.comm, e->st) != 0)
      { cudaFree(d_tab); g_last_error = "ncclAllGather of the slice table failed"; return -1; }
      CU(cudaMemcpyAsync(all.data(), d_tab + 2, sizeof(long long) * 2 * world, cudaMemcpyDeviceToHost, e->st));
      CU(cudaStreamSynchronize(e->st));
      cudaFree(d_tab);
    }
    else all = mine;
    (void)rank;
    e->rank_cb.assign(world, 0); e->rank_m.assign(world, 0); e->rank_off.assign(world, 0); e->rank_nnz.assign(world, 0);
    for(int r = 0; r < world; r++)
    {
      e->rank_cb[r] = all[2*r]; e->rank_m[r] = all[2*r+1];
      if(e->rank_cb[r] < 0 || e->rank_cb[r] + e->rank_m[r] > Mtot) { g_last_error = "inconsistent column ranges across the ranks"; return -1; }
      e->rank_off[r] = Jp[e->rank_cb[r]];
      e->rank_nnz[r] = Jp[e->rank_cb[r] + e->rank_m[r]] - Jp[e->rank_cb[r]];
    }
  }
  // tasks, range tasks and the inverse map of the gradient reduction: dlb_taskplan.cpp
  // Fused evaluation (default for unsharded solves and the gather flavour): gradient, |x|^2 and the
  // class blocks of Jt*Jt' in ONE pass over the Jacobian values; the partial gradients then come one
  // block per class task, so the plan is built without range tasks. DOGLEG_GPU_FUSED=0: the round-1
  // schedule (separate gradient pass over range tasks, class blocks on demand).
  {
    const char* fe = getenv("DOGLEG_GPU_FUSED");
    e->fused_eval = e->jv_quad && !(fe && atoi(fe) == 0);
    // Row-sharded (reduce flavour): one task per class on every rank, so the class blocks and the partial
    // gradients have the same layout everywhere and ONE grouped all-reduce per evaluation
    // ([class blocks | Jt*x | |x|^2]) gives every rank the complete blocks: both quadratic forms, the front
    // assembly, the factorization and the step are then rank-local and identical on all ranks.
    e->G_global = e->sharded && e->fused_eval;
  }
  DlbTaskPlan TP;
  {
    const char* renv = getenv("DOGLEG_GPU_RANGE");
    dlb_build_task_plan(Y, Jp, cbk, Mk, e->N, e->sm_count, !e->fused_eval && !(renv && atoi(renv) == 0), TP, e->G_global);
  }
  const std::vector<int>& task_cls = TP.task_cls; const std::vector<int>& task_m0 = TP.task_m0;
  const std::vector<int>& task_m1 = TP.task_m1;   const std::vector<int>& cls_task_ptr = TP.cls_task_ptr;
  const std::vector<long long>& task_goff = TP.task_goff; const std::vector<long long>& task_Goff = TP.task_Goff;
  const std::vector<int>& lmem_col = TP.mem_col;  const std::vector<unsigned int>& mem_pos = TP.mem_pos;
  const std::vector<int>& big_tasks = TP.big_tasks; const std::vector<int>& small_tasks = TP.small_tasks;
  const std::vector<DlbRangeTask>& rtasks = TP.rtasks; const std::vector<int>& gj_big_tasks = TP.gj_big_tasks;
  const std::vector<int>& gp_count = TP.gp_count;
  const std::vector<int>& ginv_ptr = TP.ginv_ptr; const std::vector<int>& ginv_cls = TP.ginv_cls;
  const std::vector<long long>& ginv_off = TP.ginv_off;
  const std::vector<int>& heavy_state = TP.heavy_state; const std::vector<int>& medium_state = TP.medium_state;
  const int ntasks = (int)task_cls.size(), range_kmax = TP.range_kmax, heavy_threshold = TP.heavy_threshold;
  const long long goff = TP.goff, Goff = TP.Goff;

  DlbSparseDev& S = e->S; DlbFrontDev& F = e->F;
  S.nheavy = (int)heavy_state.size(); S.heavy_threshold = heavy_threshold; S.nmedium = (int)medium_state.size();
  S.n = e->N; S.m = Mk; S.ncls = Y.ncls; S.ntasks = ntasks;
  S.nbig = (int)big_tasks.size(); S.nsmall = (int)small_tasks.size();
  S.nrange = (int)rtasks.size(); S.range_kmax = range_kmax; S.ngj_big = (int)gj_big_tasks.size();
  const std::vector<int>& mem_col_local = lmem_col;
  F.n = e->N; F.nsuper = Y.nsuper; F.ytot = (long long)Y.rows.size();
  int rc = 0;
  rc |= dev_upload(e, Y.cls_ptr, &S.cls_ptr);     rc |= dev_upload(e, Y.cls_rows, &S.cls_rows);
  rc |= dev_upload(e, Y.cls_loc, &S.cls_loc);     rc |= dev_upload(e, Y.cls_front, &S.cls_front);
  rc |= dev_upload(e, task_cls, &S.task_cls);     rc |= dev_upload(e, task_m0, &S.task_m0);
  rc |= dev_upload(e, task_m1, &S.task_m1);       rc |= dev_upload(e, task_goff, &S.task_goff);
  rc |= dev_upload(e, task_Goff, &S.task_Goff);   rc |= dev_upload(e, mem_col_local, &S.mem_col);
  rc |= dev_upload(e, mem_pos, &S.mem_pos);       rc |= dev_upload(e, ginv_ptr, &S.ginv_ptr);
  rc |= dev_upload(e, ginv_cls, &S.ginv_cls);     rc |= dev_upload(e, ginv_off, &S.ginv_off);
  rc |= dev_upload(e, heavy_state, &S.heavy_state); rc |= dev_upload(e, medium_state, &S.medium_state);
  rc |= dev_upload(e, big_tasks, &S.big_tasks);   rc |= dev_upload(e, small_tasks, &S.small_tasks);
  rc |= dev_upload(e, rtasks, &S.rtasks);         rc |= dev_upload(e, gj_big_tasks, &S.gj_big_tasks);
  rc |= dev_upload(e, gp_count, &S.gp_count);
  {
    std::vector<DlbSmallTask> info(small_tasks.size());
    int kmax = 1;
    for(size_t i = 0; i < small_tasks.size(); i++)
    {
      const int t = small_tasks[i], c = task_cls[t];
      info[i] = {Y.cls_ptr[c+1] - Y.cls_ptr[c], task_m0[t], task_m1[t] - task_m0[t], Y.cls_ptr[c], task_goff[t], task_Goff[t]};
      kmax = std::max(kmax, info[i].k);
    }
    S.small_group = kmax <= 8 ? 8 : (kmax <= 16 ? 16 : 32);
    rc |= dev_upload(e, info, &S.small_info);
  }
  rc |= dev_upload(e, Y.sn_first, &F.sn_first);   rc |= dev_upload(e, Y.rows_ptr, &F.rows_ptr);
  rc |= dev_upload(e, Y.rows, &F.rows);           rc |= dev_upload(e, Y.rel, &F.rel);
  rc |= dev_upload(e, Y.sn_parent, &F.sn_parent); rc |= dev_upload(e, Y.child_ptr, &F.child_ptr);
  rc |= dev_upload(e, Y.child_list, &F.child_list);
  { std::vector<long long> fo(Y.front_off.begin(), Y.front_off.end()); rc |= dev_upload(e, fo, &F.front_off); }
  rc |= dev_upload(e, Y.fcls_ptr, &F.fcls_ptr);   rc |= dev_upload(e, Y.fcls_list, &F.fcls_list);
  rc |= dev_upload(e, cls_task_ptr, &F.cls_task_ptr);
  S.cls_task_ptr = F.cls_task_ptr;
  {
    std::vector<int> level_sn(Y.level_sn);
    e->level_mid.assign(Y.nlevels, 0);
    e->level_big.assign(Y.nlevels, {});
    e->max_small_rows = 0;
    e->level_small_rows.assign(Y.nlevels, 0); e->level_rows.assign(Y.nlevels, 0); e->level_cols.assign(Y.nlevels, 0);
    // leaf fronts for the fused warp-per-front kernels: no children, at most 48 rows and 8 pivot
    // columns, every class a single small task of at most 4 member columns
    e->nleaf = 0; e->leaf_max_rows = 0; e->leaf_max_pairs = 0;
    std::vector<char> cls_fused(Y.ncls, 0);
    if(!e->sharded && Y.nlevels > 0)
    {
      auto eligible = [&](int sn) {
        const int r = Y.rows_ptr[sn+1] - Y.rows_ptr[sn], nc = Y.sn_first[sn+1] - Y.sn_first[sn];
        if(r > 48 || nc > 8 || Y.child_ptr[sn+1] != Y.child_ptr[sn]) return false;
        if(Y.fcls_ptr[sn+1] - Y.fcls_ptr[sn] > 32) return false;
        int npair = 0, nvals = 0, nlocs = 0;         // limits of dlb_leaf.cu
        for(int ci = Y.fcls_ptr[sn]; ci < Y.fcls_ptr[sn+1]; ci++)
        {
          const int c = Y.fcls_list[ci];
          if(cls_task_ptr[c+1] - cls_task_ptr[c] != 1) return false;
          const int t = cls_task_ptr[c];
          const int nm = task_m1[t] - task_m0[t], k = Y.cls_ptr[c+1] - Y.cls_ptr[c];
          if(k > 32) return false;
          npair += nm; nvals += nm * k; nlocs += k;
        }
        return npair <= 32 && nvals <= 256 && nlocs <= 128;
      };
      auto mid0 = std::stable_partition(level_sn.begin() + Y.level_ptr[0], level_sn.begin() + Y.level_ptr[1], eligible);
      e->nleaf = (int)(mid0 - (level_sn.begin() + Y.level_ptr[0]));
      const char* lm = getenv("DOGLEG_GPU_LEAF_MIN");
      if(e->nleaf < (lm ? atoi(lm) : 1024)) e->nleaf = 0;          // not worth a separate path
      { const char* lm2 = getenv("DOGLEG_GPU_LEAF_MMA"); e->leaf_mma = !(lm2 && atoi(lm2) == 0); }
      for(int q = Y.level_ptr[0]; q < Y.level_ptr[0] + e->nleaf; q++)
      {
        const int sn = level_sn[q];
        e->leaf_max_rows = std::max(e->leaf_max_rows, Y.rows_ptr[sn+1] - Y.rows_ptr[sn]);
        if(Y.sn_first[sn+1] - Y.sn_first[sn] > 4) e->leaf_mma = false;
        int np = 0;
        for(int ci = Y.fcls_ptr[sn]; ci < Y.fcls_ptr[sn+1]; ci++) { const int t = cls_task_ptr[Y.fcls_list[ci]]; np += task_m1[t] - task_m0[t]; }
        e->leaf_max_pairs = std::max(e->leaf_max_pairs, np);
        for(int ci = Y.fcls_ptr[sn]; ci < Y.fcls_ptr[sn+1]; ci++) cls_fused[Y.fcls_list[ci]] = 1;
      }
    }
    {
      std::vector<DlbLeaf> leaf(e->nleaf);
      for(int i = 0; i < e->nleaf; i++)
      {
        const int sn = level_sn[Y.level_ptr[0] + i];
        leaf[i] = {(long long)Y.front_off[sn], Y.sn_first[sn], Y.sn_first[sn+1] - Y.sn_first[sn],
                   Y.rows_ptr[sn+1] - Y.rows_ptr[sn], Y.rows_ptr[sn], Y.fcls_ptr[sn], Y.fcls_ptr[sn+1] - Y.fcls_ptr[sn]};
      }
      rc |= dev_upload(e, leaf, &F.leaf);
      // flat records for k_leaf_fronts_mma (strides = maxima over the leaves)
      int ps = 1, lw = 1;
      for(int i = 0; i < e->nleaf; i++)
      {
        const int sn = level_sn[Y.level_ptr[0] + i];
        int np = 0, nl = 0;
        for(int ci = Y.fcls_ptr[sn]; ci < Y.fcls_ptr[sn+1]; ci++)
        { const int c = Y.fcls_list[ci], t = cls_task_ptr[c]; np += task_m1[t] - task_m0[t]; nl += Y.cls_ptr[c+1] - Y.cls_ptr[c]; }
        ps = std::max(ps, np); lw = std::max(lw, (nl + 3) / 4);
      }
      F.leaf_ps = ps; F.leaf_lw = lw; F.leaf_max_nc = 0;
      for(int i = 0; i < e->nleaf; i++)
      { const int sn = level_sn[Y.level_ptr[0] + i]; F.leaf_max_nc = std::max(F.leaf_max_nc, Y.sn_first[sn+1] - Y.sn_first[sn]); }
      std::vector<unsigned int> lpos((size_t)e->nleaf * ps, 0u), lkl((size_t)e->nleaf * ps, 0u), lloc((size_t)e->nleaf * lw, 0u);
      for(int i = 0; i < e->nleaf && e->leaf_mma; i++)
      {
        const int sn = level_sn[Y.level_ptr[0] + i];
        int np = 0, nl = 0;
        unsigned char* lb = (unsigned char*)(lloc.data() + (size_t)i * lw);
        for(int ci = Y.fcls_ptr[sn]; ci < Y.fcls_ptr[sn+1]; ci++)
        {
          const int c = Y.fcls_list[ci], t = cls_task_ptr[c], k = Y.cls_ptr[c+1] - Y.cls_ptr[c];
          for(int m = task_m0[t]; m < task_m1[t]; m++, np++)
          { lpos[(size_t)i * ps + np] = mem_pos[m]; lkl[(size_t)i * ps + np] = (unsigned)k | ((unsigned)nl << 8); }
          for(int l = 0; l < k; l++) lb[nl + l] = (unsigned char)Y.cls_loc[Y.cls_ptr[c] + l];
          nl += k;
        }
      }
      if(!e->leaf_mma) { lpos.clear(); lkl.clear(); lloc.clear(); }
      rc |= dev_upload(e, lpos, &F.leaf_pos); rc |= dev_upload(e, lkl, &F.leaf_kl); rc |= dev_upload(e, lloc, &F.leaf_loc);
      std::vector<DlbClsInfo> cinfo(Y.ncls);
      for(int c = 0; c < Y.ncls; c++)
      {
        const int t = cls_task_ptr[c];
        cinfo[c] = {Y.cls_ptr[c+1] - Y.cls_ptr[c], t < ntasks ? task_m0[t] : 0,
                    (t < ntasks && t < cls_task_ptr[c+1]) ? task_m1[t] - task_m0[t] : 0, Y.cls_ptr[c]};
      }
      rc |= dev_upload(e, cinfo, &S.cls_info);
    }
    {
      std::vector<int> asm_small;
      std::vector<DlbSmallTask> fused_info;
      for(int t : small_tasks)
      {
        const int c = task_cls[t];
        if(!cls_fused[c]) asm_small.push_back(t);
        else fused_info.push_back({Y.cls_ptr[c+1] - Y.cls_ptr[c], task_m0[t], task_m1[t] - task_m0[t], Y.cls_ptr[c], task_goff[t], task_Goff[t]});
      }
      S.nasm_small = (int)asm_small.size(); S.nfused = (int)fused_info.size();
      rc |= dev_upload(e, asm_small, &S.asm_small_tasks);
      rc |= dev_upload(e, fused_info, &S.fused_info);
    }
    for(int l = 0; l < Y.nlevels; l++)
    {
      auto rows_of = [&](int sn) { return Y.rows_ptr[sn+1] - Y.rows_ptr[sn]; };
      const int lbeg = Y.level_ptr[l] + (l == 0 ? e->nleaf : 0);
      for(int q = Y.level_ptr[l]; q < Y.level_ptr[l+1]; q++)
      {
        const int sn = level_sn[q];
        if(q < lbeg) continue;                      // fused leaves do not shape the ordinary kernels
        e->level_rows[l] = std::max(e->level_rows[l], rows_of(sn));
        e->level_cols[l] = std::max(e->level_cols[l], Y.sn_first[sn+1] - Y.sn_first[sn]);
        if(rows_of(sn) <= DLB_SMALL_FRONT_MAX) e->level_small_rows[l] = std::max(e->level_small_rows[l], rows_of(sn));
      }
      std::stable_partition(level_sn.begin() + lbeg, level_sn.begin() + Y.level_ptr[l+1],
                            [&](int sn) { return rows_of(sn) <= DLB_SMALL_FRONT_MAX; });
      int mid = lbeg;
      while(mid < Y.level_ptr[l+1] && rows_of(level_sn[mid]) <= DLB_SMALL_FRONT_MAX)
      { e->max_small_rows = std::max(e->max_small_rows, rows_of(level_sn[mid])); mid++; }
      e->level_mid[l] = mid;
      for(int q = mid; q < Y.level_ptr[l+1]; q++)
      {
        const int sn = level_sn[q];
        e->level_big[l].push_back({(long long)Y.front_off[sn], rows_of(sn), Y.sn_first[sn+1] - Y.sn_first[sn], Y.sn_first[sn], sn});
      }
    }
    rc |= dev_upload(e, level_sn, &F.level_sn);
    rc |= upload_big_descs(e);
  }
  rc |= dev_upload(e, Y.perm, &F.perm);
  long long pool_tmp = 0, pool_scratch = 0;        // doubles behind the fronts: temporaries, gather scratch
  long long solve_scratch = 0;                     // doubles behind the rows of the solve work vector
  {
    // extend-add and forward-solve gathers of the heavy / large fronts: dlb_gatherplan.cpp
    DlbGatherParams GP;
    GP.small_front_max = DLB_SMALL_FRONT_MAX;
    // small trees (the persistent trial kernel): a few hundred targets for thousands of resident warps, and a target
    // costs its warp ~2 500 cycles per 8 sources x 128 entries (scattered sector loads) -- cut the blocks into
    // strips of 32 entries, four times as many warps share the work. Large trees stream gigabytes through the
    // gather: there the descriptor overhead per byte decides, 128-entry strips stay.
    if(Y.max_front_rows <= DLB_SMALL_FRONT_MAX && e->nleaf == 0) GP.gtile = 32;
    DlbGatherPlan plan;
    dlb_build_gather_plan(Y, GP, plan);
    e->level_gt_ptr = plan.level_gt_ptr; e->level_sg_ptr = plan.level_sg_ptr; e->level_tmp_size = plan.level_tmp_size;
    pool_tmp = plan.pool_tmp; pool_scratch = plan.pool_scratch; solve_scratch = plan.solve_scratch;
    rc |= dev_upload(e, plan.heavy_tmp_off, &F.heavy_tmp_off);
    rc |= dev_upload(e, plan.sg_flag, &F.sg_flag);
    auto upload = [&](DlbGatherList& B, DlbGather& G) {
      int r2 = 0;
      r2 |= dev_upload(e, B.dst, &G.dst);         r2 |= dev_upload(e, B.ld, &G.ld);
      r2 |= dev_upload(e, B.h, &G.h);             r2 |= dev_upload(e, B.w, &G.w);
      r2 |= dev_upload(e, B.src_ptr, &G.src_ptr); r2 |= dev_upload(e, B.gs_base, &G.gs_base);
      r2 |= dev_upload(e, B.gs_ld, &G.gs_ld);
      return r2;
    };
    rc |= upload(plan.fronts, F.fg); rc |= upload(plan.solve, F.sg);
    F.ytot = (long long)Y.rows.size() + solve_scratch;
    e->any_solve_gather = !plan.solve.dst.empty();
  }
  rc |= dev_alloc(e, (size_t)goff, &e->d_gpart);  rc |= dev_alloc(e, (size_t)std::max(ntasks, dlb_sparse_n2part_size(S, e->sm_count)), &e->d_n2part);
  rc |= dev_alloc(e, (size_t)ntasks, &e->d_jvpart);
  // class blocks per operating point; one shared buffer when no kernel reads them per point (every
  // class assembled by the fused leaf kernel: the blocks only exist for elements-only test passes)
  e->G_shared = S.nbig + S.nasm_small == 0;
  e->Goff_total = Goff;
  rc |= dev_alloc(e, (size_t)Goff, &e->slot[0].d_G);
  if(e->G_shared) e->slot[1].d_G = e->slot[0].d_G; else rc |= dev_alloc(e, (size_t)Goff, &e->slot[1].d_G);
  e->slot[0].have_G = e->slot[1].have_G = false;
  // one pool: [fronts | temporaries of the small heavy fronts | gather scratch]
  // + 128: the bulk copies of the big-front GEMM read 16-byte aligned supersets of 64-row column segments
  rc |= dev_alloc(e, (size_t)(Y.front_off[Y.nsuper] + pool_tmp + pool_scratch) + 128, &e->d_fronts);
  F.heavy_tmp = e->d_fronts ? e->d_fronts + Y.front_off[Y.nsuper] : 0;
  if(e->sharded) rc |= dev_alloc(e, (size_t)Y.front_off[Y.nsuper], &e->d_fronts_asm);
  rc |= dev_alloc(e, (size_t)F.ytot, &e->d_ywork);
  rc |= dev_alloc(e, (size_t)e->N, &e->d_zperm);
  if(rc) { g_last_error = "out of device memory for the symbolic structure / fronts"; return -1; }
  e->level_ptr = Y.level_ptr;
  e->max_front_rows = Y.max_front_rows;
  e->max_front_cols = 0;
  for(int sn = 0; sn < Y.nsuper; sn++) e->max_front_cols = std::max(e->max_front_cols, Y.sn_first[sn+1] - Y.sn_first[sn]);
  // The persistent trial kernel (dlb_trial.cu) takes the whole step between two evaluations when every
  // front fits in shared memory and no leaf kernels are involved. Its grid is a pure function of the
  // problem and the device: the partial sums (and with them the last bits of the results) depend on it.
  e->fused_trial = false;
  {
    const char* ft = getenv("DOGLEG_GPU_FUSED_TRIAL");
    bool can = e->fused_eval && !e->gather && e->nleaf == 0 && Y.nlevels > 0 && Y.nlevels <= 256 &&
               Y.max_front_rows <= DLB_SMALL_FRONT_MAX && !(ft && atoi(ft) == 0);
    for(size_t l = 0; can && l < e->level_big.size(); l++) if(!e->level_big[l].empty()) can = false;
    if(can)
    {
      const int limit = dlb_trial_max_grid(Y.max_front_rows, e->sm_count);
      int want = e->sm_count;
      for(int l = 0; l < Y.nlevels; l++) want = std::max(want, Y.level_ptr[l+1] - Y.level_ptr[l]);
      want = std::max(want, (S.nbig + S.nasm_small + dlb_trial_threads(Y.max_front_rows) / 32 - 1) / (dlb_trial_threads(Y.max_front_rows) / 32));
      e->trial_grid = std::min(limit, std::min(want, 4 * e->sm_count));
      if(e->trial_grid >= 1)
      {
        std::vector<long long> lgt(e->level_gt_ptr), lsg(e->level_sg_ptr), ltmp(e->level_tmp_size);
        lgt.resize(2 * (size_t)Y.nlevels + 1, 0); lsg.resize(2 * (size_t)Y.nlevels + 1, 0); ltmp.resize((size_t)Y.nlevels, 0);
        int r2 = 0;
        r2 |= dev_upload(e, Y.level_ptr, &e->d_level_ptr);
        r2 |= dev_upload(e, lgt, &e->d_level_gt); r2 |= dev_upload(e, lsg, &e->d_level_sg); r2 |= dev_upload(e, ltmp, &e->d_level_tmp);
        {
          // element lists: per front, every entry that receives class blocks with its sources in Gpart
          // (classes ascending, tasks ascending -- the summation order of k_front_level)
          std::vector<int> eg_ptr(Y.nsuper + 1, 0), eg_sptr{0}, eg_src;
          std::vector<unsigned int> eg_dst;
          struct Ent { unsigned int dst; int src; };
          std::vector<Ent> ents;
          bool fits = Goff < (1ll << 31);
          for(int sn = 0; sn < Y.nsuper && fits; sn++)
          {
            ents.clear();
            for(int ci = Y.fcls_ptr[sn]; ci < Y.fcls_ptr[sn+1]; ci++)
            {
              const int c = Y.fcls_list[ci];
              const int k = Y.cls_ptr[c+1] - Y.cls_ptr[c];
              const int* loc = Y.cls_loc.data() + Y.cls_ptr[c];
              for(int a = 0, q = 0; a < k; a++)
                for(int b = 0; b <= a; b++, q++)
                {
                  const int la = loc[a], lb = loc[b];
                  const unsigned int row = (unsigned int)std::max(la, lb), col = (unsigned int)std::min(la, lb);
                  for(int t = cls_task_ptr[c]; t < cls_task_ptr[c+1]; t++) ents.push_back({row | (col << 16), (int)(task_Goff[t] + q)});
                }
            }
            std::stable_sort(ents.begin(), ents.end(), [](const Ent& x, const Ent& y) { return x.dst < y.dst; });
            for(size_t i = 0; i < ents.size(); i++)
            {
              if(i == 0 || ents[i].dst != ents[i-1].dst) { if(i) eg_sptr.push_back((int)eg_src.size()); eg_dst.push_back(ents[i].dst); }
              eg_src.push_back(ents[i].src);
            }
            if(!ents.empty()) eg_sptr.push_back((int)eg_src.size());
            eg_ptr[sn+1] = (int)eg_dst.size();
            if(eg_src.size() > (size_t)1 << 30) fits = false;
          }
          if(!fits) { g_last_error = "element lists too large"; r2 = 1; }
          r2 |= dev_upload(e, eg_ptr, &e->d_eg_ptr); r2 |= dev_upload(e, eg_dst, &e->d_eg_dst);
          r2 |= dev_upload(e, eg_sptr, &e->d_eg_sptr); r2 |= dev_upload(e, eg_src, &e->d_eg_src);
        }
        r2 |= dev_alloc(e, (size_t)e->trial_grid * DLB_TRIAL_PART, &e->d_trial_part);
        r2 |= dev_alloc(e, (size_t)4, &e->d_bar);
        { const char* pe = getenv("DOGLEG_GPU_TRIAL_PROF"); e->d_prof = 0; if(pe && atoi(pe) != 0) r2 |= dev_alloc(e, (size_t)DLB_TRIAL_PROF_MAX + 1, &e->d_prof); }
        if(r2) { g_last_error = "out of device memory for the trial kernel's workspace"; return -1; }
        CU(cudaMemsetAsync(e->d_bar, 0, 4 * sizeof(unsigned int), e->st));
        e->fused_trial = true;
      }
    }
  }
  CU(cudaStreamSynchronize(e->st));
  e->pattern_set = true;
  e->pattern_verified = true;
  if(verbose)
  {
    const auto t_end = std::chrono::steady_clock::now();
    size_t fr = 0, tot = 0; cudaMemGetInfo(&fr, &tot);
    fprintf(stderr, "libdogleg-b200: pattern N=%d M=%d: %d classes, %d supernodes, %d levels, nnz(L)=%lld, fronts %.2f GB, "
            "max front %d; symbolic %.2f s, index build + upload %.2f s; device memory in use %.1f GB; fused evaluation %d, trial kernel %d (grid %d)\n",
            e->N, Mtot, Y.ncls, Y.nsuper, Y.nlevels, (long long)Y.nnzL(), 8e-9 * (double)Y.front_off[Y.nsuper], Y.max_front_rows,
            std::chrono::duration<double>(t_sym - t_begin).count(), std::chrono::duration<double>(t_end - t_sym).count(),
            1e-9 * (double)(tot - fr), (int)e->fused_eval, (int)e->fused_trial, e->trial_grid);
  }
  return 0;
}

// --------------------------------------------------------------- evaluate
extern "C" int dlb_engine_upload_p(dlb_engine_t* e, int s)
{
  cudaSetDevice(e->device);
  Slot& L = e->slot[s & 1];
  CU(cudaMemcpyAsync(L.d_p, L.h_p, sizeof(double) * e->N, cudaMemcpyHostToDevice, e->st));
  e->n_h2d += sizeof(double) * e->N;
  return 0;
}

// ---- streaming host inputs (north star: "pinned cudaMemcpyAsync on a side stream, overlapped") ----
// dlb_engine_begin_host_fill() is called right before the user's host callback writes x and the Jacobian
// values of slot s into the pinned staging buffers. A callback that fills them front to back may call
// dogleg_gpu_host_progress(n_values, n_x) as often as it likes: the newly completed pieces start their
// way to HBM on the copy stream at once, so that when the callback returns only the tail is left to
// copy -- the PCIe transfer overlaps the callback instead of following it.
static thread_local struct { dlb_engine* e; int slot; size_t wJ, wx; } g_fill = {0, 0, 0, 0};
#define DLB_FILL_MIN_BYTES (1u << 20)
extern "C" void dlb_engine_begin_host_fill(dlb_engine_t* e, int s)
{
  g_fill.e = 0;
  if(!e->host_inputs || e->type == DOGLEG_DENSE_PRODUCTS) return;
  cudaSetDevice(e->device);
  // nothing on the compute stream may still read the slot's device buffers when the pieces land
  if(cudaEventRecord(e->ev_idle, e->st) != cudaSuccess || cudaStreamWaitEvent(e->st_copy, e->ev_idle, 0) != cudaSuccess) { cudaGetLastError(); return; }
  g_fill.e = e; g_fill.slot = s & 1; g_fill.wJ = 0; g_fill.wx = 0;
}
static void fill_copy_upto(dlb_engine* e, Slot& L, size_t nJ, size_t nx, bool all)
{
  nJ = std::min(nJ, e->Jcount); nx = std::min(nx, (size_t)e->M);
  if(nx > g_fill.wx && (all || (nx - g_fill.wx) * sizeof(double) >= DLB_FILL_MIN_BYTES))
  {
    cudaMemcpyAsync(L.d_x + (e->gather ? e->col_begin : 0) + g_fill.wx, L.h_x + g_fill.wx, sizeof(double) * (nx - g_fill.wx),
                    cudaMemcpyHostToDevice, e->st_copy);
    g_fill.wx = nx;
  }
  if(nJ > g_fill.wJ && (all || (nJ - g_fill.wJ) * sizeof(double) >= DLB_FILL_MIN_BYTES))
  {
    cudaMemcpyAsync(L.d_J + (e->gather ? e->slice_off : 0) + g_fill.wJ, L.h_J + g_fill.wJ, sizeof(double) * (nJ - g_fill.wJ),
                    cudaMemcpyHostToDevice, e->st_copy);
    g_fill.wJ = nJ;
  }
}
extern "C" void dogleg_gpu_host_progress(size_t n_values_final, size_t n_x_final)
{
  dlb_engine* e = g_fill.e;
  if(!e) return;
  fill_copy_upto(e, e->slot[g_fill.slot], n_values_final, n_x_final, false);
}

extern "C" int dlb_engine_evaluate(dlb_engine_t* e, int s, int from_host, double norm2x_products)
{
  cudaSetDevice(e->device);
  Slot& L = e->slot[s & 1];
  if(e->factor_slot == (s & 1)) e->factor_slot = -1;   // the factor no longer belongs to this point
  L.have_G = L.have_cauchy = L.have_gn = false;
  if(from_host && !e->host_inputs) { g_last_error = "evaluate(from_host): this engine was created without host mirrors"; return -1; }
  if(from_host)
  {
    PhaseTimer tm(e, 0);
    if(e->type == DOGLEG_DENSE_PRODUCTS)
    {
      CU(cudaMemcpyAsync(L.d_Jtx, L.h_Jtx, sizeof(double) * e->N, cudaMemcpyHostToDevice, e->st));
      CU(cudaMemcpyAsync(L.d_J, L.h_J, sizeof(double) * e->Jcount, cudaMemcpyHostToDevice, e->st));     // the user's JtJ
      e->n_h2d += sizeof(double) * (e->N + e->Jcount);
    }
    else
    {
      size_t cnt = e->Jcount;
      if(e->type == DOGLEG_SPARSE)
      {
        cnt = (size_t)(unsigned int)L.h_Jp[e->M];
        if(cnt > (size_t)e->nnz) { g_fill.e = 0; g_last_error = "the callback wrote more nonzeros (Jt->p[Nmeas]) than NJnnz"; return -1; }
      }
      // whatever the callback has not announced yet goes now, on the copy stream; the compute stream waits for it
      if(!(g_fill.e == e && g_fill.slot == (s & 1)))
      {
        g_fill.e = e; g_fill.slot = s & 1; g_fill.wJ = 0; g_fill.wx = 0;
        CU(cudaEventRecord(e->ev_idle, e->st));
        CU(cudaStreamWaitEvent(e->st_copy, e->ev_idle, 0));
      }
      if(g_fill.wJ > cnt) g_fill.wJ = cnt;
      {
        const size_t keepJ = e->Jcount; e->Jcount = cnt;             // copy exactly the values the pattern holds
        fill_copy_upto(e, L, cnt, (size_t)e->M, true);
        e->Jcount = keepJ;
      }
      g_fill.e = 0;
      CU(cudaEventRecord(e->ev_copy, e->st_copy));
      CU(cudaStreamWaitEvent(e->st, e->ev_copy, 0));
      CU(cudaGetLastError());
      e->n_h2d += sizeof(double) * (e->M + cnt);
    }
  }
  if(e->gather && g_nccl.comm && g_nccl.world > 1)
  { // every rank's slice of x and of the Jacobian values to everybody (on the solver's stream)
    PhaseTimer tm(e, 0);
    bool ok = g_nccl.GroupStart() == 0;
    for(int r = 0; ok && r < g_nccl.world; r++)
    {
      double* px = L.d_x + e->rank_cb[r]; double* pj = L.d_J + e->rank_off[r];
      if(e->rank_m[r] > 0)   ok = ok && g_nccl.Broadcast(px, px, (size_t)e->rank_m[r], /*ncclFloat64*/ 8, r, g_nccl.comm, e->st) == 0;
      if(e->rank_nnz[r] > 0) ok = ok && g_nccl.Broadcast(pj, pj, (size_t)e->rank_nnz[r], 8, r, g_nccl.comm, e->st) == 0;
      e->allreduce_bytes += 8.0 * (double)(e->rank_m[r] + e->rank_nnz[r]);
    }
    ok = (g_nccl.GroupEnd() == 0) && ok;
    if(!ok) { g_last_error = "ncclBroadcast of the Jacobian slices failed"; return -1; }
    e->n_allreduce += 1;
  }
  if(e->type == DOGLEG_SPARSE && e->fused_eval)
  { // one pass: gradient, |x|^2 and the class blocks of this point; the reduction publishes the scalars
    if(!e->pattern_set || !e->pattern_verified) { g_last_error = "dlb_engine_set_pattern() has not been called"; return -1; }
    int n2count = 0;
    {
      PhaseTimer tm(e, 1);
      n2count = dlb_launch_sparse_eval_pass(e->S, L.d_J, L.d_x, L.d_G, e->d_gpart, e->d_n2part, e->sm_count, e->st);
    }
    if(e->G_global && g_nccl.world > 1)
    { // local partial gradient and |x|^2, then one grouped all-reduce with the class blocks, then the
      // gradient's norms (published) -- nothing else of this iteration communicates
      PhaseTimer tm(e, 3);
      dlb_launch_sparse_eval_reduce(e->S, e->d_gpart, e->d_n2part, n2count, L.d_Jtx, e->d_part, e->d_counter, e->d_sc,
                                    (DlbPublished*)0, 0ull, 1, e->sm_count, e->st);
      if(!g_nccl.comm) { g_last_error = "sharded engine without dogleg_gpu_nccl_init()"; return -1; }
      bool ok = g_nccl.GroupStart() == 0;
      ok = ok && g_nccl.AllReduce(L.d_G, L.d_G, (size_t)e->Goff_total, /*ncclFloat64*/ 8, /*ncclSum*/ 0, g_nccl.comm, e->st) == 0;
      ok = ok && g_nccl.AllReduce(L.d_Jtx, L.d_Jtx, (size_t)e->N + 1, 8, 0, g_nccl.comm, e->st) == 0;
      ok = (g_nccl.GroupEnd() == 0) && ok;
      if(!ok) { g_last_error = "ncclAllReduce of the class blocks / gradient failed"; return -1; }
      e->n_allreduce += 1; e->allreduce_bytes += 8.0 * (double)(e->Goff_total + e->N + 1);
      e->seq++;
      dlb_launch_vec_stats_Jtx_pub(L.d_Jtx, e->N, e->d_part, e->d_counter, e->d_sc, e->d_pub, e->seq, e->sm_count, e->st);
      e->n_launch += 1;
    }
    else
    {
      PhaseTimer tm(e, 3);
      e->seq++;
      dlb_launch_sparse_eval_reduce(e->S, e->d_gpart, e->d_n2part, n2count, L.d_Jtx, e->d_part, e->d_counter, e->d_sc, e->d_pub,
                                    e->seq, 0, e->sm_count, e->st);
    }
    e->n_launch += 1 + (e->S.nbig > 0) + (e->S.nasm_small > 0) + (e->S.nfused > 0);
    L.have_G = true;
    if(e->G_shared) e->slot[1 - (s & 1)].have_G = false;
    CU(cudaGetLastError());
  }
  else
  {
    PhaseTimer tm(e, 1);
    if(e->type == DOGLEG_SPARSE)
    {
      if(!e->pattern_set || !e->pattern_verified) { g_last_error = "dlb_engine_set_pattern() has not been called"; return -1; }
      dlb_launch_sparse_grad(e->S, L.d_J, L.d_x, e->d_gpart, e->d_n2part, L.d_Jtx, e->d_part, e->d_counter,
                             e->d_sc, e->sm_count, e->st);
      e->n_launch += 2;
    }
    else if(e->type == DOGLEG_DENSE)
    {
      dlb_launch_dense_grad(L.d_J, L.d_x, e->M, e->N, L.d_Jtx, e->d_work, e->d_part, e->d_counter,
                            e->d_sc, e->sm_count, e->st);
      e->n_launch += 2;
    }
    else
    {
      dlb_launch_vec_stats_Jtx(L.d_Jtx, e->N, e->d_part, e->d_counter, e->d_sc, e->sm_count, e->st);
      e->n_launch += 1;
      // a device callback left |x|^2 in DLB_BUF_NORM2X
      if(!from_host) CU(cudaMemcpyAsync(&e->d_sc->norm2_x, L.d_Jtx + e->N, sizeof(double), cudaMemcpyDeviceToDevice, e->st));
    }
    CU(cudaGetLastError());
    if(e->sharded && g_nccl.world > 1)
    { // sum the partial gradients and |x|^2 over the ranks: one all-reduce of N+1 doubles
      CU(cudaMemcpyAsync(L.d_Jtx + e->N, &e->d_sc->norm2_x, sizeof(double), cudaMemcpyDeviceToDevice, e->st));
      if(allreduce_sum(e, L.d_Jtx, (size_t)e->N + 1)) return -1;
      dlb_launch_vec_stats_Jtx(L.d_Jtx, e->N, e->d_part, e->d_counter, e->d_sc, e->sm_count, e->st);
      CU(cudaMemcpyAsync(&e->d_sc->norm2_x, L.d_Jtx + e->N, sizeof(double), cudaMemcpyDeviceToDevice, e->st));
      e->n_launch += 1;
    }
  }
  if(e->type == DOGLEG_SPARSE && e->fused_eval) { if(wait_published(e)) return -1; }
  else if(sync_scalars(e)) return -1;
  if(e->type == DOGLEG_DENSE_PRODUCTS && from_host) e->h_sc->norm2_x = norm2x_products;
  L.norm2_x = e->h_sc->norm2_x;
  L.norm2_Jtx = e->h_sc->norm2_Jtx;
  return 0;
}

static int ensure_G(dlb_engine* e, int s);
// |J v|^2 for whichever representation slot s holds -> *dst (device)
static int launch_norm2_Jv(dlb_engine* e, Slot& L, const double* d_v, double* d_dst)
{
  if(e->type == DOGLEG_SPARSE)
  {
    if(e->jv_quad && L.have_G)
      dlb_launch_sparse_jv_quad(e->S, L.d_J, L.d_G, d_v, e->d_part, e->d_counter, d_dst, e->sm_count, e->st);
    else
      dlb_launch_sparse_jv(e->S, L.d_J, d_v, e->d_part, e->d_counter, d_dst, e->sm_count, e->st);
    e->n_launch += 1;
  }
  else if(e->type == DOGLEG_DENSE)
  { dlb_launch_dense_jv(L.d_J, d_v, e->M, e->N, e->d_work, d_dst, e->sm_count, e->st); e->n_launch += 2; }
  else
  {
    if(e->packed && !e->upper)
    { g_last_error = "dense-products: v'JtJ v is only supported for unpacked or packed-upper JtJ (as in the reference)"; return -1; }
    dlb_launch_products_xAx(L.d_J, e->N, e->packed, e->upper, d_v, e->d_xAx, e->st);
    CU(cudaMemcpyAsync(d_dst, e->d_xAx, sizeof(double), cudaMemcpyDeviceToDevice, e->st));
    e->n_launch += 2;
  }
  CU(cudaGetLastError());
  if(!(e->G_global && L.have_G) && allreduce_sum(e, d_dst, 1)) return -1;      // complete class blocks: already the full sum
  return 0;
}

extern "C" int dlb_engine_cauchy(dlb_engine_t* e, int s)
{
  cudaSetDevice(e->device);
  Slot& L = e->slot[s & 1];
  if(ensure_G(e, s)) return -1;
  {
    PhaseTimer tm(e, 2);
    if(launch_norm2_Jv(e, L, L.d_Jtx, &e->d_sc->norm2_JJtx)) return -1;
    dlb_launch_cauchy(L.d_Jtx, e->N, L.d_cauchy, e->d_sc, e->sm_count, e->st);
    e->n_launch += 1;
    CU(cudaGetLastError());
  }
  if(sync_scalars(e)) return -1;
  L.have_cauchy = true; L.norm2_cauchy = e->h_sc->norm2_cauchy;
  return 0;
}

// -------------------------------------------------------------- factorize
// DOGLEG_GPU_SOLVE_PROF=1: CUDA-event stamps between the launch groups of run_solve / the level loop of the
// factorization, printed per group after a synchronisation (development aid; off = no events, no syncs)
struct EvProf
{
  bool on; cudaStream_t st; std::vector<std::pair<std::string, cudaEvent_t>> ev;
  EvProf(cudaStream_t s) : st(s) { const char* p = getenv("DOGLEG_GPU_SOLVE_PROF"); on = p && atoi(p) != 0; if(on) mark("start"); }
  void mark(const std::string& name) { if(!on) return; cudaEvent_t x; cudaEventCreate(&x); cudaEventRecord(x, st); ev.push_back({name, x}); }
  void dump(const char* what)
  {
    if(!on) return;
    cudaStreamSynchronize(st);
    fprintf(stderr, "libdogleg-b200: %s (us):", what);
    for(size_t i = 1; i < ev.size(); i++) { float ms = 0; cudaEventElapsedTime(&ms, ev[i-1].second, ev[i].second); fprintf(stderr, " %s %.1f", ev[i].first.c_str(), 1e3 * ms); }
    float tot = 0; if(ev.size() > 1) cudaEventElapsedTime(&tot, ev.front().second, ev.back().second);
    fprintf(stderr, "  total %.1f\n", 1e3 * tot);
    for(auto& x : ev) cudaEventDestroy(x.second);
    ev.clear();
  }
};

static int run_factor_levels(dlb_engine* e, const double* Gpart, double lambda)
{
  const long long big = LLONG_MAX;
  e->minor_dirty = true;
  CU(cudaMemcpyAsync(e->d_minor, &big, sizeof(big), cudaMemcpyHostToDevice, e->st));
  const int nlev = (int)e->level_ptr.size() - 1;
  EvProf prof(e->st);
  for(int l = 0; l < nlev; l++)
  {
    // large fronts start from zero (unless they arrive pre-filled) before their children are gathered in
    const int nbigl = e->level_big_ptr[l+1] - e->level_big_ptr[l];
    if(nbigl > 0 && Gpart)
    {
      dlb_launch_zero_bigfronts(e->d_big_descs + e->level_big_ptr[l], nbigl, e->level_big_max_r[l], e->d_fronts, e->st);
      e->n_launch += 1;
    }
    if(!e->level_gt_ptr.empty() && e->level_gt_ptr[2*l+2] > e->level_gt_ptr[2*l])
    {
      if(e->level_tmp_size[l] > 0)
        CU(cudaMemsetAsync(e->F.heavy_tmp, 0, sizeof(double) * (size_t)e->level_tmp_size[l], e->st));
      dlb_launch_extend_gather(e->F.fg, e->level_gt_ptr[2*l], e->level_gt_ptr[2*l+1], e->d_fronts, 0, e->st);
      dlb_launch_extend_gather(e->F.fg, e->level_gt_ptr[2*l+1], e->level_gt_ptr[2*l+2], e->d_fronts, 1, e->st);
      e->n_launch += 2;
    }
    prof.mark("g" + std::to_string(l));
    // leaf fronts of level 0, one warp each, assembled straight from the Jacobian values
    const int lbeg = e->level_ptr[l] + (l == 0 && Gpart ? e->nleaf : 0);
    if(lbeg > e->level_ptr[l])
    {
      if(e->leaf_mma)
        dlb_launch_leaf_fronts_mma(e->F, e->S, e->level_ptr[l], lbeg, e->slot[e->asm_slot].d_J, e->d_fronts, lambda,
                                   e->d_minor, e->leaf_max_rows, e->leaf_max_pairs, 1, e->sm_count, e->st);
      else
        dlb_launch_leaf_fronts(e->F, e->S, e->level_ptr[l], lbeg, e->slot[e->asm_slot].d_J, e->d_fronts, lambda,
                               e->d_minor, e->leaf_max_rows, 1, e->sm_count, e->st);
      e->n_launch += 1;
    }
    // fronts that fit in shared memory: assemble and eliminate in one kernel
    if(e->level_mid[l] > lbeg)
    {
      dlb_launch_front_level(e->F, e->S, lbeg, e->level_mid[l], e->d_fronts, Gpart, lambda,
                             e->d_minor, e->level_small_rows[l], 0, e->st);
      e->n_launch += 1;
    }
    // large fronts: assemble in global memory, then the blocked tensor-core Cholesky
    if(e->level_ptr[l+1] > e->level_mid[l])
    {
      dlb_launch_front_level(e->F, e->S, e->level_mid[l], e->level_ptr[l+1], e->d_fronts, Gpart, lambda,
                             e->d_minor, e->level_rows[l], 1, e->st);
      e->n_launch += 1;
      dlb_bigfront_factor_batch(e->d_big_descs + e->level_big_ptr[l], e->level_big_ptr[l+1] - e->level_big_ptr[l],
                                e->level_big_max_r[l], e->level_big_max_nc[l], e->d_fronts, e->d_biginv, e->d_big_cnt + e->level_big_ptr[l],
                                e->d_minor, e->st, &e->n_launch);
    }
    prof.mark("f" + std::to_string(l));
  }
  prof.dump("factorization, per level: zero + gather / fronts");
  CU(cudaGetLastError());
  return 0;
}

// all_small: also the classes that the fused leaf kernel would assemble itself (elements-only passes)
static int assemble(dlb_engine* e, Slot& L, bool all_small)
{
  PhaseTimer tm(e, 3);
  if(e->type == DOGLEG_SPARSE)
  {
    dlb_launch_sparse_assemble(e->S, L.d_J, L.d_G, all_small || e->nleaf == 0, e->sm_count, e->st); e->n_launch += 1;
    L.have_G = true;
    if(e->G_shared) e->slot[1 - (int)(&L - e->slot)].have_G = false;
  }
  return 0;
}
// the class blocks of slot s, formed once per operating point: the Cauchy step, the expected
// improvement and the factorization all use them
static int ensure_G(dlb_engine* e, int s)
{
  if(e->type != DOGLEG_SPARSE || !e->jv_quad || e->slot[s & 1].have_G) return 0;
  return assemble(e, e->slot[s & 1], false);
}
// dense types: (re)build the single front from J or the user's JtJ
static int dense_fill_front(dlb_engine* e, Slot& L)
{
  PhaseTimer tm(e, 3);
  if(e->type == DOGLEG_DENSE)
  { dlb_launch_dense_syrk(L.d_J, e->M, e->N, e->d_fronts, e->d_work, e->sm_count, e->st); e->n_launch += 2; }
  else
  { dlb_launch_products_to_front(L.d_J, e->N, e->packed, e->upper, e->d_fronts, e->st); e->n_launch += 1; }
  CU(cudaGetLastError());
  return 0;
}

extern "C" int dlb_engine_factorize(dlb_engine_t* e, int s, double lambda)
{
  cudaSetDevice(e->device);
  Slot& L = e->slot[s & 1];
  e->asm_slot = s & 1;
  // the class-local JtJ blocks only depend on J: keep them across lambda retries
  const bool have_G = L.have_G && e->type == DOGLEG_SPARSE && (!e->sharded || e->G_global);
  // DOGLEG_GPU_FORCE_REDUCE_PATH=1: take the partial-fronts path even with a single rank (tests)
  const char* fr = getenv("DOGLEG_GPU_FORCE_REDUCE_PATH");
  const bool force_reduce = fr && atoi(fr) != 0;
  const bool reduce = e->sharded && !e->G_global && (g_nccl.world > 1 || force_reduce);
  const double* Gpart = e->type == DOGLEG_SPARSE ? L.d_G : NULL;
  if(e->type == DOGLEG_SPARSE)
  {
    if(!have_G)
    {
      if(assemble(e, L, reduce)) return -1;
      if(reduce)
      { // partial (unfactored) fronts from this rank's measurement columns, summed over the ranks
        PhaseTimer tm(e, 3);
        const int nlev = (int)e->level_ptr.size() - 1;
        for(int l = 0; l < nlev; l++)
        {
          dlb_launch_front_level(e->F, e->S, e->level_ptr[l], e->level_ptr[l+1], e->d_fronts, L.d_G, -1.0,
                                 e->d_minor, e->level_rows[l], 0, e->st);
          e->n_launch += 1;
        }
        CU(cudaGetLastError());
        if(allreduce_sum(e, e->d_fronts, (size_t)e->sym->front_off[e->sym->nsuper])) return -1;
        CU(cudaMemcpyAsync(e->d_fronts_asm, e->d_fronts, sizeof(double) * (size_t)e->sym->front_off[e->sym->nsuper],
                           cudaMemcpyDeviceToDevice, e->st));
      }
    }
    else if(reduce)
      CU(cudaMemcpyAsync(e->d_fronts, e->d_fronts_asm, sizeof(double) * (size_t)e->sym->front_off[e->sym->nsuper],
                         cudaMemcpyDeviceToDevice, e->st));
    if(reduce) Gpart = NULL;       // the fronts are pre-filled: only children, lambda, elimination remain
  }
  else
  {
    if(dense_fill_front(e, L)) return -1;
    if(reduce && allreduce_sum(e, e->d_fronts, (size_t)e->N * e->N)) return -1;
  }
  {
    PhaseTimer tm(e, 4);
    // pre-filled fronts (dense types, row-sharded sparse) are selected with a NULL Gpart
    if(run_factor_levels(e, Gpart, lambda)) return -1;
    CU(cudaMemcpyAsync(e->h_minor, e->d_minor, sizeof(long long), cudaMemcpyDeviceToHost, e->st));
    CU(cudaStreamSynchronize(e->st));
    e->n_d2h += sizeof(long long);
  }
  e->factor_slot = s & 1; e->factor_lambda = lambda;
  e->n_factor += 1;
  e->h_sc->minor = (*e->h_minor == LLONG_MAX) ? -1 : *e->h_minor;
  return 0;
}

// ------------------------------------------------------------------ solves
static int run_solve(dlb_engine* e, const double* d_rhs, int nrhs)
{
  EvProf prof(e->st);
  const int nlev = (int)e->level_ptr.size() - 1;
  // fronts whose children are gathered accumulate into their (zeroed) rows of the work vector
  if(e->any_solve_gather) CU(cudaMemsetAsync(e->d_ywork, 0, sizeof(double) * (size_t)e->F.ytot * nrhs, e->st));
  for(int l = 0; l < nlev; l++)
  {
    if(e->any_solve_gather && e->level_sg_ptr[2*l+2] > e->level_sg_ptr[2*l])
      for(int rh = 0; rh < nrhs; rh++)
      {
        double* pool = e->d_ywork + (size_t)rh * e->F.ytot;
        dlb_launch_extend_gather(e->F.sg, e->level_sg_ptr[2*l], e->level_sg_ptr[2*l+1], pool, 0, e->st);
        dlb_launch_extend_gather(e->F.sg, e->level_sg_ptr[2*l+1], e->level_sg_ptr[2*l+2], pool, 1, e->st);
        e->n_launch += 2;
      }
    prof.mark("g" + std::to_string(l));
    const int lbeg = e->level_ptr[l] + (l == 0 ? e->nleaf : 0);
    if(lbeg > e->level_ptr[l])
    {
      dlb_launch_leaf_solve_fwd(e->F, e->level_ptr[l], lbeg, e->d_fronts, d_rhs, e->d_ywork, e->d_zperm, nrhs, e->sm_count, e->st);
      e->n_launch += 1;
    }
    // fronts that fit in shared memory: one CTA each; larger ones: triangle + chunked panel kernels (dlb_bigsolve.cu)
    if(e->level_mid[l] > lbeg)
    {
      dlb_launch_solve_fwd_level(e->F, lbeg, e->level_mid[l], e->d_fronts, d_rhs, e->d_ywork,
                                 e->d_zperm, nrhs, e->level_small_rows[l], std::min(e->level_cols[l], e->level_small_rows[l]), e->st);
      e->n_launch += 1;
    }
    const int nbig = e->level_big_ptr[l+1] - e->level_big_ptr[l];
    for(int rh = 0; rh < nrhs && nbig > 0; rh++)
    {
      dlb_launch_bigsolve_fwd(e->F, e->d_big_descs + e->level_big_ptr[l], nbig, e->level_big_max_r[l], e->level_big_max_nc[l],
                              e->d_fronts, e->d_biginv, d_rhs + (size_t)rh * e->N, e->d_ywork + (size_t)rh * e->F.ytot,
                              e->d_zperm + (size_t)rh * e->N, 1, e->st);
      e->n_launch += 2;
    }
    prof.mark("f" + std::to_string(l));
  }
  for(int l = nlev - 1; l >= 0; l--)
  {
    const int lbeg = e->level_ptr[l] + (l == 0 ? e->nleaf : 0);
    const int nbig = e->level_big_ptr[l+1] - e->level_big_ptr[l];
    for(int rh = 0; rh < nrhs && nbig > 0; rh++)
    {
      dlb_launch_bigsolve_bwd(e->F, e->d_big_descs + e->level_big_ptr[l], nbig, e->level_big_max_r[l], e->level_big_max_nc[l],
                              e->d_fronts, e->d_biginv, e->d_zperm + (size_t)rh * e->N, e->d_big_partial, e->d_big_part_off + e->level_big_ptr[l],
                              1, e->st);
      e->n_launch += 2;
    }
    if(e->level_mid[l] > lbeg)
      dlb_launch_solve_bwd_level(e->F, lbeg, e->level_mid[l], e->d_fronts, e->d_zperm, nrhs,
                                 e->level_small_rows[l], std::min(e->level_cols[l], e->level_small_rows[l]), e->st);
    if(lbeg > e->level_ptr[l])
      dlb_launch_leaf_solve_bwd(e->F, e->level_ptr[l], lbeg, e->d_fronts, e->d_zperm, nrhs, e->sm_count, e->st);
    e->n_launch += 1;
    prof.mark("b" + std::to_string(l));
  }
  prof.dump("solve, per level: gather / forward / backward");
  CU(cudaGetLastError());
  return 0;
}

extern "C" int dlb_engine_gauss_newton(dlb_engine_t* e, int s)
{
  cudaSetDevice(e->device);
  Slot& L = e->slot[s & 1];
  if(e->factor_slot != (s & 1)) { g_last_error = "gauss_newton: no factorization for this operating point"; return -1; }
  {
    PhaseTimer tm(e, 5);
    if(run_solve(e, L.d_Jtx, 1)) return -1;
    dlb_launch_gn_finish(e->d_zperm, e->type == DOGLEG_SPARSE ? e->F.perm : NULL, e->N, L.d_gn,
                         e->d_part, e->d_counter, e->d_sc, e->sm_count, e->st);
    e->n_launch += 1;
    CU(cudaGetLastError());
  }
  if(sync_scalars(e)) return -1;
  L.have_gn = true; L.norm2_gn = e->h_sc->norm2_gn;
  return 0;
}

__global__ void k_unpermute(const double* __restrict__ z, const int* __restrict__ perm, int n, int nrhs, double* __restrict__ out)
{
  for(size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < (size_t)n * nrhs; idx += (size_t)gridDim.x * blockDim.x)
  {
    const int rh = (int)(idx / n), k = (int)(idx - (size_t)rh * n);
    out[(size_t)rh * n + (perm ? perm[k] : k)] = z[idx];
  }
}

extern "C" int dlb_engine_solve(dlb_engine_t* e, const double* B, double* X, int nrhs)
{
  cudaSetDevice(e->device);
  if(e->factor_slot < 0) { g_last_error = "solve: no factorization available"; return -1; }
  const size_t cnt = (size_t)e->N * nrhs;
  if(nrhs > e->rhs_cap)
  {
    if(e->d_rhs) cudaFree(e->d_rhs);
    e->d_rhs = 0; e->rhs_cap = 0;
    // [rhs | zperm | ywork] for nrhs right-hand sides
    CU(cudaMalloc(&e->d_rhs, sizeof(double) * (2 * cnt + (size_t)e->F.ytot * nrhs)));
    e->rhs_cap = nrhs;
  }
  double* d_b = e->d_rhs; double* d_z = e->d_rhs + cnt; double* d_y = e->d_rhs + 2 * cnt;
  CU(cudaMemcpyAsync(d_b, B, sizeof(double) * cnt, cudaMemcpyHostToDevice, e->st));
  double* keep_z = e->d_zperm; double* keep_y = e->d_ywork;
  e->d_zperm = d_z; e->d_ywork = d_y;
  const int rc = run_solve(e, d_b, nrhs);
  e->d_zperm = keep_z; e->d_ywork = keep_y;
  if(rc) return -1;
  k_unpermute<<<std::min<size_t>((cnt + 255) / 256, 1184), 256, 0, e->st>>>(d_z, e->type == DOGLEG_SPARSE ? e->F.perm : NULL, e->N, nrhs, d_b);
  e->n_launch += 1;
  CU(cudaMemcpyAsync(X, d_b, sizeof(double) * cnt, cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  e->n_h2d += sizeof(double) * cnt; e->n_d2h += sizeof(double) * cnt;
  return 0;
}

// ------------------------------------------------------------- outlier helpers (f1)
// A = J* inv(JtJ + lambda I) J*' for every feature (featureSize consecutive measurements; featureSize*(featureSize+1)/2
// values per feature: a00 | a00 a01 a11), reference dogleg.c:2401-2791. The reference -- and round 1 here -- solves for
// inv(JtJ) j_i measurement by measurement (chunks of 4 / 64 right-hand sides: 15 625 solves + copies for a million
// measurements). For Nstate up to 16384 the inverse itself is cheaper: B = inv(JtJ + lambda I) by Nstate right-hand
// sides (the identity, generated on the device), then a_ij = sum over the nonzeros (p, q) of the two measurement
// columns of J_p B[p, q] J_q, a warp per feature, B resident in L2 / HBM. Returns 1 if the engine cannot take
// this path (too many states), -1 on errors.
__global__ void k_identity_cols(double* __restrict__ b, int n, int c0, int nc)
{
  for(size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < (size_t)n * nc; idx += (size_t)gridDim.x * blockDim.x)
  {
    const int c = (int)(idx / n), i = (int)(idx - (size_t)c * n);
    b[idx] = i == c0 + c ? 1.0 : 0.0;
  }
}
// Jp == NULL: dense row-first J (every measurement has the n entries 0..n-1)
__global__ void __launch_bounds__(256)
k_outlier_products(const double* __restrict__ Binv, int n, const int* __restrict__ Jp, const int* __restrict__ Ji,
                   const double* __restrict__ Jx, int featureSize, int nfeatures, double* __restrict__ out)
{
  const int lane = threadIdx.x & 31;
  const long long wg = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), nw = (long long)gridDim.x * (blockDim.x >> 5);
  const int npairs = featureSize * (featureSize + 1) / 2;
  for(long long f = wg; f < nfeatures; f += nw)
    for(int i = 0, ia = 0; i < featureSize; i++)
      for(int j = i; j < featureSize; j++, ia++)
      {
        const long long mi = f * featureSize + i, mj = f * featureSize + j;
        const long long pi0 = Jp ? Jp[mi] : mi * n, pi1 = Jp ? Jp[mi + 1] : (mi + 1) * n;
        const long long pj0 = Jp ? Jp[mj] : mj * n, pj1 = Jp ? Jp[mj + 1] : (mj + 1) * n;
        double acc = 0.0;
        for(long long a0 = pi0; a0 < pi1; a0 += 32)
        { // lane <-> nonzero a of measurement i; all nonzeros b of measurement j are broadcast in turn
          const long long a = a0 + lane;
          const bool on = a < pi1;
          const int ra = on ? (Jp ? Ji[a] : (int)(a - pi0)) : 0;
          const double va = on ? Jx[a] : 0.0;
          const double* Brow = Binv + (size_t)ra * n;                  // B is symmetric: row ra = column ra
          double s = 0.0;
          for(long long b0 = pj0; b0 < pj1; b0 += 32)
          {
            const long long b = b0 + lane;
            const int rb_l = b < pj1 ? (Jp ? Ji[b] : (int)(b - pj0)) : 0;
            const double vb_l = b < pj1 ? Jx[b] : 0.0;
            const int cnt = (int)(pj1 - b0 < 32 ? pj1 - b0 : 32);
            for(int u = 0; u < cnt; u++)
            {
              const int rb = __shfl_sync(0xffffffffu, rb_l, u);
              const double vb = __shfl_sync(0xffffffffu, vb_l, u);
              s = fma(Brow[rb], vb, s);
            }
          }
          acc = fma(va, s, acc);
        }
        acc = warp_sum_all(acc);
        if(lane == 0) out[f * npairs + ia] = acc;
      }
}
extern "C" int dlb_engine_outlier_products(dlb_engine_t* e, int slot, const int* Jp, const int* Ji, int featureSize,
                                           int nfeatures, double* A_host)
{
  cudaSetDevice(e->device);
  if(e->factor_slot < 0) { g_last_error = "outlier products: no factorization available"; return -1; }
  if(e->type == DOGLEG_DENSE_PRODUCTS || e->sharded) return 1;
  const int n = e->N;
  if(n > 16384 || nfeatures <= 0) return 1;
  Slot& L = e->slot[slot & 1];
  if(!L.d_J) return 1;
  const bool sparse = e->type == DOGLEG_SPARSE;
  const size_t nnz = sparse ? (size_t)Jp[(size_t)nfeatures * featureSize] : 0;
  const int npairs = featureSize * (featureSize + 1) / 2;
  double *d_B = 0, *d_out = 0; int *d_p = 0, *d_i = 0;
  auto cleanup = [&]() { cudaFree(d_B); cudaFree(d_out); cudaFree(d_p); cudaFree(d_i); cudaGetLastError(); };
  if(cudaMalloc(&d_B, sizeof(double) * (size_t)n * n) != cudaSuccess ||
     cudaMalloc(&d_out, sizeof(double) * (size_t)nfeatures * npairs) != cudaSuccess ||
     (sparse && (cudaMalloc(&d_p, sizeof(int) * ((size_t)nfeatures * featureSize + 1)) != cudaSuccess ||
                 cudaMalloc(&d_i, sizeof(int) * std::max<size_t>(nnz, 1)) != cudaSuccess)))
  { cleanup(); return 1; }
  // the inverse, 64 identity columns at a time through the level-scheduled multi-RHS solve
  const int chunk = 64;
  const size_t cnt = (size_t)n * chunk;
  if(chunk > e->rhs_cap)
  {
    if(e->d_rhs) cudaFree(e->d_rhs);
    e->d_rhs = 0; e->rhs_cap = 0;
    if(cudaMalloc(&e->d_rhs, sizeof(double) * (2 * cnt + (size_t)e->F.ytot * chunk)) != cudaSuccess) { cleanup(); return 1; }
    e->rhs_cap = chunk;
  }
  const size_t cap = (size_t)n * e->rhs_cap;
  double* d_b = e->d_rhs; double* d_z = e->d_rhs + cap; double* d_y = e->d_rhs + 2 * cap;
  if(sparse)
  {
    cudaMemcpyAsync(d_p, Jp, sizeof(int) * ((size_t)nfeatures * featureSize + 1), cudaMemcpyHostToDevice, e->st);
    cudaMemcpyAsync(d_i, Ji, sizeof(int) * nnz, cudaMemcpyHostToDevice, e->st);
    e->n_h2d += sizeof(int) * ((double)nfeatures * featureSize + 1 + (double)nnz);
  }
  int rc = 0;
  for(int c0 = 0; c0 < n && !rc; c0 += chunk)
  {
    const int nc = n - c0 < chunk ? n - c0 : chunk;
    k_identity_cols<<<std::min<size_t>(((size_t)n * nc + 255) / 256, 1184), 256, 0, e->st>>>(d_b, n, c0, nc);
    double* keep_z = e->d_zperm; double* keep_y = e->d_ywork;
    e->d_zperm = d_z; e->d_ywork = d_y;
    rc = run_solve(e, d_b, nc);
    e->d_zperm = keep_z; e->d_ywork = keep_y;
    k_unpermute<<<std::min<size_t>(((size_t)n * nc + 255) / 256, 1184), 256, 0, e->st>>>(d_z, sparse ? e->F.perm : NULL, n, nc, d_B + (size_t)c0 * n);
    e->n_launch += 2;
  }
  if(!rc)
  {
    const long long g = std::min<long long>(((long long)nfeatures + 7) / 8, (long long)e->sm_count * 8);
    k_outlier_products<<<(int)g, 256, 0, e->st>>>(d_B, n, sparse ? d_p : NULL, d_i, L.d_J + (e->gather ? e->slice_off : 0),
                                                  featureSize, nfeatures, d_out);
    e->n_launch += 1;
    if(cudaGetLastError() != cudaSuccess) rc = -1;
    cudaMemcpyAsync(A_host, d_out, sizeof(double) * (size_t)nfeatures * npairs, cudaMemcpyDeviceToHost, e->st);
    if(cudaStreamSynchronize(e->st) != cudaSuccess) { g_last_error = "outlier products: device error"; rc = -1; }
    e->n_d2h += sizeof(double) * (double)nfeatures * npairs;
  }
  cleanup();
  return rc ? -1 : 0;
}

// ------------------------------------------------------------- factor export
// The numeric factor in CHOLMOD's supernodal layout: supernode s is an r x nc column-major panel
// (leading dimension r) at x[px[s]] -- exactly the first nc columns of its front.
__global__ void k_pack_panels(DlbFrontDev F, const double* __restrict__ fronts, const int* __restrict__ px, double* __restrict__ out)
{
  const int s = blockIdx.x;
  const int nc = F.sn_first[s+1] - F.sn_first[s], r = F.rows_ptr[s+1] - F.rows_ptr[s];
  const double* A = fronts + F.front_off[s];
  double* o = out + px[s];
  for(int idx = threadIdx.x; idx < r * nc; idx += blockDim.x) o[idx] = A[idx];
}
extern "C" int dlb_engine_export_factor(dlb_engine_t* e, const int* px, long long xsize, double* x_host)
{
  cudaSetDevice(e->device);
  if(e->type != DOGLEG_SPARSE) { g_last_error = "export_factor: sparse engines only (dense factors: dlb_engine_dense_factor_to_host)"; return -1; }
  if(e->factor_slot < 0) { g_last_error = "export_factor: no factorization available"; return -1; }
  int* d_px = 0; double* d_out = 0;
  CU(cudaMalloc(&d_px, sizeof(int) * ((size_t)e->F.nsuper + 1)));
  if(cudaMalloc(&d_out, sizeof(double) * (size_t)std::max<long long>(xsize, 1)) != cudaSuccess)
  { cudaFree(d_px); cudaGetLastError(); g_last_error = "export_factor: out of device memory"; return -1; }
  CU(cudaMemcpyAsync(d_px, px, sizeof(int) * ((size_t)e->F.nsuper + 1), cudaMemcpyHostToDevice, e->st));
  k_pack_panels<<<e->F.nsuper, 256, 0, e->st>>>(e->F, e->d_fronts, d_px, d_out);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(x_host, d_out, sizeof(double) * (size_t)xsize, cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  cudaFree(d_px); cudaFree(d_out);
  e->n_launch += 1; e->n_d2h += sizeof(double) * (double)xsize;
  return 0;
}

// -------------------------------------------------------------------- step
extern "C" int dlb_engine_step(dlb_engine_t* e, int from, int to, int step_type, double delta)
{
  cudaSetDevice(e->device);
  Slot& A = e->slot[from & 1]; Slot& B = e->slot[to & 1];
  if(ensure_G(e, from)) return -1;
  {
    PhaseTimer tm(e, 6);
    dlb_launch_step(step_type, delta, A.d_p, A.d_Jtx, A.d_cauchy, A.d_gn, e->N, B.d_step, B.d_p,
                    e->d_part, e->d_counter, e->d_sc, e->sm_count, e->st);
    e->n_launch += step_type == DLB_STEP_INTERPOLATED ? 2 : 1;
    if(launch_norm2_Jv(e, A, B.d_step, &e->d_sc->norm2_Jstep)) return -1;
  }
  if(!e->lazy_p)
  {
    PhaseTimer tm(e, 7);
    CU(cudaMemcpyAsync(B.h_p, B.d_p, sizeof(double) * e->N, cudaMemcpyDeviceToHost, e->st));
    e->n_d2h += sizeof(double) * e->N;
  }
  return sync_scalars(e);
}

// ---------------------------------------------------------- fused trial step
// One cooperative launch (dlb_trial.cu) for everything between two evaluations of the callback:
// Cauchy step (unless cached for slot 'from'), Gauss-Newton step if the Cauchy step stays inside the
// trust region (factorization + solves, unless cached), step selection, p[to] = p[from] + step and
// the expected-improvement ingredients. One host round trip: the scalars (and p[to], unless lazy)
// arrive through mapped pinned memory. scalars.minor >= 0: JtJ + lambda I was not positive definite;
// nothing after the factorization was done and the caller repeats the call with a larger lambda.
extern "C" int dlb_engine_has_trial(const dlb_engine_t* e) { return e->fused_trial ? 1 : 0; }
extern "C" int dlb_engine_has_fused_eval(const dlb_engine_t* e) { return e->fused_eval ? 1 : 0; }
extern "C" int dlb_engine_trial(dlb_engine_t* e, int from, int to, double delta, double lambda)
{
  cudaSetDevice(e->device);
  if(!e->fused_trial) { g_last_error = "dlb_engine_trial: this engine has no fused trial kernel (dlb_engine_has_trial)"; return -1; }
  Slot& A = e->slot[from & 1]; Slot& B = e->slot[to & 1];
  if(!A.have_G) { g_last_error = "dlb_engine_trial: the starting point has not been evaluated"; return -1; }
  if(A.have_gn && (e->factor_slot != (from & 1))) A.have_gn = false;
  if(!A.have_gn) e->factor_slot = -1;       // the kernel starts factorizing at once (speculatively): the fronts are overwritten
  if(e->minor_dirty)
  { // the per-level schedule (or nothing yet) used the flag slots last: start from two clean ones
    static const long long big2[2] = {LLONG_MAX, LLONG_MAX};
    CU(cudaMemcpyAsync(e->d_minor, big2, sizeof(big2), cudaMemcpyHostToDevice, e->st));
    e->minor_dirty = false;
  }
  DlbTrial T;
  memset(&T, 0, sizeof(T));
  T.nlev = (int)e->level_ptr.size() - 1; T.level_ptr = e->d_level_ptr; T.level_gt = e->d_level_gt;
  T.level_sg = e->d_level_sg; T.level_tmp = e->d_level_tmp;
  T.max_rows = e->max_front_rows; T.max_cols = e->max_front_cols; T.any_solve_gather = e->any_solve_gather ? 1 : 0;
  T.small_tail = 2 * (size_t)e->N * sizeof(double) <= dlb_trial_smem_bytes(e->max_front_rows) ? 1 : 0;
  T.Jtx = A.d_Jtx; T.p_from = A.d_p; T.Gpart = A.d_G; T.cauchy = A.d_cauchy; T.gn = A.d_gn;
  T.norm2_Jtx = A.norm2_Jtx; T.norm2_cauchy = A.norm2_cauchy; T.norm2_gn = A.norm2_gn;
  T.have_cauchy = A.have_cauchy ? 1 : 0; T.have_gn = A.have_gn ? 1 : 0;
  T.step = B.d_step; T.p_to = B.d_p; T.h_p_to = e->lazy_p ? NULL : B.h_p;
  T.fronts = e->d_fronts; T.ywork = e->d_ywork; T.zperm = e->d_zperm;
  T.part = e->d_trial_part; T.bar = e->d_bar;
  T.minor = e->d_minor + (e->trial_parity & 1); T.minor_next = e->d_minor + ((e->trial_parity + 1) & 1);
  e->trial_parity++;
  T.sc = e->d_sc; T.pub = e->d_pub; T.seq = ++e->seq;
  T.delta = delta; T.lambda = lambda; T.prof = e->d_prof;
  T.eg_ptr = e->d_eg_ptr; T.eg_dst = e->d_eg_dst; T.eg_sptr = e->d_eg_sptr; T.eg_src = e->d_eg_src;
  {
    PhaseTimer tm(e, 4);
    if(dlb_launch_trial(e->S, e->F, T, e->trial_grid, e->st))
    { g_last_error = std::string("cooperative launch of the trial kernel failed: ") + cudaGetErrorString(cudaGetLastError()); return -1; }
    e->n_launch += 1;
  }
  if(wait_published(e)) return -1;
  if(e->d_prof)
  { // phase durations of this launch (CTA 0's view), microseconds
    unsigned long long h[DLB_TRIAL_PROF_MAX + 1];
    CU(cudaStreamSynchronize(e->st));
    CU(cudaMemcpy(h, e->d_prof, sizeof(h), cudaMemcpyDeviceToHost));
    const int n = (int)std::min<unsigned long long>(h[DLB_TRIAL_PROF_MAX], DLB_TRIAL_PROF_MAX);
    fprintf(stderr, "libdogleg-b200: trial kernel phases (us):");
    for(int i = 1; i < n; i++) fprintf(stderr, " %.1f", 1e-3 * (double)(h[i] - h[i-1]));
    fprintf(stderr, "  total %.1f\n", n > 0 ? 1e-3 * (double)(h[n-1] - h[0]) : 0.0);
    dlb_trial_dbg_dump();
  }
  if(!e->lazy_p) e->n_d2h += sizeof(double) * e->N;
  const dlb_scalars_t* sc = e->h_sc;
  if(!A.have_cauchy) { A.have_cauchy = true; A.norm2_cauchy = sc->norm2_cauchy; }
  if(sc->minor >= 0) { if(e->factor_slot == (from & 1)) e->factor_slot = -1; e->n_factor += 1; return 0; }
  if(sc->trial_flags != 0.0)
  {
    A.have_gn = true; A.norm2_gn = sc->norm2_gn;
    e->factor_slot = from & 1; e->factor_lambda = lambda; e->asm_slot = from & 1;
    e->n_factor += 1;
  }
  return 0;
}

// device-callback solves never read p on the host between the steps: skip the per-step copy
// (24 MB per step in the bundle-adjustment config); dlb_engine_download_p() fetches it at the end
extern "C" void dlb_engine_set_lazy_p(dlb_engine_t* e, int on) { e->lazy_p = on != 0; }
extern "C" int dlb_engine_download_p(dlb_engine_t* e, int s)
{
  cudaSetDevice(e->device);
  Slot& L = e->slot[s & 1];
  CU(cudaMemcpyAsync(L.h_p, L.d_p, sizeof(double) * e->N, cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  e->n_d2h += sizeof(double) * e->N;
  return 0;
}

extern "C" int dlb_engine_download(dlb_engine_t* e, int s)
{
  cudaSetDevice(e->device);
  Slot& L = e->slot[s & 1];
  const size_t nb = sizeof(double) * e->N;
  CU(cudaMemcpyAsync(L.h_p, L.d_p, nb, cudaMemcpyDeviceToHost, e->st));
  CU(cudaMemcpyAsync(L.h_Jtx, L.d_Jtx, nb, cudaMemcpyDeviceToHost, e->st));
  CU(cudaMemcpyAsync(L.h_cauchy, L.d_cauchy, nb, cudaMemcpyDeviceToHost, e->st));
  CU(cudaMemcpyAsync(L.h_gn, L.d_gn, nb, cudaMemcpyDeviceToHost, e->st));
  CU(cudaMemcpyAsync(L.h_step, L.d_step, nb, cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  e->n_d2h += 5 * nb;
  return 0;
}

// download x / Jacobian values too (device-callback solves: the host mirrors were never written)
extern "C" int dlb_engine_download_inputs(dlb_engine_t* e, int s)
{
  cudaSetDevice(e->device);
  Slot& L = e->slot[s & 1];
  if(!e->host_inputs) return 0;
  if(L.h_x) CU(cudaMemcpyAsync(L.h_x, L.d_x + (e->gather ? e->col_begin : 0), sizeof(double) * e->M, cudaMemcpyDeviceToHost, e->st));
  CU(cudaMemcpyAsync(L.h_J, L.d_J + (e->gather ? e->slice_off : 0), sizeof(double) * e->Jcount, cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  e->n_d2h += sizeof(double) * (e->M + e->Jcount);
  return 0;
}

// ------------------------------------------------------------------- tests
extern "C" int dlb_engine_debug_JtJ(dlb_engine_t* e, int s, double lambda, double* JtJ_out)
{
  cudaSetDevice(e->device);
  Slot& L = e->slot[s & 1];
  const size_t NN = (size_t)e->N * e->N;
  double* d_out = 0;
  CU(cudaMalloc(&d_out, sizeof(double) * NN));
  CU(cudaMemsetAsync(d_out, 0, sizeof(double) * NN, e->st));
  if(e->type == DOGLEG_SPARSE)
  {
    if(assemble(e, L, true)) return -1;
    // elements only, no elimination: lambda < 0 selects the test mode of the front kernel
    const int nlev = (int)e->level_ptr.size() - 1;
    for(int l = 0; l < nlev; l++)
      dlb_launch_front_level(e->F, e->S, e->level_ptr[l], e->level_ptr[l+1], e->d_fronts, L.d_G, -1.0,
                             e->d_minor, e->level_rows[l], 0, e->st);
  }
  else if(dense_fill_front(e, L)) return -1;
  dlb_launch_fronts_to_dense(e->F, e->d_fronts, d_out, e->st);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(JtJ_out, d_out, sizeof(double) * NN, cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  cudaFree(d_out);
  for(int i = 0; i < e->N; i++) JtJ_out[(size_t)i * e->N + i] += lambda;
  e->factor_slot = -1;
  return 0;
}

extern "C" int dlb_engine_dense_factor_to_host(dlb_engine_t* e, double* out)
{
  cudaSetDevice(e->device);
  if(e->type == DOGLEG_SPARSE) { g_last_error = "dense_factor_to_host: sparse engine"; return -1; }
  if(e->factor_slot < 0) return 0;
  const int packed = e->type == DOGLEG_DENSE ? 1 : e->packed;
  const int upper  = e->type == DOGLEG_DENSE ? 1 : e->upper;
  const size_t cnt = packed ? (size_t)e->N * (e->N + 1) / 2 : (size_t)e->N * e->N;
  double* d_out = 0;
  CU(cudaMalloc(&d_out, sizeof(double) * cnt));
  if(!packed)   // the other triangle keeps the user's values, as LAPACK leaves it
    CU(cudaMemcpyAsync(d_out, e->slot[e->factor_slot].d_J, sizeof(double) * cnt, cudaMemcpyDeviceToDevice, e->st));
  dlb_launch_front_to_reference_layout(e->d_fronts, e->N, packed, upper, d_out, e->st);
  CU(cudaMemcpyAsync(out, d_out, sizeof(double) * cnt, cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  cudaFree(d_out);
  e->n_launch += 1; e->n_d2h += sizeof(double) * cnt;
  return 0;
}
