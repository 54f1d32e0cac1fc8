"""ctypes binding of libdogleg.so (include/dogleg.h + include/dogleg_gpu.h)."""
import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

SOLVE_DENSE, SOLVE_SPARSE, SOLVE_DENSE_PRODUCTS = 0, 1, 2      # dogleg_solve_type_t
DEBUG_VNLOG = 1 << 30
BUF_P, BUF_X, BUF_JTX, BUF_CAUCHY, BUF_GN, BUF_STEP, BUF_JVALUES, BUF_JP, BUF_JI, BUF_NORM2X = range(10)
STEP_CAUCHY, STEP_GAUSSNEWTON, STEP_INTERPOLATED = 0, 1, 2
# DOGLEG_GPU_BATCH_*: why a problem of a batched solve stopped (dogleg_gpu_batch_status)
BATCH_UNFINISHED, BATCH_GRADIENT, BATCH_STEP, BATCH_TRUSTREGION, BATCH_MAX_ITERATIONS = range(5)
SYM = dict(perm=0, parent=1, colcount=2, sn_first=3, rows_ptr=4, rows=5, sn_parent=6,
           cls_of_col=7, cls_front=8, sn_level=9, rel=10, child_ptr=11, child_list=12, level_ptr=13,
           level_sn=14, cls_ptr=15, cls_rows=16, cls_loc=17, mem_ptr=18, mem_col=19)
# DLB_TP_* selectors of dlb_task_plan_get
TP = dict(task_cls=0, task_m0=1, task_m1=2, cls_task_ptr=3, task_goff=4, task_Goff=5, mem_col=6, mem_pos=7,
          big_tasks=8, small_tasks=9, gj_big_tasks=10, ranged=11, gp_count=12, gp_first=13, ginv_ptr=14,
          ginv_cls=15, ginv_off=16, heavy=17, medium=18, sizes=19, range_tasks=20)
# DLB_GP_* selectors of dlb_gather_plan_get (include/dogleg_gpu.h)
GP = dict(dst=0, src_ptr=1, src_base=2, ld=3, h=4, w=5, src_ld=6, level_ptr=7, tmp_off=8, level_tmp=9,
          sg_flag=10)


class Parameters(C.Structure):
    """dogleg_parameters2_t (reference dogleg.h:112-152); 72 bytes."""
    _fields_ = [("max_iterations", C.c_int), ("dogleg_debug", C.c_int),
                ("trustregion0", C.c_double),
                ("trustregion_decrease_factor", C.c_double), ("trustregion_decrease_threshold", C.c_double),
                ("trustregion_increase_factor", C.c_double), ("trustregion_increase_threshold", C.c_double),
                ("Jt_x_threshold", C.c_double), ("update_threshold", C.c_double),
                ("trustregion_threshold", C.c_double)]

    def set_flags(self, debug=False, packed=False, upper=False, vnlog=False):
        self.dogleg_debug = (1 if debug else 0) | (2 if packed else 0) | (4 if upper else 0) | \
                            (DEBUG_VNLOG if vnlog else 0)


class Scalars(C.Structure):
    """dlb_scalars_t (include/dogleg_gpu.h)."""
    _fields_ = [(n, C.c_double) for n in
                ("norm2_x", "norm2_Jtx", "maxabs_Jtx", "norm2_JJtx", "k_cauchy", "norm2_cauchy", "norm2_gn",
                 "norm2_step", "k_interp", "Jtx_dot_step", "maxabs_step", "norm2_Jstep", "discriminant",
                 "step_type", "trial_flags")] + [("minor", C.c_longlong)]


def lib_path():
    return os.path.join(HERE, "libdogleg.so")


def build(verbose=False):
    """Compile libdogleg.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(HERE, "csrc"), "-j8"]
    out = subprocess.run(cmd, capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("building libdogleg.so failed:\n" + out.stdout[-4000:] + out.stderr[-4000:])
    if verbose:
        print(out.stdout[-2000:])
    return lib_path()


_lib = None


def load():
    """Load libdogleg.so and declare the prototypes. Raises if it was not built:
    there is no fallback implementation."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    L = C.CDLL(path, mode=C.RTLD_LOCAL)
    dp, ip, vp = C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_void_p
    PP = C.POINTER(Parameters)
    L.dogleg_getDefaultParameters.argtypes = [PP]
    L.dogleg_getDefaultParameters.restype = None
    L.dogleg_optimize2.argtypes = [dp, C.c_uint, C.c_uint, C.c_uint, vp, vp, PP, C.POINTER(vp)]
    L.dogleg_optimize2.restype = C.c_double
    L.dogleg_optimize.argtypes = [dp, C.c_uint, C.c_uint, C.c_uint, vp, vp, C.POINTER(vp)]
    L.dogleg_optimize.restype = C.c_double
    L.dogleg_optimize_dense2.argtypes = [dp, C.c_uint, C.c_uint, vp, vp, PP, C.POINTER(vp)]
    L.dogleg_optimize_dense2.restype = C.c_double
    L.dogleg_optimize_dense.argtypes = [dp, C.c_uint, C.c_uint, vp, vp, C.POINTER(vp)]
    L.dogleg_optimize_dense.restype = C.c_double
    L.dogleg_optimize_dense_products.argtypes = [dp, C.c_uint, vp, vp, PP, C.POINTER(vp)]
    L.dogleg_optimize_dense_products.restype = C.c_double
    L.dogleg_freeContext.argtypes = [C.POINTER(vp)]
    L.dogleg_freeContext.restype = None
    L.dogleg_computeJtJfactorization.argtypes = [vp, vp]
    L.dogleg_computeJtJfactorization.restype = C.c_bool
    L.dogleg_setDebug.argtypes = [C.c_int]
    L.dogleg_setMaxIterations.argtypes = [C.c_int]
    L.dogleg_setInitialTrustregion.argtypes = [C.c_double]
    L.dogleg_setThresholds.argtypes = [C.c_double] * 3
    L.dogleg_setTrustregionUpdateParameters.argtypes = [C.c_double] * 4
    # dogleg_gpu.h
    L.dogleg_gpu_device_count.restype = C.c_int
    L.dogleg_gpu_set_device.argtypes = [C.c_int]
    L.dogleg_gpu_last_error.restype = C.c_char_p
    L.dogleg_gpu_version.restype = C.c_char_p
    L.dogleg_gpu_set_permutation.argtypes = [ip, C.c_int, C.c_int]
    L.dogleg_gpu_set_permutation.restype = None
    L.dogleg_gpu_get_stats.argtypes = [vp, dp]
    L.dogleg_gpu_get_stats.restype = None
    L.dogleg_gpu_get_phase_ms.argtypes = [dp]
    L.dogleg_gpu_get_phase_ms.restype = None
    L.dogleg_gpu_optimize_sparse.argtypes = [dp, C.c_uint, C.c_uint, C.c_uint, ip, ip, vp, vp, PP, C.POINTER(vp)]
    L.dogleg_gpu_optimize_sparse.restype = C.c_double
    L.dogleg_gpu_optimize_dense.argtypes = [dp, C.c_uint, C.c_uint, vp, vp, PP, C.POINTER(vp)]
    L.dogleg_gpu_optimize_dense.restype = C.c_double
    L.dogleg_gpu_optimize_dense_batched.argtypes = [dp, C.c_uint, C.c_uint, C.c_uint, vp, vp, PP, dp, ip]
    L.dogleg_gpu_optimize_dense_batched.restype = C.c_int
    L.dogleg_gpu_optimize_dense_products.argtypes = [dp, C.c_uint, vp, vp, PP, C.POINTER(vp)]
    L.dogleg_gpu_optimize_dense_products.restype = C.c_double
    L.dogleg_gpu_optimize_dense_products_batched.argtypes = [dp, C.c_uint, C.c_uint, vp, vp, PP, dp, ip]
    L.dogleg_gpu_optimize_dense_products_batched.restype = C.c_int
    L.dogleg_gpu_optimize_dense_batched2.argtypes = [dp, C.c_uint, C.c_uint, C.c_uint, vp, vp, PP, dp, ip, C.POINTER(vp)]
    L.dogleg_gpu_optimize_dense_batched2.restype = C.c_int
    L.dogleg_gpu_optimize_dense_products_batched2.argtypes = [dp, C.c_uint, C.c_uint, vp, vp, PP, dp, ip, C.POINTER(vp)]
    L.dogleg_gpu_optimize_dense_products_batched2.restype = C.c_int
    L.dogleg_gpu_batch_status.argtypes = [vp, ip, dp]
    L.dogleg_gpu_batch_status.restype = C.c_int
    L.dogleg_gpu_batch_solve.argtypes = [vp, dp, dp, C.c_int]
    L.dogleg_gpu_batch_solve.restype = C.c_int
    L.dogleg_gpu_batch_solve_device.argtypes = [vp, vp, vp, C.c_int, vp]
    L.dogleg_gpu_batch_solve_device.restype = C.c_int
    L.dogleg_gpu_batch_covariance.argtypes = [vp, dp, C.c_int]
    L.dogleg_gpu_batch_covariance.restype = C.c_int
    L.dogleg_gpu_batch_covariance_device.argtypes = [vp, vp, C.c_int, vp]
    L.dogleg_gpu_batch_covariance_device.restype = C.c_int
    L.dogleg_gpu_batch_free.argtypes = [C.POINTER(vp)]
    L.dogleg_gpu_batch_free.restype = None
    L.dogleg_gpu_release_batched_cache.restype = None
    L.dogleg_gpu_batched_stats.argtypes = [dp]
    L.dogleg_gpu_batched_stats.restype = None
    # row-sharded multi-GPU solves (NCCL inside the library)
    L.dogleg_gpu_nccl_get_unique_id.argtypes = [vp]
    L.dogleg_gpu_nccl_init.argtypes = [C.c_int, C.c_int, vp]
    L.dogleg_gpu_nccl_finalize.restype = None
    L.dogleg_gpu_nccl_world.restype = C.c_int
    L.dogleg_gpu_optimize_sparse_sharded.argtypes = [dp, C.c_uint, C.c_uint, ip, ip, C.c_uint, C.c_uint, vp, vp, vp, PP,
                                                     C.POINTER(vp)]
    L.dogleg_gpu_optimize_sparse_sharded.restype = C.c_double
    L.dogleg_gpu_optimize_dense_sharded.argtypes = [dp, C.c_uint, C.c_uint, C.c_uint, C.c_uint, vp, vp, vp, PP, C.POINTER(vp)]
    L.dogleg_gpu_optimize_dense_sharded.restype = C.c_double
    L.dlb_engine_create3.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_int, C.c_int, C.c_int, C.c_uint, C.c_uint]
    L.dlb_engine_create3.restype = vp
    L.dogleg_gpu_get_comm_stats.argtypes = [dp]
    L.dogleg_gpu_get_comm_stats.restype = None
    L.dlb_engine_comm_stats.argtypes = [vp, dp]
    L.dlb_engine_comm_stats.restype = None
    L.dlb_symbolic_create.argtypes = [C.c_int, C.c_int, ip, ip, ip, C.c_int]
    L.dlb_symbolic_create.restype = vp
    L.dlb_symbolic_free.argtypes = [vp]
    L.dlb_symbolic_free.restype = None
    L.dlb_symbolic_info.argtypes = [vp, C.POINTER(C.c_longlong)]
    L.dlb_symbolic_info.restype = None
    L.dlb_symbolic_get.argtypes = [vp, C.c_int, ip, C.c_longlong]
    L.dlb_symbolic_get.restype = C.c_longlong
    llp = C.POINTER(C.c_longlong)
    L.dlb_symbolic_front_off.argtypes = [vp, llp, C.c_longlong]
    L.dlb_symbolic_front_off.restype = C.c_longlong
    L.dlb_gather_plan_create.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    L.dlb_gather_plan_create.restype = vp
    L.dlb_gather_plan_free.argtypes = [vp]
    L.dlb_gather_plan_free.restype = None
    L.dlb_gather_plan_info.argtypes = [vp, llp]
    L.dlb_gather_plan_info.restype = None
    L.dlb_gather_plan_get.argtypes = [vp, C.c_int, C.c_int, llp, C.c_longlong]
    L.dlb_gather_plan_get.restype = C.c_longlong
    L.dlb_task_plan_create.argtypes = [vp, ip, C.c_int, C.c_int, C.c_int, C.c_int]
    L.dlb_task_plan_create.restype = vp
    L.dlb_task_plan_free.argtypes = [vp]
    L.dlb_task_plan_free.restype = None
    L.dlb_task_plan_get.argtypes = [vp, C.c_int, llp, C.c_longlong]
    L.dlb_task_plan_get.restype = C.c_longlong
    L.dlb_engine_create.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_int, C.c_int]
    L.dlb_engine_create.restype = vp
    L.dlb_engine_create2.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_int, C.c_int, C.c_int]
    L.dlb_engine_create2.restype = vp
    L.dogleg_gpu_release_cache.restype = None
    L.dlb_engine_destroy.argtypes = [vp]
    L.dlb_engine_destroy.restype = None
    L.dlb_engine_host_buffer.argtypes = [vp, C.c_int, C.c_int]
    L.dlb_engine_host_buffer.restype = vp
    L.dlb_engine_device_buffer.argtypes = [vp, C.c_int, C.c_int]
    L.dlb_engine_device_buffer.restype = vp
    L.dlb_engine_stream.argtypes = [vp]
    L.dlb_engine_stream.restype = vp
    L.dlb_engine_set_pattern.argtypes = [vp, ip, ip, ip, C.c_int]
    L.dlb_engine_symbolic.argtypes = [vp]
    L.dlb_engine_symbolic.restype = vp
    L.dlb_engine_evaluate.argtypes = [vp, C.c_int, C.c_int, C.c_double]
    L.dlb_engine_cauchy.argtypes = [vp, C.c_int]
    L.dlb_engine_factorize.argtypes = [vp, C.c_int, C.c_double]
    L.dlb_engine_gauss_newton.argtypes = [vp, C.c_int]
    L.dlb_engine_step.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_double]
    L.dlb_engine_has_trial.argtypes = [vp]
    L.dlb_engine_has_fused_eval.argtypes = [vp]
    L.dlb_engine_has_fused_eval.restype = C.c_int
    L.dlb_engine_trial.argtypes = [vp, C.c_int, C.c_int, C.c_double, C.c_double]
    L.dlb_engine_download.argtypes = [vp, C.c_int]
    L.dlb_engine_upload_p.argtypes = [vp, C.c_int]
    L.dlb_engine_scalars.argtypes = [vp]
    L.dlb_engine_scalars.restype = C.POINTER(Scalars)
    L.dlb_engine_solve.argtypes = [vp, dp, dp, C.c_int]
    L.dlb_engine_debug_JtJ.argtypes = [vp, C.c_int, C.c_double, dp]
    L.dlb_engine_dense_factor_to_host.argtypes = [vp, dp]
    L.dlb_engine_counters.argtypes = [vp, dp]
    L.dlb_engine_counters.restype = None
    L.dlb_engine_enable_timing.argtypes = [vp, C.c_int]
    L.dlb_engine_enable_timing.restype = None
    L.dlb_engine_phase_ms.argtypes = [vp, dp]
    L.dlb_engine_phase_ms.restype = None
    _lib = L
    return L


def default_parameters():
    P = Parameters()
    load().dogleg_getDefaultParameters(C.byref(P))
    return P
