"""Batched solves with a float Jacobian: loads tests/support/libdlb_f32jac_dev.so (f32jac_dev.cu: ragged_dev.cu's
problems with float callbacks and their widened twins) and runs dogleg_gpu_optimize_dense_batched_f32jac /
_ragged_f32jac over them, or the double entry points with the widened twin (J = (double)(float)J) or with ragged_dev.cu's
unrounded double callbacks. Used by tests/test_gpu_batched_f32jac.py and profiles/micro/batched_f32jac.py."""
import ctypes as C
import os

import numpy as np

from support import harness as H
from support import ragged as HR

vp = H.vp
_cache = {}


def lib():
    if "f32" not in _cache:
        path = os.path.join(H.ROOT, "tests", "support", "libdlb_f32jac_dev.so")
        if not os.path.exists(path):
            import __graft_entry__ as g
            g.build_support()
        L = C.CDLL(path, mode=C.RTLD_LOCAL)
        up = C.POINTER(C.c_uint)
        L.dlb_ragged_create.restype = vp
        L.dlb_ragged_create.argtypes = [C.c_int, C.c_int, up, C.c_ulonglong, H.dp]
        L.dlb_ragged_create_sample.restype = vp
        L.dlb_ragged_create_sample.argtypes = [vp, C.c_int, up]
        L.dlb_ragged_free.argtypes = [vp]
        L.dlb_ragged_free.restype = None
        L.dlb_ragged_mpad.argtypes = [vp]
        L.dlb_ragged_ncalls.argtypes = [vp]
        L.dlb_ragged_reset.argtypes = [vp]
        L.dlb_ragged_reset.restype = None
        for n in ("dlb_f32_cb_ragged", "dlb_f32_cb_ragged_twin", "dlb_ragged_cb"):
            getattr(L, n).argtypes = [vp] * 5 + [C.c_int, vp, vp]
            getattr(L, n).restype = None
        for n in ("dlb_f32_cb_uniform", "dlb_f32_cb_uniform_twin", "dlb_ragged_cb_padded"):
            getattr(L, n).argtypes = [vp] * 4 + [C.c_int, vp, vp]
            getattr(L, n).restype = None
        for n in ("dlb_f32_cb_ragged_ptr", "dlb_f32_cb_ragged_twin_ptr", "dlb_f32_cb_uniform_ptr",
                  "dlb_f32_cb_uniform_twin_ptr", "dlb_ragged_cb_ptr", "dlb_ragged_cb_padded_ptr"):
            getattr(L, n).restype = vp
        _cache["f32"] = L
    return _cache["f32"]


def create(counts, N, seed):
    """ragged.create's problems, owned by this library. Returns (dev, p0 B x N)."""
    c = HR.as_counts(counts)
    p0 = np.zeros((len(c), N))
    dev = lib().dlb_ragged_create(len(c), N, HR.as_up(c), seed, H.as_dp(p0))
    assert dev
    return dev, p0


def create_sample(prob, counts):
    c = HR.as_counts(counts)
    dev = lib().dlb_ragged_create_sample(C.cast(prob.ptr, vp), len(c), HR.as_up(c))
    assert dev
    return dev


def free(dev):
    lib().dlb_ragged_free(dev)


def ncalls(dev):
    return lib().dlb_ragged_ncalls(dev)


def reset(dev):
    lib().dlb_ragged_reset(dev)


def mpad(dev):
    return lib().dlb_ragged_mpad(dev)


# (entry point, callback) of each solve kind; the uniform kinds run on the batch padded to Nmeas = mpad(dev)
KINDS = {
    "uniform_f32": ("dogleg_gpu_optimize_dense_batched_f32jac", "dlb_f32_cb_uniform_ptr"),
    "uniform_twin": ("dogleg_gpu_optimize_dense_batched2", "dlb_f32_cb_uniform_twin_ptr"),
    "uniform_f64": ("dogleg_gpu_optimize_dense_batched2", "dlb_ragged_cb_padded_ptr"),
    "ragged_f32": ("dogleg_gpu_optimize_dense_batched_ragged_f32jac", "dlb_f32_cb_ragged_ptr"),
    "ragged_twin": ("dogleg_gpu_optimize_dense_batched_ragged", "dlb_f32_cb_ragged_twin_ptr"),
    "ragged_f64": ("dogleg_gpu_optimize_dense_batched_ragged", "dlb_ragged_cb_ptr"),
}


def solve(kind, dev, p0, N, counts=None, handle=False, **pk):
    """One solve of KINDS[kind]: (rc, p, norm2x, iterations, handle or None). counts: the ragged kinds' Nmeas."""
    L = H.dlb.load()
    entry, cb = KINDS[kind]
    P = H.make_params(L, **pk)
    p = np.ascontiguousarray(p0, dtype=np.float64).copy()
    B = p.shape[0]
    n2 = np.zeros(B)
    it = np.zeros(B, dtype=np.int32)
    h = C.c_void_p()
    meas = HR.as_up(HR.as_counts(counts)) if kind.startswith("ragged") else mpad(dev)
    rc = getattr(L, entry)(H.as_dp(p), N, meas, B, getattr(lib(), cb)(), C.c_void_p(dev), C.byref(P), H.as_dp(n2),
                           H.as_ip(it), C.byref(h) if handle else None)
    if rc < 0:
        raise RuntimeError(L.dogleg_gpu_last_error().decode())
    return rc, p, n2, it, (h if handle else None)
