"""Ragged batched solves: loads tests/support/libdlb_ragged_dev.so (ragged_dev.cu: the problems and their callbacks)
and runs dogleg_gpu_optimize_dense_batched_ragged over them, or dogleg_gpu_optimize_dense_batched2 over the same batch
zero-padded to its longest problem. Used by tests/test_gpu_batched_ragged.py and profiles/micro/batched_ragged.py."""
import ctypes as C
import os

import numpy as np

from support import harness as H

vp = H.vp
_cache = {}


def lib():
    if "ragged" not in _cache:
        path = os.path.join(H.ROOT, "tests", "support", "libdlb_ragged_dev.so")
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
        L.dlb_ragged_rows.argtypes = [vp]
        L.dlb_ragged_rows.restype = C.c_longlong
        L.dlb_ragged_ncalls.argtypes = [vp]
        L.dlb_ragged_reset.argtypes = [vp]
        L.dlb_ragged_reset.restype = None
        L.dlb_ragged_cb.argtypes = [vp] * 5 + [C.c_int, vp, vp]
        L.dlb_ragged_cb.restype = None
        L.dlb_ragged_cb_padded.argtypes = [vp] * 4 + [C.c_int, vp, vp]
        L.dlb_ragged_cb_padded.restype = None
        for n in ("dlb_ragged_cb_ptr", "dlb_ragged_cb_padded_ptr"):
            getattr(L, n).restype = vp
        _cache["ragged"] = L
    return _cache["ragged"]


def as_counts(counts):
    return np.ascontiguousarray(counts, dtype=np.uint32)


def as_up(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint))


def offsets(counts):
    return np.concatenate([[0], np.cumsum(np.asarray(counts, dtype=np.int64))])


def create(counts, N, seed):
    """Problem b = the first counts[b] rows of k_gen_batched's problem seed + b (Problem.dense(N, counts[b], seed + b)
    on the host). Returns (dev, p0 B x N)."""
    c = as_counts(counts)
    p0 = np.zeros((len(c), N))
    dev = lib().dlb_ragged_create(len(c), N, as_up(c), seed, H.as_dp(p0))
    assert dev
    return dev, p0


def create_sample(prob, counts):
    """Problem b = the reference's sample surface on its first counts[b] points."""
    c = as_counts(counts)
    dev = lib().dlb_ragged_create_sample(C.cast(prob.ptr, vp), len(c), as_up(c))
    assert dev
    return dev


def free(dev):
    lib().dlb_ragged_free(dev)


def ncalls(dev):
    return lib().dlb_ragged_ncalls(dev)


def mpad(dev):
    return lib().dlb_ragged_mpad(dev)


def solve(dev, p0, N, counts, handle=False, **pk):
    """dogleg_gpu_optimize_dense_batched_ragged: (rc, p, norm2x, iterations, handle or None)."""
    L = H.dlb.load()
    P = H.make_params(L, **pk)
    p = np.ascontiguousarray(p0, dtype=np.float64).copy()
    B = p.shape[0]
    n2 = np.zeros(B)
    it = np.zeros(B, dtype=np.int32)
    h = C.c_void_p()
    c = as_counts(counts)
    rc = L.dogleg_gpu_optimize_dense_batched_ragged(H.as_dp(p), N, as_up(c), B, lib().dlb_ragged_cb_ptr(), C.c_void_p(dev),
                                                    C.byref(P), H.as_dp(n2), H.as_ip(it), C.byref(h) if handle else None)
    if rc < 0:
        raise RuntimeError(L.dogleg_gpu_last_error().decode())
    return rc, p, n2, it, (h if handle else None)


def solve_padded(dev, p0, N, handle=False, **pk):
    """dogleg_gpu_optimize_dense_batched2 on the batch zero-padded to Nmeas = its longest count."""
    L = H.dlb.load()
    P = H.make_params(L, **pk)
    p = np.ascontiguousarray(p0, dtype=np.float64).copy()
    B = p.shape[0]
    n2 = np.zeros(B)
    it = np.zeros(B, dtype=np.int32)
    h = C.c_void_p()
    rc = L.dogleg_gpu_optimize_dense_batched2(H.as_dp(p), N, mpad(dev), B, lib().dlb_ragged_cb_padded_ptr(), C.c_void_p(dev),
                                              C.byref(P), H.as_dp(n2), H.as_ip(it), C.byref(h) if handle else None)
    if rc < 0:
        raise RuntimeError(L.dogleg_gpu_last_error().decode())
    return rc, p, n2, it, (h if handle else None)
