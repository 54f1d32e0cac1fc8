"""Dense-products solves with device callbacks: loads tests/support/libdlb_products_dev.so (the device
callbacks and their problems) and runs dogleg_gpu_optimize_dense_products(_batched) through it.
Used by tests/test_gpu_products_device.py and profiles/micro/batched_products.py."""
import ctypes as C
import os

import numpy as np

from support import harness as H

dp, ip, vp = H.dp, H.ip, H.vp
_cache = {}


def lib():
    if "prod" not in _cache:
        path = os.path.join(H.ROOT, "tests", "support", "libdlb_products_dev.so")
        if not os.path.exists(path):
            import __graft_entry__ as g
            g.build_support()
        L = C.CDLL(path, mode=C.RTLD_LOCAL)
        L.dlb_prod_problem_create_batched.restype = vp
        L.dlb_prod_problem_create_batched.argtypes = [C.c_int, C.c_int, C.c_int, C.c_ulonglong, C.c_int, dp]
        L.dlb_prod_problem_from_host.restype = vp
        L.dlb_prod_problem_from_host.argtypes = [vp, C.c_int]
        L.dlb_prod_problem_free.argtypes = [vp]
        L.dlb_prod_problem_free.restype = None
        L.dlb_prod_problem_layout.argtypes = [vp, C.c_int, C.c_int]
        L.dlb_prod_problem_layout.restype = None
        L.dlb_prod_problem_timing.argtypes = [vp, C.c_int]
        L.dlb_prod_problem_ms.argtypes = [vp]
        L.dlb_prod_problem_ms.restype = C.c_double
        L.dlb_prod_problem_ncalls.argtypes = [vp]
        for n in ("dlb_prod_cb_ptr", "dlb_prod_cb_batched_ptr"):
            getattr(L, n).restype = vp
        _cache["prod"] = L
    return _cache["prod"]


def create_batched(B, M, N, seed, stored=True):
    """B problems of the k_gen_batched family (problem b = the host's Problem.dense(N, M, seed + b)), stored in HBM or
    regenerated on every callback (stored=False). Returns (handle, p0 B x N)."""
    p0 = np.zeros((B, N))
    dev = lib().dlb_prod_problem_create_batched(B, M, N, seed, int(stored), H.as_dp(p0))
    assert dev
    return dev, p0


def from_host(prob, B=1):
    """The sample surface (B copies) or one dense host problem."""
    dev = lib().dlb_prod_problem_from_host(C.cast(prob.ptr, vp), B)
    assert dev
    return dev


def free(dev):
    lib().dlb_prod_problem_free(dev)


def ncalls(dev):
    return lib().dlb_prod_problem_ncalls(dev)


def solve_batched(dev, p0, N, packed=False, poison_inactive=False, **pk):
    """dogleg_gpu_optimize_dense_products_batched over `dev`; JtJ full or packed upper; p0 is B x N."""
    L = H.dlb.load()
    lib().dlb_prod_problem_layout(dev, int(packed), int(poison_inactive))
    P = H.make_params(L, packed=packed, upper=packed, **pk)
    p = np.ascontiguousarray(p0, dtype=np.float64).copy()
    B = p.shape[0]
    n2 = np.zeros(B)
    it = np.zeros(B, dtype=np.int32)
    rc = L.dogleg_gpu_optimize_dense_products_batched(H.as_dp(p), N, B, lib().dlb_prod_cb_batched_ptr(), C.c_void_p(dev),
                                                      C.byref(P), H.as_dp(n2), H.as_ip(it))
    if rc < 0:
        raise RuntimeError(L.dogleg_gpu_last_error().decode())
    return rc, p, n2, it


def solve_single(prob, packed=False, p0=None, keep_context=False, **pk):
    """dogleg_gpu_optimize_dense_products with the device callback (the batched one with B = 1) on a dense or
    sample host problem. keep_context: also returns the context (the caller frees it)."""
    L = H.dlb.load()
    dev = from_host(prob, 1)
    lib().dlb_prod_problem_layout(dev, int(packed), 0)
    P = H.make_params(L, packed=packed, upper=packed, **pk)
    p = (prob.p0() if p0 is None else np.array(p0, dtype=np.float64)).copy()
    ctx = C.c_void_p()
    r = L.dogleg_gpu_optimize_dense_products(H.as_dp(p), prob.N, lib().dlb_prod_cb_ptr(), C.c_void_p(dev),
                                             C.byref(P), C.byref(ctx) if keep_context else None)
    st = np.zeros(8)
    L.dogleg_gpu_get_stats(None, H.as_dp(st))
    n = ncalls(dev)
    free(dev)
    res = H.Result(norm2x=r, p=p, accepted=int(st[0]), ncalls=n, stats=st)
    return (res, ctx) if keep_context else res
