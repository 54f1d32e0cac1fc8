"""Dense-products solves with device callbacks: dogleg_gpu_optimize_dense_products_batched (the whole
trust-region automaton on the device, the callback hands over |x|^2, J'x and J'J) and the single-problem
dogleg_gpu_optimize_dense_products. Every problem must end where the reference's
dogleg_optimize_dense_products ends for the same problem: same number of accepted steps, cost within
1e-9 relative, p within 1e-7. The CPU part checks that both entry points fail loudly without a GPU."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from libdogleg_b200 import ffi
from support import products as HP

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAYOUTS = [("products-unpacked", False), ("products-packed-upper", True)]


def ref_solve(H, prob, mode, p0, **pk):
    if H.reference_lib() is not None:
        r = H.solve_reference(prob, mode, p0=p0, **pk)
        o = H.solve_oracle(prob, mode, p0=p0, **pk)
        r.accepted = o.accepted
        return r
    return H.solve_oracle(prob, mode, p0=p0, **pk)


def assert_matches(it, n2, p, ref, what=None):
    assert it == ref.accepted, (what, it, ref.accepted)
    assert abs(n2 - ref.norm2x) <= 1e-9 * ref.norm2x, (what, n2, ref.norm2x)
    assert np.max(np.abs(p - ref.p)) <= 1e-7 * max(1.0, np.max(np.abs(ref.p))), what


def test_no_gpu_means_loud_failure_for_device_products(H):
    """Without a CUDA device both products entry points return <0 and say why (no CPU fallback)."""
    L = ffi.load()
    if L.dogleg_gpu_device_count() > 0:
        pytest.skip("a GPU is present")
    cb = H.problems_lib().dlb_cb_products_ptr()          # any non-NULL function: it is never called
    p = np.zeros((4, 6))
    assert L.dogleg_gpu_optimize_dense_products_batched(H.as_dp(p), 6, 4, cb, None, None, None, None) < 0
    assert b"no CUDA device" in L.dogleg_gpu_last_error()
    assert L.dogleg_gpu_optimize_dense_products(H.as_dp(p), 6, cb, None, None, None) < 0
    assert b"no CUDA device" in L.dogleg_gpu_last_error()


@pytest.mark.gpu
@pytest.mark.parametrize("mode,packed", LAYOUTS)
@pytest.mark.parametrize("tr0", [1e3, 0.3])
def test_products_batched_synthetic_matches_reference(H, mode, packed, tr0):
    B, N, M, seed = 40, 16, 256, 1000
    dev, p0 = HP.create_batched(B, M, N, seed)
    rc, p, n2, it = HP.solve_batched(dev, p0, N, packed=packed, max_iterations=30, trustregion0=tr0)
    HP.free(dev)
    assert rc == B
    for b in range(0, B, 3):
        prob = H.Problem.dense(N, M, seed=seed + b)
        ref = ref_solve(H, prob, mode, p0[b], max_iterations=30, trustregion0=tr0)
        assert_matches(it[b], n2[b], p[b], ref, b)


@pytest.mark.gpu
@pytest.mark.parametrize("mode,packed", LAYOUTS)
def test_products_batched_sample_surface_with_rejections(H, mode, packed):
    """The reference's sample problem from 32 start points: rejected trials retry on the cached J'J of the
    current point (the callback's buffer already holds the rejected point's)."""
    prob = H.Problem.sample()
    rng = np.random.default_rng(5)
    starts = [[5, -3, 2, 1, 0, 10], [-2, 4, -1, 3, 3, 3], [0.1, 0.1, 0.1, 0, 0, 0], list(prob.p0())]
    starts += [list(rng.uniform(-3, 6, 6)) for _ in range(28)]
    p0 = np.array(starts, dtype=float)
    B = len(p0)
    dev = HP.from_host(prob, B)
    rc, p, n2, it = HP.solve_batched(dev, p0, 6, packed=packed, max_iterations=60)
    HP.free(dev)
    assert rc == B
    nrej = 0
    for b in range(B):
        ref = H.solve_oracle(prob, mode, p0=p0[b], max_iterations=60)
        nrej += sum(1 for t in ref.trials if not t.accepted)
        assert_matches(it[b], n2[b], p[b], ref, b)
    assert nrej > 10


@pytest.mark.gpu
@pytest.mark.parametrize("mode,packed", LAYOUTS)
@pytest.mark.parametrize("N", [1, 7, 8, 9, 17, 31, 32])
def test_products_batched_tile_boundaries(H, N, mode, packed):
    """Every instantiation of the kernel (8-wide state tiles) and the packed-row walk at odd sizes."""
    B, M, seed = 6, 96, 40 + N
    dev, p0 = HP.create_batched(B, M, N, seed)
    rc, p, n2, it = HP.solve_batched(dev, p0, N, packed=packed, max_iterations=25)
    HP.free(dev)
    assert rc == B
    for b in range(B):
        prob = H.Problem.dense(N, M, seed=seed + b)
        ref = ref_solve(H, prob, mode, p0[b], max_iterations=25)
        assert_matches(it[b], n2[b], p[b], ref, (N, b))


@pytest.mark.gpu
def test_products_and_dense_batched_forms_agree(H):
    B, N, M, seed = 64, 16, 256, 77
    DL = H.dev_problems_lib()
    p0 = np.zeros((B, N))
    dense = DL.dlb_dev_problem_create_batched(B, M, N, seed, H.as_dp(p0))
    assert dense
    prod, p0p = HP.create_batched(B, M, N, seed)
    assert np.array_equal(p0, p0p)
    rc_d, p_d, n2_d, it_d = H.solve_batched(dense, p0, N, M, max_iterations=30)
    rc_p, p_p, n2_p, it_p = HP.solve_batched(prod, p0, N, max_iterations=30)
    DL.dlb_dev_problem_free(dense)
    HP.free(prod)
    assert rc_d == rc_p == B
    assert np.array_equal(it_d, it_p)
    assert np.max(np.abs(p_d - p_p)) <= 1e-7 * max(1.0, np.max(np.abs(p_d)))
    assert np.max(np.abs(n2_d - n2_p) / n2_d) <= 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("packed", [False, True])
def test_products_batched_ignores_inactive_outputs(H, packed):
    """A callback that writes NaN into every output of a finished problem changes nothing."""
    B, N, M, seed = 48, 12, 128, 300
    dev, p0 = HP.create_batched(B, M, N, seed)
    a = HP.solve_batched(dev, p0, N, packed=packed, max_iterations=30)
    b = HP.solve_batched(dev, p0, N, packed=packed, poison_inactive=True, max_iterations=30)
    HP.free(dev)
    assert a[0] == b[0] == B
    assert len(set(a[3].tolist())) > 1                 # problems finish at different trials
    for u, v in zip(a[1:], b[1:]):
        assert np.array_equal(u, v)


@pytest.mark.gpu
def test_products_rejections_before_any_callback(H):
    lib = H.dlb.load()
    dev, p0 = HP.create_batched(2, 64, 33, 5)
    cbb, cb1 = HP.lib().dlb_prod_cb_batched_ptr(), HP.lib().dlb_prod_cb_ptr()
    lower = H.make_params(lib, packed=True, upper=False)
    cases = [
        (lambda: lib.dogleg_gpu_optimize_dense_products_batched(H.as_dp(p0), 33, 2, cbb, C.c_void_p(dev), None, None, None),
         b"Nstate <= 32"),
        (lambda: lib.dogleg_gpu_optimize_dense_products_batched(H.as_dp(p0), 16, 2, cbb, C.c_void_p(dev), C.byref(lower),
                                                                None, None), b"upper triangle"),
        (lambda: lib.dogleg_gpu_optimize_dense_products_batched(H.as_dp(p0), 16, 0, cbb, C.c_void_p(dev), None, None, None),
         b"bad arguments"),
        (lambda: lib.dogleg_gpu_optimize_dense_products_batched(H.as_dp(p0), 16, 2, None, C.c_void_p(dev), None, None, None),
         b"bad arguments"),
        (lambda: lib.dogleg_gpu_optimize_dense_products(H.as_dp(p0), 16, cb1, C.c_void_p(dev), C.byref(lower), None),
         b"upper triangle"),
        (lambda: lib.dogleg_gpu_optimize_dense_products(H.as_dp(p0), 0, cb1, C.c_void_p(dev), None, None), b"Nstate > 0"),
        (lambda: lib.dogleg_gpu_optimize_dense_products(H.as_dp(p0), 16, None, C.c_void_p(dev), None, None), b"callback"),
    ]
    for call, msg in cases:
        assert call() < 0
        assert msg in lib.dogleg_gpu_last_error(), (msg, lib.dogleg_gpu_last_error())
    assert HP.ncalls(dev) == 0
    HP.free(dev)


@pytest.mark.gpu
@pytest.mark.slow
def test_products_batched_beyond_hbm(H):
    """B = 40 000 problems of 65 536 measurements and 16 states: as Jacobians 336 GB, more than the
    device holds. The procedural callback regenerates the rows on every evaluation; the products form
    stores none of them."""
    lib = H.dlb.load()
    B, N, M, seed = 40000, 16, 65536, 9000
    dev, p0 = HP.create_batched(B, M, N, seed, stored=False)
    rc, p, n2, it = HP.solve_batched(dev, p0, N, packed=True, max_iterations=20)
    HP.free(dev)
    lib.dogleg_gpu_release_batched_cache()
    assert rc == B
    for b in (0, 12345, B - 1):
        prob = H.Problem.dense(N, M, seed=seed + b)
        assert np.allclose(prob.p0(), p0[b], rtol=0, atol=1e-14)    # host and procedural generators agree
        ref = ref_solve(H, prob, "products-packed-upper", p0[b], max_iterations=20)
        assert_matches(it[b], n2[b], p[b], ref, b)


@pytest.mark.gpu
def test_procedural_callback_equals_the_stored_one(H):
    """The procedural generator regenerates exactly the rows the stored batch holds."""
    B, N, M, seed = 24, 16, 256, 1000
    dev, p0 = HP.create_batched(B, M, N, seed)
    proc, p0b = HP.create_batched(B, M, N, seed, stored=False)
    assert np.array_equal(p0, p0b)
    a = HP.solve_batched(dev, p0, N, max_iterations=30)
    b = HP.solve_batched(proc, p0, N, max_iterations=30)
    HP.free(dev)
    HP.free(proc)
    assert np.array_equal(a[3], b[3])
    assert np.max(np.abs(a[1] - b[1])) <= 1e-12 * max(1.0, np.max(np.abs(a[1])))
    assert np.max(np.abs(a[2] - b[2]) / a[2]) <= 1e-12


def _context_lambda(ctx):
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "dogleg.h"\n'
           'int main(void){printf("%zu\\n", offsetof(dogleg_solverContext_t, lambda));return 0;}')
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "o.c"), "w").write(src)
        subprocess.run(["gcc", "-std=gnu11", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "compat"),
                        os.path.join(td, "o.c"), "-o", os.path.join(td, "o")], check=True)
        off = int(subprocess.run([os.path.join(td, "o")], capture_output=True, text=True, check=True).stdout)
    return C.c_double.from_address(ctx.value + off).value


@pytest.mark.gpu
@pytest.mark.parametrize("mode,packed", LAYOUTS)
@pytest.mark.parametrize("kind", ["sample", "dense40", "dense300"])
def test_single_problem_device_products_matches_reference(H, kind, mode, packed):
    prob = H.Problem.sample() if kind == "sample" else H.Problem.dense(int(kind[5:]), 2 * int(kind[5:]), seed=21)
    got = HP.solve_single(prob, packed=packed, max_iterations=50)
    ref = ref_solve(H, prob, mode, prob.p0(), max_iterations=50)
    assert got.norm2x >= 0
    assert_matches(got.accepted, got.norm2x, got.p, ref, kind)
    assert got.ncalls == ref.ncalls


@pytest.mark.gpu
@pytest.mark.parametrize("packed", [False, True])
def test_single_problem_device_products_returned_context_solve(H, packed):
    """With a returnContext, dogleg_gpu_solve works on the factor of the callback's J'J at the final point."""
    lib = H.dlb.load()
    lib.dogleg_gpu_solve.argtypes = [C.c_void_p, H.dp, H.dp, C.c_int]
    lib.dogleg_freeContext.argtypes = [C.POINTER(C.c_void_p)]
    N, M = 40, 80
    prob = H.Problem.dense(N, M, seed=33)
    got, ctx = HP.solve_single(prob, packed=packed, keep_context=True, max_iterations=50)
    assert got.norm2x >= 0 and ctx.value
    A = np.ctypeslib.as_array(prob.c.Adense, shape=(M, N))
    J = A * (1.0 + 0.3 * got.p * got.p)                   # problems.c: J = A dphi(p)
    lam = _context_lambda(ctx)
    rhs = np.asfortranarray(np.random.default_rng(8).standard_normal((N, 3)))
    X = np.zeros_like(rhs, order="F")
    assert lib.dogleg_gpu_solve(ctx, H.as_dp(rhs), H.as_dp(X), 3) == 0
    want = np.linalg.solve(J.T @ J + lam * np.eye(N), rhs)
    assert np.max(np.abs(X - want)) <= 1e-9 * np.max(np.abs(want))
    lib.dogleg_freeContext(C.byref(ctx))
