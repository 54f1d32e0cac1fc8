"""GPU parity tests of whole solves through the public dogleg.h API: the product
must request the same sequence of operating points from the callback as the
reference (that pins step type, step vector, acceptance and trust-region
evolution, SURVEY.md 7.1-0), end at the same cost and state, in the same number
of iterations. Reference = the unmodified reference code in oracle/_ref when it
is present, and always the committed golden fixtures in tests/golden/.
Tolerances (BASELINE.json): cost 1e-9 relative, p 1e-7, equal iteration count."""
import json
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
COST_RTOL, P_TOL = 1e-9, 1e-7


def close_trace(a, gold_p, gold_x):
    assert len(a.trace_norm2x) == len(gold_x), "different number of callback evaluations"
    assert np.allclose(a.trace_norm2x, gold_x, rtol=COST_RTOL, atol=0)
    assert np.max(np.abs(a.trace_p - np.asarray(gold_p))) <= P_TOL * max(1.0, np.max(np.abs(gold_p)))


@pytest.mark.parametrize("mode", ["sparse", "dense", "products-packed-upper", "products-unpacked"])
def test_sample_problem_matches_golden_trace(H, mode):
    gold = json.load(open(os.path.join(GOLD, "sample_reference.json")))[mode]
    r = H.solve_product(H.Problem.sample(), mode, max_iterations=8)
    assert r.norm2x >= 0
    assert r.ncalls == gold["ncalls"] and r.accepted == 6
    assert abs(r.norm2x - gold["norm2x"]) <= COST_RTOL * gold["norm2x"]
    assert np.max(np.abs(r.p - np.asarray(gold["p"]))) <= P_TOL
    close_trace(r, gold["trace_p"], gold["trace_norm2x"])
    assert np.max(np.abs(r.p - np.arange(1, 7))) < 5e-2          # the reference's own --check criterion


CASES = {"mrcal_2x6x12": lambda H: H.Problem.mrcal(2, 6, 12, seed=7),
         "mrcal_4x20x5": lambda H: H.Problem.mrcal(4, 20, 5, seed=2),
         "random_60x300": lambda H: H.Problem.random_sparse(60, 300, 5, seed=1),
         "ba_10x60": lambda H: H.Problem.ba(10, 60, 3, 5, 0, seed=4),
         "dense_16x256": lambda H: H.Problem.dense(16, 256, seed=3)}


@pytest.mark.parametrize("name", list(CASES))
def test_solves_match_dense_reference_fixture(H, name):
    """Sparse problems densified through the REAL reference (LAPACK) pin the sparse GPU path."""
    gold = json.load(open(os.path.join(GOLD, "dense_reference_cases.json")))[name]
    prob = CASES[name](H)
    modes = ["dense"] if name.startswith("dense") else ["sparse", "dense", "products-unpacked"]
    for mode in modes:
        r = H.solve_product(prob, mode, max_iterations=20)
        assert r.ncalls == gold["ncalls"]
        close_trace(r, gold["trace_p"], gold["trace_norm2x"])
        assert abs(r.norm2x - gold["norm2x"]) <= COST_RTOL * gold["norm2x"]


@pytest.mark.parametrize("tr0", [1e3, 0.3, 0.002])
@pytest.mark.parametrize("mode", ["sparse", "dense", "products-packed-upper", "products-unpacked"])
def test_solves_match_live_reference(H, mode, tr0):
    """Cauchy-clipped, interpolated and Gauss-Newton steps (small trust regions force the first two)."""
    prob = H.Problem.mrcal(3, 8, 6, seed=11)
    ref = H.solve_reference(prob, mode, max_iterations=30, trustregion0=tr0) if H.reference_lib() is not None \
        else H.solve_oracle(prob, mode, max_iterations=30, trustregion0=tr0)
    got = H.solve_product(prob, mode, max_iterations=30, trustregion0=tr0)
    assert got.ncalls == ref.ncalls
    close_trace(got, ref.trace_p, ref.trace_norm2x)
    assert abs(got.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)
    assert np.max(np.abs(got.p - ref.p)) <= P_TOL * max(1.0, np.max(np.abs(ref.p)))


@pytest.mark.parametrize("jv_pass", ["0", "1"])
@pytest.mark.parametrize("ranges", ["1", "0"])
def test_long_periodic_runs_match_oracle(H, monkeypatch, ranges, jv_pass):
    """Calibration layout with hundreds of points per frame and camera: the measurement columns form
    long runs of alternating x/y classes, which the gradient (and, with DOGLEG_GPU_JV_PASS=1, the
    |Jv|^2) kernels read as contiguous range tasks (DOGLEG_GPU_RANGE=0: the class-task kernels
    instead). Default |Jv|^2: v'(JtJ)v on the assembled class blocks."""
    monkeypatch.setenv("DOGLEG_GPU_RANGE", ranges)
    monkeypatch.setenv("DOGLEG_GPU_JV_PASS", jv_pass)
    monkeypatch.setenv("DOGLEG_GPU_ENGINE_CACHE", "0")
    prob = H.Problem.mrcal(3, 5, 150, seed=9)
    ref = H.solve_oracle(prob, "sparse", max_iterations=20)
    got = H.solve_product(prob, "sparse", max_iterations=20)
    assert got.ncalls == ref.ncalls and got.accepted == ref.accepted
    close_trace(got, ref.trace_p, ref.trace_norm2x)
    assert abs(got.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)


@pytest.mark.parametrize("jv_pass", ["0", "1"])
@pytest.mark.parametrize("shape", [(40, 3000, 7), (300, 20000, 40)])
def test_ragged_and_empty_columns_match_reference(H, monkeypatch, shape, jv_pass):
    """Measurement columns of every length from 0 to kmax (kmax 40: longer than a warp), runs of
    empty columns (they count in |x|^2 only), a periodic run that alternates with an empty class,
    single-entry columns. Checked against the unmodified reference on the densified problem (same
    control logic, mathematically identical JtJ) and against the sparse oracle; host and device
    callbacks."""
    monkeypatch.setenv("DOGLEG_GPU_JV_PASS", jv_pass)
    monkeypatch.setenv("DOGLEG_GPU_ENGINE_CACHE", "0")
    prob = H.Problem.ragged(*shape)
    Jp, _ = prob.pattern()
    lens = np.diff(Jp)
    assert lens.min() == 0 and lens.max() == shape[2] and (lens == 0).sum() > 200
    ref = H.solve_oracle(prob, "sparse", max_iterations=30)
    if H.reference_lib() is not None:
        dref = H.solve_reference(prob, "dense", max_iterations=30)
        assert dref.ncalls == ref.ncalls and abs(dref.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)
    got = H.solve_product(prob, "sparse", max_iterations=30)
    assert got.ncalls == ref.ncalls and got.accepted == ref.accepted
    close_trace(got, ref.trace_p, ref.trace_norm2x)
    assert abs(got.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)
    assert np.max(np.abs(got.p - ref.p)) <= P_TOL * max(1.0, np.max(np.abs(ref.p)))
    dev = H.solve_product_device(prob, "sparse", max_iterations=30)
    assert dev.ncalls == ref.ncalls and dev.accepted == ref.accepted
    assert abs(dev.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)
    assert np.max(np.abs(dev.p - ref.p)) <= P_TOL * max(1.0, np.max(np.abs(ref.p)))


TINY = [("sparse", 1, 50), ("sparse", 2, 40), ("dense", 1, 20), ("dense", 2, 30),
        ("products-packed-upper", 1, 20), ("products-unpacked", 2, 30)]


@pytest.mark.parametrize("mode,N,M", TINY)
def test_smallest_problems_match_reference(H, mode, N, M):
    """One and two states: single-column fronts, 1x1 factors, grids smaller than a warp."""
    prob = H.Problem.random_sparse(N, M, N, seed=3) if mode == "sparse" else H.Problem.dense(N, M, seed=3)
    ref_mode = "dense" if mode == "sparse" else mode      # the reference's sparse path needs CHOLMOD
    ref = H.solve_reference(prob, ref_mode, max_iterations=30) if H.reference_lib() is not None \
        else H.solve_oracle(prob, mode, max_iterations=30)
    got = H.solve_product(prob, mode, max_iterations=30)
    assert got.ncalls == ref.ncalls
    close_trace(got, ref.trace_p, ref.trace_norm2x)
    assert abs(got.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)
    assert np.max(np.abs(got.p - ref.p)) <= P_TOL * max(1.0, np.max(np.abs(ref.p)))


def test_bundle_adjustment_scalar_leaf_kernel(H, monkeypatch):
    """The scalar warp-per-front leaf kernel (what fronts with more than 4 pivot columns use), forced."""
    monkeypatch.setenv("DOGLEG_GPU_LEAF_MMA", "0")
    monkeypatch.setenv("DOGLEG_GPU_LEAF_MIN", "1")
    monkeypatch.setenv("DOGLEG_GPU_ENGINE_CACHE", "0")
    prob = H.Problem.ba(30, 600, 4, 12, 20, seed=8)
    ref = H.solve_oracle(prob, "sparse", max_iterations=20)
    got = H.solve_product(prob, "sparse", max_iterations=20)
    assert got.ncalls == ref.ncalls and got.accepted == ref.accepted
    close_trace(got, ref.trace_p, ref.trace_norm2x)


@pytest.mark.parametrize("nd", ["0", "30,16,6"])
def test_bundle_adjustment_matches_oracle(H, monkeypatch, nd):
    """Bundle-adjustment structure (config C4 in miniature: one pattern class per camera-point pair,
    thousands of 3-column leaf fronts, a banded camera system on top): warp-per-task streaming
    kernels, the block gather of the point Schur complements, fronts beyond shared memory on the
    batched DMMA path, with and without the nested-dissection ordering. Oracle = CPU restatement
    (simplicial LDL'), same callbacks."""
    monkeypatch.setenv("DOGLEG_GPU_ND", nd)
    monkeypatch.setenv("DOGLEG_GPU_ENGINE_CACHE", "0")
    monkeypatch.setenv("DOGLEG_GPU_LEAF_MIN", "1" if nd == "0" else "1000000")    # with / without the fused leaf kernels
    prob = H.Problem.ba(60, 1500, 4, 24, 0, seed=4)
    ref = H.solve_oracle(prob, "sparse", max_iterations=20)
    got = H.solve_product(prob, "sparse", max_iterations=20)
    assert got.ncalls == ref.ncalls and got.accepted == ref.accepted
    close_trace(got, ref.trace_p, ref.trace_norm2x)
    assert abs(got.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)
    assert np.max(np.abs(got.p - ref.p)) <= P_TOL * max(1.0, np.max(np.abs(ref.p)))


@pytest.mark.parametrize("p0", [[5, -3, 2, 1, 0, 10], [-2, 4, -1, 3, 3, 3], [0.1, 0.1, 0.1, 0, 0, 0]])
@pytest.mark.parametrize("mode", ["sparse", "dense", "products-unpacked"])
def test_rejected_steps_and_far_start(H, mode, p0):
    """Starts from which the first Gauss-Newton step overshoots (the reference's sample surface is
    bilinear in a,b,c): rejections, trust-region collapse to |GN|, cauchy / interpolated recovery
    must follow the reference trial by trial."""
    prob = H.Problem.sample()
    p0 = np.array(p0, dtype=float)
    ref = H.solve_reference(prob, mode, p0=p0, max_iterations=60) if H.reference_lib() is not None \
        else H.solve_oracle(prob, mode, p0=p0, max_iterations=60)
    orc = H.solve_oracle(prob, mode, p0=p0, max_iterations=60)
    got = H.solve_product(prob, mode, p0=p0, max_iterations=60)
    assert any(t.accepted == 0 for t in orc.trials), "fixture no longer produces a rejected step"
    assert {t.step_type for t in orc.trials} == {0, 1, 2}
    assert got.ncalls == ref.ncalls and got.accepted == orc.accepted
    close_trace(got, ref.trace_p, ref.trace_norm2x)
    assert abs(got.norm2x - ref.norm2x) <= COST_RTOL * ref.norm2x


def test_vnlog_output_matches_reference_text(H, capfd):
    """The vnlog convergence log libdogleg.so prints for the reference's sample problem (sample.c's data and
    start, max_iterations 8, DOGLEG_DEBUG_VNLOG) must equal the log the reference's own `sample --diag vnlog`
    printed, field for field (SURVEY.md 4.1; tests/golden/sample_reference.json)."""
    import ctypes as C
    gold = json.load(open(os.path.join(GOLD, "sample_reference.json")))
    libc = C.CDLL(None)
    for mode in ["sparse", "dense", "products-packed-upper", "products-unpacked"]:
        libc.fflush(None)                              # the library prints with stdio
        capfd.readouterr()
        r = H.solve_product(H.Problem.sample(), mode, max_iterations=8, vnlog=True)
        libc.fflush(None)
        out = capfd.readouterr().out
        assert r.norm2x >= 0
        got = [l.split() for l in out.strip().splitlines()]
        want = [l.split() for l in gold[mode]["vnlog"].strip().splitlines()]
        assert got[0] == want[0]                       # legend
        assert len(got) == len(want)
        for g, w in zip(got[1:], want[1:]):
            assert len(g) == len(w)
            for a, b in zip(g, w):
                if a == b:
                    continue
                assert np.isclose(float(a), float(b), rtol=2e-5), (g, w)   # %g prints 6 digits
        assert np.max(np.abs(r.p - np.arange(1, 7))) < 5e-2          # what `sample --check` asserts


def test_streaming_host_callback_gives_identical_results(H):
    """dogleg_gpu_host_progress: a host callback that announces its finished columns (the pinned H2D then
    overlaps the callback on a side stream) must produce the same solve, bit for bit, as the same callback
    without announcements."""
    import ctypes as C
    lib = H.dlb.load()
    res = []
    for announce in (False, True):
        prob = H.Problem.mrcal(4, 40, 125, seed=2)           # 40 000 columns: 16 waves of 2 500
        prob.c.progress = C.cast(lib.dogleg_gpu_host_progress, C.c_void_p).value if announce else None
        res.append(H.solve_product(prob, "sparse", max_iterations=30))
        prob.c.progress = None
    a, b = res
    assert a.ncalls == b.ncalls and a.norm2x == b.norm2x and np.array_equal(a.p, b.p)
    ref = H.solve_oracle(H.Problem.mrcal(4, 40, 125, seed=2), "sparse", max_iterations=30)
    assert b.ncalls == ref.ncalls and abs(b.norm2x - ref.norm2x) <= COST_RTOL * ref.norm2x


def test_full_size_mrcal_problem_matches_the_reference(H):
    """VERDICT round 1, weak #1: the FULL C2 problem (Nstate 1268, Nmeas 1e6, 22.5 M nonzeros) through
    dogleg_optimize2 with host callbacks against the unmodified reference on the same inputs: same number
    of evaluations, cost to 1e-9, p to 1e-7 (the reference needs ~15 s on one host core). Without the
    reference, p comes from the oracle restatement, which must itself reproduce the reference's recorded
    evaluation count and cost (tests/golden/c2_reference.json)."""
    gold = json.load(open(os.path.join(GOLD, "c2_reference.json")))
    prob = H.Problem.mrcal(4, 200, 625, seed=2)
    ref = H.solve_reference(prob, "sparse", max_iterations=100) if H.reference_lib() is not None \
        else H.solve_oracle(prob, "sparse", max_iterations=100)
    assert ref.ncalls == gold["ncalls"]
    assert abs(ref.norm2x - gold["norm2x"]) <= COST_RTOL * gold["norm2x"]
    got = H.solve_product(prob, "sparse", max_iterations=100)
    assert got.ncalls == ref.ncalls
    assert abs(got.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)
    assert np.max(np.abs(got.p - ref.p)) <= 1e-7 * max(1.0, np.max(np.abs(ref.p)))
    dev = H.solve_product_device(prob, "sparse", max_iterations=100)
    assert dev.ncalls == ref.ncalls
    assert abs(dev.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)
    assert np.max(np.abs(dev.p - ref.p)) <= 1e-7 * max(1.0, np.max(np.abs(ref.p)))


@pytest.mark.skipif(os.environ.get("DLB_TEST_SLOW", "0") == "0", reason="minutes of CPU time in the oracle (DLB_TEST_SLOW=1 runs it)")
def test_bundle_adjustment_tenth_scale_matches_oracle(H):
    """C4 at 1/10 scale (1 000 cameras, 100 000 points) against the oracle restatement, capped at a few
    iterations (the oracle's simplicial factorization needs ~100 s per iteration here)."""
    prob = H.Problem.ba(1000, 100000, 4, 32, 0, seed=4)
    ref = H.solve_oracle(prob, "sparse", max_iterations=2)
    got = H.solve_product_device(prob, "sparse", max_iterations=2)
    assert got.ncalls == ref.ncalls
    assert abs(got.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)
    assert np.max(np.abs(got.p - ref.p)) <= 1e-7 * max(1.0, np.max(np.abs(ref.p)))


def test_lambda_ladder_on_singular_problem(H):
    """An unobservable state: the factorization must fail at lambda=0, climb 1e-10, 1e-9, ...
    and the solve must still converge; lambda is visible through the returned context."""
    import ctypes as C
    from libdogleg_b200 import ffi
    L = ffi.load()
    prob = H.Problem.random_sparse(30, 150, 4, seed=2)
    PL = H.problems_lib()
    P = H.make_params(L, max_iterations=20)
    N = prob.N + 1

    # wrap the C callback: same problem, one extra state nobody depends on
    CB = C.CFUNCTYPE(None, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p, C.c_void_p)
    inner = C.cast(PL.dlb_cb_sparse_ptr(), CB)

    def cb(p, x, Jt, cookie):
        inner(p, x, Jt, cookie)
    cbk = CB(cb)
    p = np.append(prob.p0(), 0.25)
    ctx = C.c_void_p()
    r = L.dogleg_optimize2(H.as_dp(p), N, prob.M, prob.nnz, C.cast(cbk, C.c_void_p), C.cast(prob.ptr, C.c_void_p),
                           C.byref(P), C.byref(ctx))
    assert r >= 0 and ctx.value
    ref = H.solve_oracle(prob, "sparse", max_iterations=20)
    assert abs(r - ref.norm2x) <= 1e-6 * ref.norm2x
    assert p[-1] == 0.25                                 # the unobservable state did not move
    L.dogleg_freeContext(C.byref(ctx))
    assert not ctx.value


def test_return_context_exposes_host_state(H):
    """returnContext: beforeStep's host arrays must hold the final state (SURVEY.md 5 checkpoint row)."""
    import ctypes as C
    from libdogleg_b200 import ffi
    L = ffi.load()
    prob = H.Problem.mrcal(2, 6, 12, seed=7)
    PL = H.problems_lib()
    P = H.make_params(L, max_iterations=20)
    p = prob.p0()
    ctx = C.c_void_p()
    r = L.dogleg_optimize2(H.as_dp(p), prob.N, prob.M, prob.nnz, PL.dlb_cb_sparse_ptr(),
                           C.cast(prob.ptr, C.c_void_p), C.byref(P), C.byref(ctx))
    assert r >= 0 and ctx.value

    class Point(C.Structure):
        _fields_ = [("p", C.POINTER(C.c_double)), ("x", C.POINTER(C.c_double)), ("norm2_x", C.c_double),
                    ("Jt", C.c_void_p), ("Jt_x", C.POINTER(C.c_double)), ("updateCauchy", C.POINTER(C.c_double)),
                    ("updateGN", C.c_void_p), ("norm2_updateCauchy", C.c_double), ("norm2_updateGN", C.c_double),
                    ("bits", C.c_int * 3), ("step_to_here", C.POINTER(C.c_double)), ("norm2_step_to_here", C.c_double)]
    # beforeStep sits right after {common, callback union, cookie}
    src = r'''#include <stdio.h>
#include "dogleg.h"
int main(void){printf("%zu %zu\n", offsetof(dogleg_solverContext_t, beforeStep), offsetof(dogleg_solverContext_t, lambda));return 0;}'''
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "o.c"), "w").write(src)
        subprocess.run(["gcc", "-std=gnu11", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "compat"),
                        os.path.join(td, "o.c"), "-o", os.path.join(td, "o")], check=True)
        o_before, o_lambda = map(int, subprocess.run([os.path.join(td, "o")], capture_output=True, text=True).stdout.split())
    before = C.cast(C.c_void_p.from_address(ctx.value + o_before).value, C.POINTER(Point)).contents
    lam = C.c_double.from_address(ctx.value + o_lambda).value
    assert lam == 0.0
    assert np.allclose(np.ctypeslib.as_array(before.p, shape=(prob.N,)), p, rtol=0, atol=0)
    assert before.norm2_x == r
    x, Jx = prob.evaluate(p)
    assert np.allclose(np.ctypeslib.as_array(before.x, shape=(prob.M,)), x, rtol=1e-13, atol=1e-15)
    Jp, Ji = prob.pattern()
    g = np.zeros(prob.N)
    H.oracle_lib().orc_Jt_times_x(H.as_dp(g), prob.N, prob.M, H.as_ip(Jp), H.as_ip(Ji), H.as_dp(Jx), H.as_dp(x))
    assert np.allclose(np.ctypeslib.as_array(before.Jt_x, shape=(prob.N,)), g, rtol=1e-9, atol=1e-12)
    # the public factorization entry point works on the returned context
    assert L.dogleg_computeJtJfactorization(C.addressof(before), ctx)
    assert before.bits[0] & 0x4                       # have_factorization
    L.dogleg_freeContext(C.byref(ctx))


def test_medium_size_properties(H):
    """At a size where the dense oracle is out of reach (Nmeas = 200k) use properties:
    linearity of Jt*x in x, |J v|^2 against the scalar oracle loop, symmetry and
    positive-definiteness of the solve (residual of (JtJ) gn = -Jt x)."""
    from libdogleg_b200 import ffi
    O = H.oracle_lib()
    prob = H.Problem.mrcal(4, 40, 625, seed=2)          # Nstate 308, Nmeas 200k, nnz 4.5M
    Jp, Ji = prob.pattern()
    p = prob.p0()
    x, Jx = prob.evaluate(p)
    E = H.Engine(ffi.SOLVE_SPARSE, prob.N, prob.M, len(Ji))
    E.load_sparse(0, p, x, Jp, Ji, Jx)
    sc = E.evaluate(0)
    g = E.download(0)["Jtx"]
    g_ref = np.zeros(prob.N)
    O.orc_Jt_times_x(H.as_dp(g_ref), prob.N, prob.M, H.as_ip(Jp), H.as_ip(Ji), H.as_dp(Jx), H.as_dp(x))
    assert np.max(np.abs(g - g_ref)) <= 1e-11 * np.max(np.abs(g_ref))
    assert np.isclose(sc.norm2_x, x @ x, rtol=1e-12)
    sc = E.cauchy(0)
    assert np.isclose(sc.norm2_JJtx, O.orc_norm2_J_times_v(prob.M, H.as_ip(Jp), H.as_ip(Ji), H.as_dp(Jx), H.as_dp(g_ref)), rtol=1e-10)
    assert E.factorize(0, 0.0) == -1
    E.gauss_newton(0)
    gn = E.download(0)["gn"]
    # residual check through the scalar oracle: Jt (J gn) == -g
    import scipy.sparse as sp
    Jt = sp.csc_matrix((Jx, Ji, Jp), shape=(prob.N, prob.M))
    res = Jt @ (Jt.T @ gn) + g_ref
    assert np.max(np.abs(res)) <= 1e-8 * np.max(np.abs(g_ref))
    # linearity: evaluating with 2x gives 2 g
    E.host(0, ffi.BUF_X, prob.M)[:] = 2 * x
    sc2 = E.evaluate(0)
    assert np.array_equal(E.download(0)["Jtx"], 2 * g)
    assert sc2.norm2_x == 4 * sc.norm2_x or np.isclose(sc2.norm2_x, 4 * (x @ x), rtol=1e-12)
    E.close()


@pytest.mark.parametrize("tr0", [1e3, 0.3])
def test_device_callback_solves_match_host_callback_solves(H, tr0):
    """dogleg_gpu_optimize_sparse/_dense (Jacobian produced in HBM, no PCIe traffic per evaluation)
    must walk the same path as dogleg_optimize2 with the host version of the same model."""
    prob = H.Problem.mrcal(3, 8, 6, seed=11)
    host = H.solve_product(prob, "sparse", max_iterations=30, trustregion0=tr0)
    dev = H.solve_product_device(prob, "sparse", max_iterations=30, trustregion0=tr0)
    assert dev.ncalls == host.ncalls and dev.accepted == host.accepted
    assert abs(dev.norm2x - host.norm2x) <= COST_RTOL * host.norm2x
    assert np.max(np.abs(dev.p - host.p)) <= P_TOL * max(1.0, np.max(np.abs(host.p)))
    assert dev.stats[5] < 1e5          # H2D bytes: only p and a few scalars, no Jacobian
    dprob = H.Problem.dense(16, 256, seed=3)
    host = H.solve_product(dprob, "dense", max_iterations=30, trustregion0=tr0)
    dev = H.solve_product_device(dprob, "dense", max_iterations=30, trustregion0=tr0)
    assert dev.ncalls == host.ncalls and dev.accepted == host.accepted
    assert abs(dev.norm2x - host.norm2x) <= COST_RTOL * host.norm2x


def test_engine_cache_reuse_and_pattern_change(H):
    """Back-to-back solves reuse the cached engine; a different pattern of the same shape must be
    re-analysed, not silently reused."""
    a = H.Problem.random_sparse(40, 200, 5, seed=1)
    b = H.Problem.random_sparse(40, 200, 5, seed=2)       # same sizes, different pattern
    for prob in (a, b, a):
        ref = H.solve_oracle(prob, "sparse", max_iterations=20)
        got = H.solve_product(prob, "sparse", max_iterations=20)
        assert got.ncalls == ref.ncalls
        assert abs(got.norm2x - ref.norm2x) <= COST_RTOL * ref.norm2x


def test_cached_analysis_is_not_reused_for_a_pattern_with_one_changed_index(H):
    """ADVICE round 1 (high): a cached engine used to be matched on a strided SAMPLE of the pattern; with
    nnz > 4096 a single re-associated entry slipped through and the stale analysis was reused with the new
    values. The whole pattern is hashed now: change one interior index that no sample position covers and
    the second solve must follow the oracle of the MODIFIED problem."""
    N, M, k = 60, 3000, 5
    prob = H.Problem.random_sparse(N, M, k, seed=21)
    assert prob.nnz > 3 * 4096
    ref = H.solve_oracle(prob, "sparse", max_iterations=20)
    got = H.solve_product(prob, "sparse", max_iterations=20)
    assert got.ncalls == ref.ncalls and abs(got.norm2x - ref.norm2x) <= COST_RTOL * ref.norm2x
    Ap = np.ctypeslib.as_array(prob.c.Ap, shape=(M + 1,))
    Ai = np.ctypeslib.as_array(prob.c.Ai, shape=(prob.nnz,))
    stride = max(1, prob.nnz // 4096)
    changed = False
    for j in range(M // 3, M):                      # far from both ends of the arrays
        q = Ap[j + 1] - 1                           # last entry of the column: bump it to the next free state
        if q % stride != 0 and Ai[q] < N - 1:
            Ai[q] += 1
            changed = True
            break
    assert changed
    ref2 = H.solve_oracle(prob, "sparse", max_iterations=20)
    got2 = H.solve_product(prob, "sparse", max_iterations=20)
    assert got2.ncalls == ref2.ncalls
    assert abs(got2.norm2x - ref2.norm2x) <= COST_RTOL * ref2.norm2x
    assert np.max(np.abs(got2.p - ref2.p)) <= 1e-7 * max(1.0, np.max(np.abs(ref2.p)))


def test_pattern_with_more_nonzeros_than_declared_is_rejected(H):
    """ADVICE round 1 (medium): Jt->p[Nmeas] > NJnnz must fail the evaluation instead of over-reading the
    staging buffer and overflowing the device buffer."""
    from libdogleg_b200 import ffi
    prob = H.Problem.random_sparse(20, 100, 4, seed=3)
    Jp, Ji = prob.pattern()
    x, Jx = prob.evaluate(prob.p0())
    E = H.Engine(ffi.SOLVE_SPARSE, prob.N, prob.M, len(Ji))
    E.load_sparse(0, prob.p0(), x, Jp, Ji, Jx)
    E.evaluate(0)
    E.host(0, ffi.BUF_JP, prob.M + 1, np.int32)[prob.M] = len(Ji) + 5
    with pytest.raises(RuntimeError, match="more nonzeros"):
        E.evaluate(0)
    E.close()


def test_large_dense_solve_uses_blocked_tensor_core_path(H):
    """Nstate = 300 > 158: J'J on the DMMA SYRK kernel, blocked DMMA Cholesky, block-wide solves;
    the whole solve must still follow the reference's dense path."""
    prob = H.Problem.dense(300, 1500, seed=9)
    ref = H.solve_reference(prob, "dense", max_iterations=20) if H.reference_lib() is not None \
        else H.solve_oracle(prob, "dense", max_iterations=20)
    got = H.solve_product(prob, "dense", max_iterations=20)
    assert got.ncalls == ref.ncalls
    close_trace(got, ref.trace_p, ref.trace_norm2x)
    assert abs(got.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)
    dev = H.solve_product_device(prob, "dense", max_iterations=20)
    assert dev.ncalls == ref.ncalls and abs(dev.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)


@pytest.mark.parametrize("schedule", ["left", "right", "diag"])
@pytest.mark.parametrize("shape", [(300, 1500), (1200, 2600)])
def test_large_front_panel_schedules_agree_with_the_reference(H, monkeypatch, schedule, shape):
    """The three panel schedules of dlb_bigfront.cu (look-ahead left-looking, lazy right-looking, one diagonal CTA
    per front + product with the inverted block) on fronts of 5 and 19 panels, and the super-block triangular
    solves (1200 pivots > 1024): DOGLEG_GPU_BF_SCHEDULE forces each form in turn; every variant must
    follow the reference's dense path (dogleg.c:699-805, 867-898)."""
    monkeypatch.setenv("DOGLEG_GPU_BF_SCHEDULE", schedule)
    monkeypatch.setenv("DOGLEG_GPU_ENGINE_CACHE", "0")
    N, M = shape
    prob = H.Problem.dense(N, M, seed=4)
    ref = H.solve_reference(prob, "dense", max_iterations=6) if H.reference_lib() is not None \
        else H.solve_oracle(prob, "dense", max_iterations=6)
    got = H.solve_product_device(prob, "dense", max_iterations=6)
    assert got.ncalls == ref.ncalls
    assert abs(got.norm2x - ref.norm2x) <= COST_RTOL * abs(ref.norm2x)
    assert np.max(np.abs(got.p - ref.p)) <= 1e-7 * max(1.0, np.max(np.abs(ref.p)))
