"""Batched dense solves with a float Jacobian (dogleg_gpu_optimize_dense_batched_f32jac, _ragged_f32jac). Widening a
float to a double is exact and the kernel runs the double kernel's operations in the same order on the widened values,
so a float solve must equal the double solve driven by the widened twin callback ((double)(float)J), bit for bit:
p, cost, iterations and everything the handle holds. Also checked: per problem against the reference with a host
callback that returns the same float-rounded J; against the unrounded double solve of the same problems (a float J
moves the fixed point by about (J'J)^-1 (J_f - J)'x); the handle calls; and the refusals. The CPU part checks the
no-device failure and the prototypes."""
import ctypes as C

import numpy as np
import pytest

from libdogleg_b200 import ffi
from support import f32jac as HF
from support import harness as H
from support import ragged as HR
from test_gpu_batched_outlierness import outlierness
from test_gpu_batched_ragged import counts_for, outlierness_ragged, sample_batch, sample_prefix
from test_gpu_batched_results import batch_solve, covariance, free, status

ENTRIES = ("dogleg_gpu_optimize_dense_batched_f32jac", "dogleg_gpu_optimize_dense_batched_ragged_f32jac")


def assert_same(a, b, B, handle=True):
    """Two solves' (rc, p, norm2x, iterations, handle) bit for bit, with the handles' status, lambda and J'J (through
    dogleg_gpu_batch_covariance)."""
    assert a[0] == b[0] == B
    for u, v in zip(a[1:4], b[1:4]):
        assert np.array_equal(u, v)
    if handle:
        N = a[1].shape[1]
        for u, v in zip(status(a[4], B), status(b[4], B)):
            assert np.array_equal(u, v)
        assert np.array_equal(covariance(a[4], B, N), covariance(b[4], B, N), equal_nan=True)


# ----------------------------------------------------------------------------------------------- CPU
def test_prototypes_load():
    L = ffi.load()
    for name in ENTRIES:
        fn = getattr(L, name)
        assert fn.restype is C.c_int and len(fn.argtypes) == 10, name


def test_no_gpu_means_loud_failure_for_f32jac(H):
    L = ffi.load()
    if L.dogleg_gpu_device_count() > 0:
        pytest.skip("a GPU is present")
    p = np.zeros((4, 6))
    c = HR.as_counts([3, 0, 9, 12])
    cb = H.problems_lib().dlb_cb_dense_ptr()
    for name, call in (
            (ENTRIES[0], lambda h: L.dogleg_gpu_optimize_dense_batched_f32jac(H.as_dp(p), 6, 10, 4, cb, None, None, None,
                                                                              None, C.byref(h))),
            (ENTRIES[1], lambda h: L.dogleg_gpu_optimize_dense_batched_ragged_f32jac(H.as_dp(p), 6, HR.as_up(c), 4, cb, None,
                                                                                     None, None, None, C.byref(h)))):
        h = C.c_void_p(1234)
        assert call(h) < 0, name
        msg = L.dogleg_gpu_last_error()
        assert name.encode() + b":" in msg and b"no CUDA device" in msg, (name, msg)
        assert h.value is None


# ----------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("tr0", [1e3, 0.3])
@pytest.mark.parametrize("N", [1, 6, 8, 9, 16, 17, 24, 25, 32])
def test_uniform_equals_the_widened_twin(H, N, tr0):
    """Every kernel tile size; M below N, not a multiple of 4, and a few hundred."""
    B = 24
    for M in sorted({max(N - 1, 1), 45, 258}):
        dev, p0 = HF.create(np.full(B, M, dtype=np.uint32), N, seed=800 + N + M)
        a = HF.solve("uniform_f32", dev, p0, N, handle=True, max_iterations=30, trustregion0=tr0)
        b = HF.solve("uniform_twin", dev, p0, N, handle=True, max_iterations=30, trustregion0=tr0)
        HF.free(dev)
        assert_same(a, b, B)
        assert np.any(a[3] > 0), (N, M)
        free(a[4])
        free(b[4])


@pytest.mark.gpu
@pytest.mark.parametrize("tr0", [1e3, 0.3])
@pytest.mark.parametrize("N", [1, 6, 8, 9, 16, 17, 24, 25, 32])
def test_ragged_equals_the_widened_twin(H, N, tr0):
    """Counts 0, 1, N - 1, N, every residue mod 16 and a few hundred."""
    counts = counts_for(N, seed=40)
    B = len(counts)
    dev, p0 = HF.create(counts, N, seed=900 + N)
    a = HF.solve("ragged_f32", dev, p0, N, counts, handle=True, max_iterations=30, trustregion0=tr0)
    b = HF.solve("ragged_twin", dev, p0, N, counts, handle=True, max_iterations=30, trustregion0=tr0)
    HF.free(dev)
    assert_same(a, b, B)
    z = counts == 0
    assert np.array_equal(a[1][z], p0[z]) and np.all(a[3][z] == 0)
    free(a[4])
    free(b[4])


@pytest.mark.gpu
def test_sample_surface_equals_the_widened_twin(H):
    counts, starts = sample_batch(32)
    dev = HF.create_sample(H.Problem.sample(), counts)
    a = HF.solve("ragged_f32", dev, starts, 6, counts, handle=True, max_iterations=60)
    b = HF.solve("ragged_twin", dev, starts, 6, counts, handle=True, max_iterations=60)
    HF.free(dev)
    assert_same(a, b, len(counts))
    free(a[4])
    free(b[4])


# the reference's dense callback with J rounded to float, as the float callbacks round it
DENSE_CB = C.CFUNCTYPE(None, H.dp, H.dp, H.dp, C.c_void_p)


def rounded_callback(prob):
    inner = C.cast(H.problems_lib().dlb_cb_dense_ptr(), DENSE_CB)

    def cb(p, x, J, cookie):
        inner(p, x, J, cookie)
        a = np.ctypeslib.as_array(J, shape=(prob.M * prob.N,))
        a[:] = a.astype(np.float32)
    return DENSE_CB(cb)


def ref_solve_rounded(H, prob, p0, **pk):
    """The unmodified reference's dogleg_optimize_dense2 (the oracle restatement where it is not built) on the problem
    with a float-rounded J: Result with norm2x, p and accepted (accepted from the oracle, as test_gpu_batched.ref_solve
    does)."""
    cb = rounded_callback(prob)
    cookie = C.cast(prob.ptr, H.vp)
    P = H.make_params(ffi.load(), **pk)
    O = H.oracle_lib()
    po = np.array(p0, dtype=np.float64)
    R = H.OrcResult()
    trials = (H.OrcTrial * 4096)()
    R.trials = C.cast(trials, C.POINTER(H.OrcTrial))
    R.Ntrials_max = 4096
    prob.reset()
    n2 = O.orc_optimize_dense(H.as_dp(po), prob.N, prob.M, C.cast(cb, H.vp), cookie, C.byref(P), C.byref(R))
    res = H.Result(norm2x=n2, p=po, accepted=R.accepted_steps, trials=[trials[i] for i in range(R.Ntrials)])
    ref = H.reference_lib()
    if ref is not None:
        pr = np.array(p0, dtype=np.float64)
        prob.reset()
        res.norm2x = ref.dogleg_optimize_dense2(H.as_dp(pr), prob.N, prob.M, C.cast(cb, H.vp), cookie, C.byref(P), None)
        res.p = pr
    return res


def assert_matches_reference(p, n2, it, ref, counts_may_differ=False):
    """Cost to 1e-9 and p to 1e-7; equal accepted-step counts unless counts_may_differ (then: whether they differ)."""
    assert abs(n2 - ref.norm2x) <= 1e-9 * ref.norm2x, (n2, ref.norm2x)
    assert np.max(np.abs(p - ref.p)) <= 1e-7 * max(1.0, np.max(np.abs(ref.p)))
    if not counts_may_differ:
        assert it == ref.accepted, (it, ref.accepted)
    return int(it != ref.accepted)


@pytest.mark.gpu
@pytest.mark.parametrize("tr0", [1e3, 0.3])
def test_per_problem_against_the_reference(H, tr0):
    """Every third problem of a uniform and of a ragged batch (counts above Nstate: the others are fitted exactly and
    their cost is rounding noise, see test_gpu_batched_ragged) against the reference with the same float-rounded J."""
    N, M, seed = 16, 256, 1000
    dev, p0 = HF.create(np.full(18, M, dtype=np.uint32), N, seed)
    rc, p, n2, it, _ = HF.solve("uniform_f32", dev, p0, N, max_iterations=30, trustregion0=tr0)
    HF.free(dev)
    for b in range(0, len(p0), 3):
        prob = H.Problem.dense(N, M, seed=seed + b)
        assert np.allclose(prob.p0(), p0[b], rtol=0, atol=1e-14)
        assert_matches_reference(p[b], n2[b], it[b], ref_solve_rounded(H, prob, p0[b], max_iterations=30, trustregion0=tr0))
    counts = counts_for(N, seed=3)
    dev, p0 = HF.create(counts, N, seed)
    rc, p, n2, it, _ = HF.solve("ragged_f32", dev, p0, N, counts, max_iterations=30, trustregion0=tr0)
    HF.free(dev)
    for b in range(0, len(counts), 3):
        m = int(counts[b])
        if m <= N:
            continue
        prob = H.Problem.dense(N, m, seed=seed + b)
        assert_matches_reference(p[b], n2[b], it[b], ref_solve_rounded(H, prob, p0[b], max_iterations=30, trustregion0=tr0))


@pytest.mark.gpu
def test_sample_surface_against_the_reference_with_rejections(H):
    """With J rounded to float the Jacobian is no longer the model's derivative, so a solve ends in a tail of steps that
    converge linearly to J_f'x = 0 and change the cost only in its last bits. Whether such a step is accepted, and after
    how many of them the gradient test passes, depends on how the sums were formed, which the reference does in another
    order: on this surface a few problems end with accepted-step counts that differ from the reference's (6 against 9,
    say). Cost and p are held to the usual bounds for every problem, equal counts for at least three quarters of them
    (the dense problems of test_per_problem_against_the_reference, which converge quadratically enough, match all)."""
    counts, starts = sample_batch(32)
    dev = HF.create_sample(H.Problem.sample(), counts)
    rc, p, n2, it, _ = HF.solve("ragged_f32", dev, starts, 6, counts, max_iterations=60)
    HF.free(dev)
    nrej = ntail = 0
    for b, m in enumerate(counts):
        ref = ref_solve_rounded(H, sample_prefix(int(m)), starts[b], max_iterations=60)
        nrej += sum(1 for t in ref.trials if not t.accepted)
        ntail += assert_matches_reference(p[b], n2[b], it[b], ref, counts_may_differ=True)
    assert nrej > 10
    print(f"accepted-step counts differ from the reference's for {ntail} of {len(counts)} problems")
    assert ntail <= len(counts) // 4, ntail


def first_order_shift(N, M, seed, p):
    """|(J'J)^-1 (J_f - J)'x| at p for Problem.dense(N, M, seed): how far rounding J to float moves the fixed point."""
    prob = H.Problem.dense(N, M, seed=seed)
    A = np.ctypeslib.as_array(prob.c.Adense, shape=(M, N))
    bv = np.ctypeslib.as_array(prob.c.b, shape=(M,))
    x = A @ (p + 0.1 * p ** 3) - bv
    J = A * (1.0 + 0.3 * p * p)
    Jf = J.astype(np.float32).astype(np.float64)
    return np.max(np.abs(np.linalg.solve(J.T @ J, (Jf - J).T @ x)))


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,M", [(100000, 16, 256), (20000, 25, 100)])
def test_float_against_double(H, B, N, M):
    """The float-J solve against the ordinary double-J solve of the same problems (C3's shape and one more N). The
    synthetic model has a unique minimum, which rounding J to float moves by about (J'J)^-1 (J_f - J)'x; a problem that
    misses the p bound is reported with that prediction beside the observed difference."""
    seed = 3000 + N
    dev, p0 = HF.create(np.full(B, M, dtype=np.uint32), N, seed)
    f = HF.solve("uniform_f32", dev, p0, N, max_iterations=100)
    d = HF.solve("uniform_f64", dev, p0, N, max_iterations=100)
    HF.free(dev)
    assert f[0] == d[0] == B
    cost_rel = np.abs(f[2] - d[2]) / d[2]
    assert np.all(cost_rel <= 1e-9), (np.argmax(cost_rel), cost_rel.max())
    dp = np.max(np.abs(f[1] - d[1]), axis=1) / np.maximum(1.0, np.max(np.abs(d[1]), axis=1))
    bad = np.nonzero(dp > 1e-7)[0]
    report = [(int(b), float(dp[b]), float(first_order_shift(N, M, seed + int(b), d[1][b]))) for b in bad[:10]]
    assert len(bad) == 0, f"{len(bad)} problems miss the p bound; (problem, observed, first-order prediction): {report}"


def widened_xJ(kind, dev, p, N, counts=None):
    """x and the widened float J at p from the twin callback (device), as numpy."""
    import torch
    L = HF.lib()
    B = p.shape[0]
    d_p = torch.from_numpy(np.ascontiguousarray(p)).cuda()
    if kind == "ragged":
        off = HR.offsets(counts)
        rows = int(off[-1])
        d_off = torch.from_numpy(off).cuda()
        d_x = torch.empty(rows, dtype=torch.float64, device="cuda")
        d_J = torch.empty((rows, N), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        L.dlb_f32_cb_ragged_twin(d_p.data_ptr(), d_x.data_ptr(), d_J.data_ptr(), d_off.data_ptr(), None, B,
                                 torch.cuda.current_stream().cuda_stream, dev)
    else:
        M = HF.mpad(dev)
        d_x = torch.empty((B, M), dtype=torch.float64, device="cuda")
        d_J = torch.empty((B, M, N), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        L.dlb_f32_cb_uniform_twin(d_p.data_ptr(), d_x.data_ptr(), d_J.data_ptr(), None, B,
                                  torch.cuda.current_stream().cuda_stream, dev)
    torch.cuda.synchronize()
    return d_x.cpu().numpy(), d_J.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["uniform", "ragged"])
def test_handle_calls(H, kind):
    """Status, solves and covariances (host and device forms) and the outlierness factors of a float solve's handle
    equal those of the twin solve's handle, bit for bit; outlierness takes the widened J."""
    torch = pytest.importorskip("torch")
    L = ffi.load()
    N, seed = 16, 1000
    counts = counts_for(N, seed=5)
    counts[counts < N + 2] += N + 2
    if kind == "uniform":
        counts[:] = 130
    B = len(counts)
    dev, p0 = HF.create(counts, N, seed)
    a = HF.solve(kind + "_f32", dev, p0, N, counts, handle=True, max_iterations=30)
    b = HF.solve(kind + "_twin", dev, p0, N, counts, handle=True, max_iterations=30)
    assert_same(a, b, B)
    ha, hb = a[4], b[4]
    assert np.array_equal(covariance(ha, B, N, packed=True), covariance(hb, B, N, packed=True))
    R = np.random.default_rng(4).standard_normal((B, 3, N))
    assert np.array_equal(batch_solve(ha, R), batch_solve(hb, R))
    stream = torch.cuda.current_stream().cuda_stream
    d_R = torch.from_numpy(R).cuda()
    dev_out = []
    for h in (ha, hb):
        d_cov = torch.full((B, N * N), float("nan"), dtype=torch.float64, device="cuda")
        d_X = torch.full_like(d_R, float("nan"))
        assert L.dogleg_gpu_batch_covariance_device(h, d_cov.data_ptr(), 0, stream) == 0
        assert L.dogleg_gpu_batch_solve_device(h, d_R.data_ptr(), d_X.data_ptr(), 3, stream) == 0
        torch.cuda.synchronize()
        dev_out.append((d_cov.cpu().numpy(), d_X.cpu().numpy()))
    for u, v in zip(*dev_out):
        assert np.array_equal(u, v)
    x, J = widened_xJ(kind, dev, a[1], N, counts)
    HF.free(dev)
    for fs in (1, 2):
        if kind == "uniform":
            M = int(counts[0])
            fa = outlierness(ha, x, J, fs, M // fs)
            fb = outlierness(hb, x, J, fs, M // fs)
        else:
            fa = outlierness_ragged(ha, x, J, fs, scale=np.full(B, -1.0))
            fb = outlierness_ragged(hb, x, J, fs, scale=np.full(B, -1.0))
        assert np.array_equal(fa[0], fb[0], equal_nan=True) and np.array_equal(fa[1], fb[1])
        assert np.all(np.isfinite(fa[1]))
    for u, v in zip(status(ha, B), status(hb, B)):                   # the ladder may have raised lambda: alike
        assert np.array_equal(u, v)
    free(ha)
    free(hb)


@pytest.mark.gpu
def test_bad_arguments_are_refused_before_the_first_callback(H):
    L = ffi.load()
    N = 8
    counts = HR.as_counts([5, 0, 30, 12])
    dev, p0 = HF.create(counts, N, 31)
    P = H.make_params(L, max_iterations=10)
    huge = HR.as_counts([2 ** 31 - 1] * 40)
    over = HR.as_counts([5, 2 ** 31, 30, 12])
    p40 = np.zeros((40, 32))
    p4k = np.zeros((40000, 32))
    fu, fr = HF.lib().dlb_f32_cb_uniform_ptr(), HF.lib().dlb_f32_cb_ragged_ptr()
    uniform = [  # (p, Nstate, Nmeas, B, callback, message)
        (p0, 0, 30, 4, fu, b"Nstate"),
        (p0, 33, 30, 4, fu, b"Nstate"),
        (p0, N, 30, 0, fu, b"bad arguments"),
        (None, N, 30, 4, fu, b"bad arguments"),
        (p0, N, 30, 4, None, b"bad arguments"),
        (p0, N, 2 ** 31, 4, fu, b"Nmeas exceeds INT_MAX"),
        (p4k, 32, 2 ** 30, 40000, fu, b"out of device memory"),
    ]
    ragged = [
        (p0, 0, counts, 4, fr, b"Nstate"),
        (p0, 33, counts, 4, fr, b"Nstate"),
        (p0, N, counts, 0, fr, b"bad arguments"),
        (p0, N, None, 4, fr, b"bad arguments"),
        (None, N, counts, 4, fr, b"bad arguments"),
        (p0, N, counts, 4, None, b"bad arguments"),
        (p0, N, over, 4, fr, b"Nmeas[1] = 2147483648 exceeds INT_MAX"),
        (p40, 32, huge, 40, fr, b"out of device memory"),
    ]
    for name, cases in ((ENTRIES[0], uniform), (ENTRIES[1], ragged)):
        for p, n, c, B, f, want in cases:
            q = None if p is None else p.copy()
            h = C.c_void_p(1234)
            meas = c if name == ENTRIES[0] else (None if c is None else HR.as_up(c))
            rc = getattr(L, name)(None if q is None else H.as_dp(q), n, meas, B, f, C.c_void_p(dev), C.byref(P), None, None,
                                  C.byref(h))
            msg = L.dogleg_gpu_last_error()
            assert rc < 0 and name.encode() + b":" in msg and want in msg, (name, n, B, msg)
            assert h.value is None
            assert HF.ncalls(dev) == 0
            if q is not None:
                assert np.array_equal(q, p)
    HF.free(dev)
