"""The final state of a batched solve (dogleg_gpu_optimize_dense_batched2 / _dense_products_batched2 with a
dogleg_gpu_batch_t): per-problem JtJ + lambda I at the returned p, solves and covariances with it, lambda and
the termination status. Checked against numpy, the oracle and the single-problem path; the CPU part checks the
argument handling without a device."""
import ctypes as C

import numpy as np
import pytest

from libdogleg_b200 import ffi
from support import harness as H
from support import products as HP

GRADIENT, STEP, TRUSTREGION, MAX_ITERATIONS = (ffi.BATCH_GRADIENT, ffi.BATCH_STEP, ffi.BATCH_TRUSTREGION,
                                               ffi.BATCH_MAX_ITERATIONS)
FORMS = [("dense", False), ("products", False), ("products", True)]


def solve2(form, dev, p0, N, M=0, packed=False, handle=True, **pk):
    """One `2` call over a device problem set: (rc, p, norm2x, iterations, handle or None)."""
    L = ffi.load()
    P = H.make_params(L, packed=packed, upper=packed, **pk)
    p = np.ascontiguousarray(p0, dtype=np.float64).copy()
    B = p.shape[0]
    n2 = np.zeros(B)
    it = np.zeros(B, dtype=np.int32)
    h = C.c_void_p()
    hp = C.byref(h) if handle else None
    if form == "dense":
        rc = L.dogleg_gpu_optimize_dense_batched2(H.as_dp(p), N, M, B, H.dev_problems_lib().dlb_dev_cb_dense_batched_ptr(),
                                                  C.c_void_p(dev), C.byref(P), H.as_dp(n2), H.as_ip(it), hp)
    else:
        HP.lib().dlb_prod_problem_layout(dev, int(packed), 0)
        rc = L.dogleg_gpu_optimize_dense_products_batched2(H.as_dp(p), N, B, HP.lib().dlb_prod_cb_batched_ptr(),
                                                           C.c_void_p(dev), C.byref(P), H.as_dp(n2), H.as_ip(it), hp)
    if rc < 0:
        raise RuntimeError(L.dogleg_gpu_last_error().decode())
    assert bool(h.value) == handle
    return rc, p, n2, it, (h if handle else None)


def create(form, B, M, N, seed):
    """The k_gen_batched family (problem b = Problem.dense(N, M, seed + b)) for either form: (dev, p0, free)."""
    if form == "dense":
        DL = H.dev_problems_lib()
        p0 = np.zeros((B, N))
        dev = DL.dlb_dev_problem_create_batched(B, M, N, seed, H.as_dp(p0))
        assert dev
        return dev, p0, DL.dlb_dev_problem_free
    dev, p0 = HP.create_batched(B, M, N, seed)
    return dev, p0, HP.free


def status(h, B):
    st = np.full(B, -1, dtype=np.int32)
    lam = np.full(B, np.nan)
    assert ffi.load().dogleg_gpu_batch_status(h, H.as_ip(st), H.as_dp(lam)) == 0
    return st, lam


def covariance(h, B, N, packed=False, expect=0):
    out = np.full((B, N * (N + 1) // 2 if packed else N * N), np.nan)
    assert ffi.load().dogleg_gpu_batch_covariance(h, H.as_dp(out), int(packed)) == expect
    return out


def batch_solve(h, R):
    """R: B x nrhs x N (problem b's block column-major); returns X alike."""
    R = np.ascontiguousarray(R, dtype=np.float64)
    X = np.full_like(R, np.nan)
    assert ffi.load().dogleg_gpu_batch_solve(h, H.as_dp(R), H.as_dp(X), R.shape[1]) == 0
    return X


def free(h):
    ffi.load().dogleg_gpu_batch_free(C.byref(h))
    assert h.value is None


def final_JtJ(N, M, seed, p):
    """J'J of Problem.dense(N, M, seed) at p: J = A diag(1 + 0.3 p^2) (problems.c dlb_cb_dense)."""
    prob = H.Problem.dense(N, M, seed=seed)
    A = np.ctypeslib.as_array(prob.c.Adense, shape=(M, N))
    J = A * (1.0 + 0.3 * p * p)
    return J.T @ J


def assert_rel(got, want, tol=1e-9):
    assert np.max(np.abs(got - want)) <= tol * np.max(np.abs(want)), np.max(np.abs(got - want)) / np.max(np.abs(want))


# ----------------------------------------------------------------------------------------------- CPU
def test_no_gpu_means_loud_failure_for_batched2(H):
    L = ffi.load()
    if L.dogleg_gpu_device_count() > 0:
        pytest.skip("a GPU is present")
    p = np.zeros((4, 6))
    h = C.c_void_p(1234)
    assert L.dogleg_gpu_optimize_dense_batched2(H.as_dp(p), 6, 16, 4, H.problems_lib().dlb_cb_dense_ptr(), None, None,
                                                None, None, C.byref(h)) < 0
    assert b"no CUDA device" in L.dogleg_gpu_last_error()
    assert h.value is None
    h = C.c_void_p(1234)
    assert L.dogleg_gpu_optimize_dense_products_batched2(H.as_dp(p), 6, 4, H.problems_lib().dlb_cb_products_ptr(), None,
                                                         None, None, None, C.byref(h)) < 0
    assert b"no CUDA device" in L.dogleg_gpu_last_error()
    assert h.value is None


def test_null_batch_handle_is_refused(H):
    L = ffi.load()
    x = np.zeros(64)
    st = np.zeros(4, dtype=np.int32)
    calls = [
        ("dogleg_gpu_batch_status", lambda: L.dogleg_gpu_batch_status(None, H.as_ip(st), H.as_dp(x))),
        ("dogleg_gpu_batch_solve", lambda: L.dogleg_gpu_batch_solve(None, H.as_dp(x), H.as_dp(x), 1)),
        ("dogleg_gpu_batch_solve_device", lambda: L.dogleg_gpu_batch_solve_device(None, x.ctypes.data, x.ctypes.data, 1, None)),
        ("dogleg_gpu_batch_covariance", lambda: L.dogleg_gpu_batch_covariance(None, H.as_dp(x), 0)),
        ("dogleg_gpu_batch_covariance_device", lambda: L.dogleg_gpu_batch_covariance_device(None, x.ctypes.data, 1, None)),
    ]
    for name, call in calls:
        assert call() < 0, name
        msg = L.dogleg_gpu_last_error()
        assert name.encode() in msg and b"NULL handle" in msg, (name, msg)
    h = C.c_void_p()
    L.dogleg_gpu_batch_free(C.byref(h))
    assert h.value is None
    L.dogleg_gpu_batch_free(None)


# ----------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("form,packed", FORMS)
@pytest.mark.parametrize("tr0", [1e3, 0.3])
def test_handle_changes_nothing(H, form, packed, tr0):
    B, N, M, seed = 40, 16, 256, 1000
    dev, p0, release = create(form, B, M, N, seed)
    a = solve2(form, dev, p0, N, M, packed=packed, handle=False, max_iterations=30, trustregion0=tr0)
    b = solve2(form, dev, p0, N, M, packed=packed, handle=True, max_iterations=30, trustregion0=tr0)
    release(dev)
    free(b[4])
    assert a[0] == b[0] == B
    for u, v in zip(a[1:4], b[1:4]):
        assert np.array_equal(u, v)


@pytest.mark.gpu
@pytest.mark.parametrize("tr0", [1e3, 0.3])
def test_covariance_and_lambda_against_numpy_and_oracle(H, tr0):
    B, N, M, seed = 40, 16, 256, 1000
    covs = {}
    for form, packed in FORMS:
        dev, p0, release = create(form, B, M, N, seed)
        rc, p, n2, it, h = solve2(form, dev, p0, N, M, packed=packed, max_iterations=30, trustregion0=tr0)
        release(dev)
        assert rc == B
        st, lam = status(h, B)
        covs[(form, packed)] = (covariance(h, B, N), covariance(h, B, N, packed=True))
        free(h)
        if form != "dense":
            continue
        for b in range(B):
            want = np.linalg.inv(final_JtJ(N, M, seed + b, p[b]) + lam[b] * np.eye(N))
            assert_rel(covs[(form, packed)][0][b].reshape(N, N), want)
        for b in range(0, B, 3):
            ref = H.solve_oracle(H.Problem.dense(N, M, seed=seed + b), "dense", p0=p0[b], max_iterations=30, trustregion0=tr0)
            assert it[b] == ref.accepted
            assert lam[b] == ref.lam, (b, lam[b], ref.lam)
    full_d, packed_d = covs[("dense", False)]
    for key, (full, pk) in covs.items():
        for b in range(B):
            assert_rel(full[b], full_d[b])
            assert np.array_equal(pk[b], full[b].reshape(N, N)[np.triu_indices(N)])


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 7, 8, 9, 17, 31, 32])
def test_every_instantiation(H, N):
    """Every tile size of k_batched_factor, both forms, 1 / 5 / 40 right-hand sides (40: two 32-column chunks)."""
    B, M, seed = 6, 96, 40 + N
    rng = np.random.default_rng(N)
    for form, packed in (("dense", False), ("products", N % 2 == 1)):
        dev, p0, release = create(form, B, M, N, seed)
        rc, p, n2, it, h = solve2(form, dev, p0, N, M, packed=packed, max_iterations=25)
        release(dev)
        assert rc == B
        st, lam = status(h, B)
        A = [final_JtJ(N, M, seed + b, p[b]) + lam[b] * np.eye(N) for b in range(B)]
        for nrhs in (1, 5, 40):
            R = rng.standard_normal((B, nrhs, N))
            X = batch_solve(h, R)
            for b in range(B):
                assert_rel(X[b].T, np.linalg.solve(A[b], R[b].T))
        full, pk = covariance(h, B, N), covariance(h, B, N, packed=True)
        for b in range(B):
            assert_rel(full[b].reshape(N, N), np.linalg.inv(A[b]))
            assert np.array_equal(pk[b], full[b].reshape(N, N)[np.triu_indices(N)])
        free(h)


@pytest.mark.gpu
def test_batch_solve_matches_the_single_problem_path(H):
    """dogleg_gpu_solve on the context of dogleg_gpu_optimize_dense, same problem, same right-hand sides."""
    L = ffi.load()
    L.dogleg_gpu_solve.argtypes = [C.c_void_p, H.dp, H.dp, C.c_int]
    B, N, M, seed = 12, 16, 256, 1000
    dev, p0, release = create("dense", B, M, N, seed)
    rc, p, n2, it, h = solve2("dense", dev, p0, N, M, max_iterations=30)
    release(dev)
    R = np.random.default_rng(3).standard_normal((B, 4, N))
    X = batch_solve(h, R)
    free(h)
    DL = H.dev_problems_lib()
    for b in (0, 5, 11):
        prob = H.Problem.dense(N, M, seed=seed + b)
        d1 = DL.dlb_dev_problem_create(C.cast(prob.ptr, C.c_void_p))
        P = H.make_params(L, max_iterations=30)
        q = p0[b].copy()
        ctx = C.c_void_p()
        L.dogleg_gpu_optimize_dense(H.as_dp(q), N, M, DL.dlb_dev_cb_dense_ptr(), C.c_void_p(d1), C.byref(P), C.byref(ctx))
        DL.dlb_dev_problem_free(d1)
        assert ctx.value
        rhs = np.asfortranarray(R[b].T)
        Xs = np.zeros_like(rhs, order="F")
        assert L.dogleg_gpu_solve(ctx, H.as_dp(rhs), H.as_dp(Xs), 4) == 0
        L.dogleg_freeContext(C.byref(ctx))
        assert np.max(np.abs(q - p[b])) <= 1e-7 * max(1.0, np.max(np.abs(p[b])))
        assert_rel(X[b].T, Xs)


def expected_status(ref, max_iterations, gmax, Jt_x_threshold):
    """Why the oracle's run stopped, from its trial record and the gradient at its final p."""
    converged = not (gmax > Jt_x_threshold)
    if not ref.trials:                                  # stopped at the initial point
        return GRADIENT if converged else MAX_ITERATIONS
    last = ref.trials[-1]
    if not last.accepted:
        return TRUSTREGION
    if not np.isfinite(last.norm2x_after):              # the step was computed, never evaluated
        return STEP
    if converged:
        return GRADIENT
    assert ref.accepted >= max_iterations
    return MAX_ITERATIONS


def dense_gmax(prob, p):
    A = np.ctypeslib.as_array(prob.c.Adense, shape=(prob.M, prob.N))
    b = np.ctypeslib.as_array(prob.c.b, shape=(prob.M,))
    x = A @ (p + 0.1 * p ** 3) - b
    return np.max(np.abs((A * (1.0 + 0.3 * p * p)).T @ x))


def sample_gmax(prob, p):
    x, Jx = prob.evaluate(p)
    Jp, Ji = prob.pattern()
    g = np.zeros(prob.N)
    for i in range(prob.M):
        np.add.at(g, Ji[Jp[i]:Jp[i + 1]], Jx[Jp[i]:Jp[i + 1]] * x[i])
    return np.max(np.abs(g))


@pytest.mark.gpu
def test_termination_status_matches_the_oracle(H):
    B, N, M, seed = 40, 16, 256, 1000
    runs = [dict(max_iterations=0), dict(max_iterations=30, Jt_x_threshold=1e300), dict(max_iterations=3),
            dict(max_iterations=100, Jt_x_threshold=1e-4, update_threshold=0.0),
            dict(max_iterations=100, Jt_x_threshold=0.0, update_threshold=1e-3)]
    seen = set()
    dev, p0, release = create("dense", B, M, N, seed)
    for pk in runs:
        rc, p, n2, it, h = solve2("dense", dev, p0, N, M, **pk)
        st, lam = status(h, B)
        free(h)
        for b in range(B):
            prob = H.Problem.dense(N, M, seed=seed + b)
            ref = H.solve_oracle(prob, "dense", p0=p0[b], **pk)
            assert it[b] == ref.accepted, (pk, b)
            thr = pk.get("Jt_x_threshold", 1e-8)
            assert st[b] == expected_status(ref, pk["max_iterations"], dense_gmax(prob, ref.p), thr), (pk, b, st[b])
            seen.add(int(st[b]))
    release(dev)
    # the sample surface from far starts, where trials are rejected: a coarse trust-region threshold ends a problem at
    # its first rejection that shrinks the region below 1 (well before the cost reaches rounding noise)
    prob = H.Problem.sample()
    rng = np.random.default_rng(5)
    starts = np.array([[5, -3, 2, 1, 0, 10], [-2, 4, -1, 3, 3, 3]] + [list(rng.uniform(-3, 6, 6)) for _ in range(14)])
    DL = H.dev_problems_lib()
    sdev = DL.dlb_dev_problem_create_sample_batched(C.cast(prob.ptr, C.c_void_p), len(starts))
    pk = dict(max_iterations=60, trustregion_threshold=1.0)
    rc, p, n2, it, h = solve2("dense", sdev, starts, 6, prob.M, **pk)
    DL.dlb_dev_problem_free(sdev)
    st, lam = status(h, len(starts))
    free(h)
    for b in range(len(starts)):
        ref = H.solve_oracle(prob, "dense", p0=starts[b], **pk)
        assert it[b] == ref.accepted
        assert st[b] == expected_status(ref, pk["max_iterations"], sample_gmax(prob, ref.p), 1e-8), (b, st[b])
        seen.add(int(st[b]))
    assert {GRADIENT, STEP, TRUSTREGION, MAX_ITERATIONS} <= seen, seen


@pytest.mark.gpu
def test_lambda_ladder_on_a_singular_final_matrix(H):
    """State 3 enters no measurement, so J'J is singular. Stopped at the initial point the solve never factored
    it (lambda 0): the covariance call climbs the ladder, stores the lambda and matches numpy at it. Solved for
    real, the trial kernel's lambda is the oracle's."""
    N, M, dead = 8, 64, 3
    prob = H.Problem.dense(N, M, seed=71)
    A = np.ctypeslib.as_array(prob.c.Adense, shape=(M, N))
    A[:, dead] = 0.0
    for pk in (dict(max_iterations=0), dict(max_iterations=20)):
        dev = HP.from_host(prob, 1)
        rc, p, n2, it, h = solve2("products", dev, prob.p0()[None, :], N, **pk)
        HP.free(dev)
        st0, lam0 = status(h, 1)
        cov = covariance(h, 1, N)[0].reshape(N, N)
        st1, lam1 = status(h, 1)
        ref = H.solve_oracle(prob, "products-unpacked", **pk)
        assert lam0[0] == ref.lam
        if pk["max_iterations"] == 0:
            assert st0[0] == MAX_ITERATIONS and lam0[0] == 0.0
        assert lam1[0] >= 1e-10
        k = np.log10(lam1[0] / 1e-10)
        assert abs(k - round(k)) < 1e-9                      # a rung of 1e-10 * 10^k
        J = A * (1.0 + 0.3 * p[0] * p[0])
        want = np.linalg.inv(J.T @ J + lam1[0] * np.eye(N))
        live = [i for i in range(N) if i != dead]
        assert_rel(cov[np.ix_(live, live)], want[np.ix_(live, live)])
        assert abs(cov[dead, dead] - 1.0 / lam1[0]) <= 1e-9 / lam1[0]
        free(h)


@pytest.mark.gpu
def test_host_and_device_forms_are_bit_identical(H):
    torch = pytest.importorskip("torch")
    L = ffi.load()
    B, N, M, seed = 40, 16, 256, 1000
    dev, p0, release = create("dense", B, M, N, seed)
    rc, p, n2, it, h = solve2("dense", dev, p0, N, M, max_iterations=30)
    release(dev)
    stream = torch.cuda.current_stream().cuda_stream
    for packed in (False, True):
        d_out = torch.full((B, N * (N + 1) // 2 if packed else N * N), float("nan"), dtype=torch.float64, device="cuda")
        assert L.dogleg_gpu_batch_covariance_device(h, d_out.data_ptr(), int(packed), stream) == 0
        torch.cuda.synchronize()
        assert np.array_equal(d_out.cpu().numpy(), covariance(h, B, N, packed=packed))
    for nrhs in (1, 40):
        R = np.random.default_rng(nrhs).standard_normal((B, nrhs, N))
        d_R = torch.from_numpy(R).cuda()
        d_X = torch.full_like(d_R, float("nan"))
        assert L.dogleg_gpu_batch_solve_device(h, d_R.data_ptr(), d_X.data_ptr(), nrhs, stream) == 0
        torch.cuda.synchronize()
        assert np.array_equal(d_X.cpu().numpy(), batch_solve(h, R))
    free(h)


@pytest.mark.gpu
def test_handle_outlives_the_workspace(H):
    L = ffi.load()
    B, N, M, seed = 40, 16, 256, 1000
    dev, p0, release = create("dense", B, M, N, seed)
    rc, p, n2, it, h = solve2("dense", dev, p0, N, M, max_iterations=30)
    before = covariance(h, B, N)
    st_before = status(h, B)
    solve2("dense", dev, p0 + 0.25, N, M, handle=False, max_iterations=30)     # reuses the same workspace
    release(dev)
    L.dogleg_gpu_release_batched_cache()
    L.dogleg_gpu_release_cache()
    assert np.array_equal(covariance(h, B, N), before)
    for u, v in zip(status(h, B), st_before):
        assert np.array_equal(u, v)
    free(h)
    free(h)                                                          # freeing a NULL handle is harmless
