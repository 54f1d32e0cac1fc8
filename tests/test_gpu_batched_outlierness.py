"""Outlierness factors of every problem of a batched solve (dogleg_gpu_batch_outlierness / _device) on the returned
dogleg_gpu_batch_t, with x and J evaluated at the returned p. Checked against numpy's
J* inv(JtJ + lambda I) J*' and the reference's formula, against dogleg_getOutliernessFactors on the single-problem
path, and for bit-reproducibility; the CPU part checks the NULL-handle refusals without a device."""
import ctypes as C

import numpy as np
import pytest

from libdogleg_b200 import ffi
from support import products as HP
from support.harness import as_dp
from test_gpu_batched_results import FORMS, TRUSTREGION, covariance, create, free, solve2, status
from test_gpu_outliers import before_offset

DBL_MAX = np.finfo(np.float64).max


def dense_xJ(H, N, M, seed, p):
    """x and J of Problem.dense(N, M, seed) at p: x = A (p + 0.1 p^3) - b, J = A diag(1 + 0.3 p^2) (problems.c)."""
    prob = H.Problem.dense(N, M, seed=seed)
    A = np.ctypeslib.as_array(prob.c.Adense, shape=(M, N))
    b = np.ctypeslib.as_array(prob.c.b, shape=(M,))
    return A @ (p + 0.1 * p ** 3) - b, A * (1.0 + 0.3 * p * p)


def batch_xJ(H, N, M, seed, p):
    xs, Js = zip(*(dense_xJ(H, N, M, seed + b, p[b]) for b in range(p.shape[0])))
    return np.array(xs), np.array(Js)


def numpy_outlierness(x, J, lam, fs, nfeat, nout=0, scale=-1.0):
    """dogleg_getOutliernessFactors of one problem (dogleg_outliers.c / dogleg.c:2294-2399), in numpy."""
    M, N = J.shape
    if not scale > 0:
        Nok = M - nout * fs
        scale = Nok / (4.0 * ((N + 1) * float(x @ x) / (Nok - N - 1)))
    inv = np.linalg.inv(J.T @ J + lam * np.eye(N))
    f = np.zeros(nfeat)
    for i in range(nfeat):
        r = J[i * fs:(i + 1) * fs]
        a = r @ inv @ r.T
        xf = x[i * fs:(i + 1) * fs]
        if fs == 1:
            d = 1.0 - a[0, 0]
            if abs(d) < 1e-8:
                f[i] = DBL_MAX
                continue
            f[i] = xf[0] ** 2 / d
        else:
            det = (1.0 - a[0, 0]) * (1.0 - a[1, 1]) - a[0, 1] ** 2
            if abs(det) < 1e-8:
                f[i] = DBL_MAX
                continue
            Bm = np.array([[a[1, 1] - 1.0, -a[0, 1]], [-a[0, 1], a[0, 0] - 1.0]])
            v = Bm @ xf
            f[i] = xf @ v / det + v @ v / det ** 2
        f[i] *= scale / 8.0
    return f, scale


def outlierness(h, x, J, fs, nfeat, nout=None, scale=None, expect=0):
    """The host form: (factors B x nfeat, scale B)."""
    B, M = x.shape
    x = np.ascontiguousarray(x, dtype=np.float64)
    J = np.ascontiguousarray(J, dtype=np.float64)
    sc = np.full(B, -1.0) if scale is None else np.array(scale, dtype=np.float64)
    f = np.full((B, nfeat), np.nan)
    no = None if nout is None else np.ascontiguousarray(nout, dtype=np.int32)
    rc = ffi.load().dogleg_gpu_batch_outlierness(h, as_dp(x), as_dp(J), M, fs, nfeat,
                                                 None if no is None else no.ctypes.data_as(C.POINTER(C.c_int)),
                                                 as_dp(sc), as_dp(f))
    assert rc == expect, (rc, ffi.load().dogleg_gpu_last_error())
    return f, sc


def assert_factors(got, want, tol=1e-7):
    assert np.allclose(got, want, rtol=tol, atol=1e-12 * np.max(np.abs(want))), \
        np.max(np.abs(got - want) / (np.abs(want) + 1e-300))


# ----------------------------------------------------------------------------------------------- CPU
def test_null_handle_is_refused_by_outlierness(H):
    L = ffi.load()
    x = np.zeros(64)
    calls = [
        ("dogleg_gpu_batch_outlierness",
         lambda: L.dogleg_gpu_batch_outlierness(None, H.as_dp(x), H.as_dp(x), 8, 1, 8, None, H.as_dp(x), H.as_dp(x))),
        ("dogleg_gpu_batch_outlierness_device",
         lambda: L.dogleg_gpu_batch_outlierness_device(None, x.ctypes.data, x.ctypes.data, 8, 1, 8, None, x.ctypes.data,
                                                       x.ctypes.data, None)),
    ]
    for name, call in calls:
        assert call() < 0, name
        msg = L.dogleg_gpu_last_error()
        assert name.encode() in msg and b"NULL handle" in msg, (name, msg)


# ----------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("fs", [1, 2])
@pytest.mark.parametrize("tr0", [1e3, 0.3])
def test_factors_match_numpy_at_the_returned_p(H, tr0, fs):
    B, N, M, seed = 40, 16, 256, 1000
    nfeat = M // fs
    out = {}
    for form, packed in FORMS:
        dev, p0, release = create(form, B, M, N, seed)
        rc, p, n2, it, h = solve2(form, dev, p0, N, M, packed=packed, max_iterations=30, trustregion0=tr0)
        release(dev)
        st, lam = status(h, B)
        x, J = batch_xJ(H, N, M, seed, p)
        f, sc = outlierness(h, x, J, fs, nfeat)
        free(h)
        for b in range(B):
            fw, sw = numpy_outlierness(x[b], J[b], lam[b], fs, nfeat)
            assert_factors(f[b], fw)
            assert abs(sc[b] - sw) <= 1e-9 * abs(sw)
        out[(form, packed)] = f
    for f in out.values():
        assert_factors(f, out[("dense", False)])


@pytest.mark.gpu
@pytest.mark.parametrize("fs", [1, 2])
def test_factors_match_the_single_problem_path(H, fs):
    """dogleg_getOutliernessFactors on the context of dogleg_optimize_dense2 for the same problem and start. The two
    paths reach p within about 1e-7 of each other, hence the looser bound."""
    L = ffi.load()
    B, N, M, seed = 12, 16, 256, 1000
    nfeat = M // fs
    dev, p0, release = create("dense", B, M, N, seed)
    rc, p, n2, it, h = solve2("dense", dev, p0, N, M, max_iterations=30)
    release(dev)
    x, J = batch_xJ(H, N, M, seed, p)
    f, sc = outlierness(h, x, J, fs, nfeat)
    free(h)
    L.dogleg_getOutliernessFactors.restype = C.c_bool
    L.dogleg_getOutliernessFactors.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int, C.c_int, C.c_int,
                                               C.c_void_p, C.c_void_p]
    off = before_offset()
    for b in (0, 5, 11):
        prob = H.Problem.dense(N, M, seed=seed + b)
        P = H.make_params(L, max_iterations=30)
        q = p0[b].copy()
        ctx = C.c_void_p()
        assert L.dogleg_optimize_dense2(H.as_dp(q), N, M, H.problems_lib().dlb_cb_dense_ptr(), C.cast(prob.ptr, C.c_void_p),
                                        C.byref(P), C.byref(ctx)) >= 0
        point = C.c_void_p.from_address(ctx.value + off).value
        fs1 = np.zeros(nfeat)
        s1 = C.c_double(-1.0)
        assert L.dogleg_getOutliernessFactors(as_dp(fs1), C.byref(s1), fs, nfeat, 0, point, ctx)
        L.dogleg_freeContext(C.byref(ctx))
        assert np.max(np.abs(q - p[b])) <= 1e-7 * max(1.0, np.max(np.abs(p[b])))
        assert_factors(f[b], fs1, tol=1e-6)
        assert abs(sc[b] - s1.value) <= 1e-6 * abs(s1.value)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 7, 8, 9, 17, 31, 32])
def test_every_instantiation_and_chunk_edge(H, N):
    """Every tile size of k_batched_outlierness. Nmeas = 77: three 32-row chunks, the last one partial, and odd for
    pairs. The features cover all of Nmeas, or stop short of it: the trailing measurements count in the scale only."""
    B, M, seed = 6, 77, 40 + N
    for form, packed in (("dense", False), ("products", N % 2 == 1)):
        dev, p0, release = create(form, B, M, N, seed)
        rc, p, n2, it, h = solve2(form, dev, p0, N, M, packed=packed, max_iterations=25)
        release(dev)
        st, lam = status(h, B)
        x, J = batch_xJ(H, N, M, seed, p)
        for fs, nfeat in ((1, M), (1, M - 13), (2, M // 2), (2, 20)):
            f, sc = outlierness(h, x, J, fs, nfeat)
            for b in range(B):
                fw, sw = numpy_outlierness(x[b], J[b], lam[b], fs, nfeat)
                assert_factors(f[b], fw)
                assert abs(sc[b] - sw) <= 1e-9 * abs(sw)
        free(h)


@pytest.mark.gpu
@pytest.mark.parametrize("fs", [1, 2])
def test_rejected_trials_factors_at_the_returned_p(H, fs):
    """The sample surface from far starts: problems stop on a rejected trial (TRUSTREGION), so the last point the
    callback evaluated is not the returned p. The handle's JtJ is that of the returned p, and so are the factors."""
    prob = H.Problem.sample()
    rng = np.random.default_rng(5)
    starts = np.array([[5, -3, 2, 1, 0, 10], [-2, 4, -1, 3, 3, 3]] + [list(rng.uniform(-3, 6, 6)) for _ in range(14)])
    DL = H.dev_problems_lib()
    sdev = DL.dlb_dev_problem_create_sample_batched(C.cast(prob.ptr, C.c_void_p), len(starts))
    rc, p, n2, it, h = solve2("dense", sdev, starts, 6, prob.M, max_iterations=60, trustregion_threshold=1.0)
    DL.dlb_dev_problem_free(sdev)
    st, lam = status(h, len(starts))
    assert TRUSTREGION in st
    xs, Js = [], []
    for b in range(len(starts)):
        x, Jx = prob.evaluate(p[b])
        xs.append(x)
        Js.append(Jx.reshape(prob.M, 6))                 # the sample's Jt is dense: 6 entries per measurement
    x, J = np.array(xs), np.array(Js)
    nfeat = prob.M // fs
    f, sc = outlierness(h, x, J, fs, nfeat)
    free(h)
    for b in range(len(starts)):
        fw, sw = numpy_outlierness(x[b], J[b], lam[b], fs, nfeat)
        assert_factors(f[b], fw)
        assert abs(sc[b] - sw) <= 1e-9 * abs(sw)


@pytest.mark.gpu
@pytest.mark.parametrize("fs", [1, 2])
def test_planted_outlier(H, fs):
    """One corrupted measurement of one problem is that problem's largest factor, at least 1; every other problem's
    factors do not change by a bit."""
    B, N, M, seed = 40, 16, 256, 1000
    nfeat = M // fs
    dev, p0, release = create("dense", B, M, N, seed)
    rc, p, n2, it, h = solve2("dense", dev, p0, N, M, max_iterations=30)
    release(dev)
    x, J = batch_xJ(H, N, M, seed, p)
    f0, s0 = outlierness(h, x, J, fs, nfeat)
    bad_b, bad_m = 17, 101
    x[bad_b, bad_m] += 1.0
    f1, s1 = outlierness(h, x, J, fs, nfeat)
    free(h)
    assert np.argmax(f1[bad_b]) == bad_m // fs
    assert f1[bad_b, bad_m // fs] >= 1.0
    others = np.arange(B) != bad_b
    assert np.array_equal(f1[others], f0[others])
    assert np.array_equal(s1[others], s0[others])


@pytest.mark.gpu
def test_lambda_ladder_on_a_singular_final_matrix(H):
    """The singular final J'J of test_gpu_batched_results' ladder test (state 3 enters no measurement; stopped at
    the initial point, lambda 0): outlierness climbs the ladder to the rung covariance alone would take and stores
    it; the factors and a later covariance match numpy at that lambda."""
    N, M, dead = 8, 64, 3
    prob = H.Problem.dense(N, M, seed=71)
    A = np.ctypeslib.as_array(prob.c.Adense, shape=(M, N))
    A[:, dead] = 0.0
    bvec = np.ctypeslib.as_array(prob.c.b, shape=(M,))
    handles = []
    for _ in range(2):
        dev = HP.from_host(prob, 1)
        rc, p, n2, it, h = solve2("products", dev, prob.p0()[None, :], N, max_iterations=0)
        HP.free(dev)
        assert status(h, 1)[1][0] == 0.0
        handles.append(h)
    q = p[0]
    x = A @ (q + 0.1 * q ** 3) - bvec
    J = A * (1.0 + 0.3 * q * q)
    cov_alone = covariance(handles[1], 1, N)
    lam_c = status(handles[1], 1)[1][0]
    f, sc = outlierness(handles[0], x[None, :], J[None, :], 1, M)
    lam_o = status(handles[0], 1)[1][0]
    assert lam_o == lam_c and lam_o >= 1e-10
    fw, sw = numpy_outlierness(x, J, lam_o, 1, M)
    assert_factors(f[0], fw)
    assert np.array_equal(covariance(handles[0], 1, N), cov_alone)
    for h in handles:
        free(h)


@pytest.mark.gpu
def test_scale_in_and_out(H):
    """A positive scale is kept bit for bit; NoutlierFeatures changes the computed one exactly as the formula says."""
    B, N, M, seed, fs = 40, 16, 256, 1000, 2
    nfeat = M // fs
    dev, p0, release = create("dense", B, M, N, seed)
    rc, p, n2, it, h = solve2("dense", dev, p0, N, M, max_iterations=30)
    release(dev)
    st, lam = status(h, B)
    x, J = batch_xJ(H, N, M, seed, p)
    given = np.where(np.arange(B) % 3 == 0, 0.37 + np.arange(B), -1.0)
    f, sc = outlierness(h, x, J, fs, nfeat, scale=given)
    nout = (np.arange(B) * 7) % 23
    fn, scn = outlierness(h, x, J, fs, nfeat, nout=nout)
    f0, sc0 = outlierness(h, x, J, fs, nfeat)
    free(h)
    for b in range(B):
        if given[b] > 0:
            assert sc[b] == given[b]
            assert_factors(f[b], numpy_outlierness(x[b], J[b], lam[b], fs, nfeat, scale=given[b])[0])
        else:
            assert sc[b] == sc0[b]
        fw, sw = numpy_outlierness(x[b], J[b], lam[b], fs, nfeat, nout=nout[b])
        assert abs(scn[b] - sw) <= 1e-9 * abs(sw)
        assert_factors(fn[b], fw)
        # the same |x|^2 in both: the ratio is the formula's
        Nok = M - nout[b] * fs
        assert abs(scn[b] / sc0[b] - (Nok * (Nok - N - 1)) / (M * (M - N - 1))) <= 1e-14


@pytest.mark.gpu
def test_host_and_device_forms_are_bit_identical(H):
    """x and J from the test model's device callback at the returned p; the device form runs on a torch stream."""
    torch = pytest.importorskip("torch")
    L = ffi.load()
    B, N, M, seed = 40, 16, 256, 1000
    dev, p0, release = create("dense", B, M, N, seed)
    rc, p, n2, it, h = solve2("dense", dev, p0, N, M, max_iterations=30)
    stream = torch.cuda.Stream()
    DL = H.dev_problems_lib()
    DL.dlb_dev_cb_dense_batched.argtypes = [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_void_p]
    DL.dlb_dev_cb_dense_batched.restype = None
    d_p = torch.from_numpy(p).cuda()
    d_x = torch.empty((B, M), dtype=torch.float64, device="cuda")
    d_J = torch.empty((B, M, N), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    DL.dlb_dev_cb_dense_batched(d_p.data_ptr(), d_x.data_ptr(), d_J.data_ptr(), None, B, stream.cuda_stream, dev)
    torch.cuda.synchronize()
    release(dev)
    x, J = d_x.cpu().numpy(), d_J.cpu().numpy()
    xw, Jw = batch_xJ(H, N, M, seed, p)
    assert np.allclose(x, xw, rtol=1e-12, atol=1e-14) and np.allclose(J, Jw, rtol=1e-12, atol=1e-14)
    for fs in (1, 2):
        nfeat = M // fs
        nout = np.arange(B, dtype=np.int32) % 4
        with torch.cuda.stream(stream):
            d_scale = torch.full((B,), -1.0, dtype=torch.float64, device="cuda")
            d_f = torch.full((B, nfeat), float("nan"), dtype=torch.float64, device="cuda")
            d_nout = torch.from_numpy(nout).cuda()
        assert L.dogleg_gpu_batch_outlierness_device(h, d_x.data_ptr(), d_J.data_ptr(), M, fs, nfeat, d_nout.data_ptr(),
                                                     d_scale.data_ptr(), d_f.data_ptr(), stream.cuda_stream) == 0
        stream.synchronize()
        f, sc = outlierness(h, x, J, fs, nfeat, nout=nout)
        assert np.array_equal(d_f.cpu().numpy(), f)
        assert np.array_equal(d_scale.cpu().numpy(), sc)
        f2, sc2 = outlierness(h, x, J, fs, nfeat, nout=nout)             # and run to run
        assert np.array_equal(f2, f) and np.array_equal(sc2, sc)
    free(h)


@pytest.mark.gpu
def test_handle_is_unchanged(H):
    B, N, M, seed = 40, 16, 256, 1000
    dev, p0, release = create("dense", B, M, N, seed)
    rc, p, n2, it, h = solve2("dense", dev, p0, N, M, max_iterations=30)
    release(dev)
    before = covariance(h, B, N)
    st0, lam0 = status(h, B)
    x, J = batch_xJ(H, N, M, seed, p)
    outlierness(h, x, J, 2, M // 2)
    st1, lam1 = status(h, B)
    assert np.array_equal(covariance(h, B, N), before)
    assert np.array_equal(st0, st1) and np.array_equal(lam0, lam1)
    free(h)


@pytest.mark.gpu
def test_bad_arguments_are_refused(H):
    L = ffi.load()
    B, N, M, seed = 4, 8, 40, 7
    dev, p0, release = create("dense", B, M, N, seed)
    rc, p, n2, it, h = solve2("dense", dev, p0, N, M, max_iterations=10)
    release(dev)
    x = np.zeros((B, M))
    J = np.zeros((B, M, N))
    sc = np.full(B, -1.0)
    f = np.full((B, M), np.nan)
    dx, dJ, dsc, df = (as_dp(a) for a in (x, J, sc, f))
    bad = [  # (x, J, Nmeas, featureSize, Nfeatures, scale, factors, message)
        (None, dJ, M, 1, M, dsc, df, b"bad arguments"),
        (dx, None, M, 1, M, dsc, df, b"bad arguments"),
        (dx, dJ, M, 1, M, None, df, b"bad arguments"),
        (dx, dJ, M, 1, M, dsc, None, b"bad arguments"),
        (dx, dJ, M, 3, 10, dsc, df, b"featureSize > 2"),
        (dx, dJ, M, 1, 0, dsc, df, b"Nfeatures"),
        (dx, dJ, 0, 1, 1, dsc, df, b"Nmeas"),
        (dx, dJ, M, 2, M // 2 + 1, dsc, df, b"exceeds Nmeas"),
        (dx, dJ, M, 1, M + 1, dsc, df, b"exceeds Nmeas"),
    ]
    for name in ("dogleg_gpu_batch_outlierness", "dogleg_gpu_batch_outlierness_device"):
        for xa, Ja, m, fs, nf, s, fa, want in bad:
            if name.endswith("_device"):
                args = [C.cast(a, C.c_void_p) if a is not None else None for a in (xa, Ja)]
                rc = L.dogleg_gpu_batch_outlierness_device(h, args[0], args[1], m, fs, nf, None,
                                                           C.cast(s, C.c_void_p) if s is not None else None,
                                                           C.cast(fa, C.c_void_p) if fa is not None else None, None)
            else:
                rc = L.dogleg_gpu_batch_outlierness(h, xa, Ja, m, fs, nf, None, s, fa)
            msg = L.dogleg_gpu_last_error()
            assert rc < 0 and name.encode() + b":" in msg and want in msg, (name, fs, nf, m, msg)
    assert np.all(np.isnan(f)) and np.all(sc == -1.0)
    # featureSize <= 1 means 1, as in the reference
    f1, s1 = outlierness(h, x + 1.0, J, 0, M)
    f2, s2 = outlierness(h, x + 1.0, J, 1, M)
    assert np.array_equal(f1, f2) and np.array_equal(s1, s2)
    free(h)
