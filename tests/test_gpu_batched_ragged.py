"""Ragged batched dense solves (dogleg_gpu_optimize_dense_batched_ragged): problems with different numbers of
measurements, stored without padding, and the outlierness factors of their handles. The solve must equal
dogleg_gpu_optimize_dense_batched2 on the same batch zero-padded to its longest problem, bit for bit: a problem's first
Nmeas[b] rows form the same 4-row groups in both layouts, and zero rows add exact zeros to every sum. Also checked
against the reference per problem, against numpy, and for the argument refusals; the CPU part checks the host-side
layout and the refusals without a device."""
import ctypes as C

import numpy as np
import pytest

from libdogleg_b200 import ffi
from support import harness as H
from support import ragged as HR
from test_gpu_batched import ref_solve
from test_gpu_batched_outlierness import assert_factors, numpy_outlierness, outlierness
from test_gpu_batched_results import (GRADIENT, MAX_ITERATIONS, STEP, TRUSTREGION, assert_rel, batch_solve, covariance,
                                      dense_gmax, expected_status, free, solve2, status)

ip = C.POINTER(C.c_int)


def counts_for(N, seed=0):
    """0, 1, N - 1, N, every residue mod 16 (row groups of 4 x a ring of 4) and a few hundred, shuffled."""
    c = np.array([0, 1, max(N - 1, 0), N] + [48 + r for r in range(16)] + [300, 517], dtype=np.uint32)
    return c[np.random.default_rng(seed + N).permutation(len(c))]


def ragged_xJ(N, counts, seed, p):
    """x and J of the dense kind at p, in the ragged layout (numpy, from the host's Problem.dense)."""
    xs, Js = [], []
    for b, m in enumerate(counts):
        if m == 0:
            continue
        prob = H.Problem.dense(N, int(m), seed=seed + b)
        A = np.ctypeslib.as_array(prob.c.Adense, shape=(int(m), N))
        bv = np.ctypeslib.as_array(prob.c.b, shape=(int(m),))
        xs.append(A @ (p[b] + 0.1 * p[b] ** 3) - bv)
        Js.append(A * (1.0 + 0.3 * p[b] * p[b]))
    return np.concatenate(xs), np.concatenate(Js)


def outlierness_ragged(h, x, J, fs, nfeat=None, nout=None, scale=None, factors=None, expect=0):
    """The host form: (factors laid out like x, scale B)."""
    L = ffi.load()
    sc = np.array(scale, dtype=np.float64)
    f = np.full(len(x), np.nan) if factors is None else np.array(factors, dtype=np.float64)
    nf = None if nfeat is None else np.ascontiguousarray(nfeat, dtype=np.int32)
    no = None if nout is None else np.ascontiguousarray(nout, dtype=np.int32)
    rc = L.dogleg_gpu_batch_outlierness_ragged(h, H.as_dp(np.ascontiguousarray(x)), H.as_dp(np.ascontiguousarray(J)), fs,
                                               None if nf is None else nf.ctypes.data_as(ip),
                                               None if no is None else no.ctypes.data_as(ip), H.as_dp(sc), H.as_dp(f))
    assert rc == expect, (rc, L.dogleg_gpu_last_error())
    return f, sc


# ----------------------------------------------------------------------------------------------- CPU
def test_layout_matches_numpy(H):
    L = ffi.load()
    rng = np.random.default_rng(1)
    for counts in (counts_for(16), rng.integers(0, 200000, 3000), np.array([5]), np.array([0, 0, 70000, 3, 70000, 3])):
        c = HR.as_counts(counts)
        off = np.zeros(len(c) + 1, dtype=np.int64)
        order = np.zeros(len(c), dtype=np.int32)
        assert L.dlb_batched_ragged_layout(HR.as_up(c), len(c), off.ctypes.data_as(C.POINTER(C.c_longlong)),
                                           order.ctypes.data_as(ip)) == 0
        assert np.array_equal(off, HR.offsets(c))
        assert np.array_equal(order, np.argsort(-c.astype(np.int64), kind="stable"))     # longest first, ties by index
    c = HR.as_counts([3, 2 ** 31])
    off = np.zeros(3, dtype=np.int64)
    order = np.zeros(2, dtype=np.int32)
    assert L.dlb_batched_ragged_layout(HR.as_up(c), 2, off.ctypes.data_as(C.POINTER(C.c_longlong)), order.ctypes.data_as(ip)) < 0


def test_no_gpu_means_loud_failure_for_ragged(H):
    L = ffi.load()
    if L.dogleg_gpu_device_count() > 0:
        pytest.skip("a GPU is present")
    p = np.zeros((4, 6))
    c = HR.as_counts([3, 0, 9, 12])
    h = C.c_void_p(1234)
    assert L.dogleg_gpu_optimize_dense_batched_ragged(H.as_dp(p), 6, HR.as_up(c), 4, H.problems_lib().dlb_cb_dense_ptr(),
                                                      None, None, None, None, C.byref(h)) < 0
    msg = L.dogleg_gpu_last_error()
    assert b"dogleg_gpu_optimize_dense_batched_ragged" in msg and b"no CUDA device" in msg
    assert h.value is None


def test_null_handle_is_refused_by_ragged_outlierness(H):
    L = ffi.load()
    x = np.zeros(64)
    calls = [
        ("dogleg_gpu_batch_outlierness_ragged",
         lambda: L.dogleg_gpu_batch_outlierness_ragged(None, H.as_dp(x), H.as_dp(x), 1, None, None, H.as_dp(x), H.as_dp(x))),
        ("dogleg_gpu_batch_outlierness_ragged_device",
         lambda: L.dogleg_gpu_batch_outlierness_ragged_device(None, x.ctypes.data, x.ctypes.data, 1, None, None,
                                                              x.ctypes.data, x.ctypes.data, None)),
    ]
    for name, call in calls:
        assert call() < 0, name
        msg = L.dogleg_gpu_last_error()
        assert name.encode() + b":" in msg and b"NULL handle" in msg, (name, msg)


# ----------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("tr0", [1e3, 0.3])
@pytest.mark.parametrize("N", [1, 6, 8, 9, 16, 17, 24, 25, 32])
def test_ragged_equals_zero_padded(H, N, tr0):
    counts = counts_for(N)
    B = len(counts)
    dev, p0 = HR.create(counts, N, seed=500 + N)
    assert HR.mpad(dev) == 517
    a = HR.solve(dev, p0, N, counts, handle=True, max_iterations=30, trustregion0=tr0)
    b = HR.solve_padded(dev, p0, N, handle=True, max_iterations=30, trustregion0=tr0)
    HR.free(dev)
    assert a[0] == b[0] == B
    for u, v in zip(a[1:4], b[1:4]):
        assert np.array_equal(u, v)
    sa, sb = status(a[4], B), status(b[4], B)
    assert np.array_equal(sa[0], sb[0]) and np.array_equal(sa[1], sb[1])
    assert np.array_equal(covariance(a[4], B, N), covariance(b[4], B, N))
    z = counts == 0                                      # no measurement: stops at its start point, converged
    assert np.array_equal(a[1][z], p0[z]) and np.all(a[3][z] == 0) and np.all(a[2][z] == 0.0)
    assert np.all(sa[0][z] == GRADIENT)
    free(a[4])
    free(b[4])


@pytest.mark.gpu
@pytest.mark.parametrize("tr0", [1e3, 0.3])
def test_per_problem_against_the_reference(H, tr0):
    """Every third problem against the reference's dense path on its own Nmeas[b]. A problem with no more measurements
    than states is fitted exactly, so its cost ends in rounding noise (about 1e-28) where a relative bound means nothing:
    the cost bound has an absolute floor of 1e-20, far below the cost of any problem that is not fitted exactly. At that
    noise level the last trial's acceptance depends on the last bits of sums the reference forms in another order, and
    with fewer measurements than states p is not fixed by the cost, so the steps and p are compared for problems with
    more measurements than states."""
    N, seed = 16, 1000
    counts = counts_for(N, seed=3)
    dev, p0 = HR.create(counts, N, seed)
    rc, p, n2, it, _ = HR.solve(dev, p0, N, counts, max_iterations=30, trustregion0=tr0)
    HR.free(dev)
    assert rc == len(counts)
    for b in range(0, len(counts), 3):
        m = int(counts[b])
        if m == 0:
            assert it[b] == 0 and np.array_equal(p[b], p0[b])
            continue
        prob = H.Problem.dense(N, m, seed=seed + b)
        assert np.allclose(prob.p0(), p0[b], rtol=0, atol=1e-14)      # host and device generators agree
        ref = ref_solve(H, prob, p0[b], max_iterations=30, trustregion0=tr0)
        assert abs(n2[b] - ref.norm2x) <= 1e-9 * ref.norm2x + 1e-20, (b, m, n2[b], ref.norm2x)
        if m > N:
            assert it[b] == ref.accepted, (b, m, it[b], ref.accepted)
            assert np.max(np.abs(p[b] - ref.p)) <= 1e-7 * max(1.0, np.max(np.abs(ref.p))), (b, m)


def sample_prefix(m):
    prob = H.Problem.sample()
    prob.c.M = m
    prob.M = m
    return prob


def sample_batch(B, seed=5):
    """Prefixes of at least 30 points. The grid's points run x-major, so a prefix of fewer than 21 points has at most two
    distinct x: then x^2, x and 1 are dependent, JtJ is singular and the steps depend on the last bits of every sum."""
    rng = np.random.default_rng(seed)
    counts = np.concatenate([[100, 30, 57, 33], rng.integers(30, 101, B - 4)]).astype(np.uint32)
    starts = np.array([[5, -3, 2, 1, 0, 10], [-2, 4, -1, 3, 3, 3]] + [list(rng.uniform(-3, 6, 6)) for _ in range(B - 2)])
    return counts, starts


@pytest.mark.gpu
def test_sample_surface_prefixes_with_rejections(H):
    counts, starts = sample_batch(32)
    prob = H.Problem.sample()
    dev = HR.create_sample(prob, counts)
    rc, p, n2, it, _ = HR.solve(dev, starts, 6, counts, max_iterations=60)
    HR.free(dev)
    assert rc == len(counts)
    nrej = 0
    for b, m in enumerate(counts):
        ref = H.solve_oracle(sample_prefix(int(m)), "dense", p0=starts[b], max_iterations=60)
        nrej += sum(1 for t in ref.trials if not t.accepted)
        assert it[b] == ref.accepted, (b, m, it[b], ref.accepted)
        assert abs(n2[b] - ref.norm2x) <= 1e-9 * ref.norm2x
        assert np.max(np.abs(p[b] - ref.p)) <= 1e-7 * max(1.0, np.max(np.abs(ref.p)))
    assert nrej > 10        # the batch really exercises the rejection path


@pytest.mark.gpu
def test_permuting_the_problems_permutes_every_output(H):
    counts, starts = sample_batch(40, seed=9)
    perm = np.random.default_rng(2).permutation(len(counts))
    prob = H.Problem.sample()
    out = []
    for c, s in ((counts, starts), (counts[perm], starts[perm])):
        dev = HR.create_sample(prob, c)
        rc, p, n2, it, h = HR.solve(dev, s, 6, c, handle=True, max_iterations=60, trustregion0=0.3)
        HR.free(dev)
        out.append((p, n2, it) + status(h, len(c)) + (covariance(h, len(c), 6),))
        free(h)
    for u, v in zip(out[0], out[1]):
        assert np.array_equal(u[perm], v)


@pytest.mark.gpu
def test_equal_counts_give_the_uniform_form(H):
    """Every count equal: the uniform form's outputs on the test model's own uniform batch (problems_dev.cu)."""
    B, N, M, seed = 24, 13, 77, 600
    DL = H.dev_problems_lib()
    pu = np.zeros((B, N))
    udev = DL.dlb_dev_problem_create_batched(B, M, N, seed, H.as_dp(pu))
    u = solve2("dense", udev, pu, N, M, max_iterations=30)
    DL.dlb_dev_problem_free(udev)
    counts = np.full(B, M, dtype=np.uint32)
    dev, p0 = HR.create(counts, N, seed)
    assert np.array_equal(p0, pu)
    r = HR.solve(dev, p0, N, counts, handle=True, max_iterations=30)
    HR.free(dev)
    for a, b in zip(u[:4], r[:4]):
        assert np.array_equal(a, b)
    for a, b in zip(status(u[4], B), status(r[4], B)):
        assert np.array_equal(a, b)
    assert np.array_equal(covariance(u[4], B, N), covariance(r[4], B, N))
    free(u[4])
    free(r[4])


@pytest.mark.gpu
def test_ragged_handle(H):
    """Termination codes against the oracle's trial record; covariance and dogleg_gpu_batch_solve against numpy's
    inv(JtJ + lambda I) at the returned p (problems with at least Nstate measurements: the others are singular up to
    lambda); the _device forms equal the host forms. A problem with no more measurements than states is fitted exactly:
    its cost ends in rounding noise, where accepting the last trial depends on the last bits of sums that the oracle
    forms in another order, so only problems with more measurements than states are held to the oracle's record (every
    problem equals the zero-padded uniform solve bit for bit in test_ragged_equals_zero_padded)."""
    torch = pytest.importorskip("torch")
    L = ffi.load()
    N, seed = 16, 1000
    counts = counts_for(N, seed=3)
    B = len(counts)
    dev, p0 = HR.create(counts, N, seed)
    for pk in (dict(max_iterations=0), dict(max_iterations=3), dict(max_iterations=30),
               dict(max_iterations=100, Jt_x_threshold=0.0, update_threshold=1e-3)):
        rc, p, n2, it, h = HR.solve(dev, p0, N, counts, handle=True, **pk)
        st, lam = status(h, B)
        for b, m in enumerate(counts):
            if m == 0:
                assert st[b] == GRADIENT
                continue
            if m <= N:
                assert st[b] in (GRADIENT, STEP, TRUSTREGION, MAX_ITERATIONS), (pk, b, st[b])
                continue
            prob = H.Problem.dense(N, int(m), seed=seed + b)
            ref = H.solve_oracle(prob, "dense", p0=p0[b], **pk)
            assert it[b] == ref.accepted, (pk, b)
            thr = pk.get("Jt_x_threshold", 1e-8)
            assert st[b] == expected_status(ref, pk["max_iterations"], dense_gmax(prob, ref.p), thr), (pk, b, st[b])
        if pk["max_iterations"] == 30:
            cov = covariance(h, B, N)
            st, lam = status(h, B)                     # the ladder may have raised lambda of a singular problem
            R = np.random.default_rng(4).standard_normal((B, 3, N))
            X = batch_solve(h, R)
            x, J = ragged_xJ(N, counts, seed, p)
            off = HR.offsets(counts)
            for b, m in enumerate(counts):
                if m < N:
                    assert np.all(np.isfinite(cov[b])) and lam[b] > 0.0
                    continue
                Jb = J[off[b]:off[b + 1]]
                A = Jb.T @ Jb + lam[b] * np.eye(N)
                assert_rel(cov[b].reshape(N, N), np.linalg.inv(A))
                assert_rel(X[b].T, np.linalg.solve(A, R[b].T))
            stream = torch.cuda.current_stream().cuda_stream
            d_out = torch.full((B, N * N), float("nan"), dtype=torch.float64, device="cuda")
            assert L.dogleg_gpu_batch_covariance_device(h, d_out.data_ptr(), 0, stream) == 0
            d_R = torch.from_numpy(R).cuda()
            d_X = torch.full_like(d_R, float("nan"))
            assert L.dogleg_gpu_batch_solve_device(h, d_R.data_ptr(), d_X.data_ptr(), 3, stream) == 0
            torch.cuda.synchronize()
            assert np.array_equal(d_out.cpu().numpy(), cov) and np.array_equal(d_X.cpu().numpy(), X)
        free(h)
    HR.free(dev)


def ragged_numpy_outlierness(x, J, counts, lam, fs, nfeat, off):
    fw, sw = {}, np.zeros(len(counts))
    for b in range(len(counts)):
        fw[b], sw[b] = numpy_outlierness(x[off[b]:off[b + 1]], J[off[b]:off[b + 1]], lam[b], fs, int(nfeat[b]))
    return fw, sw


@pytest.mark.gpu
@pytest.mark.parametrize("fs", [1, 2])
@pytest.mark.parametrize("tr0", [1e3, 0.3])
def test_outlierness_against_numpy(H, tr0, fs):
    """Nfeatures NULL, short of Nmeas[b] (trailing rows count in the scale only) and 0 for some problems. Counts of at
    least Nstate + 2 keep the reference's scale finite."""
    N, seed = 16, 1000
    counts = np.random.default_rng(7).integers(N + 2, 400, 30).astype(np.uint32)
    counts[5] = 77
    B = len(counts)
    off = HR.offsets(counts)
    dev, p0 = HR.create(counts, N, seed)
    rc, p, n2, it, h = HR.solve(dev, p0, N, counts, handle=True, max_iterations=30, trustregion0=tr0)
    HR.free(dev)
    st, lam = status(h, B)
    x, J = ragged_xJ(N, counts, seed, p)
    full = (counts // fs).astype(np.int32)
    short = np.where(np.arange(B) % 4 == 0, 0, np.maximum(full - 3, 0)).astype(np.int32)
    for nfeat in (None, short):
        f, sc = outlierness_ragged(h, x, J, fs, nfeat=nfeat, scale=np.full(B, -1.0))
        nf = full if nfeat is None else nfeat
        fw, sw = ragged_numpy_outlierness(x, J, counts, lam, fs, nf, off)
        for b in range(B):
            if nf[b] > 0:
                assert_factors(f[off[b]:off[b] + nf[b]], fw[b])
            assert np.all(np.isnan(f[off[b] + nf[b]:off[b + 1]]))          # no feature: not written
            assert abs(sc[b] - sw[b]) <= 1e-9 * abs(sw[b])
    free(h)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [6, 9, 17, 25])
def test_outlierness_equals_the_padded_handle(H, N):
    """With positive input scales every factor equals dogleg_gpu_batch_outlierness's on the zero-padded handle and data,
    bit for bit (counts 0, 1, N - 1 and N included); and the handle is unchanged afterwards."""
    counts = counts_for(N, seed=11)
    B = len(counts)
    off = HR.offsets(counts)
    seed = 700 + N
    dev, p0 = HR.create(counts, N, seed)
    Mp = HR.mpad(dev)
    rr = HR.solve(dev, p0, N, counts, handle=True, max_iterations=30)
    rp = HR.solve_padded(dev, p0, N, handle=True, max_iterations=30)
    HR.free(dev)
    hr, hp = rr[4], rp[4]
    p = rr[1]
    x, J = ragged_xJ(N, counts, seed, p)
    xp, Jp = np.zeros((B, Mp)), np.zeros((B, Mp, N))
    for b, m in enumerate(counts):
        xp[b, :m], Jp[b, :m] = x[off[b]:off[b + 1]], J[off[b]:off[b + 1]]
    scale = 0.5 + np.arange(B)
    before = (covariance(hr, B, N),) + status(hr, B)
    for fs in (1, 2):
        f, sc = outlierness_ragged(hr, x, J, fs, scale=scale)
        fp, scp = outlierness(hp, xp, Jp, fs, Mp // fs, scale=scale)
        assert np.array_equal(sc, scp)
        for b, m in enumerate(counts):
            assert np.array_equal(f[off[b]:off[b] + m // fs], fp[b, :m // fs]), b
    after = (covariance(hr, B, N),) + status(hr, B)
    for u, v in zip(before, after):
        assert np.array_equal(u, v)
    free(hr)
    free(hp)


@pytest.mark.gpu
def test_outlierness_host_and_device_forms_and_refusals(H):
    """x and J from the ragged callback on a torch stream; the device form equals the host form bit for bit, run to run.
    A bad Nfeatures[b] is refused by the host form (naming b) and gives that problem a NaN scale and no factors in the
    device form. Ragged and uniform handles are refused by each other's calls."""
    torch = pytest.importorskip("torch")
    L = ffi.load()
    N, seed = 16, 1000
    counts = counts_for(N, seed=5)
    counts[counts < N + 2] += N + 2
    B = len(counts)
    off = HR.offsets(counts)
    rows = int(off[-1])
    dev, p0 = HR.create(counts, N, seed)
    rc, p, n2, it, h = HR.solve(dev, p0, N, counts, handle=True, max_iterations=30)
    stream = torch.cuda.Stream()
    d_p = torch.from_numpy(p).cuda()
    d_off = torch.from_numpy(off).cuda()
    d_x = torch.empty(rows, dtype=torch.float64, device="cuda")
    d_J = torch.empty((rows, N), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    HR.lib().dlb_ragged_cb(d_p.data_ptr(), d_x.data_ptr(), d_J.data_ptr(), d_off.data_ptr(), None, B, stream.cuda_stream, dev)
    torch.cuda.synchronize()
    HR.free(dev)
    x, J = d_x.cpu().numpy(), d_J.cpu().numpy()
    xw, Jw = ragged_xJ(N, counts, seed, p)
    assert np.allclose(x, xw, rtol=1e-12, atol=1e-14) and np.allclose(J, Jw, rtol=1e-12, atol=1e-14)
    nout = np.arange(B, dtype=np.int32) % 3
    for fs in (1, 2):
        nfeat = (counts // fs - np.arange(B) % 5).astype(np.int32)
        with torch.cuda.stream(stream):
            d_scale = torch.full((B,), -1.0, dtype=torch.float64, device="cuda")
            d_f = torch.full((rows,), float("nan"), dtype=torch.float64, device="cuda")
            d_nf = torch.from_numpy(nfeat).cuda()
            d_nout = torch.from_numpy(nout).cuda()
        assert L.dogleg_gpu_batch_outlierness_ragged_device(h, d_x.data_ptr(), d_J.data_ptr(), fs, d_nf.data_ptr(),
                                                            d_nout.data_ptr(), d_scale.data_ptr(), d_f.data_ptr(),
                                                            stream.cuda_stream) == 0
        stream.synchronize()
        f, sc = outlierness_ragged(h, x, J, fs, nfeat=nfeat, nout=nout, scale=np.full(B, -1.0))
        assert np.array_equal(d_f.cpu().numpy(), f, equal_nan=True) and np.array_equal(d_scale.cpu().numpy(), sc)
        f2, sc2 = outlierness_ragged(h, x, J, fs, nfeat=nfeat, nout=nout, scale=np.full(B, -1.0))
        assert np.array_equal(f2, f, equal_nan=True) and np.array_equal(sc2, sc)
        # bad counts: refused by the host form, NaN scale and no factors in the device form
        bad = nfeat.copy()
        bad[3] = counts[3] // fs + 1
        bad[7] = -1
        sentinel = np.full(rows, 7.0)
        for b_bad, arr in ((3, bad), (7, np.where(np.arange(B) == 3, nfeat, bad).astype(np.int32))):
            f3, sc3 = outlierness_ragged(h, x, J, fs, nfeat=arr, nout=nout, scale=np.full(B, -1.0), factors=sentinel,
                                         expect=-1)
            msg = L.dogleg_gpu_last_error()
            assert b"dogleg_gpu_batch_outlierness_ragged:" in msg and f"b = {b_bad},".encode() in msg, msg
            assert np.all(f3 == 7.0) and np.all(sc3 == -1.0)
        with torch.cuda.stream(stream):
            d_scale = torch.full((B,), -1.0, dtype=torch.float64, device="cuda")
            d_f = torch.full((rows,), 7.0, dtype=torch.float64, device="cuda")
            d_nf = torch.from_numpy(bad).cuda()
        assert L.dogleg_gpu_batch_outlierness_ragged_device(h, d_x.data_ptr(), d_J.data_ptr(), fs, d_nf.data_ptr(),
                                                            d_nout.data_ptr(), d_scale.data_ptr(), d_f.data_ptr(),
                                                            stream.cuda_stream) == 0
        stream.synchronize()
        fd, sd = d_f.cpu().numpy(), d_scale.cpu().numpy()
        for b in range(B):
            seg = slice(off[b], off[b + 1])
            if b in (3, 7):
                assert np.isnan(sd[b]) and np.all(fd[seg] == 7.0)
            else:
                assert sd[b] == sc[b] and np.array_equal(fd[off[b]:off[b] + nfeat[b]], f[off[b]:off[b] + nfeat[b]])
    # cross refusals
    M = 40
    DL = H.dev_problems_lib()
    up0 = np.zeros((4, N))
    ud = DL.dlb_dev_problem_create_batched(4, M, N, 77, H.as_dp(up0))
    hu = solve2("dense", ud, up0, N, M, max_iterations=5)[4]
    DL.dlb_dev_problem_free(ud)
    xs, fs_ = np.zeros(4 * M * N + rows * N), np.zeros(4 * M + rows)
    scs = np.full(B, -1.0)
    for name, call in (
            ("dogleg_gpu_batch_outlierness", lambda: L.dogleg_gpu_batch_outlierness(h, H.as_dp(xs), H.as_dp(xs), M, 1, M, None,
                                                                                     H.as_dp(scs), H.as_dp(fs_))),
            ("dogleg_gpu_batch_outlierness_device",
             lambda: L.dogleg_gpu_batch_outlierness_device(h, d_x.data_ptr(), d_J.data_ptr(), M, 1, M, None,
                                                           d_scale.data_ptr(), d_f.data_ptr(), None)),
            ("dogleg_gpu_batch_outlierness_ragged",
             lambda: L.dogleg_gpu_batch_outlierness_ragged(hu, H.as_dp(xs), H.as_dp(xs), 1, None, None, H.as_dp(scs),
                                                           H.as_dp(fs_))),
            ("dogleg_gpu_batch_outlierness_ragged_device",
             lambda: L.dogleg_gpu_batch_outlierness_ragged_device(hu, d_x.data_ptr(), d_J.data_ptr(), 1, None, None,
                                                                  d_scale.data_ptr(), d_f.data_ptr(), None))):
        assert call() < 0, name
        msg = L.dogleg_gpu_last_error()
        assert name.encode() + b":" in msg and (b"ragged solve" in msg or b"uniform batched solve" in msg), (name, msg)
    assert np.all(scs == -1.0) and np.all(fs_ == 0.0)
    free(h)
    free(hu)


@pytest.mark.gpu
def test_bad_arguments_are_refused_before_the_first_callback(H):
    L = ffi.load()
    N = 8
    counts = HR.as_counts([5, 0, 30, 12])
    dev, p0 = HR.create(counts, N, 31)
    cb = HR.lib().dlb_ragged_cb_ptr()
    P = H.make_params(L, max_iterations=10)
    huge = HR.as_counts([2 ** 31 - 1] * 40)
    over = HR.as_counts([5, 2 ** 31, 30, 12])
    p40 = np.zeros((40, 32))
    cases = [  # (p, Nstate, Nmeas, B, callback, message)
        (p0, 0, counts, 4, cb, b"Nstate"),
        (p0, 33, counts, 4, cb, b"Nstate"),
        (p0, N, counts, 0, cb, b"bad arguments"),
        (p0, N, None, 4, cb, b"bad arguments"),
        (None, N, counts, 4, cb, b"bad arguments"),
        (p0, N, counts, 4, None, b"bad arguments"),
        (p0, N, over, 4, cb, b"Nmeas[1] = 2147483648 exceeds INT_MAX"),
        (p40, 32, huge, 40, cb, b"out of device memory"),
    ]
    for p, n, c, B, f, want in cases:
        q = None if p is None else p.copy()
        h = C.c_void_p(1234)
        rc = L.dogleg_gpu_optimize_dense_batched_ragged(None if q is None else H.as_dp(q), n,
                                                        None if c is None else HR.as_up(c), B, f, C.c_void_p(dev),
                                                        C.byref(P), None, None, C.byref(h))
        msg = L.dogleg_gpu_last_error()
        assert rc < 0 and b"dogleg_gpu_optimize_dense_batched_ragged:" in msg and want in msg, (n, B, msg)
        assert h.value is None
        assert HR.ncalls(dev) == 0
        if q is not None:
            assert np.array_equal(q, p)
    HR.free(dev)
