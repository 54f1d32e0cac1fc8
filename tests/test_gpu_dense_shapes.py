"""The dense single-problem path (DOGLEG_DENSE, DOGLEG_DENSE_PRODUCTS) one engine call at a time, at every shape
where its kernels switch, up to C5's 4096 states, against high-precision references and LAPACK.

Every tolerance is an a-priori first-order rounding-error bound c*n*u*(the same sum taken over absolute values),
u = 2^-53, c <= 4 (Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed., ch. 3, 8, 10). Such a bound
holds for any summation order, so it covers the fixed-order sums, the DMMA tiles, the rsqrt pivots and the
inverted diagonal blocks alike (DESIGN.md section 5, divergences 7 and 10). The largest ratio of error to bound
each check met is printed at the end of the module (pytest -s)."""
import ctypes

import numpy as np
import pytest
import scipy.linalg

from libdogleg_b200 import ffi

pytestmark = pytest.mark.gpu
U = 2.0 ** -53
LD = np.longdouble

# ---------------------------------------------------------------- the kernels' plans, restated
# dlb_dense.cu: SY_T, SY_K, SY_DMMA_MIN_N; dlb_bigfront.cu: BF_NB; dlb_bigsolve.cu: BS_SUPER; dlb_engine.cu:
# DLB_SMALL_FRONT_MAX; dlb_front.cu: the thread counts of k_front_level
SY_T, SY_K, SY_DMMA_MIN_N, SJ_T = 64, 16, 96, 128
BF_NB, BS_SUPER, SMALL_FRONT_MAX = 64, 512, 158


def syrk_plan(M, N, sm_count):
    """syrk_plan of dlb_dense.cu: (tile size, tiles, row slices, rows per slice)."""
    T = SJ_T if N >= SY_DMMA_MIN_N else SY_T
    nt = (N + T - 1) // T
    ntile = nt * (nt + 1) // 2
    nslice = (2 * sm_count) // ntile
    if ntile > sm_count and N >= SY_DMMA_MIN_N:
        best = 0.0
        for ns in range(1, 9):
            total = ntile * ns
            waves = (total + sm_count - 1) // sm_count
            eff = total / (waves * sm_count)
            if eff > best + 0.02:
                best, nslice = eff, ns
    nslice = max(1, min(nslice, (M + 255) // 256))
    rows_per = (M + nslice - 1) // nslice
    rows_per = (rows_per + SY_K - 1) // SY_K * SY_K
    nslice = max(1, (M + rows_per - 1) // rows_per)
    return T, ntile, nslice, rows_per


def bs_super(nc):
    """bs_super of dlb_bigsolve.cu: columns per launch of the triangular solves."""
    return BS_SUPER if nc > 2 * BS_SUPER else nc


def branches(N, M, sm_count):
    """What the dense path does at (N, M) on a GPU with sm_count SMs."""
    T, ntile, nslice, rows_per = syrk_plan(M, N, sm_count)
    b = dict(tile=T, wave_sliced=ntile > sm_count and T == SJ_T, nslice=nslice,
             odd16=nslice > 1 and rows_per % 32 == 16, partial_last=M - (nslice - 1) * rows_per < rows_per)
    if N <= SMALL_FRONT_MAX:                  # one front in shared memory: k_front_level
        b.update(front="smem", threads=512 if N > 64 else 256 if N > 40 else 128)
    else:                                     # dlb_bigfront.cu, lazy right-looking (one front: 1 * N/64 row tiles)
        npanel = (N + BF_NB - 1) // BF_NB
        cmax = bs_super(N)
        b.update(front="hbm", panels=npanel, below=N - (npanel - 1) * BF_NB - 1,
                 supers=(N + cmax - 1) // cmax, last_super=N - (N - 1) // cmax * cmax)
    return b


# (N, M, the branches this fixture is here for), computed for 148 SMs and asserted on the device the test runs on
SHAPES = [
    (1, 50, dict(front="smem", threads=128)),
    (7, 300, dict(threads=128, nslice=2)),
    (8, 300, dict(threads=128, nslice=2)),
    (40, 700, dict(threads=128, nslice=3, odd16=True, partial_last=True)),
    (41, 700, dict(threads=256, nslice=3, odd16=True)),
    (64, 900, dict(threads=256, tile=64)),
    (65, 900, dict(threads=512, tile=64)),
    (95, 5000, dict(tile=64, nslice=20)),
    (96, 5000, dict(tile=128, nslice=20)),
    (158, 3000, dict(front="smem", threads=512)),
    (159, 3000, dict(front="hbm", panels=3)),
    (192, 3000, dict(panels=3, below=63)),
    (193, 3000, dict(panels=4, below=0)),
    (255, 3000, dict(panels=4, below=62)),
    (1024, 4000, dict(panels=16, supers=1)),
    (1025, 4000, dict(panels=17, below=0, supers=3, last_super=1)),
    (2049, 5000, dict(wave_sliced=True, nslice=8, below=0, supers=5, last_super=1)),
    (2112, 6000, dict(wave_sliced=True, nslice=8, odd16=True, partial_last=True, supers=5)),
    (4096, 8176, dict(wave_sliced=True, nslice=7, odd16=True, panels=64, supers=8)),
]
SHAPE_IDS = ["%dx%d" % (N, M) for N, M, _ in SHAPES]
GRADED = (1025, 4000)          # J diag(10^linspace(-3, 3, N)): cond(J'J) ~ 1e13


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize("N,M,claims", SHAPES, ids=SHAPE_IDS)
def test_each_fixture_reaches_the_branches_it_claims(N, M, claims):
    """A fixture that no longer reaches its branch (a changed constant, another GPU) fails here instead of
    quietly covering less."""
    got = branches(N, M, sm_count())
    assert {k: got.get(k) for k in claims} == claims, got


def test_the_fixtures_cover_every_branch():
    """The fixtures together cover every switch of the dense path (on a 148-SM B200)."""
    b = [branches(N, M, 148) for N, M, _ in SHAPES]
    assert {x["threads"] for x in b if x["front"] == "smem"} == {128, 256, 512}
    assert {x["tile"] for x in b} == {SY_T, SJ_T}
    assert any(x["wave_sliced"] and x["odd16"] and x["partial_last"] for x in b)
    assert any(x["wave_sliced"] and x["nslice"] > 1 and not x["partial_last"] for x in b)
    assert any(x["front"] == "hbm" and x["below"] == 0 for x in b)
    assert any(x.get("last_super") == 1 for x in b) and max(x.get("supers", 0) for x in b) == 8
    assert max(N for N, _, _ in SHAPES) == 4096


# ---------------------------------------------------------------- fixtures and references
def make_problem(N, M, graded=False):
    rng = np.random.default_rng(1000 * N + M + graded)
    J = rng.standard_normal((M, N))
    if graded:
        J *= 10.0 ** np.linspace(-3, 3, N)
    return J, rng.standard_normal(M), rng.standard_normal(N)


RATIO = {}


def within(where, name, err, bound):
    """err <= bound entry by entry; remembers the largest ratio of each check over all shapes."""
    err, bound = np.broadcast_arrays(np.asarray(err, dtype=np.float64), np.asarray(bound, dtype=np.float64))
    bad = ~(err <= bound)
    assert not bad.any(), "%s, %s: %d entries beyond the bound, worst %r > %r" % (
        where, name, bad.sum(), err[bad].max() if np.isfinite(err[bad]).all() else np.nan, bound[bad][0])
    nz = bound > 0
    if nz.any():                              # graded, schedule and singular-column checks reported on their own
        key = where.split()[0] + ": " + name if where.split()[0] in ("graded", "left", "right", "diag") else name
        RATIO[key] = max(RATIO.get(key, 0.0), float((err[nz] / bound[nz]).max()))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if RATIO:
        print("\nlargest error / bound of test_gpu_dense_shapes.py:")
        for k in sorted(RATIO):
            print("  %-44s %.3g" % (k, RATIO[k]))


def unpack_upper(packed, N):
    """Row-first packed upper (dpptrf's layout of L', the layout of dlb_engine_dense_factor_to_host) -> L."""
    Up = np.zeros((N, N))
    Up[np.triu_indices(N)] = packed
    return Up.T.copy()


def factor_of(E):
    out = np.full(E.N * (E.N + 1) // 2 if E.packed or E.type == ffi.SOLVE_DENSE else E.N * E.N, np.nan)
    E.check(E.L.dlb_engine_dense_factor_to_host(E.h, out.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
    return out


def residual_ld(A, X, B):
    """B - A X with the products and sums in long double, rounded to double."""
    return (B.astype(LD) - A.astype(LD) @ X.astype(LD)).astype(np.float64)


def check_factor(tag, A, L, lam, lapack=True, scaled=False):
    """L from the GPU against A + lam I (the matrix the GPU assembled)."""
    N = A.shape[0]
    Al = A + lam * np.eye(N)
    assert np.isfinite(L).all()
    assert not np.triu(L, 1).any()
    # Cholesky backward error |dA| <= gamma_{N+1} |L||L'| (Higham Thm 10.3), plus gamma_N for forming L L' here
    within(tag, ("singular column: " if lam == 1e-10 else "") + "|LL'-A| <= 2(N+1)u|L||L'|", np.abs(L @ L.T - Al), 2 * (N + 1) * U * (np.abs(L) @ np.abs(L).T))
    if not lapack:
        return
    cf = scipy.linalg.cho_factor(Al, lower=True)
    Lr = np.tril(cf[0])
    ev = np.linalg.eigvalsh(Al)
    # forward error of both factors: ||dL|| <~ kappa_2(A) ||dA|| / ||A|| ||L|| (Higham Thm 10.8), ||dA|| <= (N+1)u ||A||
    within(tag, "|L-L_lapack| <= 8Nu k2(A) max|L|", np.abs(L - Lr).max(), 8 * N * U * (ev[-1] / ev[0]) * np.abs(L).max())
    if scaled:
        # the same bound on S A S, S = diag(A)^-1/2: chol(S A S) = S L, and the elimination is scale-invariant
        s = 1.0 / np.sqrt(np.diag(Al))
        es = np.linalg.eigvalsh(s[:, None] * Al * s[None, :])
        within(tag, "|S(L-L_lapack)| <= 8Nu k2(SAS) max|SL|", np.abs(s[:, None] * (L - Lr)).max(),
               8 * N * U * (es[-1] / es[0]) * np.abs(s[:, None] * L).max())
    return cf, Al, ev[-1] / ev[0]


def check_solve(tag, what, Al, cf, kappa, X, B):
    """X from the GPU solves Al X = B (columns): normwise backward error, forward error against LAPACK's."""
    N = Al.shape[0]
    B = B.reshape(N, -1)
    X = X.reshape(N, -1)
    assert np.isfinite(X).all()
    X0 = scipy.linalg.cho_solve(cf, B)
    R0 = residual_ld(Al, X0, B)
    steps = 3 if kappa * U > 1e-12 else 1                # contraction kappa*u per step
    Xr = X0 + scipy.linalg.cho_solve(cf, R0)             # iterative refinement, residuals in long double
    for _ in range(steps - 1):
        Xr = Xr + scipy.linalg.cho_solve(cf, residual_ld(Al, Xr, B))
    # b - A x for the GPU's x: R0 from long double, the small correction A (x - x0) in double
    R = R0 - Al @ (X - X0)
    nA = np.abs(Al).sum(axis=1).max()
    eta = np.abs(R).max(axis=0) / (nA * np.abs(X).max(axis=0) + np.abs(B).max(axis=0))
    # Cholesky solves are normwise backward stable: (A + dA) x = b, ||dA|| <= c N u ||A|| (Higham Thm 10.4)
    within(tag, what + " backward error <= 4Nu", eta, 4 * N * U)
    nx = np.abs(Xr).max(axis=0)
    fe = np.abs(X - Xr).max(axis=0).max() / nx.max()
    fe_lapack = np.abs(X0 - Xr).max(axis=0).max() / nx.max()
    within(tag, what + " forward error <= 10 lapack + 4Nu", fe, 10 * fe_lapack + 4 * N * U)


def run_dense_checks(H, N, M, graded=False, label=""):
    tag = label or ("%dx%d" % (N, M))
    J, x, p = make_problem(N, M, graded)
    Jl, xl = J.astype(LD), x.astype(LD)
    aJ = np.abs(J)
    E = H.Engine(ffi.SOLVE_DENSE, N, M)
    try:
        E.load_dense(0, p, x, J)
        # ---- evaluation: J'x, |x|^2, max|J'x|
        sc = E.evaluate(0)
        g = E.download(0)["Jtx"]
        g_ref = (Jl.T @ xl).astype(np.float64)
        ax = aJ.T @ np.abs(x)
        within(tag, "J'x", np.abs(g - g_ref), (M + 2) * U * ax)
        within(tag, "|x|^2", abs(sc.norm2_x - float(np.sum(xl * xl))), (M + 2) * U * float(x @ x))
        assert sc.maxabs_Jtx == np.abs(g).max()
        within(tag, "max|J'x|", abs(sc.maxabs_Jtx - np.abs(g_ref).max()), (M + 2) * U * ax.max())
        gl = g.astype(LD)
        within(tag, "|J'x|^2", abs(sc.norm2_Jtx - float(np.sum(gl * gl))), (N + 2) * U * float(g @ g))
        # ---- |J J'x|^2 (the Cauchy step), v = the GPU's own J'x: sum_i (sum_k J_ik v_k)^2
        sc = E.cauchy(0)
        y = Jl @ gl
        z = aJ @ np.abs(g)
        within(tag, "|J J'x|^2", abs(sc.norm2_JJtx - float(np.sum(y * y))), (2 * N + M + 2) * U * float(z @ z))
        # ---- the assembled J'J (before factorize: debug_JtJ runs the SYRK again and drops the factor)
        A = E.JtJ(0, 0.0)
        assert np.array_equal(A, A.T)
        aa = aJ.T @ aJ
        within(tag, "J'J vs BLAS", np.abs(A - J.T @ J), 2 * (M + 2) * U * aa)
        edges = sorted({k for k in (0, 63, 64, 127, 128, N - 1) if 0 <= k < N})
        Ae = (Jl[:, edges].T @ Jl).astype(np.float64)        # whole rows (= columns) at the tile edges
        within(tag, "J'J tile-edge rows, long double", np.abs(A[edges] - Ae), (M + 1) * U * aa[edges])
        rng = np.random.default_rng(N)
        I = rng.integers(0, N, 2000)
        K = rng.integers(0, N, 2000)
        for c in range(0, 2000, 500):
            i, k = I[c:c + 500], K[c:c + 500]
            a_ref = np.einsum("mi,mi->i", Jl[:, i], Jl[:, k]).astype(np.float64)
            within(tag, "J'J 2000 entries, long double", np.abs(A[i, k] - a_ref), (M + 1) * U * aa[i, k])
        # ---- factor, Gauss-Newton step, solves
        for lam in (0.5, 0.0):
            assert E.factorize(0, lam) == -1
            L = unpack_upper(factor_of(E), N)
            cf, Al, kappa = check_factor(tag, A, L, lam, scaled=graded)
            E.gauss_newton(0)
            gn = E.download(0)["gn"]
            check_solve(tag, "Gauss-Newton", Al, cf, kappa, -gn, g)
            if lam == 0.0:
                for nrhs in (1, 3, 64):
                    B = rng.standard_normal((N, nrhs))
                    check_solve(tag, "solve(B)", Al, cf, kappa, E.solve(B), B)
        # ---- |J step|^2 of the Gauss-Newton step
        sc = E.step(0, 1, ffi.STEP_GAUSSNEWTON, 1e9)
        st = E.download(1)["step"]
        assert np.array_equal(st, gn)
        y = Jl @ st.astype(LD)
        z = aJ @ np.abs(st)
        within(tag, "|J step|^2", abs(sc.norm2_Jstep - float(np.sum(y * y))), (2 * N + M + 2) * U * float(z @ z))
    finally:
        E.close()


@pytest.mark.parametrize("N,M", [s[:2] for s in SHAPES], ids=SHAPE_IDS)
def test_dense_engine_at_the_branch_shapes(H, N, M):
    run_dense_checks(H, N, M)


def test_graded_columns_keep_the_factor_scale_invariant(H):
    """cond(J'J) ~ 1e13, cond of the equilibrated matrix ~ 40: the Cholesky factor, its pivots and the inverted
    diagonal blocks of the solves are scale-invariant, so the solves stay as accurate as LAPACK's."""
    run_dense_checks(H, *GRADED, graded=True, label="graded %dx%d" % GRADED)


@pytest.mark.parametrize("N,M", [s[:2] for s in SHAPES], ids=SHAPE_IDS)
def test_exact_singular_columns_are_reported_at_their_column(H, N, M):
    """A zero column k of J makes pivot k an exact 0: factorize(0, 0) reports minor == k; the first rung of the
    lambda ladder (1e-10) then factorizes, within the backward bound of A + 1e-10 I."""
    J, x, p = make_problem(N, M)
    E = H.Engine(ffi.SOLVE_DENSE, N, M)
    try:
        for k in [k for k in (0, 63, 64, 157, 158, 511, 512, 1023, 1024, N - 1) if k < N]:
            Jk = J.copy()
            Jk[:, k] = 0.0
            E.load_dense(0, p, x, Jk)
            E.evaluate(0)
            A = E.JtJ(0, 0.0)
            assert not A[k].any() and not A[:, k].any()
            assert E.factorize(0, 0.0) == k
            assert E.factorize(0, 1e-10) == -1
            check_factor("singular column %d of %dx%d" % (k, N, M), A, unpack_upper(factor_of(E), N), 1e-10, lapack=False)
    finally:
        E.close()


@pytest.mark.parametrize("sched", ["left", "right", "diag"])
@pytest.mark.parametrize("N,M", [(193, 3000), (1025, 4000)])
def test_every_panel_schedule_on_one_dense_front(H, N, M, sched, monkeypatch):
    """A single dense front only ever takes the right-looking schedule; the left-looking and throughput ones
    (sparse big fronts) must factorize and solve it just as well."""
    monkeypatch.setenv("DOGLEG_GPU_BF_SCHEDULE", sched)
    J, x, p = make_problem(N, M)
    E = H.Engine(ffi.SOLVE_DENSE, N, M)
    try:
        E.load_dense(0, p, x, J)
        E.evaluate(0)
        g = E.download(0)["Jtx"]
        A = E.JtJ(0, 0.0)
        tag = "%s %d" % (sched, N)
        for lam in (0.5, 0.0):
            assert E.factorize(0, lam) == -1
            cf, Al, kappa = check_factor(tag, A, unpack_upper(factor_of(E), N), lam)
            E.gauss_newton(0)
            check_solve(tag, "Gauss-Newton", Al, cf, kappa, -E.download(0)["gn"], g)
            B = np.random.default_rng(N).standard_normal((N, 3))
            check_solve(tag, "solve(B)", Al, cf, kappa, E.solve(B), B)
    finally:
        E.close()


LAYOUTS = {"packed-upper": (1, 1), "full": (0, 0), "packed-lower": (1, 0)}


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("N,M", [(159, 3000), (1025, 4000)])
def test_products_engine_equals_the_dense_engine_bit_for_bit(H, N, M, layout):
    """Fed the dense engine's own J'J and J'x, a dense-products engine runs the same kernels on the same front:
    the same factor and Gauss-Newton step to the last bit, in every layout."""
    packed, upper = LAYOUTS[layout]
    J, x, p = make_problem(N, M)
    D = H.Engine(ffi.SOLVE_DENSE, N, M)
    try:
        D.load_dense(0, p, x, J)
        D.evaluate(0)
        g = D.download(0)["Jtx"]
        A = D.JtJ(0, 0.0)
        assert D.factorize(0, 0.0) == -1
        fac = factor_of(D)
        D.gauss_newton(0)
        gn = D.download(0)["gn"]
    finally:
        D.close()
    if packed and upper:
        lay = A[np.triu_indices(N)]
    elif packed:
        lay = A[np.tril_indices(N)]
    else:
        lay = A.ravel().copy()
    P = H.Engine(ffi.SOLVE_DENSE_PRODUCTS, N, 0, 0, packed, upper)
    try:
        P.load_products(0, p, g, lay)
        P.evaluate(0, float(x @ x))
        assert P.factorize(0, 0.0) == -1
        out = factor_of(P)
        L = np.zeros((N, N))
        if packed and upper:
            L = unpack_upper(out, N)
        elif packed:                                        # row-first packed lower: L itself
            L[np.tril_indices(N)] = out
        else:                                               # Fortran 'L' of the row-first array: L' in its upper half
            F = out.reshape(N, N)
            L = np.triu(F).T
            assert np.array_equal(F[np.tril_indices(N, -1)], A[np.tril_indices(N, -1)])   # the user's values stay
        assert np.array_equal(L[np.tril_indices(N)], unpack_upper(fac, N)[np.tril_indices(N)])
        P.gauss_newton(0)
        assert np.array_equal(P.download(0)["gn"], gn)
        if packed and not upper:
            with pytest.raises(RuntimeError):              # as in the reference (dogleg.c:597-601)
                P.cauchy(0)
    finally:
        P.close()


def test_c5_shape_is_bit_reproducible(H):
    """DESIGN.md section 4: fixed summation order everywhere, so two fresh engines agree to the last bit."""
    N, M = 4096, 8176
    J, x, p = make_problem(N, M)
    B = np.random.default_rng(5).standard_normal((N, 3))
    outs = []
    for _ in range(2):
        E = H.Engine(ffi.SOLVE_DENSE, N, M)
        try:
            E.load_dense(0, p, x, J)
            sc = E.evaluate(0)
            o = [np.array([sc.norm2_x, sc.norm2_Jtx, sc.maxabs_Jtx]), E.download(0)["Jtx"], E.JtJ(0, 0.0)]
            assert E.factorize(0, 0.0) == -1
            o.append(factor_of(E))
            sc = E.gauss_newton(0)
            o += [np.array([sc.norm2_gn]), E.download(0)["gn"], E.solve(B)]
            outs.append(o)
        finally:
            E.close()
    for a, b in zip(*outs):
        assert np.array_equal(a, b)
