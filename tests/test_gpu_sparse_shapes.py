"""The sparse multifrontal path (DOGLEG_SPARSE) one engine call at a time, on fixtures whose front shapes are built
to reach every branch of the factorization and the solves, against a-priori rounding-error bounds.

Each fixture is a tree of cliques: node v owns c_v states and touches s_v states of its parent's front, so with
DOGLEG_GPU_RELAX=0 and the postorder injected as the ordering its front has exactly c_v + s_v rows and c_v pivots.
Every fixture restates the dispatch rule it is there for from the engine's symbolic analysis, asserts it, and
checks the restatement against the number of kernel launches one factorization makes.

Every tolerance is a first-order bound c*(m*u*|J|'|J| + k*u*|L||L'|), u = 2^-53, c <= 4, k the number of terms of
the factor's inner products (Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed., ch. 3, 8, 10). Such a
bound holds for any summation order, so it covers the DMMA tiles, the inverted diagonal blocks and the gathers
alike. The largest ratio of error to bound each check met is printed at the end of the module (pytest -s)."""
import ctypes as C
import os

import numpy as np
import pytest
import scipy.linalg

from libdogleg_b200 import ffi

pytestmark = pytest.mark.gpu
U = 2.0 ** -53
LD = np.longdouble
CB = 4                                  # the constant of every bound

# ---------------------------------------------------------------- the kernels' plans, restated
# dlb_engine.cu: DLB_SMALL_FRONT_MAX, the leaf-front eligibility; dlb_bigfront.cu: BF_NB and the schedule thresholds;
# dlb_bigsolve.cu: BS_SUPER; dlb_gatherplan.h: heavy (two passes over source lists longer than gsplit are read from the
# plan itself); dlb_trial.cu: the thread count and shared memory of k_trial
SMALL_FRONT_MAX, BF_NB, BS_SUPER = 158, 64, 512
HEAVY, LEAF_ROWS, LEAF_COLS, LEAF_MMA_COLS = 4, 48, 8, 4
SYM_SN_FIRST, SYM_ROWS_PTR, SYM_ROWS, SYM_CHILD_PTR, SYM_LEVEL_PTR, SYM_LEVEL_SN = 3, 4, 5, 11, 13, 14
GP_SRC_PTR, GP_LEVEL_PTR = 1, 7
ENV = {"DOGLEG_GPU_RELAX": "0", "DOGLEG_GPU_ENGINE_CACHE": "0"}
LEAF_MIN = 100                         # DOGLEG_GPU_LEAF_MIN for the leaf fixtures (default 1024)


def front_threads(rows):
    """dlb_launch_front_level: threads of k_front_level for a level whose largest small front has `rows` rows."""
    return 512 if rows > 64 else 256 if rows > 40 else 128


def bf_schedule(nf, max_r, forced=None):
    """dlb_bigfront_factor_batch: (front, 64-row tile) pairs pick the panel schedule."""
    if forced:
        return forced
    pairs = nf * ((max_r + 63) // 64)
    return "diag" if pairs > 2 * 296 else "right" if pairs < 2 * 148 else "left"


def bf_launches(nf, max_r, max_nc, forced=None):
    """kernel launches of dlb_bigfront_factor_batch for one level"""
    sched = bf_schedule(nf, max_r, forced)
    nsteps = (max_nc + BF_NB - 1) // BF_NB
    nt = (max_r - 1 + 63) // 64
    if sched == "diag":                        # k_bf_diag + k_bf_trsm per panel, then the Schur complement
        return 2 * nsteps + (nt > 0)
    if sched == "left":                        # one k_bf_step per panel, then the Schur complement
        return nsteps + (nt > 0)
    below = max_r - (nsteps - 1) * BF_NB - 1   # right-looking: one k_bf_step per panel, the last update behind them
    return nsteps + (below > 0)


def trial_threads(max_rows):
    return 512 if max_rows > 112 else 256


def trial_smem(max_rows):
    return 8 * ((max_rows + 2) * max_rows + 2 * max_rows + 8)


TRIAL_SMEM_MAX = 200 * 1024             # the dynamic shared memory k_trial opts into: 157 rows fit, 158 do not


# ---------------------------------------------------------------- fixtures
class Fixture:
    """Jt in CCS (measurement columns grouped in classes of one pattern) for a tree of cliques.
    nodes: (c, s, parent) with parents before children; leaves with chunk > 0 split their separator into chunks of
    that many states, one class of nm measurement columns per chunk (the bundle-adjustment shape the leaf kernels
    take); every other node has c + 8 measurement columns over its whole front."""

    def __init__(self, name, nodes, seed, chunk=0, nm=2, graded=False):
        rng = np.random.default_rng(seed)
        self.name, self.nodes = name, nodes
        C_, S_, nid = [], [], 0
        for c, s, par in nodes:
            C_.append(np.arange(nid, nid + c))
            nid += c
            pool = np.concatenate([C_[par], S_[par]]) if par >= 0 else np.zeros(0, int)
            assert s <= len(pool)
            S_.append(np.sort(rng.choice(pool, s, replace=False)) if s else np.zeros(0, int))
        N = nid
        kids = [[] for _ in nodes]
        order = []
        for v, (_, _, par) in enumerate(nodes):
            if par >= 0:
                kids[par].append(v)

        def visit(v):
            for ch in kids[v]:
                visit(ch)
            order.append(v)
        for v, (_, _, par) in enumerate(nodes):
            if par < 0:
                visit(v)
        label = rng.permutation(N)                  # internal id -> state: the ordering is not the identity
        self.perm = label[np.concatenate([C_[v] for v in order])].astype(np.int32)
        self.node_states = [label[C_[v]] for v in range(len(nodes))]
        # values on a grid of 2^-16 (|J'J| sums stay below 2^53 of its units: the reference J'J is exact in double),
        # graded columns: any doubles, the reference in long double
        self.graded = graded
        scale = 10.0 ** np.linspace(-3, 3, N)[rng.permutation(N)] if graded else np.ones(N)
        quant = (lambda v: v) if graded else (lambda v: np.round(v * 65536.0) / 65536.0)
        self.classes = []                           # (states ascending, m x k values)
        for v, (c, s, par) in enumerate(nodes):
            if chunk and not kids[v] and par >= 0:
                parts = [S_[v][i:i + chunk] for i in range(0, s, chunk)]
                groups = [(np.concatenate([C_[v], q]), nm) for q in parts]
            else:
                groups = [(np.concatenate([C_[v], S_[v]]), c + 8)]
            for internal, m in groups:
                st = np.sort(label[internal])
                self.classes.append((st, quant(rng.standard_normal((m, len(st))) * scale[st])))
        self.N = N
        self.M = sum(V.shape[0] for _, V in self.classes)
        self.rebuild()
        self.x = rng.standard_normal(self.M)
        self.p = rng.standard_normal(N)

    def rebuild(self):
        Jp, Ji, Jx = [0], [], []
        for st, V in self.classes:
            for row in V:
                Ji.append(st)
                Jx.append(row)
                Jp.append(Jp[-1] + len(st))
        self.Jp = np.array(Jp, dtype=np.int32)
        self.Ji = np.concatenate(Ji).astype(np.int32)
        self.Jx = np.concatenate(Jx)
        self.nnz = len(self.Ji)

    def zero_state(self, k):
        """J with the column of state k zeroed (the pattern keeps its explicit zeros)"""
        self.classes = [(st, np.where(st[None, :] == k, 0.0, V)) for st, V in self.classes]
        self.rebuild()

    def reference(self, lam):
        """(J'J + lam I in long double, |J|'|J| + lam I, the number of roundings m_ij + 1 of each entry)"""
        if getattr(self, "_ref", None) is None or self._ref[0] is not self.classes:
            N = self.N
            A = np.zeros((N, N), dtype=LD)
            aa = np.zeros((N, N))
            m = np.ones((N, N))
            for st, V in self.classes:
                ix = np.ix_(st, st)
                A[ix] += (V.T @ V).astype(LD) if not self.graded else V.T.astype(LD) @ V.astype(LD)
                aa[ix] += np.abs(V).T @ np.abs(V)
                m[ix] += V.shape[0]
            self._ref = (self.classes, A, aa, m)
        _, A, aa, m = self._ref
        A, aa = A.copy(), aa.copy()
        d = np.arange(self.N)
        A[d, d] += lam
        aa[d, d] += lam
        return A, aa, m


def clique_tree(levels, seed):
    """levels: (count per parent, c, s) from the root down"""
    nodes = [(levels[0][1], 0, -1)]
    prev = [0]
    for cnt, c, s in levels[1:]:
        cur = []
        for par in prev:
            for _ in range(cnt):
                nodes.append((c, s, par))
                cur.append(len(nodes) - 1)
        prev = cur
    return nodes


def star(root_c, kids, extra_roots=()):
    """a root of root_c states with children (c, s) and separate single-front trees of extra_roots states"""
    return [(root_c, 0, -1)] + [(c, s, 0) for c, s in kids] + [(c, 0, -1) for c in extra_roots]


def _children(seed, n, rlo, rhi, clo, chi):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        c = int(rng.integers(clo, chi + 1))
        out.append((c, int(rng.integers(rlo, rhi + 1)) - c))
    return out


def _leaves(n, cs):
    out = []
    for i in range(n):
        c = cs[i % len(cs)]
        r = LEAF_ROWS if i % 3 == 0 else 36 + i % 12
        out.append((c, r - c))
    return out


def _gather_tree():
    nodes = [(112, 0, -1), (10, 50, 0), (12, 60, 0)]
    nodes += [(4, 56, 1)] * 30 + [(6, 50, 2)] * 5
    return nodes


# name: (nodes, fixture options, environment, the branches the fixture is there for)
FIXTURES = {
    # k_front_level at 40 / 41 / 64 / 65 / 158 rows, small-front solves both sides of 64, a 159-row root without update block
    "ladder": (clique_tree([(1, 159, 0), (1, 30, 128), (2, 10, 55), (2, 10, 54), (2, 6, 35), (2, 4, 36)], 1), {}, {},
               dict(threads={128, 256, 512}, level_rows={40, 41, 64, 65, 158}, solve_threads={128, 512}, big_nc={159},
                    rootless_update=True)),
    # big fronts of different r and nc in one level (159 rows; nc 1, 63, 64, 65, 130), right-looking
    "bigs": (star(193, [(1, 158), (63, 137), (64, 106), (65, 165), (130, 170), (8, 50)]), {}, {},
             dict(schedules={"right"}, big_nc={1, 63, 64, 65, 130, 193}, big_rows={159})),
    # big fronts of 159 and 160 rows with children: they fit the shared-memory variant of k_front_level, which must
    # keep the update matrices gathered into them (it used to start them from zero)
    "big-smem": ([(160, 0, -1), (30, 128, 0), (159, 0, -1), (20, 100, 2)], {}, {},
                 dict(schedules={"right"}, big_rows={159, 160}, rootless_update=True)),
    "left": (star(200, _children(3, 80, 159, 192, 1, 8), [193]), {}, {}, dict(schedules={"left", "right"})),
    "diag": (star(200, _children(4, 160, 159, 192, 1, 8), [193]), {}, {}, dict(schedules={"diag", "right"})),
    # a 1030-pivot root: super-block solves
    "super": (star(1030, [(20, 100)] * 6), {}, {}, dict(super=True)),
    # heavy fronts with 5 and 30 children, two-pass gathers, strips of 32 (trial-kernel tree), k_trial<256> at 112 rows
    "gather": (_gather_tree(), {}, {}, dict(heavy={5, 30}, two_pass=True, trial=256, max_rows=112)),
    "trial113": (star(113, [(8, 90)] * 3), {}, {}, dict(trial=512, max_rows=113)),
    # 160 fronts of 157 rows in one level: more fronts than k_trial<512> has CTAs (158 rows do not fit its shared memory)
    "trial157": (star(157, [(2, 155)] * 160), {}, {}, dict(trial=512, max_rows=157, wide=True)),
    # leaf fronts: <= 4 pivots (MMA), 5 and 8 pivots (scalar), the MMA shapes on the scalar kernel
    "leaf34": (star(60, _leaves(120, [3, 4])), dict(chunk=9, nm=2), {"DOGLEG_GPU_LEAF_MIN": str(LEAF_MIN)},
               dict(leaf="mma", leaf_nc={3, 4}, leaf_rows=LEAF_ROWS)),
    "leaf58": (star(60, _leaves(120, [5, 8])), dict(chunk=9, nm=3), {"DOGLEG_GPU_LEAF_MIN": str(LEAF_MIN)},
               dict(leaf="scalar", leaf_nc={5, 8}, leaf_rows=LEAF_ROWS)),
    "leaf34-scalar": (star(60, _leaves(120, [3, 4])), dict(chunk=9, nm=2),
                      {"DOGLEG_GPU_LEAF_MIN": str(LEAF_MIN), "DOGLEG_GPU_LEAF_MMA": "0"},
                      dict(leaf="scalar", leaf_nc={3, 4}, leaf_rows=LEAF_ROWS)),
}
NAMES = list(FIXTURES)
_cache = {}


def fixture(name, graded=False):
    key = (name, graded)
    if key not in _cache:
        nodes, opts, _, _ = FIXTURES[name]
        _cache[key] = Fixture(name, nodes, seed=7 + NAMES.index(name), graded=graded, **opts)
    return _cache[key]


@pytest.fixture(scope="module", autouse=True)
def _module_env():
    """no relaxed amalgamation (the fronts are the fixtures' cliques), no engine reuse across environments"""
    saved = {k: os.environ.get(k) for k in ENV}
    os.environ.update(ENV)
    ffi.load().dogleg_gpu_release_cache()
    yield
    for k, v in saved.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v
    if RATIO:
        print("\nlargest error / bound of test_gpu_sparse_shapes.py:")
        for k in sorted(RATIO):
            print("  %-52s %.3g" % (k, RATIO[k]))


def set_env(monkeypatch, name, extra=None):
    for k, v in dict(FIXTURES[name][2], **(extra or {})).items():
        monkeypatch.setenv(k, v)


def engine(H, F):
    E = H.Engine(ffi.SOLVE_SPARSE, F.N, F.M, F.nnz)
    E.load_sparse(0, F.p, F.x, F.Jp, F.Ji, F.Jx, perm=F.perm, postorder=0)
    return E


# ---------------------------------------------------------------- the engine's structure
def sym_get(E, what):
    S = E.L.dlb_engine_symbolic(E.h)
    n = E.L.dlb_symbolic_get(S, what, None, 0)
    out = np.zeros(max(n, 1), dtype=np.int32)
    E.L.dlb_symbolic_get(S, what, out.ctypes.data_as(C.POINTER(C.c_int)), n)
    return out[:n]


def gather_get(E, what):
    L = E.L
    G = L.dlb_gather_plan_create(L.dlb_engine_symbolic(E.h), SMALL_FRONT_MAX, -1, 0, 0, 0)
    assert G
    try:
        n = L.dlb_gather_plan_get(G, 0, what, None, 0)
        out = np.zeros(max(n, 1), dtype=np.int64)
        L.dlb_gather_plan_get(G, 0, what, out.ctypes.data_as(C.POINTER(C.c_longlong)), n)
        return out[:n]
    finally:
        L.dlb_gather_plan_free(G)


def plan(E, env, forced=None):
    """What the engine does with this symbolic analysis, restated from dlb_engine.cu (set_pattern,
    run_factor_levels), and the kernel launches of one factorization that follow from it."""
    first, rptr = sym_get(E, SYM_SN_FIRST), sym_get(E, SYM_ROWS_PTR)
    cptr, lptr, lsn = sym_get(E, SYM_CHILD_PTR), sym_get(E, SYM_LEVEL_PTR), sym_get(E, SYM_LEVEL_SN)
    nsuper = len(first) - 1
    r = np.diff(rptr)
    nc = np.diff(first)
    nch = np.diff(cptr)
    nlev = len(lptr) - 1
    level0 = lsn[lptr[0]:lptr[1]]
    eligible = [s for s in level0 if r[s] <= LEAF_ROWS and nc[s] <= LEAF_COLS and nch[s] == 0]
    nleaf = len(eligible) if len(eligible) >= int(env.get("DOGLEG_GPU_LEAF_MIN", 1024)) else 0
    leaves = set(eligible) if nleaf else set()
    gptr = gather_get(E, GP_LEVEL_PTR)
    srcs = np.diff(gather_get(E, GP_SRC_PTR))
    b = dict(nsuper=nsuper, nlev=nlev, rows=r, nc=nc, nchildren=nch, nleaf=nleaf, threads=set(), level_rows=set(),
             solve_threads=set(), schedules=set(), big_nc=set(), big_rows=set(), super=False,
             leaf_nc={int(nc[s]) for s in leaves}, leaf_rows=max([int(r[s]) for s in leaves], default=0),
             leaf=("mma" if max(nc[s] for s in leaves) <= LEAF_MMA_COLS and env.get("DOGLEG_GPU_LEAF_MMA") != "0"
                   else "scalar") if leaves else None,
             heavy={int(nch[s]) for s in range(nsuper) if nch[s] > HEAVY},
             two_pass=any(gptr[2 * l + 1] > gptr[2 * l] for l in range(nlev)),
             longest_list=int(srcs.max()) if len(srcs) else 0, max_rows=int(r.max()),
             rootless_update=any(r[s] == nc[s] > SMALL_FRONT_MAX for s in range(nsuper)))
    launches = 0
    for l in range(nlev):
        sns = [s for s in lsn[lptr[l]:lptr[l + 1]] if s not in leaves]
        big = [s for s in sns if r[s] > SMALL_FRONT_MAX]
        small = [s for s in sns if r[s] <= SMALL_FRONT_MAX]
        if small:
            rows = max(r[s] for s in small)
            b["threads"].add(front_threads(rows))
            b["level_rows"].add(int(rows))
            b["solve_threads"].add(128 if rows <= 64 else 512)
        launches += 2 * (gptr[2 * l + 2] > gptr[2 * l]) + (l == 0 and bool(leaves)) + bool(small)
        if big:
            max_r, max_nc = max(r[s] for s in big), max(nc[s] for s in big)
            b["schedules"].add(bf_schedule(len(big), max_r, forced))
            b["big_nc"] |= {int(nc[s]) for s in big}
            b["big_rows"] |= {int(r[s]) for s in big}
            b["super"] |= max_nc > 2 * BS_SUPER
            launches += 2 + bf_launches(len(big), max_r, max_nc, forced)     # zero-fill + assembly + panels
    b["launches"] = launches
    # dlb_engine.cu: the persistent trial kernel takes trees without leaf kernels whose fronts all fit its shared memory
    b["has_trial"] = nleaf == 0 and 0 < nlev <= 256 and r.max() <= SMALL_FRONT_MAX and trial_smem(int(r.max())) <= TRIAL_SMEM_MAX
    b["trial"] = trial_threads(int(r.max())) if b["has_trial"] else None
    # more fronts in a level than k_trial has CTAs: at most one CTA per SM fits (228 KB of shared memory)
    b["wide"] = b["has_trial"] and max(np.diff(lptr)) > sm_count() and 2 * trial_smem(int(r.max())) > 228 * 1024
    return b


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def launches(E):
    out = np.zeros(4)
    E.L.dlb_engine_counters(E.h, out.ctypes.data_as(C.POINTER(C.c_double)))
    return out[0]


def check_branches(E, F, name, forced=None):
    """the fronts are the fixture's cliques, the fixture reaches its branches, and one factorization makes the
    launches the restated rules predict"""
    env = dict(FIXTURES[name][2], **({"DOGLEG_GPU_BF_SCHEDULE": forced} if forced else {}))
    b = plan(E, env, forced)
    assert b["nsuper"] == len(F.nodes)
    assert sorted(zip(b["nc"].tolist(), b["rows"].tolist())) == sorted((c, c + s) for c, s, _ in F.nodes)
    for k, v in FIXTURES[name][3].items():
        if k == "schedules" and forced:
            v = {forced}
        got = b[k]
        if isinstance(v, set) and k in ("big_nc", "big_rows", "level_rows"):
            assert v <= got, (k, got)
        else:
            assert got == v, (k, got)
    assert E.has_trial() == b["has_trial"]
    return b


# ---------------------------------------------------------------- checks
RATIO = {}


def within(tag, name, err, bound):
    err, bound = np.broadcast_arrays(np.asarray(err, dtype=np.float64), np.asarray(bound, dtype=np.float64))
    bad = ~(err <= bound)
    assert not bad.any(), "%s, %s: %d entries beyond the bound, worst %r > %r" % (
        tag, name, bad.sum(), err[bad].max() if np.isfinite(err[bad]).all() else np.nan, bound[bad][0])
    nz = bound > 0
    if nz.any():
        RATIO[name] = max(RATIO.get(name, 0.0), float((err[nz] / bound[nz]).max()))


def export_factor(E, b):
    """the factor straight from the fronts (dlb_engine_export_factor: r x nc column-major panels, ld r),
    as a dense lower-triangular matrix in the elimination order"""
    L = E.L
    L.dlb_engine_export_factor.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_longlong, C.POINTER(C.c_double)]
    L.dlb_engine_export_factor.restype = C.c_int
    sizes = (b["rows"] * b["nc"]).astype(np.int64)
    px = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    x = np.full(int(px[-1]), np.nan)
    E.check(L.dlb_engine_export_factor(E.h, px.ctypes.data_as(C.POINTER(C.c_int)), int(px[-1]),
                                       x.ctypes.data_as(C.POINTER(C.c_double))))
    return x, px


def factor_matrix(E, b, x, px):
    first, rows, rptr = sym_get(E, SYM_SN_FIRST), sym_get(E, SYM_ROWS), sym_get(E, SYM_ROWS_PTR)
    N = E.N
    Lm = np.zeros((N, N))
    panels = []
    for s in range(b["nsuper"]):
        rs = rows[rptr[s]:rptr[s + 1]]
        nc = first[s + 1] - first[s]
        P = x[px[s]:px[s] + len(rs) * nc].reshape((nc, len(rs))).T
        P = np.where(np.arange(len(rs))[:, None] >= np.arange(nc)[None, :], P, 0.0)   # fronts leave the upper part undefined
        for c in range(nc):
            Lm[rs[c:], first[s] + c] = P[c:, c]
        panels.append((rs, P))
    return Lm, panels


def check_assembly(tag, F, E, lam):
    A, aa, m = F.reference(lam)
    Ag = E.JtJ(0, lam)               # entries shared by several fronts are summed in any order: both triangles checked
    assert np.array_equal(Ag != 0, A != 0)
    within(tag, "J'J + lam I, entry by entry", np.abs(Ag - A.astype(np.float64)), CB * m * U * aa)
    return A, aa, m


def check_factor(tag, F, E, b, A, aa, m, what="factor"):
    x, px = export_factor(E, b)
    Lm, panels = factor_matrix(E, b, x, px)
    assert np.isfinite(Lm).all()
    perm = F.perm
    PA = A[np.ix_(perm, perm)]
    LL = np.zeros(A.shape, dtype=LD)
    for rs, P in panels:                                  # L L' as a sum of panel products, in long double
        Pl = P.astype(LD)
        LL[np.ix_(rs, rs)] += Pl @ Pl.T
    aL = np.abs(Lm)
    cnt = (Lm != 0).sum(axis=1)
    k = np.minimum.outer(cnt, cnt)
    bound = CB * (m[np.ix_(perm, perm)] * U * aa[np.ix_(perm, perm)] + k * U * (aL @ aL.T))
    within(tag, what + ": |LL'-PAP'| <= c(m u|J|'|J| + k u|L||L'|)", np.abs((LL - PA).astype(np.float64)), bound)
    return Lm, x


def check_solve(tag, what, F, A, aa, m, Lm, X, B, steps=1):
    """X from the GPU solves A X = B (original ordering): componentwise backward error, forward error against
    LAPACK's on the same matrix"""
    N = F.N
    B = B.reshape(N, -1)
    X = X.reshape(N, -1)
    assert np.isfinite(X).all()
    perm = F.perm
    iperm = np.argsort(perm)
    kmax = int((Lm != 0).sum(axis=1).max())
    aL = np.abs(Lm)
    R = (B.astype(LD) - A @ X.astype(LD)).astype(np.float64)
    Xp = np.abs(X[perm])
    LLx = (aL @ (aL.T @ Xp))[iperm]                       # |L||L'||x| in the original ordering
    bound = CB * (m.max() * U * (aa @ np.abs(X)) + kmax * U * (LLx + np.abs(B)))
    within(tag, what + " backward error", np.abs(R), bound)
    Ad = A.astype(np.float64)
    cf = scipy.linalg.cho_factor(Ad, lower=True)
    X0 = scipy.linalg.cho_solve(cf, B)
    Xr = X0.copy()
    for _ in range(steps):                                # iterative refinement, residuals in long double
        Xr = Xr + scipy.linalg.cho_solve(cf, (B.astype(LD) - A @ Xr.astype(LD)).astype(np.float64))
    nx = np.abs(Xr).max()
    fe = np.abs(X - Xr).max() / nx
    fe_lapack = np.abs(X0 - Xr).max() / nx
    within(tag, what + " forward error <= 10 lapack + 4ku", fe, 10 * fe_lapack + 4 * kmax * U)


def solve_checks(tag, F, E, b, lam, rng, nrhs_list=(1, 3, 64), check=True, steps=1):
    """factorize, Gauss-Newton step, solves; checked against the bounds unless check=False (then only the
    outputs are returned, for the bit-for-bit comparison of two engines)"""
    if check:
        A, aa, m = check_assembly(tag, F, E, lam)
    n0 = launches(E)
    assert E.factorize(0, lam) == -1
    assert launches(E) - n0 == b["launches"], (launches(E) - n0, b["launches"])
    if check:
        Lm, x = check_factor(tag, F, E, b, A, aa, m)
    else:
        x = export_factor(E, b)[0]
    E.gauss_newton(0)
    d = E.download(0)
    gn, g = d["gn"], d["Jtx"]
    out = {"factor": x, "gn": gn}
    if check:
        check_solve(tag, "Gauss-Newton", F, A, aa, m, Lm, -gn, g, steps)
    for nrhs in nrhs_list:
        B = rng.standard_normal((F.N, nrhs))
        out[nrhs] = X = E.solve(B)
        if check:
            check_solve(tag, "solve(B)", F, A, aa, m, Lm, X, B, steps)
    return out


# ---------------------------------------------------------------- tests
@pytest.mark.parametrize("name", NAMES)
def test_sparse_engine_at_the_branch_shapes(H, name, monkeypatch):
    """assembly, factor, Gauss-Newton step and solves with 1, 3 and 64 right-hand sides at lambda = 0.5 and 0;
    a second engine gives the same bits"""
    set_env(monkeypatch, name)
    F = fixture(name)
    outs = []
    for rep in range(2):
        E = engine(H, F)
        try:
            b = check_branches(E, F, name)
            E.evaluate(0)
            got = {}
            for lam in (0.5, 0.0):
                got[lam] = solve_checks("%s lam=%g" % (name, lam), F, E, b, lam, np.random.default_rng(11),
                                        check=rep == 0)
            outs.append(got)
        finally:
            E.close()
    for lam in (0.5, 0.0):                                 # reproducibility: two engines, the same bits
        for k in outs[0][lam]:
            assert np.array_equal(outs[0][lam][k], outs[1][lam][k]), (name, lam, k)


@pytest.mark.parametrize("sched", ["left", "right", "diag"])
def test_every_panel_schedule_on_unequal_big_fronts(H, sched, monkeypatch):
    """DOGLEG_GPU_BF_SCHEDULE forces each schedule on a level of big fronts with different r and nc"""
    name = "bigs"
    set_env(monkeypatch, name, {"DOGLEG_GPU_BF_SCHEDULE": sched})
    F = fixture(name)
    E = engine(H, F)
    try:
        b = check_branches(E, F, name, forced=sched)
        E.evaluate(0)
        rng = np.random.default_rng(12)
        for lam in (0.5, 0.0):
            solve_checks("%s %s lam=%g" % (name, sched, lam), F, E, b, lam, rng, (3,))
    finally:
        E.close()


def test_graded_columns(H, monkeypatch):
    """columns of J graded over six decades: cond(J'J) ~ 1e12, the bounds are componentwise and hold as they are"""
    name = "ladder"
    set_env(monkeypatch, name)
    F = fixture(name, graded=True)
    E = engine(H, F)
    try:
        b = check_branches(E, F, name)
        E.evaluate(0)
        rng = np.random.default_rng(13)
        for lam in (0.5, 0.0):
            solve_checks("graded lam=%g" % lam, F, E, b, lam, rng, (1, 3), steps=3)
    finally:
        E.close()


TRIAL = [n for n in NAMES if FIXTURES[n][3].get("trial")]


@pytest.mark.parametrize("name", TRIAL)
def test_trial_kernel_steps(H, name, monkeypatch):
    """k_trial (one launch per trial step): its factor is where export_factor finds it and meets the factor bound;
    its Gauss-Newton, Cauchy and interpolated steps meet the solve bounds and the step formulas"""
    set_env(monkeypatch, name)
    F = fixture(name)
    E = engine(H, F)
    try:
        b = check_branches(E, F, name)
        assert E.has_trial()
        N = F.N
        Jl = [(st, V.astype(LD)) for st, V in F.classes]
        for lam in (0.5, 0.0):
            tag = "%s trial lam=%g" % (name, lam)
            sc = E.evaluate(0)
            A, aa, m = check_assembly(tag, F, E, lam)
            E.evaluate(0)
            sc = E.trial(0, 1, 1e300, lam)
            assert sc.minor == -1 and sc.step_type == ffi.STEP_GAUSSNEWTON and sc.trial_flags != 0
            d0, d1 = E.download(0), E.download(1)
            g = d0["Jtx"]
            assert np.array_equal(d1["step"], d0["gn"])
            Lm, _ = check_factor(tag, F, E, b, A, aa, m, "trial factor")
            check_solve(tag, "trial Gauss-Newton", F, A, aa, m, Lm, -d0["gn"], g)
            # the Cauchy point -(|g|^2/|Jg|^2) g from the GPU's g, in long double
            gl = g.astype(LD)
            y2 = LD(0)
            z2 = 0.0
            for st, V in Jl:
                y = V @ gl[st]
                y2 += np.sum(y * y)
                z = np.abs(V.astype(np.float64)) @ np.abs(g[st])
                z2 += float(z @ z)
            kc = -np.sum(gl * gl) / y2
            cau = d0["cauchy"]
            kmax_J = max(len(st) for st, _ in F.classes)
            rel = (N + 4) * U + (2 * kmax_J + F.M + 2) * U * z2 / float(y2)
            within(tag, "trial Cauchy point", np.abs(cau - (kc * gl).astype(np.float64)), CB * rel * np.abs(float(kc) * g))
            ncau = float(np.sqrt(np.sum(cau.astype(LD) ** 2)))
            ngn = float(np.sqrt(np.sum(d0["gn"].astype(LD) ** 2)))
            # Cauchy step: the Cauchy point cut to the trust region
            delta = 0.5 * ncau
            sc = E.trial(0, 1, delta, lam)
            assert sc.step_type == ffi.STEP_CAUCHY
            st_ = E.download(1)["step"]
            ref = (cau.astype(LD) * (LD(delta) / np.sqrt(np.sum(cau.astype(LD) ** 2)))).astype(np.float64)
            within(tag, "trial Cauchy step", np.abs(st_ - ref), CB * (N + 4) * U * np.abs(ref))
            # interpolated step between the Cauchy point and the Gauss-Newton step, |step| = delta
            assert ncau < ngn
            delta = np.sqrt(ncau * ngn)
            sc = E.trial(0, 1, delta, lam)
            assert sc.step_type == ffi.STEP_INTERPOLATED
            st_ = E.download(1)["step"]
            a_, g_ = cau.astype(LD), d0["gn"].astype(LD)
            dd = a_ - g_
            l2, negc = np.sum(dd * dd), np.sum(dd * a_)
            disc = negc * negc - l2 * (np.sum(a_ * a_) - LD(delta) ** 2)
            k = (negc + np.sqrt(disc)) / l2
            absd = np.abs(dd)
            scale = (np.sum(absd * np.abs(a_)) + np.sqrt(negc * negc + l2 * (np.sum(a_ * a_) + LD(delta) ** 2))) / l2
            within(tag, "trial k_interp", abs(sc.k_interp - float(k)), CB * (N + 4) * U * float(scale))
            ref = (a_ + k * (g_ - a_)).astype(np.float64)
            within(tag, "trial interpolated step", np.abs(st_ - ref),
                   CB * (N + 4) * U * (np.abs(cau) + float(scale) * np.abs(d0["gn"] - cau)))
            within(tag, "trial |interpolated step| = delta", abs(float(np.sqrt(np.sum(st_.astype(LD) ** 2))) - delta),
                   CB * (N + 4) * U * delta * float(scale))
    finally:
        E.close()


# (fixture, forced schedule, the front whose state is zeroed, its pivot inside the front, the branch)
SINGULAR = [
    ("leaf34", None, 5, 1, "leaf front"),
    ("ladder", None, 4, 3, "small front"),
    ("bigs", "right", 5, 70, "big front, right-looking"),
    ("bigs", "left", 5, 70, "big front, left-looking"),
    ("bigs", "diag", 5, 70, "big front, throughput"),
    ("left", None, 81, 100, "big front, natural left-looking"),
    ("gather", None, 1, 3, "trial kernel"),
]


@pytest.mark.parametrize("name,forced,node,j,branch", SINGULAR, ids=[s[4] for s in SINGULAR])
def test_exact_singular_columns_are_reported_at_their_pivot(H, name, forced, node, j, branch, monkeypatch):
    """A zero column of J makes that state's pivot an exact 0: the factorization reports minor = its position in
    the elimination order (perm[minor] = the state, CHOLMOD's L->minor); at lambda = 1e-10 it is positive
    definite and meets the factor bound"""
    set_env(monkeypatch, name, {"DOGLEG_GPU_BF_SCHEDULE": forced} if forced else None)
    F = Fixture(name, FIXTURES[name][0], seed=7 + NAMES.index(name), **FIXTURES[name][1])
    state = int(F.node_states[node][j])
    F.zero_state(state)
    E = engine(H, F)
    try:
        b = check_branches(E, F, name, forced)
        pos = int(np.nonzero(F.perm == state)[0][0])
        E.evaluate(0)
        tag = "%s singular" % name
        A, aa, m = check_assembly(tag, F, E, 0.0)
        assert not A[state].any()
        E.evaluate(0)
        if branch == "trial kernel":
            sc = E.trial(0, 1, 1e300, 0.0)
            assert sc.minor == pos
            sc = E.trial(0, 1, 1e300, 1e-10)
            assert sc.minor == -1 and sc.step_type == ffi.STEP_GAUSSNEWTON
        else:
            assert E.factorize(0, 0.0) == pos
            assert E.factorize(0, 1e-10) == -1
        A, aa, m = F.reference(1e-10)
        check_factor(tag, F, E, b, A, aa, m, "singular column, lambda 1e-10")
    finally:
        E.close()
