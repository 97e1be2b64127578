"""The supernodal LDLt kernels at their routing and staging edges, entry by entry against an extended-precision residual.

`fpsb_ldlt.cu` sends every supernode down one route (flat one-wide leaf kernels, a warp of a bundle, a whole CTA) and
stages its fronts in fixed-size passes (Schur update: 64 rows of a descendant, TRSM: 128 rows of L21, backward solve:
1024 gathered rows).  The structures below are built from dense Jacobian blocks with a user ordering so that one
factorisation covers several routes and every pass boundary sits one row short of full, exactly full and one row past.
`SymbolicAnalysis.routes()` (the predicates the launches use) proves that each structure reaches what it is there for.

Bars (oracle/fps_oracle.c, long double, independent of conditioning):
  factor  |(P K P' - L^ D^ L^')_ij| <= (c_ij + 4) 2^-53 (|L^| |D^| |L^'|)_ij  for every (i, j) of the pattern of L,
          c_ij = #{k < j : L(i,k) L(j,k) structurally nonzero}; the diagonals of regularised pivots are skipped
  solve   |b - K~ x^|_i <= (3c + 10) 2^-53 (P' |L^| |D^| |L^'| P |x^|)_i,  c = largest row / column count of L,
          K~ = K with the pivot changes of the regularised pivots
The relaxed amalgamation's explicit zeros are not in the pattern of L, but the solves read whole panels: a slot that is
not exactly 0 breaks the solve bar.

FPSB_LDLT_MODE is read once per process: `python tests/test_gpu_ldlt_edges.py --worker <mode> <out.npz>` runs every
structure in that mode (single instance, both batched entries, the failing factorisations) and the GPU tests compare
the files with the oracle and with each other.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SQRT_EPS = float(np.sqrt(np.finfo(float).eps))
MODES = ["0", "1", "2"]
NINST = 3


# ---------------------------------------------------------------------------------------------------------------------
# structures: dense Jacobian blocks placed block-diagonally, eliminated in a chosen order
# ---------------------------------------------------------------------------------------------------------------------
class _Build:
    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.nv = self.nc = 0
        self.rows, self.cols, self.vals, self.order = [], [], [], []
        self.dup_rows = []          # (row, copy of row): identical values (rank-deficient rows)
        self.zero_rows = []         # rows whose values are all 0.0 in the failing factorisations

    def var(self, k):
        self.nv += k
        return list(range(self.nv - k, self.nv))

    def con(self, k):
        self.nc += k
        return list(range(self.nc - k, self.nc))

    def dense(self, C, V):
        for c in C:
            for v in V:
                self.rows.append(c); self.cols.append(v)

    def elim(self, *groups):
        for kind, idx in groups:
            self.order += [("v" if kind == "v" else "c", i) for i in idx]

    def front(self, W, r, n2=2, n1=2, dup=None, zero=None):
        """The last of the n1 variables V1 and W - 1 constraints C1 form one supernode of width W whose r rows below
        are the constraints C2; C2 and the n2 variables V2 form the next chain, which takes the Schur update of that
        supernode (nrow = r, ncol = min(r, 64), wd = W).  dup = (a, b): C1[b] repeats C1[a]; zero: C1[zero] is 0."""
        V1 = self.var(n1); C1 = self.con(W - 1); C2 = self.con(r); V2 = self.var(n2)
        self.dense(C1 + C2, V1); self.dense(C2, V2)
        self.elim(("v", V1), ("c", C1), ("c", C2), ("v", V2))
        if dup is not None:
            self.dup_rows.append((C1[dup[0]], C1[dup[1]]))
        if zero is not None:
            self.zero_rows.append(C1[zero])

    def star(self, nr):
        """A constraint x between two variables (one-wide leaves of nr = 1) and nr variables that also meet a
        constraint y: x is a supernode of width 1 above the leaves with nr rows below.  A free variable eliminated
        just before x keeps the relaxed amalgamation from merging the last leaf into it."""
        V1 = self.var(2); z = self.var(1); x = self.con(1); V2 = self.var(nr); y = self.con(1)
        self.dense(x, V1 + V2); self.dense(y, V2)
        self.elim(("v", V1), ("v", z), ("c", x), ("v", V2), ("c", y))

    def tiny(self, m=1, n=2, dup=False, zero=False):
        """m constraints x n variables, variables first: n - 1 one-wide leaves, then the last variable and the
        constraints as one supernode of width m + 1 without rows below."""
        V = self.var(n); C = self.con(m)
        self.dense(C, V)
        self.elim(("v", V), ("c", C))
        if dup:
            self.dup_rows.append((C[0], C[m - 1]))
        if zero:
            self.zero_rows.append(C[m - 1])

    def zero_slot(self):
        """v0, c, v1 with c meeting both: the relaxed amalgamation merges the three columns and stores (v1, v0), which
        is not in the pattern of L, as an explicit zero."""
        V = self.var(2); c = self.con(1)
        self.dense(c, V)
        self.elim(("v", V[:1]), ("c", c), ("v", V[1:]))

    def wide_leaf(self, k, zero=False):
        """A constraint eliminated before its k variables, which meet nothing else: a leaf of width k + 1 whose first
        pivot is -delta."""
        c = self.con(1); V = self.var(k)
        self.dense(c, V)
        self.elim(("c", c), ("v", V))
        if zero:
            self.zero_rows.append(c[0])

    def free(self, nvar=0, ncon=0):
        """Variables without Jacobian entries and empty constraint rows: one-wide leaves with nr = 0."""
        self.elim(("v", self.var(nvar)), ("c", self.con(ncon)))

    def duplicate_entries(self, k):
        """Repeat k existing COO entries (the assembly sums every source of a slot)."""
        pick = self.rng.choice(len(self.rows), size=k, replace=False)
        self.rows += [self.rows[i] for i in pick]; self.cols += [self.cols[i] for i in pick]

    def finish(self, delta, zero_values=False):
        rows, cols = np.array(self.rows, np.int64), np.array(self.cols, np.int64)
        vals = self.rng.standard_normal(len(rows))
        for a, b in self.dup_rows:
            ia, ib = np.flatnonzero(rows == a), np.flatnonzero(rows == b)
            va = {c: v for c, v in zip(cols[ia], vals[ia])}
            vals[ib] = [va[c] for c in cols[ib]]
        if zero_values:
            for z in self.zero_rows:
                vals[rows == z] = 0.0
        P = np.array([i if k == "v" else self.nv + i for k, i in self.order], np.int64)
        assert sorted(P.tolist()) == list(range(self.nv + self.nc))
        return dict(nvar=self.nv, ncon=self.nc, rows=rows, cols=cols, vals=vals, P=P, delta=delta)


def _trsm():
    # TRSM passes of 128 rows: nr = 127, 128, 129, 257 below CTA supernodes of width 9, 31, 32, 33
    b = _Build(11)
    for W, r in ((9, 127), (31, 128), (32, 129), (33, 257)):
        b.front(W, r)
    b.duplicate_entries(3)
    return b.finish(0.5)


def _schur():
    # Schur update passes of 64 rows: nrow = 63, 64, 65 from sources of width 63, 64, 40; ncol = 63 and 65 - 64 = 1
    b = _Build(12)
    for W, r in ((63, 63), (64, 64), (40, 65)):
        b.front(W, r)
    b.duplicate_entries(3)
    return b.finish(0.5)


def _solve():
    # backward-solve staging of 1024 rows: nr = 1023, 1024, 1025 below supernodes of width 64; their variables are
    # one-wide leaves with nr > 1000
    b = _Build(13)
    for r in (1023, 1024, 1025):
        b.front(64, r, n2=1)
    return b.finish(0.5)


def _warp():
    # the warp-level predicate on both sides (w = 8: nr = 56 / 57; w = 1 above the leaves: nr = 511 / 512), bundles of
    # 7, 8 and 8 + 1 warp-level supernodes in one level between CTA-level ones, free variables and empty rows
    b = _Build(14)
    b.front(8, 56); b.front(8, 57)
    b.star(511); b.star(512)
    for run in (7, 8, 9):
        for _ in range(run):
            b.tiny()
        b.tiny(10, 2)
    b.free(nvar=2, ncon=2)
    b.zero_slot()
    return b.finish(0.5)


def _reg():
    # delta below the pivot tolerance: a regularised pivot in every route — an empty row (one-wide leaf), a repeated row
    # in a warp-level supernode above the leaves, a repeated row at column 7 of a CTA supernode above the leaves (the
    # later columns of its block and its rows below use it), the first pivot of a wide leaf, scalar routines (w = 12)
    # and warp (w = 4); explicit zero slots and repeated entries
    b = _Build(15)
    b.free(ncon=1)
    b.tiny(3, 4, dup=True)
    b.front(20, 30, n2=5, n1=60, dup=(2, 6))
    b.wide_leaf(11); b.wide_leaf(3)
    b.zero_slot(); b.zero_slot()
    b.duplicate_entries(4)
    return b.finish(1e-10)


STRUCTS = {"trsm": _trsm, "schur": _schur, "solve": _solve, "warp": _warp, "reg": _reg}


# one zero pivot, in one route only, with the regularisation off: the factorisation must fail and hand the right-hand
# sides back (delta = 0, the zero rows' values 0.0)
def _fail_leaf1():
    b = _Build(21); b.tiny(2, 3); b.free(ncon=1)
    return b.finish(0.0, True)


def _fail_warp():
    b = _Build(22); b.tiny(2, 3); b.tiny(3, 4, zero=True)
    return b.finish(0.0, True)


def _fail_block():
    b = _Build(23); b.front(20, 30, n2=5, n1=60, zero=6)
    return b.finish(0.0, True)


def _fail_wide_leaf():
    b = _Build(24); b.tiny(2, 3); b.wide_leaf(11, zero=True)
    return b.finish(0.0, True)


FAILS = {"leaf1": _fail_leaf1, "warp": _fail_warp, "block": _fail_block, "wide_leaf": _fail_wide_leaf}

_CACHE = {}


def _struct(name):
    if name not in _CACHE:
        _CACHE[name] = STRUCTS[name]() if name in STRUCTS else FAILS[name[5:]]()
    return _CACHE[name]


def _rhs(s, seed):
    rng = np.random.default_rng(seed)
    n, m = s["nvar"], s["ncon"]
    return rng.standard_normal(n), rng.standard_normal(m), rng.standard_normal(n)


def _batch_vals(s, seed):
    """NINST perturbed copies of the values, with their own deltas and right-hand sides."""
    rng = np.random.default_rng(seed)
    n, m = s["nvar"], s["ncon"]
    J = s["vals"][None, :] * (1.0 + 0.05 * rng.standard_normal((NINST, len(s["vals"]))))
    delta = s["delta"] * (1.0 + 0.5 * rng.random(NINST))
    return J, delta, rng.standard_normal((NINST, n)), rng.standard_normal((NINST, m)), rng.standard_normal((NINST, n))


def _routes_host(s):
    from fpsb200.symbolic import SymbolicAnalysis
    return SymbolicAnalysis(s["nvar"], s["ncon"], s["rows"], s["cols"], s["P"]).routes()


# ---------------------------------------------------------------------------------------------------------------------
# host: every structure reaches its edges, the symbolic analysis is the oracle's, the bars hold for the oracle's factor
# ---------------------------------------------------------------------------------------------------------------------
EDGES = {
    "trsm": ("cta_w33_63", "trsm_multi", "trsm_tail_m1", "trsm_tail_0", "trsm_tail_1", "upd_multi", "upd_wd4"),
    "schur": ("cta_w64", "cta_w33_63", "upd_multi", "upd_nrow8", "upd_ncol8", "upd_wd4", "upd_tail_m1", "upd_tail_0",
              "upd_tail_1", "multi_src"),
    "solve": ("cta_w64", "solve_multi", "solve_tail_m1", "solve_tail_0", "solve_tail_1", "leaf1"),
    "warp": ("warp_nonleaf", "bundles", "full_bundles", "cta", "zero_slots", "leaf_wide"),
    "reg": ("leaf1", "leaf_wide", "warp", "warp_nonleaf", "cta", "zero_slots", "multi_src", "leaf_contrib"),
}


@pytest.mark.parametrize("name", list(STRUCTS))
def test_structure_reaches_its_edges(name):
    rt = _routes_host(_struct(name))
    missing = [k for k in EDGES[name] if rt[k] == 0]
    assert not missing, (name, missing, rt)
    if name == "solve":
        assert rt["max_nr"] > 1000 and rt["leaf1"] == 3


def _alone(fn, *args):
    b = _Build(0)
    fn(b, *args)
    return _routes_host(b.finish(0.5))


@pytest.mark.parametrize("W,r,counter", [
    (64, 1023, "solve_tail_m1"), (64, 1024, "solve_tail_0"), (64, 1025, "solve_tail_1"),
    (9, 127, "trsm_tail_m1"), (31, 128, "trsm_tail_0"), (32, 129, "trsm_tail_1"), (33, 257, "trsm_tail_1"),
    (63, 63, "upd_tail_m1"), (64, 64, "upd_tail_0"), (40, 65, "upd_tail_1"),
])
def test_pass_boundaries(W, r, counter):
    """Each front of the structures above, alone, ends a staging pass where it is meant to: its first supernode's nr
    (backward solve, TRSM) or the nrow of the Schur update pair it sends (r) is one row short of a full pass, exactly
    full or one row past a full pass."""
    rt = _alone(_Build.front, W, r)
    assert rt[counter] >= 1, rt
    assert rt["solve_multi"] == (1 if r > 1024 else 0) and rt["trsm_multi"] >= (1 if r > 128 else 0), rt


def test_warp_level_predicate_boundary():
    """w <= 8 and w (w + nr) <= 512: w = 8 with nr = 56 is warp-level, nr = 57 CTA-level; a width-1 supernode above
    the leaves with nr = 511 is warp-level, nr = 512 CTA-level.  (The 513-wide chain below the second star leaves a
    width-1 tail without rows, which is warp-level: the warp count of the stars stays at one.)"""
    lo, hi = _alone(_Build.front, 8, 56), _alone(_Build.front, 8, 57)
    assert (lo["warp_nonleaf"], lo["cta"]) == (1, 1) and (hi["warp_nonleaf"], hi["cta"]) == (0, 2), (lo, hi)
    lo, hi = _alone(_Build.star, 511), _alone(_Build.star, 512)
    assert hi["cta"] == lo["cta"] + 1 and lo["warp_nonleaf"] == hi["warp_nonleaf"] == 1, (lo, hi)
    assert lo["max_nr"] == 511 and hi["max_nr"] == 512


def test_every_counter_is_reached():
    """Every route counter is nonzero on some structure."""
    from fpsb200._lib import LDLT_ROUTE_KEYS
    seen = {k: 0 for k in LDLT_ROUTE_KEYS}
    for name in STRUCTS:
        for k, v in _routes_host(_struct(name)).items():
            seen[k] += v
    assert not [k for k, v in seen.items() if v == 0], seen


@pytest.mark.parametrize("name", list(STRUCTS) + ["fail_" + k for k in FAILS])
def test_symbolic_bit_exact_and_oracle_bars(oracle, name):
    """The product's symbolic analysis equals the oracle's for the user ordering; the oracle's own double L, D pass the
    factor and solve bars (the bars are met by a correct factorisation in any summation order), and moving one
    entry of L by twice its bound fails the factor bar."""
    from fpsb200.symbolic import SymbolicAnalysis
    s = _struct(name)
    g = SymbolicAnalysis(s["nvar"], s["ncon"], s["rows"], s["cols"], s["P"]).get()
    lo = oracle.LDLtOracle(s["nvar"], s["ncon"], s["rows"], s["cols"], s["P"])
    r1, r2, r3 = _rhs(s, 1)
    ref = lo.solve_two_mixed(s["vals"], s["delta"], r1, r2)
    assert ref[4]
    for key in ("P", "parent", "Lnz", "Lp", "Li"):      # Li: filled by the numeric pass
        assert np.array_equal(g[key], lo.symbolic()[key]), key
    if name.startswith("fail_"):
        off = oracle.LDLtOracle(s["nvar"], s["ncon"], s["rows"], s["cols"], s["P"], 0.0, 0.0, 0.0)
        assert not off.solve_two_mixed(s["vals"], s["delta"], r1, r2)[4]
        return
    Lx, D = lo.numeric()
    reg = lo.regularised()
    assert bool(reg.any()) == (name == "reg")
    f = lo.check_factor(Lx, D, reg)
    assert f["ratio"] <= 1.0, f["ratio"]
    n = s["nvar"]
    for x, b in _solutions(ref, lo.solve_two_least_squares(r1, r3), r1, r2, r3, n, s["ncon"]):
        assert lo.check_solve(Lx, D, x, b, reg)[0] <= 1.0
    # one entry moved by twice its bound: at the worst off-diagonal position and at the middle of Lx
    col = np.repeat(np.arange(len(D)), np.diff(g["Lp"]))
    for p in {min(f["where"], len(Lx) - 1), len(Lx) // 2}:
        bad = Lx.copy()
        bad[p] += 2.0 * f["bound"][p] / abs(D[col[p]])
        assert lo.check_factor(bad, D, reg)["ratio"] > 1.0, p


def _solutions(mixed, ls, r1, r2, r3, n, m):
    """(x, b) of the four systems: mixed [r1; 0], [0; r2] and least squares [r1; 0], [r3; 0]."""
    z_n, z_m = np.zeros(n), np.zeros(m)
    return [(np.r_[mixed[0], mixed[1]], np.r_[r1, z_m]), (np.r_[mixed[2], mixed[3]], np.r_[z_n, r2]),
            (np.r_[ls[0], ls[1]], np.r_[r1, z_m]), (np.r_[ls[2], ls[3]], np.r_[r3, z_m])]


# ---------------------------------------------------------------------------------------------------------------------
# GPU worker: one process per FPSB_LDLT_MODE
# ---------------------------------------------------------------------------------------------------------------------
def _work(mode, path):
    import fpsb200
    out = {}
    for name in STRUCTS:
        s = _struct(name)
        n, m = s["nvar"], s["ncon"]
        H = fpsb200.B200Handle(n, m, s["rows"], s["cols"])
        H.set_jac_values(s["vals"])
        H.ldlt_analyze(s["P"], 0, None)
        out[f"{name}.routes"] = np.array(list(H.ldlt_routes().values()))
        r1, r2, r3 = _rhs(s, 1)
        mx = H.ldlt_solve_two_mixed(s["delta"], r1, r2)
        Lx, D = H.ldlt_get_factor()
        ls = H.ldlt_solve_two_least_squares(r1, r3)
        out[f"{name}.Lx"], out[f"{name}.D"] = Lx, D
        out[f"{name}.ok"] = np.array([mx[4], ls[4]])
        for i in range(4):
            out[f"{name}.mixed.{i}"], out[f"{name}.ls.{i}"] = mx[i], ls[i]
        J, delta, b1, b2, b3 = _batch_vals(s, 2)
        bm = H.ldlt_batch_solve_two_mixed(delta, J, b1, b2)
        bl = H.ldlt_batch_solve_two_least_squares(b1, b3)
        for i in range(5):
            out[f"{name}.bmixed.{i}"], out[f"{name}.bls.{i}"] = np.asarray(bm[i]), np.asarray(bl[i])
        for k in range(NINST):
            H.set_jac_values(J[k])
            sm = H.ldlt_solve_two_mixed(delta[k], b1[k], b2[k])
            sl = H.ldlt_solve_two_least_squares(b1[k], b3[k])
            for i in range(4):
                out[f"{name}.smixed{k}.{i}"], out[f"{name}.sls{k}.{i}"] = sm[i], sl[i]
            out[f"{name}.sok{k}"] = np.array([sm[4], sl[4]])
    off = fpsb200.LdltOpts()
    off.ldlt_tol, off.ldlt_r1, off.ldlt_r2 = 0.0, 0.0, 0.0
    for name in FAILS:
        s = _struct("fail_" + name)
        n, m = s["nvar"], s["ncon"]
        H = fpsb200.B200Handle(n, m, s["rows"], s["cols"])
        H.set_jac_values(s["vals"])
        H.ldlt_analyze(s["P"], 0, off)
        out[f"fail_{name}.routes"] = np.array(list(H.ldlt_routes().values()))
        r1, r2, r3 = _rhs(s, 1)
        mx = H.ldlt_solve_two_mixed(0.0, r1, r2)
        ls = H.ldlt_solve_two_least_squares(r1, r3)
        bm = H.ldlt_batch_solve_two_mixed(0.0, s["vals"][None, :], r1[None, :], r2[None, :])
        for i in range(4):
            out[f"fail_{name}.mixed.{i}"], out[f"fail_{name}.ls.{i}"] = mx[i], ls[i]
            out[f"fail_{name}.bmixed.{i}"] = np.asarray(bm[i])[0]
        out[f"fail_{name}.ok"] = np.array([mx[4], ls[4], bool(np.asarray(bm[4])[0])])
    np.savez(path, **out)


WORKER_TIMEOUT = 300


@pytest.fixture(scope="session")
def ldlt_runs(tmp_path_factory):
    cache = {}
    base = tmp_path_factory.mktemp("ldlt_edges")

    def get(mode):
        if mode not in cache:
            path = str(base / f"mode{mode}.npz")
            child = {k: v for k, v in os.environ.items() if not k.startswith("FPSB_")}
            child["FPSB_LDLT_MODE"] = mode
            child["PYTHONPATH"] = os.pathsep.join([ROOT] + [p for p in sys.path if p])
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", mode, path], env=child, cwd=ROOT,
                               capture_output=True, text=True, timeout=WORKER_TIMEOUT)
            if r.returncode != 0:
                raise AssertionError(f"worker mode {mode} exited with {r.returncode}:\n{r.stderr[-4000:]}")
            with np.load(path) as z:
                cache[mode] = {k: z[k] for k in z.files}
        return cache[mode]

    return get


_ORACLE = {}


def _oracle_run(oracle, name):
    if name not in _ORACLE:
        s = _struct(name)
        lo = oracle.LDLtOracle(s["nvar"], s["ncon"], s["rows"], s["cols"], s["P"])
        r1, r2, r3 = _rhs(s, 1)
        mixed = lo.solve_two_mixed(s["vals"], s["delta"], r1, r2)
        _, D = lo.numeric()
        _ORACLE[name] = dict(lo=lo, r=(r1, r2, r3), mixed=mixed, ls=lo.solve_two_least_squares(r1, r3), D=D,
                             reg=lo.regularised())
    return _ORACLE[name]


RESULTS = {}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(STRUCTS))
def test_factor_and_solve_bars(ldlt_runs, oracle, name, mode):
    """The GPU factor and the four solutions (mixed and least squares) meet the bars; the plan's routes on the handle
    equal the host query; the regularised pivots and the signs of D are the double oracle's."""
    r = ldlt_runs(mode)
    s = _struct(name)
    assert list(r[f"{name}.routes"]) == list(_routes_host(s).values())
    o = _oracle_run(oracle, name)
    lo = o["lo"]
    assert r[f"{name}.ok"].all() and o["mixed"][4]
    Lx, D = r[f"{name}.Lx"], r[f"{name}.D"]
    f = lo.check_factor(Lx, D, o["reg"])
    gpu_reg = np.abs(f["dpre"]) < SQRT_EPS
    assert np.array_equal(gpu_reg, o["reg"]), np.flatnonzero(gpu_reg != o["reg"])
    assert np.array_equal(np.sign(D), np.sign(o["D"]))
    mixed = [r[f"{name}.mixed.{i}"] for i in range(4)]
    ls = [r[f"{name}.ls.{i}"] for i in range(4)]
    sol = [lo.check_solve(Lx, D, x, b, o["reg"])[0]
           for x, b in _solutions(mixed, ls, *o["r"], s["nvar"], s["ncon"])]
    RESULTS[(name, mode)] = (f["ratio"], max(sol))
    assert f["ratio"] <= 1.0, (f["ratio"], f["where"])
    assert max(sol) <= 1.0, sol


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(STRUCTS))
def test_batch_bitwise_single(ldlt_runs, name, mode):
    """Both batched entries give, for each of the perturbed instances, bitwise what the single path gives."""
    r = ldlt_runs(mode)
    for k in range(NINST):
        assert bool(r[f"{name}.bmixed.4"][k]) == bool(r[f"{name}.sok{k}"][0])
        assert bool(r[f"{name}.bls.4"][k]) == bool(r[f"{name}.sok{k}"][1])
        for i in range(4):
            assert np.array_equal(r[f"{name}.bmixed.{i}"][k], r[f"{name}.smixed{k}.{i}"]), (k, i)
            assert np.array_equal(r[f"{name}.bls.{i}"][k], r[f"{name}.sls{k}.{i}"]), (k, i)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(STRUCTS))
def test_modes_zero_and_one_bitwise(ldlt_runs, name):
    """The scalar routines (mode 0) and the staged fronts (mode 1) factorise in the same operation order: the same
    factor, bit for bit.  Their solves sum in the same order as long as every backward solve fits one staging pass
    (the staged routine subtracts one partial sum per 1024-row pass) and no supernode pulls from more than eight
    descendants (one partial sum per warp): then the solutions agree bit for bit as well."""
    a, b = ldlt_runs("0"), ldlt_runs("1")
    for key in ("Lx", "D"):
        assert np.array_equal(a[f"{name}.{key}"], b[f"{name}.{key}"]), key
    if _routes_host(_struct(name))["solve_multi"]:
        return
    for key in [f"{k}.{i}" for k in ("mixed", "ls") for i in range(4)]:
        assert np.array_equal(a[f"{name}.{key}"], b[f"{name}.{key}"]), key


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(FAILS))
def test_zero_pivot_passthrough(ldlt_runs, oracle, name, mode):
    """With the regularisation off a zero pivot in any one route fails the factorisation (single and batched), as in
    the oracle, and the outputs hold the right-hand sides."""
    r = ldlt_runs(mode)
    s = _struct("fail_" + name)
    assert list(r[f"fail_{name}.routes"]) == list(_routes_host(s).values())
    assert not r[f"fail_{name}.ok"].any()
    lo = oracle.LDLtOracle(s["nvar"], s["ncon"], s["rows"], s["cols"], s["P"], 0.0, 0.0, 0.0)
    r1, r2, r3 = _rhs(s, 1)
    assert not lo.solve_two_mixed(s["vals"], 0.0, r1, r2)[4]
    z_n, z_m = np.zeros(s["nvar"]), np.zeros(s["ncon"])
    for kind, want in (("mixed", (r1, z_m, z_n, r2)), ("bmixed", (r1, z_m, z_n, r2)), ("ls", (r1, z_m, r3, z_m))):
        for i in range(4):
            assert np.array_equal(r[f"fail_{name}.{kind}.{i}"], want[i]), (kind, i)


def test_route_of_failing_structures():
    """Each failing structure holds its zero pivot in the route it names."""
    rt = {k: _routes_host(_struct("fail_" + k)) for k in FAILS}
    assert rt["warp"]["warp_nonleaf"] >= 2 and rt["warp"]["cta"] == 0
    assert rt["block"]["cta"] >= 1
    assert rt["wide_leaf"]["leaf_wide"] == 1 and rt["wide_leaf"]["cta"] == 0
    assert rt["leaf1"]["leaf1"] >= 3 and rt["leaf1"]["cta"] == 0


@pytest.mark.gpu
def test_print_ratio_table():
    """The worst factor / solve ratios of every structure in every mode (printed for the record)."""
    if not RESULTS:
        pytest.skip("no bar results in this session")
    lines = ["structure " + " ".join(f"mode{m}(factor/solve)" for m in MODES)]
    for name in STRUCTS:
        lines.append(name + " " + " ".join("%.3f/%.3f" % RESULTS[(name, m)] if (name, m) in RESULTS else "-"
                                           for m in MODES))
    print("\n" + "\n".join(lines))


if __name__ == "__main__":
    if len(sys.argv) == 4 and sys.argv[1] == "--worker":
        if ROOT not in sys.path:
            sys.path.insert(0, ROOT)
        _work(sys.argv[2], sys.argv[3])
    else:
        sys.exit("usage: python tests/test_gpu_ldlt_edges.py --worker <mode> <out.npz>")
