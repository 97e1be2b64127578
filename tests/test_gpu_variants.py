"""GPU: the kernel variants the rest of the suite never runs.

The run-time switches of the Krylov loop (`FPSB_LOOP*`, `FPSB_INFLIGHT`, `FPSB_NO_CUTS`) and of the LDLt factorisation
(`FPSB_LDLT_MODE`) are read once per process, so every configuration here runs in a worker process of its own:
`python tests/test_gpu_variants.py --worker <case set> <env name> <out.npz>` builds its operators from fixed seeds, runs
the solves and writes every output vector, stats record, `loop_info()` and launch count to `out.npz`.  The tests compare
those files with each other and with the CPU oracle.

A. Scheduling invariance.  The persistent loop kernel reduces in an order fixed by its grid and the tile map alone
   (DESIGN.md, "Determinism"), so ring stages, in-flight tiles, speculative tiles, early row sums and the iterations per
   launch must not change a single bit.  Every forced configuration is compared bitwise with the default run of the same
   operator, and `loop_info()` shows which geometry each operator reached.
B. Chunk boundaries and slot retirement at fixed iteration counts, against the oracle, on the default loop, on one
   launch per half iteration (`FPSB_LOOP=0`) and on one iteration per launch (`FPSB_LOOP_CHUNK=1`).
C. LDLt modes 0 (scalar routines), 1 (staged fronts, the default) and 2 (DMMA Schur update) through the single-instance
   path and both batched entries.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SQRT_EPS = float(np.sqrt(np.finfo(float).eps))
STAT_KEYS = ("niter", "solved", "inconsistent", "status", "rnorm", "arnorm", "anorm", "acond", "xnorm")
LOOP_KEYS = ("persistent", "early", "nstage", "grid", "stage_bytes", "inflight", "nspec", "chunk")

# ---------------------------------------------------------------------------------------------------------------------
# configurations: one worker process each
# ---------------------------------------------------------------------------------------------------------------------
ENVS = {
    "default": {},
    "loop1": {"FPSB_LOOP": "1"},
    "nstage2": {"FPSB_LOOP_NSTAGE": "2"},
    "nstage4": {"FPSB_LOOP_NSTAGE": "4"},
    "nstage6": {"FPSB_LOOP_NSTAGE": "6"},
    "inflight1": {"FPSB_INFLIGHT": "1"},
    "inflight3": {"FPSB_INFLIGHT": "3"},
    "nspec0": {"FPSB_LOOP_NSPEC": "0"},
    "nspec1": {"FPSB_LOOP_NSPEC": "1"},
    "chunk1": {"FPSB_LOOP_CHUNK": "1"},
    "chunk5": {"FPSB_LOOP_CHUNK": "5"},
    "chunk7": {"FPSB_LOOP_CHUNK": "7"},
    "nocuts": {"FPSB_NO_CUTS": "1"},
    "step": {"FPSB_LOOP": "0"},
    "mode0": {"FPSB_LDLT_MODE": "0"},
    "mode1": {"FPSB_LDLT_MODE": "1"},
    "mode2": {"FPSB_LDLT_MODE": "2"},
}
KNOB_ENVS = [e for e in ENVS if e not in ("default", "nocuts", "step") and not e.startswith("mode")]

# Part A operators: (m, n, nnz per row, window) of models.window_random_jacobian, or the Poisson-control stencil.  The
# geometry each one is there to reach is asserted in test_loop_geometry_reached; the comments give what loop_info()
# reported on a B200 (148 SMs) as stages / grid / bytes per ring stage.  (With 9 entries per row instead of 5 the
# operator of test_fixed_iteration_parity needs 32 768-byte stages and gets 4.)
OPS = {
    "small8": (700, 1500, 5, 24),        # 8 / 3 / 22 528: grid below the SM count
    "stage6": (2000, 4000, 6, 100),      # 6 / 8 / 26 880
    "stage2": (2000, 8000, 40, 700),     # 2 / 35 / 55 424: wide windows and long rows, a stage above a quarter of the ring
    "grid": (40000, 80000, 9, 24),       # 4 / 148 / 32 256: >= 148 tiles in A and A', grid = SMs, no row cuts
    "cuts": (80000, 160000, 6, 24),      # 6 / 148 / 24 576: >= 4 x 148 tiles in A', re-cut into a multiple of the grid
    "poisson": 256,                      # 6 / 148 / 32 000: multi-segment windows
}
# the stencil needs thousands of iterations at the reference tolerances: capped (the comparison is bitwise either way;
# 60 iterations cross two launch boundaries)
POISSON_CAP = 60

# Part B: the operator of test_gpu_krylov.py::test_fixed_iteration_parity, iteration counts around the first three
# launch boundaries (24 iterations per launch; the first half iteration runs in a step kernel before the loop)
FIXED_OP = (700, 1500, 9, 24)
FIXED_KS = (23, 24, 25, 26, 47, 48, 49, 50, 73)
FIXED_DELTAS = (0.0, 0.3)
ASYM = ((5, 49), (49, 5), (5, 5), (49, 49))
CUTS_K = 30


def _fixed_kw(k_ls, k_ln=None, k_ne=None):
    k_ln = k_ls if k_ln is None else k_ln
    k_ne = k_ls if k_ne is None else k_ne
    return dict(ls_atol=0.0, ls_rtol=0.0, ls_itmax=k_ls, ln_atol=0.0, ln_rtol=0.0, ln_btol=0.0, ln_itmax=k_ln,
                ne_atol=0.0, ne_rtol=0.0, ne_etol=0.0, ne_itmax=k_ne)


# Part C: the shapes of test_gpu_ldlt.py (m, n, nnz per row, window, delta, ordering)
LDLT_CASES = [(1, 10, 9, 4, 0.0, None), (30, 60, 5, 8, 0.25, None), (30, 60, 5, 8, 0.0, "id"),
              (30, 60, 5, 8, 1e-2, "rand"), (500, 1000, 10, 32, 1e-2, None),
              (500, 1000, 10, 32, 0.0, "rand"), (5000, 10000, 10, 64, SQRT_EPS, None),
              (20000, 40000, 20, 64, 1e-8, None)]
BATCH_BIG = (2000, 4000, 5, 32)
BATCH_BIG_NINST = 6


# ---------------------------------------------------------------------------------------------------------------------
# operators and inputs (shared by the worker and the parent)
# ---------------------------------------------------------------------------------------------------------------------
def _op_matrix(name):
    from fpsb200 import models
    spec = OPS[name]
    if name == "poisson":
        return sp.csr_matrix(models.poisson_control(spec).A)
    m, n, k, w = spec
    return models.window_random_jacobian(m, n, k, w=w, seed=5)


def _fixed_matrix():
    from fpsb200 import models
    m, n, k, w = FIXED_OP
    return models.window_random_jacobian(m, n, k, w=w, seed=21)


def _rhs(n, m, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(n), rng.standard_normal(m), rng.standard_normal(n)


def _ldlt_matrix(case):
    from fpsb200 import models
    m, n, k, w, _, _ = case
    return models.window_random_jacobian(m, n, k, w=w, seed=17)


def _ldlt_ordering(case):
    m, n, _, _, _, pk = case
    if pk is None:
        return None
    return np.arange(n + m) if pk == "id" else np.random.default_rng(5).permutation(n + m)


def _rank_deficient_matrix():
    from fpsb200 import models
    return models.sparse_qp(2000, 1000, nnz_per_row=8, w=16, seed=3, rank_deficient_frac=0.02).A


def _mix_problem():
    """The healthy / regularised / failing instances of test_gpu_ldlt_batch.py."""
    from fpsb200 import models
    A = models.window_random_jacobian(60, 120, 6, w=10, seed=4).tolil()
    A[7] = A[8]
    A = A.tocsr()
    coo = sp.coo_matrix(A)
    rng = np.random.default_rng(8)
    ninst = 6
    J = coo.data[None, :] * (1.0 + 0.1 * rng.standard_normal((ninst, coo.nnz)))
    J[2, coo.row == 7] = J[2, coo.row == 8]
    J[4] = 0.0
    delta = np.array([0.0, 1e-2, 0.0, 0.25, 0.0, SQRT_EPS])
    r1, r2, r3 = rng.standard_normal((ninst, 120)), rng.standard_normal((ninst, 60)), rng.standard_normal((ninst, 120))
    return A, J, delta, r1, r2, r3


def _big_batch_problem():
    from fpsb200 import models
    m, n, k, w = BATCH_BIG
    A = models.window_random_jacobian(m, n, k, w=w, seed=31)
    coo = sp.coo_matrix(A)
    rng = np.random.default_rng(m + n)
    ninst = BATCH_BIG_NINST
    J = coo.data[None, :] * (1.0 + 0.1 * rng.standard_normal((ninst, coo.nnz)))
    delta = np.array([(0.0, SQRT_EPS, 0.25, 1e-2)[i % 4] for i in range(ninst)])
    return A, J, delta, rng.standard_normal((ninst, n)), rng.standard_normal((ninst, m)), rng.standard_normal((ninst, n))


# ---------------------------------------------------------------------------------------------------------------------
# worker
# ---------------------------------------------------------------------------------------------------------------------
def _handle(A, **opts):
    import ctypes
    import fpsb200
    coo = sp.coo_matrix(A)
    H = fpsb200.B200Handle(A.shape[1], A.shape[0], coo.row, coo.col)
    H.set_jac_values(coo.data)
    if opts:
        o = fpsb200.IterOpts()
        fpsb200._lib.lib().fpsb_iter_default_opts(ctypes.c_int64(A.shape[1]), ctypes.c_int64(A.shape[0]), ctypes.byref(o))
        for k, v in opts.items():
            setattr(o, k, v)
        H.iter_setup(o)
    return H


class _Out(dict):
    def vecs(self, key, arrays):
        for i, a in enumerate(arrays):
            self[f"{key}.{i}"] = np.asarray(a)

    def stats(self, key, st):
        self[f"{key}.stats"] = np.array([[float(s[k]) for k in STAT_KEYS] for s in st])

    def solve(self, H, key, fn, *args):
        l0 = H.launch_count()
        got = fn(*args)
        self[f"{key}.launches"] = np.array(H.launch_count() - l0)
        self[f"{key}.loop"] = np.array([H.loop_info()[k] for k in LOOP_KEYS])
        self.vecs(key, got[:-1])
        self.stats(key, got[-1])


def _work_sched(out, env):
    names = list(OPS)
    if env == "nocuts":
        names = ["cuts"]
    for name in names:
        A = _op_matrix(name)
        m, n = A.shape
        opts = dict(ls_itmax=POISSON_CAP, ln_itmax=POISSON_CAP, ne_itmax=POISSON_CAP) if name == "poisson" else {}
        H = _handle(A, **opts)
        ts = H.tile_stats()
        out[f"{name}.tiles"] = np.array([ts[o][k] for o in ("A", "At") for k in ("tiles", "windowed", "multi_segment")])
        r1, r2, r3 = _rhs(n, m, 1234)
        if env != "nocuts":
            out.solve(H, f"{name}.mixed0", H.iter_solve_two_mixed, 0.0, r1, r2)
            out.solve(H, f"{name}.mixed2", H.iter_solve_two_mixed, 1e-2, r1, r2)
            out.solve(H, f"{name}.ls", H.iter_solve_two_least_squares, 1e-2, r1, r3)
            out.solve(H, f"{name}.extras", H.iter_solve_two_extras, 1e-2, r1, r2)
            out.solve(H, f"{name}.again", H.iter_solve_two_mixed, 1e-2, r1, r2)
        if name == "cuts":
            # fixed iteration count on the operator whose tiles FPSB_NO_CUTS changes (compared with the oracle)
            H = _handle(A, **_fixed_kw(CUTS_K))
            out.solve(H, f"{name}.fixed", H.iter_solve_two_mixed, 1e-2, r1, r2)


def _work_fixed(out, env):
    A = _fixed_matrix()
    m, n = A.shape
    r1, r2, r3 = _rhs(n, m, 8)
    for k in FIXED_KS:
        H = _handle(A, **_fixed_kw(k))
        for d in FIXED_DELTAS:
            out.solve(H, f"k{k}.d{d}.mixed", H.iter_solve_two_mixed, d, r1, r2)
            out.solve(H, f"k{k}.d{d}.ls", H.iter_solve_two_least_squares, d, r1, r3)
            out.solve(H, f"k{k}.d{d}.extras", H.iter_solve_two_extras, d, r1, r2)
    for kl, kc in ASYM:
        H = _handle(A, **_fixed_kw(kl, kc))
        out.solve(H, f"asym{kl}_{kc}", H.iter_solve_two_mixed, 1e-2, r1, r2)
    H = _handle(A, **_fixed_kw(49))
    out.solve(H, "zero.mixed", H.iter_solve_two_mixed, 1e-2, r1, np.zeros(m))
    out.solve(H, "zero.ls", H.iter_solve_two_least_squares, 1e-2, r1, np.zeros(n))


def _work_ldlt(out, env):
    import fpsb200
    for ci, case in enumerate(LDLT_CASES):
        A = _ldlt_matrix(case)
        m, n = A.shape
        delta = case[4]
        coo = sp.coo_matrix(A)
        H = fpsb200.B200Handle(n, m, coo.row, coo.col)
        H.set_jac_values(coo.data)
        H.ldlt_analyze(_ldlt_ordering(case), 0, None)
        r1, r2, r3 = _rhs(n, m, 5 + ci)
        p = H.ldlt_solve_two_mixed(delta, r1, r2)
        out.vecs(f"c{ci}.mixed", p[:4]); out[f"c{ci}.mixed.ok"] = np.array(p[4])
        Lx, D = H.ldlt_get_factor()
        out[f"c{ci}.Lx"], out[f"c{ci}.D"] = Lx, D
        for key, v in H.ldlt_symbolic().items():
            out[f"c{ci}.sym.{key}"] = v
        info = H.ldlt_plan_info()
        out[f"c{ci}.plan"] = np.array([info["nsuper"], info["nleaf"], info["nlevels"]])
        p = H.ldlt_solve_two_least_squares(r1, r3)
        out.vecs(f"c{ci}.ls", p[:4]); out[f"c{ci}.ls.ok"] = np.array(p[4])
    # rank deficient, delta = 0: regularised pivots
    A = _rank_deficient_matrix()
    m, n = A.shape
    coo = sp.coo_matrix(A)
    H = fpsb200.B200Handle(n, m, coo.row, coo.col)
    H.set_jac_values(coo.data)
    H.ldlt_analyze(None, 0, None)
    rng = np.random.default_rng(1)
    r1 = rng.standard_normal(n); r2 = A @ rng.standard_normal(n)
    p = H.ldlt_solve_two_mixed(0.0, r1, r2)
    out.vecs("rd.mixed", p[:4]); out["rd.ok"] = np.array(p[4])
    out["rd.D"] = H.ldlt_get_factor()[1]
    out["rd.P"] = H.ldlt_symbolic()["P"]
    # batched against single, healthy / regularised / failing instances and one shape with non-leaf supernodes
    A, J, delta, r1, r2, r3 = _mix_problem()
    o = fpsb200.LdltOpts()
    o.ldlt_tol, o.ldlt_r1, o.ldlt_r2 = 0.0, 0.0, 0.0
    for tag, opts, keep in (("mixreg", None, list(range(6))), ("mixoff", o, [0, 1, 3, 4, 5])):
        _batch_and_single(out, tag, A, J[keep], delta[keep], r1[keep], r2[keep], r3[keep], opts)
    A, J, delta, r1, r2, r3 = _big_batch_problem()
    _batch_and_single(out, "big", A, J, delta, r1, r2, r3, None)


def _batch_and_single(out, tag, A, J, delta, r1, r2, r3, opts):
    import fpsb200
    m, n = A.shape
    coo = sp.coo_matrix(A)
    H = fpsb200.B200Handle(n, m, coo.row, coo.col)
    H.ldlt_analyze(None, 0, opts)
    info = H.ldlt_plan_info()
    out[f"{tag}.plan"] = np.array([info["nsuper"], info["nleaf"], info["nlevels"]])
    bm = H.ldlt_batch_solve_two_mixed(delta, J, r1, r2)
    bl = H.ldlt_batch_solve_two_least_squares(r1, r3)
    out.vecs(f"{tag}.bmixed", bm); out.vecs(f"{tag}.bls", bl)
    for i in range(J.shape[0]):
        H.set_jac_values(J[i])
        sm = H.ldlt_solve_two_mixed(delta[i], r1[i], r2[i])
        sl = H.ldlt_solve_two_least_squares(r1[i], r3[i])
        out.vecs(f"{tag}.smixed{i}", list(sm[:4]) + [np.array(sm[4])])
        out.vecs(f"{tag}.sls{i}", list(sl[:4]) + [np.array(sl[4])])


WORK = {"sched": _work_sched, "fixed": _work_fixed, "ldlt": _work_ldlt}


def _worker(argv):
    case_set, env, path = argv
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    out = _Out()
    WORK[case_set](out, env)
    np.savez(path, **out)


# ---------------------------------------------------------------------------------------------------------------------
# parent: one worker process per (case set, environment), run in sequence and cached for the session
# ---------------------------------------------------------------------------------------------------------------------
WORKER_TIMEOUT = 300


@pytest.fixture(scope="session")
def runs(tmp_path_factory):
    cache = {}
    base = tmp_path_factory.mktemp("variants")

    def get(case_set, env):
        key = (case_set, env)
        if key not in cache:
            path = str(base / f"{case_set}-{env}.npz")
            child = {k: v for k, v in os.environ.items() if not (k.startswith("FPSB_") or k == "FPSB200_LIB")}
            child.update(ENVS[env])
            if "FPSB200_LIB" in os.environ:
                child["FPSB200_LIB"] = os.environ["FPSB200_LIB"]
            child["PYTHONPATH"] = os.pathsep.join([ROOT] + [p for p in sys.path if p])
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", case_set, env, path], env=child,
                               cwd=ROOT, capture_output=True, text=True, timeout=WORKER_TIMEOUT)
            if r.returncode != 0:
                raise AssertionError(f"worker {case_set} / {env} exited with {r.returncode}:\n{r.stderr[-4000:]}")
            with np.load(path) as z:
                cache[key] = {k: z[k] for k in z.files}
        return cache[key]

    return get


@pytest.fixture(scope="session")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _loop(run, key):
    return dict(zip(LOOP_KEYS, (int(v) for v in run[f"{key}.loop"])))


def _solve_keys(name):
    return [f"{name}.{s}" for s in ("mixed0", "mixed2", "ls", "extras", "again")]


def _as_again(run):
    """The first run of the repeated solve under the name of the second."""
    return {k.replace(".mixed2.", ".again."): v for k, v in run.items() if ".mixed2." in k}


def _nvec(key):
    return 2 if key.endswith("extras") else 4


def _bitwise(a, b, key):
    for i in range(_nvec(key)):
        if not np.array_equal(a[f"{key}.{i}"], b[f"{key}.{i}"]):
            return f"{key}.{i}: rel {_rel(a[f'{key}.{i}'], b[f'{key}.{i}']):.3e}"
    if not np.array_equal(a[f"{key}.stats"], b[f"{key}.stats"], equal_nan=True):
        return f"{key}.stats: {a[f'{key}.stats']} vs {b[f'{key}.stats']}"
    return None


# ---------------------------------------------------------------------------------------------------------------------
# A. scheduling invariance
# ---------------------------------------------------------------------------------------------------------------------
def test_loop_geometry_reached(runs, num_sms):
    """The default run reaches every geometry the operators are there for: ring stages 2, 4, 6 and 8 (all four
    naturally, under the 40 KB / 44 KB tile caps), a grid below and equal to the SM count, row cuts on and off,
    multi-segment windows."""
    d = runs("sched", "default")
    info = {name: _loop(d, f"{name}.mixed2") for name in OPS}
    for name, li in info.items():
        assert li["persistent"] == 1 and li["early"] == 1 and li["chunk"] == 24, (name, li)
        assert li["nspec"] == min(3, li["nstage"] - 1), (name, li)
        for key in _solve_keys(name)[:-1]:
            assert _loop(d, key)["persistent"] == 1, key      # extras: its LSQR half runs the loop, MINRES the step kernel
    assert info["small8"]["nstage"] == 8 and info["small8"]["grid"] < num_sms, info["small8"]
    assert info["stage6"]["nstage"] == 6, info["stage6"]
    assert info["stage2"]["nstage"] == 2, info["stage2"]
    assert info["grid"]["nstage"] == 4 and info["grid"]["grid"] == num_sms, info["grid"]
    assert info["cuts"]["grid"] == num_sms, info["cuts"]
    # row cuts: A' has >= 4 tiles per SM and was re-cut into a multiple of the grid; A (fewer tiles) was not
    t = d["cuts.tiles"]
    assert t[3] >= 4 * num_sms and t[3] % num_sms == 0, t
    g = d["grid.tiles"]
    assert g[0] >= num_sms and g[3] >= num_sms and g[3] < 4 * num_sms, g
    # multi-segment windows (as test_gpu_multiseg.py checks them)
    p = d["poisson.tiles"]
    assert p[2] > 0, p
    print("\nloop geometry (default run):", {k: (v["nstage"], v["grid"], v["stage_bytes"]) for k, v in info.items()})


@pytest.mark.parametrize("env", KNOB_ENVS)
def test_scheduling_knob_is_bitwise_invariant(runs, env):
    """Every forced configuration gives bitwise the default run's p1, q1, p2, q2 (u1, u2) and stats, and reports the
    geometry it forced."""
    d, r = runs("sched", "default"), runs("sched", env)
    knob = ENVS[env]
    for name in OPS:
        nat = _loop(d, f"{name}.mixed2")
        li = _loop(r, f"{name}.mixed2")
        assert li["persistent"] == 1, (name, li)
        assert li["grid"] == nat["grid"] and li["stage_bytes"] == nat["stage_bytes"], (name, li, nat)
        want_nstage = min(nat["nstage"], int(knob.get("FPSB_LOOP_NSTAGE", 8)))
        assert li["nstage"] == want_nstage, (name, li)
        assert li["early"] == (0 if "FPSB_LOOP" in knob else 1), (name, li)
        assert li["chunk"] == int(knob.get("FPSB_LOOP_CHUNK", 24)), (name, li)
        assert li["nspec"] == min(int(knob.get("FPSB_LOOP_NSPEC", 3)), li["nstage"] - 1), (name, li)
        assert li["inflight"] <= max(1, int(knob.get("FPSB_INFLIGHT", 2))), (name, li)
        for key in _solve_keys(name):
            diff = _bitwise(r, d, key)
            assert diff is None, f"{env} changed {diff}"
        # the same solve twice in one process
        assert _bitwise(r, _as_again(r), f"{name}.again") is None


def test_default_runs_repeat_bitwise(runs):
    d = runs("sched", "default")
    for name in OPS:
        assert _bitwise(d, _as_again(d), f"{name}.again") is None, name


def test_no_row_cuts_against_oracle(runs, oracle, num_sms):
    """FPSB_NO_CUTS changes the tiles and with them the reduction order: both tilings are held to the oracle at a fixed
    iteration count that crosses a launch boundary."""
    d, r = runs("sched", "default"), runs("sched", "nocuts")
    assert not np.array_equal(d["cuts.tiles"], r["cuts.tiles"])
    assert r["cuts.tiles"][3] % num_sms != 0 or r["cuts.tiles"][3] < d["cuts.tiles"][3]
    A = _op_matrix("cuts")
    m, n = A.shape
    r1, r2, _ = _rhs(n, m, 1234)
    ref = oracle.IterativeOracle(A, **_fixed_kw(CUTS_K)).solve_two_mixed(1e-2, r1, r2)
    for run in (d, r):
        assert _loop(run, "cuts.fixed")["persistent"] == 1
        for s in range(2):
            assert run["cuts.fixed.stats"][s][0] == ref[4][s]["niter"] == CUTS_K
        e = [_rel(run[f"cuts.fixed.{i}"], ref[i]) for i in range(4)]
        print(f"\ncuts operator, {CUTS_K} iterations: relative difference to the oracle", [f"{x:.1e}" for x in e])
        assert max(e) < BAR_B
    for i in range(4):
        assert _rel(d[f"cuts.fixed.{i}"], r[f"cuts.fixed.{i}"]) < BAR_B


# ---------------------------------------------------------------------------------------------------------------------
# B. chunk boundaries and slot retirement at fixed iteration counts
# ---------------------------------------------------------------------------------------------------------------------
BAR_B = 1e-10          # 30 iterations on the "cuts" operator, with and without row cuts: measured 4.8e-12 at most
_ORACLE_CACHE = {}


def _fixed_oracle(oracle, kind, k, d, k_ln=None):
    key = (kind, k, d, k_ln)
    if key not in _ORACLE_CACHE:
        A = _fixed_matrix()
        m, n = A.shape
        r1, r2, r3 = _rhs(n, m, 8)
        o = oracle.IterativeOracle(A, **_fixed_kw(k, k_ln))
        if kind == "mixed":
            _ORACLE_CACHE[key] = o.solve_two_mixed(d, r1, r2)
        elif kind == "ls":
            _ORACLE_CACHE[key] = o.solve_two_least_squares(d, r1, r3)
        elif kind == "extras":
            _ORACLE_CACHE[key] = o.solve_two_extras(d, r1, r2)
        elif kind == "zero.mixed":
            _ORACLE_CACHE[key] = o.solve_two_mixed(d, r1, np.zeros(m))
        else:
            _ORACLE_CACHE[key] = o.solve_two_least_squares(d, r1, np.zeros(n))
    return _ORACLE_CACHE[key]


def _bar_b(kind, d, i, k):
    """Bar of the fixed-iteration comparisons (iterate relative difference) after k iterations.

    Measured on a B200 (FIXED_OP, all three Krylov entries, delta in {0, 0.3}):
      * up to 26 iterations (across the first launch boundary) loop and step path agree to 1.1e-15 and both agree with
        the oracle to the same order: the project's roundoff bar of 1e-11 holds with four orders to spare;
      * from about 30 iterations on, LSQR and CRAIG have converged to machine precision on this operator and every
        further iteration roughly doubles the roundoff difference between two implementations (loop vs step path at
        47 / 48 / 49 / 50 / 73 iterations, LSQR x without damping: 1.0e-10 / 2.2e-10 / 4.3e-10 / 1.0e-9 / 2.8e-9,
        largest of all vectors 4.8e-9; against the oracle the same vector: 1.3e-9 / 2.8e-9 / 5.5e-9 / 1.3e-8 / 2.5e-8,
        the largest of all comparisons).  The difference grows smoothly through the boundaries at 24 and 48, the two
        GPU implementations agree with each other five to ten times more closely than with the oracle, and one
        iteration per launch is bitwise the default loop (test_chunk_of_one_equals_default_at_fixed_counts): this is
        roundoff growth, not a hand-over error, which would show at the first boundary and at O(1).  Bar: 2e-7,
        eight times the largest measured spread."""
    return 1e-11 if k <= 26 else 2e-7


def _table(title, errs):
    """errs: {(kind, delta, vector index): {k: relative difference}} -> printed one line per vector."""
    print(f"\n{title}")
    for g in sorted(errs):
        print("  ", g, " ".join(f"{k}:{e:.1e}" for k, e in sorted(errs[g].items())))


@pytest.mark.parametrize("env", ["default", "step", "chunk1"])
def test_fixed_iterations_across_chunk_boundaries(runs, oracle, env):
    """All tolerances 0 and itmax = k: the same iteration count as the oracle, iterates within _bar_b of it."""
    r = runs("fixed", env)
    errs, reached = {}, set()
    for k in FIXED_KS:
        for d in FIXED_DELTAS:
            for kind in ("mixed", "ls", "extras"):
                key = f"k{k}.d{d}.{kind}"
                li = _loop(r, key)
                assert li["persistent"] == (0 if env == "step" else 1), (key, li)
                ref = _fixed_oracle(oracle, kind, k, d)
                for s in range(2):
                    # (a converged LSQR may stop on its machine-precision test before k: 49 with delta = 0.3, 61 at
                    # k = 73 without damping, on both sides)
                    assert int(r[f"{key}.stats"][s][0]) == ref[-1][s]["niter"], (key, s)
                    reached.add(int(ref[-1][s]["niter"]))
                for i in range(_nvec(key)):
                    errs.setdefault((kind, d, i), {})[k] = _rel(r[f"{key}.{i}"], ref[i])
    _table(f"{env}: relative difference to the oracle", errs)
    assert {23, 24, 25, 26, 47, 48, 49, 50} <= reached, reached            # both sides of the first two boundaries
    for (kind, d, i), ek in errs.items():
        for k, e in ek.items():
            assert e < _bar_b(kind, d, i, k), (kind, d, i, k, e)


def test_loop_against_step_path(runs):
    """The persistent loop and one launch per half iteration are two implementations of the same recurrences."""
    a, b = runs("fixed", "default"), runs("fixed", "step")
    errs = {}
    for k in FIXED_KS:
        for d in FIXED_DELTAS:
            for kind in ("mixed", "ls", "extras"):
                key = f"k{k}.d{d}.{kind}"
                assert np.array_equal(a[f"{key}.stats"][:, 0], b[f"{key}.stats"][:, 0])
                for i in range(_nvec(key)):
                    errs.setdefault((kind, d, i), {})[k] = _rel(a[f"{key}.{i}"], b[f"{key}.{i}"])
    _table("loop vs step path: relative difference", errs)
    for (kind, d, i), ek in errs.items():
        for k, e in ek.items():
            assert e < _bar_b(kind, d, i, k), (kind, d, i, k, e)


def test_chunk_of_one_equals_default_at_fixed_counts(runs):
    """One iteration per launch hands the state over at every iteration: bitwise the default loop."""
    a, b = runs("fixed", "default"), runs("fixed", "chunk1")
    for key in [k[:-len(".stats")] for k in a if k.endswith(".stats")]:
        assert _bitwise(b, a, key) is None, key


@pytest.mark.parametrize("env", ["default", "step", "chunk1"])
def test_retired_slot_is_left_alone(runs, oracle, env):
    """One slot stops at 5 iterations while the other runs on to 49 inside the same launches (and the reverse); a zero
    right-hand side retires its slot at iteration 0.  The retired slot equals the oracle and, bitwise, the run in which
    both slots stop at its count."""
    r = runs("fixed", env)
    for kl, kc in ASYM:
        key = f"asym{kl}_{kc}"
        ref = _fixed_oracle(oracle, "mixed", kl, 1e-2, kc)
        st = r[f"{key}.stats"]
        assert int(st[0][0]) == ref[4][0]["niter"] == kl and int(st[1][0]) == ref[4][1]["niter"] == kc, key
        errs = {(key, i): _rel(r[f"{key}.{i}"], ref[i]) for i in range(4)}
        print(f"\n{env} {key}: relative difference to the oracle", {i: f"{e:.1e}" for (_, i), e in errs.items()})
        for i in range(4):
            assert errs[(key, i)] < _bar_b("mixed", 1e-2, i, kl if i < 2 else kc), (key, i)
    # LSQR (slot 0: p1, q1) retired at 5 while CRAIG ran on; CRAIG (slot 1: p2, q2) retired at 5 while LSQR ran on
    for i in (0, 1):
        assert np.array_equal(r[f"asym5_49.{i}"], r[f"asym5_5.{i}"]), i
        assert np.array_equal(r[f"asym49_5.{i}"], r[f"asym49_49.{i}"]), i
    for i in (2, 3):
        assert np.array_equal(r[f"asym49_5.{i}"], r[f"asym5_5.{i}"]), i
        assert np.array_equal(r[f"asym5_49.{i}"], r[f"asym49_49.{i}"]), i
    assert np.array_equal(r["asym5_49.stats"][0], r["asym5_5.stats"][0], equal_nan=True)
    assert np.array_equal(r["asym49_5.stats"][1], r["asym5_5.stats"][1], equal_nan=True)
    for kind in ("zero.mixed", "zero.ls"):
        ref = _fixed_oracle(oracle, kind, 49, 1e-2)
        st = r[f"{kind}.stats"]
        assert int(st[0][0]) == ref[4][0]["niter"] == 49 and int(st[1][0]) == ref[4][1]["niter"] == 0, kind
        assert st[1][1] == 1.0, kind                                       # solved
        for i in (0, 1):
            e = _rel(r[f"{kind}.{i}"], ref[i])
            print(f"{env} {kind}.{i}: {e:.1e}")
            assert e < _bar_b("mixed" if kind == "zero.mixed" else "ls", 1e-2, i, 49), (kind, i)
        for i in (2, 3):
            assert np.array_equal(r[f"{kind}.{i}"], ref[i]) and not r[f"{kind}.{i}"].any(), (kind, i)


# ---------------------------------------------------------------------------------------------------------------------
# C. LDLt modes
# ---------------------------------------------------------------------------------------------------------------------
MODES = ["mode0", "mode1", "mode2"]
_LDLT_ORACLE = {}


def _ldlt_oracle(oracle, ci, P):
    if ci not in _LDLT_ORACLE:
        case = LDLT_CASES[ci]
        A = _ldlt_matrix(case)
        m, n = A.shape
        coo = sp.coo_matrix(A)
        lo = oracle.LDLtOracle(n, m, coo.row, coo.col, P)
        r1, r2, r3 = _rhs(n, m, 5 + ci)
        mixed = lo.solve_two_mixed(coo.data, case[4], r1, r2)
        sym = lo.symbolic()
        Lx, D = lo.numeric()
        ls = lo.solve_two_least_squares(r1, r3)
        _LDLT_ORACLE[ci] = dict(A=A, r=(r1, r2, r3), mixed=mixed, ls=ls, sym=sym, Lx=Lx, D=D)
    return _LDLT_ORACLE[ci]


@pytest.mark.parametrize("mode", MODES)
def test_ldlt_mode_single_instance_against_oracle(runs, oracle, mode):
    """Symbolic analysis bit-exact, factor to 1e-10, solutions to 1e-8 (1e-5 with regularised pivots), residual 1e-10,
    for the mixed and the least-squares solves."""
    r = runs("ldlt", mode)
    for ci, case in enumerate(LDLT_CASES):
        o = _ldlt_oracle(oracle, ci, r[f"c{ci}.sym.P"])
        for key in ("P", "parent", "Lnz", "Lp", "Li"):
            assert np.array_equal(r[f"c{ci}.sym.{key}"], o["sym"][key]), (ci, key)
        assert _rel(r[f"c{ci}.D"], o["D"]) < 1e-10 and _rel(r[f"c{ci}.Lx"], o["Lx"]) < 1e-10, ci
        assert bool(r[f"c{ci}.mixed.ok"]) and bool(r[f"c{ci}.ls.ok"]) and o["mixed"][4], ci
        perturbed = bool(np.any(np.abs(np.abs(o["D"]) - SQRT_EPS) < 1e-12))
        bar = 1e-5 if perturbed else 1e-8
        for kind in ("mixed", "ls"):
            for i in range(4):
                assert _rel(r[f"c{ci}.{kind}.{i}"], o[kind][i]) < bar, (ci, kind, i)
        if not perturbed:
            A, delta = o["A"], case[4]
            (r1, r2, r3), g = o["r"], [r[f"c{ci}.mixed.{i}"] for i in range(4)]
            e1 = np.r_[g[0] + A.T @ g[1] - r1, A @ g[0] - delta * g[1]]
            e2 = np.r_[g[2] + A.T @ g[3], A @ g[2] - delta * g[3] - r2]
            assert np.linalg.norm(e1) / np.linalg.norm(r1) < 1e-10 and np.linalg.norm(e2) / np.linalg.norm(r2) < 1e-10, ci
            g = [r[f"c{ci}.ls.{i}"] for i in range(4)]
            e1 = np.r_[g[0] + A.T @ g[1] - r1, A @ g[0] - delta * g[1]]
            e2 = np.r_[g[2] + A.T @ g[3] - r3, A @ g[2] - delta * g[3]]
            assert np.linalg.norm(e1) / np.linalg.norm(r1) < 1e-10 and np.linalg.norm(e2) / np.linalg.norm(r3) < 1e-10, ci
    # the largest shape has supernodes above the leaves, whose Schur updates run through the mode's routines
    nsuper, nleaf, _ = r[f"c{len(LDLT_CASES) - 1}.plan"]
    assert nsuper > nleaf


@pytest.mark.parametrize("mode", MODES)
def test_ldlt_mode_rank_deficient_regularisation(runs, oracle, mode):
    """Duplicated Jacobian rows with delta = 0: the regularised pivots and their signs are the oracle's."""
    r = runs("ldlt", mode)
    A = _rank_deficient_matrix()
    m, n = A.shape
    coo = sp.coo_matrix(A)
    lo = oracle.LDLtOracle(n, m, coo.row, coo.col, r["rd.P"])
    rng = np.random.default_rng(1)
    r1 = rng.standard_normal(n); r2 = A @ rng.standard_normal(n)
    ref = lo.solve_two_mixed(coo.data, 0.0, r1, r2)
    _, oD = lo.numeric()
    assert bool(r["rd.ok"]) and ref[4]
    reg = np.abs(np.abs(oD) - SQRT_EPS) < 1e-12
    assert reg.sum() >= 10
    D = r["rd.D"]
    assert np.array_equal(np.abs(np.abs(D) - SQRT_EPS) < 1e-12, reg)
    assert np.array_equal(np.sign(D), np.sign(oD))


@pytest.mark.parametrize("mode", MODES)
def test_ldlt_mode_batch_bitwise_single(runs, mode):
    """Both batched entries equal, bitwise, the single path run on each instance alone, under every mode: healthy,
    regularised and failing instances, and a shape whose plan has supernodes above the leaves."""
    r = runs("ldlt", mode)
    for tag, ninst in (("mixreg", 6), ("mixoff", 5), ("big", BATCH_BIG_NINST)):
        for i in range(ninst):
            for kind in ("mixed", "ls"):
                for j in range(4):
                    assert np.array_equal(r[f"{tag}.b{kind}.{j}"][i], r[f"{tag}.s{kind}{i}.{j}"]), (tag, kind, i, j)
                assert bool(r[f"{tag}.b{kind}.4"][i]) == bool(r[f"{tag}.s{kind}{i}.4"]), (tag, kind, i)
    assert r["mixreg.bmixed.4"].all()
    assert list(r["mixoff.bmixed.4"]) == [True, True, True, False, True]
    nsuper, nleaf, _ = r["big.plan"]
    assert nsuper > nleaf


def test_ldlt_modes_zero_and_one_agree(runs):
    """Modes 0 and 1 follow the reference's operation order: their factors agree to 1e-14 relative.  (On a B200 all 16
    factor arrays of LDLT_CASES came out bitwise equal.)"""
    a, b = runs("ldlt", "mode0"), runs("ldlt", "mode1")
    same = []
    for ci in range(len(LDLT_CASES)):
        for key in ("Lx", "D"):
            assert _rel(a[f"c{ci}.{key}"], b[f"c{ci}.{key}"]) < 1e-14, (ci, key)
            same.append(np.array_equal(a[f"c{ci}.{key}"], b[f"c{ci}.{key}"]))
    print(f"\nmodes 0 and 1: {sum(same)} of {len(same)} factor arrays bitwise equal")


if __name__ == "__main__":
    if len(sys.argv) == 5 and sys.argv[1] == "--worker":
        _worker(sys.argv[2:])
    else:
        sys.exit("usage: python tests/test_gpu_variants.py --worker <sched|fixed|ldlt> <env name> <out.npz>")
