"""GPU: every exit branch of the Krylov recurrences, and the full stats record against the oracle.

The stats record (niter, solved, inconsistent, status, rnorm, arnorm, anorm, acond, xnorm) comes from scalar recurrences
fed by partial sums the row epilogues compute (`acc1` of MD_LSQR_V / MD_CRAIG_U, `xx` of MINRES_E2, ...).  The iterates
never read them, so only a comparison of the record itself catches a wrong partial: with it a solve stops one iteration
early or late, or leaves by the wrong branch.  The recurrences run in four places, each fed by its own partial-sum code:
the last CTA of the step kernel (`FPSB_LOOP=0`, and MINRES / CGLS everywhere), the persistent loop kernel, the finish of
the row-partitioned handle (world size 1 here) and thread 0 of the batched extras kernel.

1. Fixed iteration counts (tolerances 0, itmax = k): the record equals the oracle's, counts and flags exactly, norms to
   1e-11 relative, on every path.
2. Every exit branch, built from structure where it can be (the deciding quantity is exactly zero), on every path that
   can reach it: status, solved, inconsistent and niter exactly, the rest of the record and the vectors to 1e-11.
3. One slot of solve_two_mixed exits strangely (LSQR on A r = 0 after its first product, CRAIG inconsistent in the
   middle of its first iteration) while the other runs on: the running slot is bitwise the run whose other right-hand
   side is zero.
4. The consumers of the flags: IterativeSolver warns exactly when the oracle's solve fails, TR_fused returns the
   oracle's MINRES `solved`.

The FPSB_LOOP switch is read once per process, so the step path runs in a worker process:
`python tests/test_gpu_krylov_exits.py --worker <default|step> <out.npz>` runs every solve of its path(s) and writes the
vectors, stats records and loop_info() to out.npz.  Stopping decisions that are not exact zeros are shown not to be near
ties by the unmarked `test_exit_margin` tests, which need only the oracle.
"""
import os
import subprocess
import sys
import types
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SQRT_EPS = float(np.sqrt(np.finfo(float).eps))
STAT_KEYS = ("niter", "solved", "inconsistent", "status", "rnorm", "arnorm", "anorm", "acond", "xnorm")
FLAG_KEYS = STAT_KEYS[:4]
NORM_KEYS = STAT_KEYS[4:]
BAR = 1e-11
ZERO_RHS, SOLVED, ZERO_RESID, FWD_ERR, TIRED, ILLCOND_LIM, INCONSISTENT, ZERO_ATB = 1, 2, 3, 4, 5, 7, 8, 9

# ---------------------------------------------------------------------------------------------------------------------
# operators
# ---------------------------------------------------------------------------------------------------------------------
FIXED_KS = (1, 2, 4, 5, 6, 7, 20)          # the err_lbnd window opens at iteration 5
DELTAS = (0.0, 0.3)
PAD = 3                                     # structurally empty rows and columns of the "struct" operator


def _fixed_matrix():
    from fpsb200 import models
    return models.window_random_jacobian(2000, 4000, 10, w=32, seed=21)


def _struct_matrix():
    """window_random_jacobian(2000, 4000) with PAD empty rows and PAD empty columns appended."""
    from fpsb200 import models
    A0 = models.window_random_jacobian(2000, 4000, 10, w=32, seed=41)
    return sp.bmat([[A0, None], [None, sp.csr_matrix((PAD, PAD))]]).tocsr()


def _select_matrix():
    """S[i, 2 i] = 2: S S' = 4 I, and S' S e_j = 4 e_j on every selected column j."""
    m, n = 2000, 4000
    return sp.csr_matrix((np.full(m, 2.0), (np.arange(m), 2 * np.arange(m))), shape=(m, n))


def _wellcond_matrix():
    """S[i, 2 i] = sqrt(1 + 0.1 i / m): the nonzero spectrum of S S' and S' S fills [1, 1.1], so every method gains a
    factor of about 40 per iteration and a converged solve crosses its threshold far from a tie."""
    m, n = 2000, 4000
    return sp.csr_matrix((np.sqrt(1.0 + 0.1 * np.arange(m) / m), (np.arange(m), 2 * np.arange(m))), shape=(m, n))


MATRICES = {"fixed": _fixed_matrix, "struct": _struct_matrix, "select": _select_matrix, "wellcond": _wellcond_matrix}
_MAT_CACHE = {}


def _matrix(name):
    if name not in _MAT_CACHE:
        _MAT_CACHE[name] = MATRICES[name]()
    return _MAT_CACHE[name]


def _fixed_kw(k):
    return dict(ls_atol=0.0, ls_rtol=0.0, ls_itmax=k, ln_atol=0.0, ln_rtol=0.0, ln_btol=0.0, ln_itmax=k,
                ne_atol=0.0, ne_rtol=0.0, ne_etol=0.0, ne_itmax=k)


# ---------------------------------------------------------------------------------------------------------------------
# part 2 cases: (name, operator, kind, delta, right-hand sides, IterOpts overrides, expected statuses of the two slots)
# kind "ldlt" is the LDLt path's solve_two_extras (CGLS + MINRES); "ls" is solve_two_least_squares.
# ---------------------------------------------------------------------------------------------------------------------
def _rhs(op, spec):
    A = _matrix(op)
    m, n = A.shape
    rng = np.random.default_rng(7)
    r1, r2, r3 = rng.standard_normal(n), rng.standard_normal(m), rng.standard_normal(n)
    out = []
    for s in spec:
        if s == "zero_n":
            out.append(np.zeros(n))
        elif s == "zero_m":
            out.append(np.zeros(m))
        elif s == "rand_n":
            out.append(r1)
        elif s == "rand_n2":
            out.append(r3)
        elif s == "rand_m":
            out.append(r2)
        elif s == "range_n":            # A' y: LSQR on A' is consistent
            out.append(A.T @ r2)
        elif s == "empty_cols":         # supported only on the empty columns: A r = 0 exactly
            v = np.zeros(n); v[n - PAD:] = rng.standard_normal(PAD); out.append(v)
        elif s == "empty_row":          # e_i on an empty row: A' e_i = 0 exactly
            v = np.zeros(m); v[m - 2] = 1.5; out.append(v)
        elif s == "selected_col":       # one entry on a selected column of S
            v = np.zeros(n); v[2 * 777] = 3.0; out.append(v)
        elif s == "selected_col2":
            v = np.zeros(n); v[2 * 1500] = -0.75; out.append(v)
        else:
            raise ValueError(s)
    return out


def _cases():
    c = []
    for kind, spec in (("mixed", ("zero_n", "zero_m")), ("ls", ("zero_n", "zero_n")), ("extras", ("zero_n", "zero_m")),
                       ("ldlt", ("zero_n", "zero_m"))):
        c.append(dict(name=f"zero_rhs.{kind}", op="struct", kind=kind, delta=0.3, rhs=spec, kw={},
                      want=(ZERO_RHS, ZERO_RHS)))
    for d in DELTAS:
        c.append(dict(name=f"zero_atb.mixed.d{d}", op="struct", kind="mixed", delta=d, rhs=("empty_cols", "zero_m"),
                      kw={}, want=(ZERO_ATB, ZERO_RHS)))
        c.append(dict(name=f"lsqr_beta0.mixed.d{d}", op="select", kind="mixed", delta=d, rhs=("selected_col", "zero_m"),
                      kw={}, want=(ZERO_RESID if d == 0 else SOLVED, ZERO_RHS)))
        c.append(dict(name=f"craig_inconsistent.d{d}", op="struct", kind="mixed", delta=d, rhs=("zero_n", "empty_row"),
                      kw={}, want=(ZERO_RHS, INCONSISTENT)))
        c.append(dict(name=f"minres_early.d{d}", op="select", kind="extras", delta=d, rhs=("zero_n", "rand_m"), kw={},
                      want=(ZERO_RHS, ZERO_ATB)))
        c.append(dict(name=f"minres_early.ldlt.d{d}", op="select", kind="ldlt", delta=d, rhs=("zero_n", "rand_m"),
                      kw={}, want=(ZERO_RHS, ZERO_ATB)))
        # ln_conlim / ne_conlim lowered below the condition estimate of iteration 1 (CRAIG: 4.1 at delta = 0, 10.1 at
        # 0.3; MINRES: gmax / gmin = 1 exactly).  No later iteration of these operators grows the estimate by the 4x
        # that a 2x margin on both sides would need, and iteration 0 runs no conditioning test.
        c.append(dict(name=f"craig_conlim.d{d}", op="struct", kind="mixed", delta=d, rhs=("zero_n", "rand_m"),
                      kw=dict(ln_conlim=1.0), want=(ZERO_RHS, ILLCOND_LIM)))
        c.append(dict(name=f"minres_conlim.d{d}", op="struct", kind="extras", delta=d, rhs=("zero_n", "rand_m"),
                      kw=dict(ne_conlim=0.25), want=(ZERO_RHS, ILLCOND_LIM)))
    c.append(dict(name="zero_atb.ls", op="struct", kind="ls", delta=0.3, rhs=("empty_cols", "empty_cols"), kw={},
                  want=(ZERO_ATB, ZERO_ATB)))
    c.append(dict(name="zero_atb.extras", op="struct", kind="extras", delta=0.3, rhs=("empty_cols", "zero_m"), kw={},
                  want=(ZERO_ATB, ZERO_RHS)))
    c.append(dict(name="lsqr_beta0.ls", op="select", kind="ls", delta=0.0, rhs=("selected_col", "selected_col2"),
                  kw={}, want=(ZERO_RESID, ZERO_RESID)))
    # converged solves at the reference tolerances, on the operator whose spectrum makes the crossing sharp (margins:
    # test_exit_margin)
    c.append(dict(name="converged.lsqr", op="wellcond", kind="mixed", delta=0.0, rhs=("rand_n", "zero_m"), kw={},
                  want=(SOLVED, ZERO_RHS)))
    c.append(dict(name="converged.lsqr_consistent", op="wellcond", kind="mixed", delta=0.0, rhs=("range_n", "zero_m"),
                  kw={}, want=(ZERO_RESID, ZERO_RHS)))
    c.append(dict(name="converged.craig", op="wellcond", kind="mixed", delta=0.0, rhs=("zero_n", "rand_m"), kw={},
                  want=(ZERO_RHS, SOLVED)))
    c.append(dict(name="converged.minres", op="wellcond", kind="extras", delta=0.3, rhs=("zero_n", "rand_m"), kw={},
                  want=(ZERO_RHS, ZERO_RESID)))
    c.append(dict(name="converged.fwd_err", op="wellcond", kind="extras", delta=0.0, rhs=("zero_n", "rand_m"),
                  kw=dict(ne_atol=1e-14, ne_rtol=1e-14, ne_etol=3e-3), want=(ZERO_RHS, FWD_ERR)))
    c.append(dict(name="converged.ldlt", op="wellcond", kind="ldlt", delta=0.3, rhs=("rand_n", "zero_m"), kw={},
                  want=(SOLVED, ZERO_RHS)))
    return c


CASES = _cases()
CASE_BY_NAME = {c["name"]: c for c in CASES}
# part 3: (name, operator, delta, rhs, slot that keeps running, rhs of the reference run).  The running slot has its
# tolerances off and stops at RETIRE_K; the other slot's exit is structural and does not look at a tolerance.
RETIRE_K = 41
RETIRE_VEC_BAR = 1e-10
RETIRE = [("atb_vs_craig", "struct", 0.3, ("empty_cols", "rand_m"), 1, ("zero_n", "rand_m")),
          ("incons_vs_lsqr", "struct", 0.3, ("rand_n", "empty_row"), 0, ("rand_n", "zero_m"))]


def _case_inputs(case):
    return _matrix(case["op"]), _rhs(case["op"], case["rhs"])


# ---------------------------------------------------------------------------------------------------------------------
# oracle side
# ---------------------------------------------------------------------------------------------------------------------
_ORACLE_CACHE = {}


def _ldlt_extras_oracle(O, A, delta, r1, r2, scale=1.0, itmax=0):
    """fo_ldlt_solve_two_extras spelled out: cgls(A', r1, tau) and minres(A A' + tau I, r2) at Krylov.jl's defaults,
    every threshold multiplied by `scale` (conlim divided by it)."""
    tau = max(delta, 1e-14)
    u1, s1 = O.cgls(A, r1, lam=tau, atol=SQRT_EPS * scale, rtol=SQRT_EPS * scale, itmax=itmax, transpose=True)
    u2, s2 = O.minres_normal(A, r2, tau, atol=SQRT_EPS / 100 * scale, rtol=SQRT_EPS / 100 * scale,
                             etol=SQRT_EPS * scale, conlim=1 / SQRT_EPS / scale, itmax=itmax)
    return u1, u2, [s1, s2]


def _oracle_solve(O, A, kind, delta, r1, r2, kw):
    if kind == "ldlt":
        return _ldlt_extras_oracle(O, A, delta, r1, r2)
    o = O.IterativeOracle(A, **kw)
    return {"mixed": o.solve_two_mixed, "ls": o.solve_two_least_squares, "extras": o.solve_two_extras}[kind](
        delta, r1, r2)


def _case_oracle(O, case):
    key = ("case", case["name"])
    if key not in _ORACLE_CACHE:
        A, (r1, r2) = _case_inputs(case)
        _ORACLE_CACHE[key] = _oracle_solve(O, A, case["kind"], case["delta"], r1, r2, case["kw"])
    return _ORACLE_CACHE[key]


def _fixed_oracle(O, kind, k, d):
    key = ("fixed", kind, k, d)
    if key not in _ORACLE_CACHE:
        A = _matrix("fixed")
        r1, r2, r3 = _rhs("fixed", ("rand_n", "rand_m", "rand_n2"))
        _ORACLE_CACHE[key] = _oracle_solve(O, A, kind, d, r1, r3 if kind == "ls" else r2, _fixed_kw(k))
    return _ORACLE_CACHE[key]


def _scaled_outcome(O, case, s):
    """Exit (niter, status, solved, inconsistent) of both slots with every stopping threshold multiplied by s (conlim
    divided by s): tolerances x2 loosen every test, x1/2 tighten it."""
    A, (r1, r2) = _case_inputs(case)
    d, kw = case["delta"], case["kw"]
    if case["kind"] == "ldlt":
        st = _ldlt_extras_oracle(O, A, d, r1, r2, scale=s)[2]
    else:
        t = O.IterativeOracle(A, **kw).tol
        lam = np.sqrt(d) if case["kind"] != "extras" else np.sqrt(max(d, 1e-14))
        lsqr = lambda b: O.lsqr(A, b, lam=lam, atol=t.ls_atol * s, rtol=t.ls_rtol * s, itmax=t.ls_itmax,
                                transpose=True, axtol=SQRT_EPS * s, btol=SQRT_EPS * s, etol=SQRT_EPS * s,
                                conlim=1 / SQRT_EPS / s)[1]
        st = [lsqr(r1)]
        if case["kind"] == "mixed":
            st.append(O.craig(A, -r2, delta=d, atol=t.ln_atol * s, rtol=t.ln_rtol * s, btol=t.ln_btol * s,
                              conlim=t.ln_conlim / s, itmax=t.ln_itmax)[2])
        elif case["kind"] == "ls":
            st.append(lsqr(r2))
        else:
            st.append(O.minres_normal(A, r2, max(d, 1e-14), atol=t.ne_atol * s, rtol=t.ne_rtol * s,
                                      etol=t.ne_etol * s, conlim=t.ne_conlim / s, itmax=t.ne_itmax)[1])
    return [tuple(x[k] for k in FLAG_KEYS) for x in st]


# ---------------------------------------------------------------------------------------------------------------------
# margins (oracle only: no GPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", [c["name"] for c in CASES])
def test_exit_margin(oracle, name):
    """Each case reaches its intended exit in the oracle, and the decision is not a near tie: with every stopping
    threshold loosened 2x the solve still runs to the same iteration (no test was within 2x of firing one iteration
    earlier) and with every threshold tightened 2x it still stops there by the same branch (the deciding ratio is at
    least 2x inside its threshold).  The exact-zero constructions pass trivially; the machine-precision tests
    (1 + x <= 1) have no threshold to scale and decide none of these cases."""
    case = CASE_BY_NAME[name]
    st = _case_oracle(oracle, case)[-1]
    for s, w in zip(st, case["want"]):
        if w is not None:
            assert s["status"] == w, (name, s)
    base = [tuple(x[k] for k in FLAG_KEYS) for x in st]
    assert _scaled_outcome(oracle, case, 1.0) == base, name
    for scale in (2.0, 0.5):
        assert _scaled_outcome(oracle, case, scale) == base, (name, scale)


def test_exit_statuses_covered(oracle):
    """Part 2 reaches statuses 1, 2, 3, 4, 7, 8 and 9 in the oracle; 5 (itmax) is what part 1 runs into."""
    seen = {s["status"] for c in CASES for s in _case_oracle(oracle, c)[-1]}
    assert {ZERO_RHS, SOLVED, ZERO_RESID, FWD_ERR, ILLCOND_LIM, INCONSISTENT, ZERO_ATB} <= seen, seen
    st = _fixed_oracle(oracle, "mixed", 4, 0.0)[-1]
    assert all(s["status"] == TIRED and s["niter"] == 4 for s in st)


def test_retirement_exits(oracle):
    """Part 3 in the oracle: the running slot runs to RETIRE_K, the other leaves by its structural branch at once."""
    for name, op, d, rhs, run, ref_rhs in RETIRE:
        st = _retire_oracle(oracle, name, op, d, rhs)[-1]
        assert st[run]["niter"] == RETIRE_K and st[run]["status"] == TIRED, (name, st)
        assert st[1 - run]["niter"] == 0 and st[1 - run]["status"] == (ZERO_ATB if run == 1 else INCONSISTENT), st
        st = _retire_oracle(oracle, name + ".ref", op, d, ref_rhs)[-1]
        assert st[1 - run]["status"] == ZERO_RHS


def _retire_oracle(O, name, op, d, rhs):
    return _case_oracle(O, dict(name="retire." + name, op=op, kind="mixed", delta=d, rhs=rhs, kw=_fixed_kw(RETIRE_K)))


# ---------------------------------------------------------------------------------------------------------------------
# worker
# ---------------------------------------------------------------------------------------------------------------------
def _opts(A, kw):
    import ctypes
    import fpsb200
    o = fpsb200.IterOpts()
    fpsb200._lib.lib().fpsb_iter_default_opts(ctypes.c_int64(A.shape[1]), ctypes.c_int64(A.shape[0]), ctypes.byref(o))
    for k, v in kw.items():
        setattr(o, k, v)
    return o


_HANDLES = {}


def _handle(op, kw):
    """One handle per operator (worker process), set up with the options of the next solve."""
    import fpsb200
    A = _matrix(op)
    if ("h", op) not in _HANDLES:
        coo = sp.coo_matrix(A)
        H = fpsb200.B200Handle(A.shape[1], A.shape[0], coo.row, coo.col)
        H.set_jac_values(coo.data)
        _HANDLES[("h", op)] = H
    H = _HANDLES[("h", op)]
    H.iter_setup(_opts(A, kw))
    return H


def _dist(op, kw):
    """The row-partitioned handle of world size 1 (one per operator), set up with the options of the next solve."""
    from fpsb200.partition import RowPartition, DistHandle
    A = _matrix(op)
    if ("d", op) not in _HANDLES:
        coo = sp.coo_matrix(A)
        m, n = A.shape
        D = DistHandle(RowPartition(n, m, coo.row.astype(np.int64), coo.col.astype(np.int64), 1), 0, device=0)
        D.set_jac_values(coo.data)
        _HANDLES[("d", op)] = D
    D = _HANDLES[("d", op)]
    D.H.iter_setup(_opts(A, kw))
    return D


class _Out(dict):
    def put(self, key, got, loop=None):
        for i, a in enumerate(got[:-1]):
            self[f"{key}.{i}"] = np.asarray(a)
        self[f"{key}.stats"] = np.array([[float(s[k]) for k in STAT_KEYS] for s in got[-1]])
        if loop is not None:
            self[f"{key}.persistent"] = np.array(loop["persistent"])


def _iter_call(H, kind, d, r1, r2):
    return {"mixed": H.iter_solve_two_mixed, "ls": H.iter_solve_two_least_squares,
            "extras": H.iter_solve_two_extras}[kind](d, r1, r2)


def _dist_call(D, kind, d, r1, r2):
    return {"mixed": D.solve_two_mixed, "ls": D.solve_two_least_squares, "extras": D.solve_two_extras}[kind](d, r1, r2)


def _batch_stats(st, i):
    return [{k: st[k][i, j].item() for k in STAT_KEYS} for j in range(2)]


def _work(out, env):
    import fpsb200
    path = "step" if env == "step" else "loop"
    # part 1: fixed iteration counts
    A = _matrix("fixed")
    coo = sp.coo_matrix(A)
    r1, r2, r3 = _rhs("fixed", ("rand_n", "rand_m", "rand_n2"))
    for k in FIXED_KS:
        H = _handle("fixed", _fixed_kw(k))
        D = _dist("fixed", _fixed_kw(k)) if env == "default" else None
        for d in DELTAS:
            for kind in ("mixed", "ls", "extras"):
                b = r3 if kind == "ls" else r2
                out.put(f"fixed.k{k}.d{d}.{kind}.{path}", _iter_call(H, kind, d, r1, b), H.loop_info())
                if D is not None:
                    out.put(f"fixed.k{k}.d{d}.{kind}.dist", _dist_call(D, kind, d, r1, b))
            if env == "default":
                o = fpsb200.ExtrasOpts()
                o.cg_atol = o.cg_rtol = 0.0
                o.cg_itmax = k
                o.mr_atol = o.mr_rtol = o.mr_etol = 0.0
                o.mr_conlim = 1 / SQRT_EPS
                o.mr_itmax = k
                J = np.stack([coo.data, 0.5 * coo.data])
                u1, u2, st = H.ldlt_batch_solve_two_extras(d, J, np.stack([r1, r3]), np.stack([r2, -r2]), opts=o)
                for i in range(2):
                    out.put(f"fixed.k{k}.d{d}.ldlt.batch{i}", (u1[i], u2[i], _batch_stats(st, i)))
    # part 2: exit branches
    for case in CASES:
        A, (r1, r2) = _case_inputs(case)
        kind, d, name = case["kind"], case["delta"], case["name"]
        H = _handle(case["op"], case["kw"])
        if kind == "ldlt":
            if env != "default":
                continue
            out.put(f"{name}.ldlt", H.ldlt_solve_two_extras(d, r1, r2))
            coo = sp.coo_matrix(A)
            J = np.stack([coo.data, 0.5 * coo.data])
            u1, u2, st = H.ldlt_batch_solve_two_extras(d, J, np.stack([r1, r1]), np.stack([r2, r2]))
            for i in range(2):
                out.put(f"{name}.batch{i}", (u1[i], u2[i], _batch_stats(st, i)))
            continue
        out.put(f"{name}.{path}", _iter_call(H, kind, d, r1, r2), H.loop_info())
        if env == "default":
            out.put(f"{name}.dist", _dist_call(_dist(case["op"], case["kw"]), kind, d, r1, r2))
    # part 3: one slot retires early while the other runs on
    for name, op, d, rhs, run, ref_rhs in RETIRE:
        H = _handle(op, _fixed_kw(RETIRE_K))
        for tag, spec in (("", rhs), (".ref", ref_rhs)):
            r1, r2 = _rhs(op, spec)
            out.put(f"retire.{name}{tag}.{path}", H.iter_solve_two_mixed(d, r1, r2), H.loop_info())


def _worker(argv):
    env, path = argv
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    out = _Out()
    _work(out, env)
    np.savez(path, **out)


# ---------------------------------------------------------------------------------------------------------------------
# parent
# ---------------------------------------------------------------------------------------------------------------------
ENVS = {"default": {}, "step": {"FPSB_LOOP": "0"}}
WORKER_TIMEOUT = 600


@pytest.fixture(scope="session")
def exit_runs(tmp_path_factory):
    cache = {}
    base = tmp_path_factory.mktemp("krylov_exits")

    def get(env):
        if env not in cache:
            path = str(base / f"{env}.npz")
            child = {k: v for k, v in os.environ.items() if not (k.startswith("FPSB_") or k == "FPSB200_LIB")}
            child.update(ENVS[env])
            if "FPSB200_LIB" in os.environ:
                child["FPSB200_LIB"] = os.environ["FPSB200_LIB"]
            child["PYTHONPATH"] = os.pathsep.join([ROOT] + [p for p in sys.path if p])
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", env, path], env=child, cwd=ROOT,
                               capture_output=True, text=True, timeout=WORKER_TIMEOUT)
            if r.returncode != 0:
                raise AssertionError(f"worker {env} exited with {r.returncode}:\n{r.stderr[-4000:]}")
            with np.load(path) as z:
                cache[env] = {k: z[k] for k in z.files}
        return cache[env]

    return get


PATHS = {"loop": "default", "step": "step", "dist": "default"}


def _rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _stats(run, key):
    return [dict(zip(STAT_KEYS, row)) for row in run[f"{key}.stats"]]


def _compare(run, key, ref, nvec, rhs, vec_bar=BAR):
    """Flags exactly; norms and vectors to BAR relative.  Two quantities are roundoff once a solve has reached its
    answer, and are held to the problem's scale instead of their own: rnorm / arnorm (measured on a B200: MINRES's
    early exit at iteration 1 reports rnorm 3.6e-15 where the oracle has 8.0e-14, both eps-level for |b| = 45) get
    1e-13 |b| max(1, anorm) absolute, and a vector whose norm is below |b| (p = r - A'q of a consistent system) is
    compared relative to |b|.  The decisions themselves are the exact flags."""
    got = _stats(run, key)
    worst = 0.0
    bnorm = max(np.linalg.norm(r) for r in rhs)
    for s, (g, o) in enumerate(zip(got, ref[-1])):
        for k in FLAG_KEYS:
            assert g[k] == float(o[k]), (key, s, k, g, o)
        for k in NORM_KEYS:
            e = abs(g[k] - o[k])
            floor = 1e-13 * bnorm * max(1.0, o["anorm"]) if k in ("rnorm", "arnorm") else 0.0
            assert e <= BAR * abs(o[k]) + floor or g[k] == o[k], (key, s, k, g[k], o[k])
            worst = max(worst, e / max(abs(o[k]), floor / BAR) if o[k] else 0.0)
    for i in range(nvec):
        a, b = run[f"{key}.{i}"], ref[i]
        if not b.any():
            assert not a.any(), (key, i)
            continue
        e = float(np.linalg.norm(a - b) / max(np.linalg.norm(b), bnorm))
        assert e < vec_bar, (key, i, e)
        worst = max(worst, e)
    return worst


def _nvec(kind):
    return 2 if kind in ("extras", "ldlt") else 4


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["loop", "step", "dist", "batch"])
def test_stats_at_fixed_counts(exit_runs, oracle, path):
    """Tolerances 0, itmax = k: the whole stats record equals the oracle's on each place the recurrences run."""
    run = exit_runs("step" if path == "step" else "default")
    A = _matrix("fixed")
    worst = 0.0
    for k in FIXED_KS:
        for d in DELTAS:
            if path == "batch":
                r1, r2, r3 = _rhs("fixed", ("rand_n", "rand_m", "rand_n2"))
                for i, (Ai, b1, b2) in enumerate(((A, r1, r2), (0.5 * A, r3, -r2))):
                    ref = _batch_fixed_oracle(oracle, Ai, d, b1, b2, k)
                    assert ref[2][0]["niter"] == ref[2][1]["niter"] == k
                    worst = max(worst, _compare(run, f"fixed.k{k}.d{d}.ldlt.batch{i}", ref, 2, (b1, b2)))
                continue
            for kind in ("mixed", "ls", "extras"):
                key = f"fixed.k{k}.d{d}.{kind}.{path}"
                ref = _fixed_oracle(oracle, kind, k, d)
                assert all(s["niter"] == k for s in ref[-1])
                if path in ("loop", "step"):
                    assert int(run[f"{key}.persistent"]) == (1 if path == "loop" else 0), key
                r1, r2, r3 = _rhs("fixed", ("rand_n", "rand_m", "rand_n2"))
                worst = max(worst, _compare(run, key, ref, _nvec(kind), (r1, r3 if kind == "ls" else r2)))
    print(f"\nfixed counts {FIXED_KS}, {path}: largest relative difference to the oracle {worst:.1e}")


def _batch_fixed_oracle(O, Ai, d, r1, r2, k):
    tau = max(d, 1e-14)
    Ai = sp.csr_matrix(Ai)
    u1, s1 = O.cgls(Ai, r1, lam=tau, atol=0.0, rtol=0.0, itmax=k, transpose=True)
    u2, s2 = O.minres_normal(Ai, r2, tau, 0.0, 0.0, 0.0, conlim=1 / SQRT_EPS, itmax=k)
    return u1, u2, [s1, s2]


def _case_paths(case):
    return ["ldlt", "batch0", "batch1"] if case["kind"] == "ldlt" else ["loop", "step", "dist"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in CASES])
def test_exit_branch(exit_runs, oracle, name):
    """The case's exit, on every path that can reach it: flags exactly, the rest of the record and the vectors to
    1e-11 relative (exact where the oracle's vector is zero), plus the closed forms."""
    case = CASE_BY_NAME[name]
    A, (r1, r2) = _case_inputs(case)
    ref = _case_oracle(oracle, case)
    for path in _case_paths(case):
        run = exit_runs("step" if path == "step" else "default")
        key = f"{name}.{path}"
        if path.startswith("batch"):
            i = int(path[-1])
            Ai = A if i == 0 else 0.5 * A
            r = _ldlt_extras_oracle(oracle, sp.csr_matrix(Ai), case["delta"], r1, r2)
        else:
            r = ref
        worst = _compare(run, key, r, _nvec(case["kind"]), (r1, r2))
        st = _stats(run, key)
        if path in ("loop", "step") and case["kind"] != "extras":
            # (extras: LSQR runs on the loop, MINRES on the step kernels; loop_info describes the last solve)
            loops = int(run[f"{key}.persistent"])
            assert loops == (1 if path == "loop" else 0) or st[0]["status"] in (ZERO_RHS, ZERO_ATB), (key, loops)
        print(f"\n{name:28s} {path:6s} status {[int(s['status']) for s in st]} niter {[int(s['niter']) for s in st]}"
              f" largest relative difference {worst:.1e}", end="")
        # closed forms
        if name.startswith("zero_atb") and case["kind"] in ("mixed", "ls"):
            assert st[0]["niter"] == 0 and np.array_equal(run[f"{key}.0"], r1) and not run[f"{key}.1"].any()
            if case["kind"] == "ls":
                assert np.array_equal(run[f"{key}.2"], r2) and not run[f"{key}.3"].any()
        if name.startswith("craig_inconsistent"):
            assert st[1]["niter"] == 0 and st[1]["inconsistent"] == 1
            assert not run[f"{key}.2"].any() and not run[f"{key}.3"].any()
        if name.startswith("minres_early"):
            tau = max(case["delta"], 1e-14)
            assert st[1]["niter"] == 1
            c = 4.0 * (1.0 if path != "batch1" else 0.25) + tau
            assert _rel(run[f"{key}.1"], r2 / c) < 1e-14, key
        if name.startswith("zero_rhs"):
            for i in range(_nvec(case["kind"])):
                assert not run[f"{key}.{i}"].any()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["loop", "step"])
def test_slot_exits_while_other_runs(exit_runs, oracle, path):
    """LSQR leaves on A r = 0 right after its first product (slot 0) while CRAIG runs 40+ iterations, and CRAIG leaves
    inconsistent in the middle of its first iteration (slot 1, pending x update) while LSQR runs on.  The running
    slot's vectors and stats are bitwise those of the run whose other right-hand side is zero, and match the oracle.

    At 41 iterations the vectors carry more roundoff than at the counts of part 1 (measured on a B200: 2.2e-11 for p2 on
    the step path, 1.4e-12 on the loop; test_gpu_variants.py documents the growth past about 26 iterations): they are
    held to RETIRE_VEC_BAR, the stats record to the usual bars."""
    run = exit_runs("step" if path == "step" else "default")
    for name, op, d, rhs, keep, ref_rhs in RETIRE:
        key, rkey = f"retire.{name}.{path}", f"retire.{name}.ref.{path}"
        assert int(run[f"{key}.persistent"]) == (1 if path == "loop" else 0)
        vec = (0, 1) if keep == 0 else (2, 3)
        for i in vec:
            assert np.array_equal(run[f"{key}.{i}"], run[f"{rkey}.{i}"]), (name, i)
        assert np.array_equal(run[f"{key}.stats"][keep], run[f"{rkey}.stats"][keep]), name
        worst = _compare(run, key, _retire_oracle(oracle, name, op, d, rhs), 4, _rhs(op, rhs), vec_bar=RETIRE_VEC_BAR)
        st = _stats(run, key)
        print(f"\n{name} {path}: status {[int(s['status']) for s in st]} niter {[int(s['niter']) for s in st]}"
              f" largest relative difference {worst:.1e}", end="")


# ---------------------------------------------------------------------------------------------------------------------
# part 4: the consumers of the flags
# ---------------------------------------------------------------------------------------------------------------------
def _fpnlp(A, delta, **kw):
    from fpsb200 import models
    from fpsb200.qdsolver import IterativeSolver
    m, n = A.shape
    nlp = models.SparseQPModel(np.ones(n), np.zeros(n), A, np.zeros(m))
    return types.SimpleNamespace(qdsolver=IterativeSolver(nlp, **kw), delta=delta, nlp=nlp,
                                 explicit_linear_constraints=False), nlp


WARN_CASES = [c["name"] for c in CASES if c["kind"] != "ldlt"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", WARN_CASES)
def test_iterative_solver_warns_exactly_on_failure(oracle, name):
    from fpsb200 import qdsolver
    case = CASE_BY_NAME[name]
    A, (r1, r2) = _case_inputs(case)
    ost = _case_oracle(oracle, case)[-1]
    fp, nlp = _fpnlp(sp.csr_matrix(A), case["delta"], **case["kw"])
    fn = {"mixed": qdsolver.solve_two_mixed, "ls": qdsolver.solve_two_least_squares,
          "extras": qdsolver.solve_two_extras}[case["kind"]]
    x = np.zeros(A.shape[1])
    fp.qdsolver.handle.set_jac_values(nlp.jac_coord(x))     # least squares / extras trust the last mixed solve's values
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        fn(fp, x, r1, r2)
    failed = [str(w.message) for w in rec if "Failed solving" in str(w.message)]
    want = sum(1 for s in ost if not s["solved"])
    assert len(failed) == want, (name, failed, ost)
    assert [s["solved"] for s in fp.qdsolver.last_stats] == [s["solved"] for s in ost]


@pytest.mark.gpu
def test_tr_fused_reports_oracle_minres_solved(oracle):
    """The feasibility step's Gauss-Newton solve at delta = 0 on a Jacobian with duplicated rows: TR_fused returns the
    oracle's MINRES `solved`, and warns exactly when it is false."""
    from fpsb200 import models
    from fpsb200.fps_solve import TR_fused
    A = models.window_random_jacobian(600, 1200, 8, w=16, seed=3).tolil()
    for i in range(0, 600, 50):
        A[i + 1] = A[i]
    A = A.tocsr()
    m, n = A.shape
    rng = np.random.default_rng(2)
    results = []
    for cz in (A @ rng.standard_normal(n), rng.standard_normal(m)):     # in the range of A, and not
        fp, nlp = _fpnlp(A, 0.0)
        ref = oracle.IterativeOracle(A).solve_two_extras(0.0, np.zeros(n), cz)[2][1]
        with warnings.catch_warnings(record=True) as rec:
            warnings.simplefilter("always")
            _, _, _, solved = TR_fused(fp.qdsolver, nlp, np.zeros(n), cz, 1e-8, 10.0, np.linalg.norm(cz))
        assert solved == ref["solved"], ref
        assert any("Fail minres" in str(w.message) for w in rec) == (not ref["solved"])
        results.append((ref["niter"], ref["status"], solved))
    print("\nTR_fused (oracle niter, status, GPU solved):", results)


if __name__ == "__main__":
    if len(sys.argv) == 4 and sys.argv[1] == "--worker":
        _worker(sys.argv[2:])
    else:
        sys.exit("usage: python tests/test_gpu_krylov_exits.py --worker <default|step> <out.npz>")
