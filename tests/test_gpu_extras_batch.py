"""GPU: batched LDLt solve_two_extras (fpsb_ldlt_batch_solve_two_extras) — CGLS and MINRES for many instances of one
Jacobian pattern in one launch.

Every (instance, method) pair runs inside one CTA with fixed-order reductions, so the batch is bitwise reproducible and
independent of the batch; against the single-instance entry (whose reductions span many CTAs) and the CPU oracle it is
held to the bars of test_gpu_krylov.py::test_solve_two_extras, and to 1e-11 at fixed iteration counts."""
import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

SQRT_EPS = float(np.sqrt(np.finfo(float).eps))
DELTAS = (0.0, SQRT_EPS, 0.25, 1e-2)
KEYS = ("niter", "solved", "inconsistent", "status", "rnorm", "arnorm", "anorm", "acond", "xnorm")


def _rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def _handle(A):
    import fpsb200
    coo = sp.coo_matrix(A)
    m, n = A.shape
    return fpsb200.B200Handle(n, m, coo.row, coo.col), coo


def _inputs(coo, n, m, ninst, rng):
    J = coo.data[None, :] * (1.0 + 0.1 * rng.standard_normal((ninst, coo.nnz)))
    delta = np.array([DELTAS[i % len(DELTAS)] for i in range(ninst)])
    return J, delta, rng.standard_normal((ninst, n)), rng.standard_normal((ninst, m))


def _st(st, i, j):
    """stats of instance i, method j (0 CGLS, 1 MINRES) as a KrylovStats.as_dict()-like dict"""
    return {k: st[k][i, j].item() for k in KEYS}


def _bars(s_cg, s_mr, u1, u2, r_cg, r_mr, ref1, ref2, niter=1, u2_bar=2e-4):
    """the bars of test_gpu_krylov.py::test_solve_two_extras between two implementations"""
    assert s_cg["solved"] == r_cg["solved"] and abs(s_cg["niter"] - r_cg["niter"]) <= niter, (s_cg, r_cg)
    assert _rel(u1, ref1) < 1e-6
    assert s_mr["solved"] == r_mr["solved"] and abs(s_mr["niter"] - r_mr["niter"]) <= niter, (s_mr, r_mr)
    assert _rel(u2, ref2) < u2_bar


def _true_residual(Ai, tau, u2, r2, s_mr):
    true_res = np.linalg.norm(Ai @ (Ai.T @ u2) + tau * u2 - r2)
    assert abs(true_res - s_mr["rnorm"]) <= 0.05 * true_res + 1e-12     # the reported rNorm is the real one
    return true_res / np.linalg.norm(r2)


def _poisson():
    from fpsb200 import models
    return models.poisson_control(20).A


# (m, n, nnz per row, window): from one constraint up to a working set that does not fit shared memory
SHAPES = [(1, 10, 9, 4), (30, 60, 5, 8), (500, 1000, 10, 32), (2000, 4000, 5, 32), "poisson"]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: s if isinstance(s, str) else "x".join(map(str, s[:2])))
def test_batch_matches_single_instance_and_oracle(oracle, shape):
    from fpsb200 import models
    if shape == "poisson":
        A = _poisson()
    else:
        m, n, k, w = shape
        A = models.window_random_jacobian(m, n, k, w=w, seed=31)
    m, n = A.shape
    H, coo = _handle(A)
    rng = np.random.default_rng(m + n)
    ninst = 40
    J, delta, r1, r2 = _inputs(coo, n, m, ninst, rng)
    u1, u2, st = H.ldlt_batch_solve_two_extras(delta, J, r1, r2)
    assert u1.shape == (ninst, m) and u2.shape == (ninst, m)
    assert all(st[k].shape == (ninst, 2) for k in KEYS)
    # MINRES on A A' of the Poisson-control operator runs about m iterations, and Krylov.jl's stopping test
    # (rNorm <= tol * Anorm * xNorm) leaves relative residuals of a few 1e-3: there the reference itself (the oracle)
    # misses the 1e-3 residual bar, and the single-instance path is up to 2 iterations and 1.4e-3 away from it (measured
    # on 80 instances).  The batch is held to that spread and to the oracle's own residual.
    bars = dict(niter=2, u2_bar=5e-3) if shape == "poisson" else {}
    lo = oracle.LDLtOracle(n, m, coo.row, coo.col, np.arange(n + m))
    for i in sorted(set(range(0, ninst, 7)) | {1, 2, 3, ninst - 1}):
        s_cg, s_mr = _st(st, i, 0), _st(st, i, 1)
        H.set_jac_values(J[i])
        v1, v2, sst = H.ldlt_solve_two_extras(delta[i], r1[i], r2[i])
        _bars(s_cg, s_mr, u1[i], u2[i], sst[0], sst[1], v1, v2, **bars)
        lo.jvals = J[i]
        o1, o2, ost = lo.solve_two_extras(delta[i], r1[i], r2[i])
        _bars(s_cg, s_mr, u1[i], u2[i], ost[0], ost[1], o1, o2, **bars)
        Ai = sp.csr_matrix((J[i], (coo.row, coo.col)), shape=(m, n))
        tau = max(delta[i], 1e-14)
        res = _true_residual(Ai, tau, u2[i], r2[i], s_mr)
        if shape == "poisson":
            assert res < 2 * np.linalg.norm(Ai @ (Ai.T @ o2) + tau * o2 - r2[i]) / np.linalg.norm(r2[i])
        else:
            assert res < 1e-3


@pytest.mark.parametrize("delta", [0.0, 0.3])
@pytest.mark.parametrize("iters", [1, 2, 3, 7, 20])
def test_fixed_iteration_parity(oracle, delta, iters):
    """Tolerances off, itmax = iters: every instance runs exactly `iters` iterations of both methods and agrees with
    the oracle's CGLS / MINRES to roundoff."""
    import fpsb200
    from fpsb200 import models
    m, n = 700, 1500
    A = models.window_random_jacobian(m, n, 9, w=24, seed=21)
    H, coo = _handle(A)
    rng = np.random.default_rng(8)
    ninst = 3
    J = coo.data[None, :] * (1.0 + 0.1 * rng.standard_normal((ninst, coo.nnz)))
    r1, r2 = rng.standard_normal((ninst, n)), rng.standard_normal((ninst, m))
    o = fpsb200.ExtrasOpts()
    o.cg_atol = o.cg_rtol = 0.0
    o.cg_itmax = iters
    o.mr_atol = o.mr_rtol = o.mr_etol = 0.0
    o.mr_conlim = 1 / SQRT_EPS
    o.mr_itmax = iters
    u1, u2, st = H.ldlt_batch_solve_two_extras(delta, J, r1, r2, opts=o)
    assert (st["niter"] == iters).all()
    tau = max(delta, 1e-14)
    for i in range(ninst):
        Ai = sp.csr_matrix((J[i], (coo.row, coo.col)), shape=(m, n))
        x1, s1 = oracle.cgls(Ai, r1[i], lam=tau, atol=0.0, rtol=0.0, itmax=iters, transpose=True)
        x2, s2 = oracle.minres_normal(Ai, r2[i], tau, 0.0, 0.0, 0.0, itmax=iters)
        assert s1["niter"] == s2["niter"] == iters
        assert _rel(u1[i], x1) < 1e-11
        assert _rel(u2[i], x2) < 1e-11


def test_independent_of_batch_position_and_buffers():
    """10 240 instances, easy (delta = 0.25) and hard (delta = 0, two nearly equal Jacobian rows), so the items run
    different iteration counts: each instance is bitwise what it is alone or elsewhere in a batch, host and device
    buffers agree bitwise, and a second run repeats the first."""
    import torch
    from fpsb200 import models
    A = models.window_random_jacobian(30, 60, 5, w=8, seed=4).tolil()
    A[7] = A[8]                                       # same pattern in both rows
    A = A.tocsr()
    H, coo = _handle(A)
    m, n = A.shape
    rng = np.random.default_rng(17)
    ninst = 10240
    J = coo.data[None, :] * (1.0 + 0.1 * rng.standard_normal((ninst, coo.nnz)))
    hard = np.arange(ninst) % 3 == 0
    J[np.ix_(hard, coo.row == 7)] = J[np.ix_(hard, coo.row == 8)] * (1.0 + 1e-7)
    delta = np.where(hard, 0.0, 0.25)
    r1, r2 = rng.standard_normal((ninst, n)), rng.standard_normal((ninst, m))
    host = H.ldlt_batch_solve_two_extras(delta, J, r1, r2)
    it = host[2]["niter"]
    assert it[hard].mean() > it[~hard].mean()         # the work items really differ
    again = H.ldlt_batch_solve_two_extras(delta, J, r1, r2)
    dev = torch.device("cuda", 0)
    t = lambda a: torch.as_tensor(a, device=dev)
    got = H.ldlt_batch_solve_two_extras(t(delta), t(J), t(r1), t(r2))
    for a, b, c in zip(host[:2], again[:2], got[:2]):
        assert np.array_equal(a, b) and np.array_equal(a, c.cpu().numpy())
    for k in KEYS:
        assert np.array_equal(host[2][k], again[2][k], equal_nan=True)
        assert np.array_equal(host[2][k], got[2][k].cpu().numpy(), equal_nan=True)
    for i in (0, 1, 4097, 7000, ninst - 1):
        one = H.ldlt_batch_solve_two_extras(delta[i:i + 1], J[i:i + 1], r1[i:i + 1], r2[i:i + 1])
        lo = max(0, i - 5)
        part = H.ldlt_batch_solve_two_extras(delta[lo:i + 9], J[lo:i + 9], r1[lo:i + 9], r2[lo:i + 9])
        for a, b, c in zip(host[:2], one[:2], part[:2]):
            assert np.array_equal(a[i], b[0]) and np.array_equal(a[i], c[i - lo]), i
        for k in KEYS:
            assert np.array_equal(host[2][k][i], one[2][k][0], equal_nan=True), (i, k)


def test_edge_instances_and_arguments():
    import torch
    from fpsb200 import models
    A = models.window_random_jacobian(40, 90, 6, w=10, seed=9)
    H, coo = _handle(A)
    m, n = A.shape
    rng = np.random.default_rng(2)
    J, delta, r1, r2 = _inputs(coo, n, m, 6, rng)
    r1[1] = 0.0                                       # CGLS: zero right-hand side
    r2[2] = 0.0                                       # MINRES: zero right-hand side
    J[3] = 0.0                                        # zero Jacobian
    delta[3] = 0.25
    u1, u2, st = H.ldlt_batch_solve_two_extras(delta, J, r1, r2)
    assert not u1[1].any() and st["status"][1, 0] == 1 and st["niter"][1, 0] == 0 and st["solved"][1, 0]
    assert not u2[2].any() and st["status"][2, 1] == 1 and st["niter"][2, 1] == 0 and st["solved"][2, 1]
    assert not u1[3].any()
    assert np.allclose(u2[3], r2[3] / 0.25, rtol=1e-12, atol=0.0)
    # no instance, host and device
    dev = torch.device("cuda", 0)
    t = lambda a: torch.as_tensor(a, device=dev)
    for args in ((delta[:0], J[:0], r1[:0], r2[:0]), (t(delta[:0]), t(J[:0]), t(r1[:0]), t(r2[:0]))):
        e1, e2, est = H.ldlt_batch_solve_two_extras(*args)
        assert tuple(e1.shape) == (0, m) and tuple(e2.shape) == (0, m)
        assert all(tuple(est[k].shape) == (0, 2) for k in KEYS)
    # wrong shapes
    bad = [(delta, J[:, :-1], r1, r2), (delta, J, r1[:, :-1], r2), (delta, J, r1, r2[:, :-1]), (delta[:-1], J, r1, r2),
           (delta, J[:-1], r1, r2), (delta, J, r1.ravel(), r2)]
    for args in bad:
        with pytest.raises(ValueError):
            H.ldlt_batch_solve_two_extras(*args)
    # a scalar delta is used for every instance
    s = H.ldlt_batch_solve_two_extras(0.25, J, r1, r2)
    v = H.ldlt_batch_solve_two_extras(np.full(6, 0.25), J, r1, r2)
    assert np.array_equal(s[0], v[0]) and np.array_equal(s[1], v[1])
    assert all(np.array_equal(s[2][k], v[2][k], equal_nan=True) for k in KEYS)


def test_leaves_factors_and_single_instance_state_alone():
    from fpsb200 import models
    A = models.window_random_jacobian(200, 400, 6, w=16, seed=12)
    H, coo = _handle(A)
    H.ldlt_analyze()
    m, n = A.shape
    rng = np.random.default_rng(3)
    J, delta, r1, r2 = _inputs(coo, n, m, 16, rng)
    r3 = rng.standard_normal((16, n))
    # single-instance state: values, factor and Krylov workspaces
    H.set_jac_values(coo.data)
    sm = H.ldlt_solve_two_mixed(1e-2, r1[0], r2[0])
    se = H.ldlt_solve_two_extras(1e-2, r1[1], r2[1])
    # Val(1) order over a batch: mixed -> least squares -> extras (another ninst) -> least squares
    H.ldlt_batch_solve_two_mixed(delta, J, r1, r2)
    l1 = H.ldlt_batch_solve_two_least_squares(r1, r3)
    H.ldlt_batch_solve_two_extras(delta[:5], J[:5], r1[:5], r2[:5])
    l2 = H.ldlt_batch_solve_two_least_squares(r1, r3)
    assert all(np.array_equal(a, b) for a, b in zip(l1, l2))
    sm2 = H.ldlt_solve_two_mixed(1e-2, r1[0], r2[0])
    se2 = H.ldlt_solve_two_extras(1e-2, r1[1], r2[1])
    assert all(np.array_equal(a, b) for a, b in zip(sm[:4], sm2[:4])) and sm[4] == sm2[4]
    assert np.array_equal(se[0], se2[0]) and np.array_equal(se[1], se2[1]) and se[2] == se2[2]


def _model(name):
    from fpsb200 import models
    if name == "mgh01feas":
        Ar = np.array
        return models.CallableModel(lambda x: 0.0, lambda x: np.zeros(2), lambda x: Ar([-x[0], 10 * (x[1] - x[0] ** 2)]),
                                    lambda x: Ar([[-1.0, 0.0], [-20 * x[0], 10.0]]), lambda x: np.zeros((2, 2)),
                                    lambda x, j: np.zeros((2, 2)) if j == 0 else Ar([[-20.0, 0.0], [0.0, 0.0]]),
                                    [-1.2, 1.0], 2, lcon=[-1.0, 0.0], ucon=[-1.0, 0.0], lin=[0], name=name)
    return models.reference_test_problem(name)


@pytest.mark.parametrize("name,explicit", [("hs8", False), ("hs61", False), ("hs26", False), ("mgh01feas", True)])
def test_model_level_batch_matches_loop(name, explicit):
    import warnings
    import fpsb200
    nlp = _model(name)
    qds = fpsb200.LDLtSolver(nlp, 0.0, explicit_linear_constraints=explicit)
    f = fpsb200.FletcherPenaltyNLP(nlp, 0.5, 0.0, 1e-3, 2, qds=qds, explicit_linear_constraints=explicit)
    rng = np.random.default_rng(11)
    n, npen = f.nvar, f.npen
    ninst = 64
    X = nlp.meta.x0[None, :] + 0.3 * rng.standard_normal((ninst, n))
    r1, r2 = rng.standard_normal((ninst, n)), rng.standard_normal((ninst, npen))
    with warnings.catch_warnings():
        warnings.simplefilter("error")                # like the single LDLt solve_two_extras: no warning
        u1, u2 = fpsb200.solve_two_extras_batch(f, X, r1, r2)
    st = qds.last_batch_stats
    assert u1.shape == (ninst, npen) and u2.shape == (ninst, npen)
    assert all(st[k].shape == (ninst, 2) for k in KEYS)
    for i in range(ninst):
        v1, v2 = fpsb200.solve_two_extras(f, X[i], r1[i], r2[i])
        _bars(_st(st, i, 0), _st(st, i, 1), u1[i], u2[i], qds.last_stats[0], qds.last_stats[1], v1, v2)
    # per-instance delta
    d = np.linspace(0.0, 0.5, ninst)
    u1, u2 = fpsb200.solve_two_extras_batch(f, X, r1, r2, delta=d)
    st = qds.last_batch_stats
    for i in (0, 31, 63):
        f.delta = d[i]
        v1, v2 = fpsb200.solve_two_extras(f, X[i], r1[i], r2[i])
        _bars(_st(st, i, 0), _st(st, i, 1), u1[i], u2[i], qds.last_stats[0], qds.last_stats[1], v1, v2)


def test_model_level_type_error_for_iterative_solver():
    import fpsb200
    nlp = _model("hs8")
    f = fpsb200.FletcherPenaltyNLP(nlp, 0.5, 0.0, 1e-3, 2, qds=fpsb200.IterativeSolver(nlp, 0.0))
    X = np.zeros((2, f.nvar))
    with pytest.raises(TypeError):
        fpsb200.solve_two_extras_batch(f, X, np.ones((2, f.nvar)), np.ones((2, f.npen)))
