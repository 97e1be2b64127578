"""GPU: batched LDLt path (fpsb_ldlt_batch_solve_two_*) — many instances of one Jacobian pattern in one call.

Every instance is checked against the single-instance path run on that instance alone (bitwise: the batch kernel runs
the same per-supernode routines in the same order) and against the CPU oracle with the bars of test_gpu_ldlt.py."""
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

SQRT_EPS = float(np.sqrt(np.finfo(float).eps))
DELTAS = (0.0, SQRT_EPS, 0.25, 1e-2)


def _rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def _ordering(kind, n, m, coo, rng):
    if kind == "amd":
        return None
    if kind == "id":
        return np.arange(n + m)
    if kind == "rand":
        return rng.permutation(n + m)
    from fpsb200.symbolic import order_dissection
    return order_dissection(n, m, coo.row, coo.col)


def _handle(A, P=None, opts=None):
    import fpsb200
    coo = sp.coo_matrix(A)
    m, n = A.shape
    H = fpsb200.B200Handle(n, m, coo.row, coo.col)
    H.ldlt_analyze(P, 0, opts)
    return H, coo


def _batch_inputs(coo, n, m, ninst, rng):
    J = coo.data[None, :] * (1.0 + 0.1 * rng.standard_normal((ninst, coo.nnz)))
    delta = np.array([DELTAS[i % len(DELTAS)] for i in range(ninst)])
    return J, delta, rng.standard_normal((ninst, n)), rng.standard_normal((ninst, m)), rng.standard_normal((ninst, n))


def _single(H, jv, delta, r1, r2, r3):
    H.set_jac_values(jv)
    mixed = H.ldlt_solve_two_mixed(delta, r1, r2)
    lsq = H.ldlt_solve_two_least_squares(r1, r3)
    return mixed, lsq


def _equal(batch, i, single):
    return all(np.array_equal(batch[k][i], single[k]) for k in range(4)) and bool(batch[4][i]) == single[4]


CASES = [(1, 10, 9, 4, "amd"), (1, 10, 9, 4, "id"), (30, 60, 5, 8, "amd"), (30, 60, 5, 8, "id"),
         (30, 60, 5, 8, "rand"), (30, 60, 5, 8, "dissection"), (500, 1000, 10, 32, "amd"),
         (500, 1000, 10, 32, "dissection"), (2000, 4000, 5, 32, "amd"), (2000, 4000, 5, 32, "dissection")]


@pytest.mark.parametrize("m,n,k,w,ordering", CASES)
def test_batch_bitwise_single_instance_and_oracle(oracle, m, n, k, w, ordering):
    from fpsb200 import models
    A = models.window_random_jacobian(m, n, k, w=w, seed=31)
    rng = np.random.default_rng(m + n)
    coo = sp.coo_matrix(A)
    H, coo = _handle(A, _ordering(ordering, n, m, coo, rng))
    ninst = 40
    J, delta, r1, r2, r3 = _batch_inputs(coo, n, m, ninst, rng)
    bm = H.ldlt_batch_solve_two_mixed(delta, J, r1, r2)
    bl = H.ldlt_batch_solve_two_least_squares(r1, r3)
    assert bm[4].all() and bl[4].all()
    assert all(a.shape == (ninst, s) for a, s in zip(bm[:4], (n, m, n, m)))
    sym = H.ldlt_symbolic()
    lo = oracle.LDLtOracle(n, m, coo.row, coo.col, sym["P"])
    for i in sorted(set(range(0, ninst, 7)) | {1, 2, 3, ninst - 1}):
        mixed, lsq = _single(H, J[i], delta[i], r1[i], r2[i], r3[i])
        assert _equal(bm, i, mixed), f"mixed, instance {i}"
        assert _equal(bl, i, lsq), f"least squares, instance {i}"
        # oracle bars of test_gpu_ldlt.py
        o = lo.solve_two_mixed(J[i], delta[i], r1[i], r2[i])
        _, oD = lo.numeric()
        perturbed = bool(np.any(np.abs(np.abs(oD) - SQRT_EPS) < 1e-12))
        bar = 1e-5 if perturbed else 1e-8
        for a, b in zip((bm[0][i], bm[1][i], bm[2][i], bm[3][i]), o[:4]):
            assert _rel(a, b) < bar
        if not perturbed:
            Ai = sp.csr_matrix((J[i], (coo.row, coo.col)), shape=(m, n))
            e1 = np.r_[bm[0][i] + Ai.T @ bm[1][i] - r1[i], Ai @ bm[0][i] - delta[i] * bm[1][i]]
            e2 = np.r_[bm[2][i] + Ai.T @ bm[3][i], Ai @ bm[2][i] - delta[i] * bm[3][i] - r2[i]]
            assert np.linalg.norm(e1) / np.linalg.norm(r1[i]) < 1e-10
            assert np.linalg.norm(e2) / np.linalg.norm(r2[i]) < 1e-10
        o = lo.solve_two_least_squares(r1[i], r3[i])
        for a, b in zip((bl[0][i], bl[1][i], bl[2][i], bl[3][i]), o[:4]):
            assert _rel(a, b) < bar


def test_batch_healthy_rank_deficient_and_failing_instances():
    """Duplicated Jacobian rows with delta = 0 get regularised pivots with the default options (bitwise equal to the
    single path); with regularisation off an instance with a zero Jacobian and delta = 0 (exactly zero pivots) fails
    alone and returns its right-hand sides."""
    import fpsb200
    from fpsb200 import models
    A = models.window_random_jacobian(60, 120, 6, w=10, seed=4).tolil()
    A[7] = A[8]                                       # same pattern in both rows
    A = A.tocsr()
    coo = sp.coo_matrix(A)
    rng = np.random.default_rng(8)
    ninst = 6
    J = coo.data[None, :] * (1.0 + 0.1 * rng.standard_normal((ninst, coo.nnz)))
    J[2, coo.row == 7] = J[2, coo.row == 8]           # instance 2: rows 7 and 8 equal (rank deficient)
    J[4] = 0.0                                        # instance 4: zero Jacobian
    delta = np.array([0.0, 1e-2, 0.0, 0.25, 0.0, SQRT_EPS])
    r1, r2, r3 = rng.standard_normal((ninst, 120)), rng.standard_normal((ninst, 60)), rng.standard_normal((ninst, 120))
    # regularisation on: every instance factorises, the regularised ones equal to the single path
    H, _ = _handle(A)
    got = H.ldlt_batch_solve_two_mixed(delta, J, r1, r2)
    assert got[4].all()
    for i in range(ninst):
        H.set_jac_values(J[i])
        assert _equal(got, i, H.ldlt_solve_two_mixed(delta[i], r1[i], r2[i])), i
        if i in (2, 4):
            _, D = H.ldlt_get_factor()
            assert np.any(np.abs(np.abs(D) - SQRT_EPS) < 1e-12)      # a pivot was regularised
    # regularisation off: only instance 4 fails
    o = fpsb200.LdltOpts()
    o.ldlt_tol, o.ldlt_r1, o.ldlt_r2 = 0.0, 0.0, 0.0
    H, _ = _handle(A, None, o)
    keep = [0, 1, 3, 4, 5]
    p1, q1, p2, q2, ok = H.ldlt_batch_solve_two_mixed(delta[keep], J[keep], r1[keep], r2[keep])
    assert list(ok) == [True, True, True, False, True]
    assert np.array_equal(p1[3], r1[4]) and not q1[3].any() and not p2[3].any() and np.array_equal(q2[3], r2[4])
    for k, i in enumerate(keep):
        H.set_jac_values(J[i])
        assert _equal((p1, q1, p2, q2, ok), k, H.ldlt_solve_two_mixed(delta[i], r1[i], r2[i])), i
    P1, Q1, P2, Q2, ok2 = H.ldlt_batch_solve_two_least_squares(r1[keep], r3[keep])
    assert np.array_equal(ok2, ok)
    assert np.array_equal(P1[3], r1[4]) and np.array_equal(P2[3], r3[4]) and not Q1[3].any() and not Q2[3].any()


def test_batch_factor_reuse_and_state():
    import fpsb200
    from fpsb200 import models
    A = models.window_random_jacobian(200, 400, 6, w=16, seed=12)
    H, coo = _handle(A)
    rng = np.random.default_rng(3)
    ninst = 16
    J, delta, r1, r2, r3 = _batch_inputs(coo, 400, 200, ninst, rng)
    # least squares before any batched mixed call
    with pytest.raises(fpsb200.FpsbError, match="FPSB_ESTATE"):
        H.ldlt_batch_solve_two_least_squares(r1, r3)
    # the single-instance factor is left alone by batched calls
    H.set_jac_values(coo.data)
    H.ldlt_solve_two_mixed(1e-2, r1[0], r2[0])
    before = H.ldlt_solve_two_least_squares(r1[1], r3[1])
    H.ldlt_batch_solve_two_mixed(delta, J, r1, r2)
    bl = H.ldlt_batch_solve_two_least_squares(r1, r3)
    after = H.ldlt_solve_two_least_squares(r1[1], r3[1])
    assert all(np.array_equal(a, b) for a, b in zip(before[:4], after[:4])) and before[4] == after[4]
    # another ninst
    with pytest.raises(fpsb200.FpsbError, match="FPSB_ESTATE"):
        H.ldlt_batch_solve_two_least_squares(r1[:5], r3[:5])
    # per instance: single mixed followed by single least squares
    for i in range(ninst):
        _, lsq = _single(H, J[i], delta[i], r1[i], r2[i], r3[i])
        assert _equal(bl, i, lsq), i


def test_batch_device_and_host_buffers_and_sizes():
    import torch
    from fpsb200 import models
    A = models.window_random_jacobian(3, 10, 4, w=4, seed=2)
    H, coo = _handle(A)
    rng = np.random.default_rng(5)
    ninst = 10240                                     # many times the grid
    J, delta, r1, r2, r3 = _batch_inputs(coo, 10, 3, ninst, rng)
    host = H.ldlt_batch_solve_two_mixed(delta, J, r1, r2)
    hl = H.ldlt_batch_solve_two_least_squares(r1, r3)
    dev = torch.device("cuda", 0)
    t = lambda a: torch.as_tensor(a, device=dev)
    got = H.ldlt_batch_solve_two_mixed(t(delta), t(J), t(r1), t(r2))
    gl = H.ldlt_batch_solve_two_least_squares(t(r1), t(r3))
    for a, b in zip(host, got):
        assert np.array_equal(a, b.cpu().numpy())
    for a, b in zip(hl, gl):
        assert np.array_equal(a, b.cpu().numpy())
    assert host[4].all()
    for i in (0, 4097, ninst - 1):
        H.set_jac_values(J[i])
        assert _equal(host, i, H.ldlt_solve_two_mixed(delta[i], r1[i], r2[i]))
    # a scalar delta is used for every instance
    s = H.ldlt_batch_solve_two_mixed(0.25, J[:3], r1[:3], r2[:3])
    v = H.ldlt_batch_solve_two_mixed(np.full(3, 0.25), J[:3], r1[:3], r2[:3])
    assert all(np.array_equal(a, b) for a, b in zip(s, v))
    # one instance, no instance
    one = H.ldlt_batch_solve_two_mixed(delta[:1], J[:1], r1[:1], r2[:1])
    assert all(np.array_equal(a[0], b[0]) for a, b in zip(one, host))
    for args in ((delta[:0], J[:0], r1[:0], r2[:0]), (t(delta[:0]), t(J[:0]), t(r1[:0]), t(r2[:0]))):
        out = H.ldlt_batch_solve_two_mixed(*args)
        assert [tuple(a.shape) for a in out] == [(0, 10), (0, 3), (0, 10), (0, 3), (0,)]
    # reproducible from run to run
    again = H.ldlt_batch_solve_two_mixed(delta, J, r1, r2)
    assert all(np.array_equal(a, b) for a, b in zip(host, again))


@pytest.mark.parametrize("name,explicit", [("hs8", False), ("hs61", False), ("hs26", False), ("mgh01feas", True)])
def test_model_level_batch_equals_loop(name, explicit):
    import fpsb200
    from fpsb200 import models
    if name == "mgh01feas":
        Ar = np.array
        nlp = models.CallableModel(lambda x: 0.0, lambda x: np.zeros(2), lambda x: Ar([-x[0], 10 * (x[1] - x[0] ** 2)]),
                                   lambda x: Ar([[-1.0, 0.0], [-20 * x[0], 10.0]]), lambda x: np.zeros((2, 2)),
                                   lambda x, j: np.zeros((2, 2)) if j == 0 else Ar([[-20.0, 0.0], [0.0, 0.0]]),
                                   [-1.2, 1.0], 2, lcon=[-1.0, 0.0], ucon=[-1.0, 0.0], lin=[0], name=name)
    else:
        nlp = models.reference_test_problem(name)
    qds = fpsb200.LDLtSolver(nlp, 0.0, explicit_linear_constraints=explicit)
    f = fpsb200.FletcherPenaltyNLP(nlp, 0.5, 0.0, 1e-3, 2, qds=qds, explicit_linear_constraints=explicit)
    rng = np.random.default_rng(11)
    n, npen = f.nvar, f.npen
    X = nlp.meta.x0[None, :] + 0.3 * rng.standard_normal((64, n))
    r1, r2, r3 = rng.standard_normal((64, n)), rng.standard_normal((64, npen)), rng.standard_normal((64, n))
    got = fpsb200.solve_two_mixed_batch(f, X, r1, r2)
    gl = fpsb200.solve_two_least_squares_batch(f, X, r1, r3)
    for i in range(64):
        ref = fpsb200.solve_two_mixed(f, X[i], r1[i], r2[i])
        assert all(np.array_equal(a[i], b) for a, b in zip(got, ref)), i
        ref = fpsb200.solve_two_least_squares(f, X[i], r1[i], r3[i])
        assert all(np.array_equal(a[i], b) for a, b in zip(gl, ref)), i
    # per-instance delta
    d = np.linspace(0.0, 0.5, 64)
    got = fpsb200.solve_two_mixed_batch(f, X, r1, r2, delta=d)
    for i in (0, 31, 63):
        f.delta = d[i]
        ref = fpsb200.solve_two_mixed(f, X[i], r1[i], r2[i])
        assert all(np.array_equal(a[i], b) for a, b in zip(got, ref)), i


def test_model_level_warnings_and_type():
    import fpsb200
    from fpsb200 import models
    A = np.array
    # c(x) = [x1, x1 x2]: J(0, 1) = [1 0; 1 0] (exactly singular K with delta = 0 and no regularisation)
    nlp = models.CallableModel(lambda x: 0.0, lambda x: np.zeros(2), lambda x: A([x[0], x[0] * x[1]]),
                               lambda x: A([[1.0, 0.0], [x[1], x[0]]]), lambda x: np.zeros((2, 2)),
                               lambda x, j: np.zeros((2, 2)) if j == 0 else A([[0.0, 1.0], [1.0, 0.0]]),
                               [0.0, 1.0], 2, name="dup")
    # natural ordering: the variables are eliminated before the constraint rows (whose diagonal is -delta = 0)
    qds = fpsb200.LDLtSolver(nlp, 0.0, ldlt_tol=0.0, ldlt_r1=0.0, ldlt_r2=0.0, P=np.arange(4))
    f = fpsb200.FletcherPenaltyNLP(nlp, 0.5, 0.0, 0.0, 2, qds=qds)
    X = A([[0.0, 1.0], [1.0, 2.0], [0.0, 1.0]])
    r1, r2 = np.ones((3, 2)), np.ones((3, 2))
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        p1, q1, p2, q2 = fpsb200.solve_two_mixed_batch(f, X, r1, r2)
    assert sum("failed _factorization" in str(x.message) for x in w) == 2
    assert np.array_equal(p1[0], r1[0]) and np.array_equal(q2[2], r2[2])
    fi = fpsb200.FletcherPenaltyNLP(nlp, 0.5, 0.0, 0.0, 2, qds=fpsb200.IterativeSolver(nlp, 0.0))
    with pytest.raises(TypeError):
        fpsb200.solve_two_mixed_batch(fi, X, r1, r2)
    with pytest.raises(TypeError):
        fpsb200.solve_two_least_squares_batch(fi, X, r1, r1)


@pytest.mark.parametrize("n,m", [(10, 3), (20, 12), (3, 2)])
def test_batch_agrees_with_dense_batch(n, m):
    import fpsb200
    rng = np.random.default_rng(n + m)
    ninst = 300
    A = rng.standard_normal((ninst, m, n))
    rows, cols = np.meshgrid(np.arange(m), np.arange(n), indexing="ij")
    H = fpsb200.B200Handle(n, m, rows.ravel(), cols.ravel())
    H.ldlt_analyze(np.arange(n + m))
    r1, r2 = rng.standard_normal((ninst, n)), rng.standard_normal((ninst, m))
    got = H.ldlt_batch_solve_two_mixed(1e-2, A.reshape(ninst, -1), r1, r2)
    ref = fpsb200.batch_solve_two(A, 1e-2, r1, r2)
    assert got[4].all() and ref[4].all()
    for a, b in zip(got[:4], ref[:4]):
        for i in range(ninst):
            assert _rel(a[i], b[i]) < 1e-8
