"""GPU: BatchFletcherPenaltyNLP (K points of one model in lock-step), the batched Jacobian products and the batched
Steihaug–Toint CG, against a loop of DeviceFletcherPenaltyNLP / _steihaug_device and the numpy _steihaug."""
import ctypes as C
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu


def _qp(n=200, m=80, seed=7):
    from fpsb200 import models
    return models.sparse_qp(n, m, nnz_per_row=6, w=24, seed=seed)


def _curved(n=200, m=80, seed=7):
    from fpsb200 import models
    qp = _qp(n, m, seed)
    rng = np.random.default_rng(seed + 1)
    return models.CurvedQPModel(qp.Q, qp.q, qp.A, qp.b, 0.3 * rng.standard_normal(m))


def _bits(t):
    a = np.atleast_1d(t.detach().cpu().numpy())
    return a.view(np.int64) if a.dtype == np.float64 else a


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _inputs(K, n, seed=3):
    import torch
    rng = np.random.default_rng(seed)
    X = torch.tensor(0.5 * rng.standard_normal((K, n)), device="cuda")
    V = torch.tensor(rng.standard_normal((K, n)), device="cuda")
    sigma = 1.0 + 9.0 * rng.random(K)
    delta = np.where(rng.random(K) < 0.5, 0.0, 1e-2)
    return X, V, sigma, delta


def _csr_cons_qp(qp):
    """DeviceSparseQP whose single `cons` is the batched CSR-order product of one row: the stock `cons` goes through the
    tiled SELL-32 product, which rounds A x differently in the last bits"""
    import fpsb200

    class CsrCons(fpsb200.DeviceSparseQP):
        def cons(self, x):
            return self._op().batch_jprod(self._vals, x[None])[0] - self.b

    return CsrCons(qp)


@pytest.mark.parametrize("K", [1, 7, 300])
def test_batch_is_bitwise_the_single_evaluator(K):
    """rho = eta = 0: ys, gs, v, w, grad and the Val(2) hprod bitwise equal to DeviceFletcherPenaltyNLP per instance on
    the same c(x) (the batched LDLt solves are bitwise the single path and the combinations keep its operation order);
    obj to 1e-13 (its sums run in one CTA instead of across the grid).  Against the stock model, whose c(x) comes from
    the SELL-32 product, everything agrees to 1e-13."""
    import torch
    import fpsb200
    qp = _qp()
    dm = fpsb200.DeviceSparseQP(qp)
    X, V, sigma, delta = _inputs(K, qp.meta.nvar)
    B = fpsb200.BatchFletcherPenaltyNLP(dm, sigma, 0.0, delta, 2, qds=fpsb200.LDLtSolver(dm, 0.0, ordering="amd"))
    phi, g = B.objgrad(X)
    Hv = B.hprod(X, V, obj_weight=0.7)
    rel = lambda a, b: float(torch.linalg.norm(a - b) / max(float(torch.linalg.norm(b)), 1e-300))
    for model, bitwise in ((_csr_cons_qp(qp), True), (dm, False)):
        qs = fpsb200.LDLtSolver(model, 0.0, ordering="amd")
        for i in range(K):
            S = fpsb200.DeviceFletcherPenaltyNLP(model, float(sigma[i]), 0.0, float(delta[i]), 2, qds=qs)
            f = S.obj(X[i])
            pairs = [(B.ys[i], S.ys), (B.gs[i], S.gs), (B.v[i], S.v), (B.w[i], S.w), (g[i], S.grad(X[i])),
                     (Hv[i], S.hprod(X[i], V[i], obj_weight=0.7))]
            for k, (a, b) in enumerate(pairs):
                assert (_same(a, b) if bitwise else rel(a, b) <= 1e-13), (i, k, bitwise)
            scale = max(1.0, abs(S.fx) + abs(float(S.cx @ S.ys)))
            assert abs(float(phi[i]) - f) <= 1e-13 * scale, i


def test_batch_with_penalty_and_proximal_terms():
    """rho > 0 and eta > 0 per instance (some 0): the CSR-order batched Jacobian products against the SELL-order single
    ones, to 1e-13."""
    import torch
    import fpsb200
    qp = _qp()
    dm = fpsb200.DeviceSparseQP(qp)
    K, n = 7, qp.meta.nvar
    X, V, sigma, delta = _inputs(K, n, seed=5)
    rng = np.random.default_rng(6)
    rho = np.array([0.0, 2.0, 0.5, 0.0, 3.0, 1.0, 2.0])
    eta = np.array([0.3, 0.0, 1.0, 0.0, 0.2, 0.7, 1.5])
    xk = torch.tensor(rng.standard_normal((K, n)), device="cuda")
    B = fpsb200.BatchFletcherPenaltyNLP(dm, sigma, rho, delta, 2, qds=fpsb200.LDLtSolver(dm, 0.0, ordering="amd"))
    B.eta, B.xk = eta, xk
    phi, g = B.objgrad(X)
    Hv = B.hprod(X, V)
    qs = fpsb200.LDLtSolver(dm, 0.0, ordering="amd")
    rel = lambda a, b: float(torch.linalg.norm(a - b) / max(float(torch.linalg.norm(b)), 1e-300))
    for i in range(K):
        S = fpsb200.DeviceFletcherPenaltyNLP(dm, float(sigma[i]), float(rho[i]), float(delta[i]), 2, qds=qs)
        S.eta, S.xk = float(eta[i]), xk[i].clone()
        f = S.obj(X[i])
        scale = max(1.0, abs(S.fx) + abs(float(S.cx @ S.ys)) + rho[i] / 2 * float(S.cx @ S.cx))
        assert abs(float(phi[i]) - f) <= 1e-13 * scale, i
        assert rel(g[i], S.grad(X[i])) <= 1e-13, i
        assert rel(Hv[i], S.hprod(X[i], V[i])) <= 1e-13, i


def test_val1_hprod_matches_the_single_evaluator():
    import torch
    import fpsb200
    cm = _curved()
    dcm = fpsb200.DeviceCurvedQP(cm)
    K = 5
    X, V, sigma, delta = _inputs(K, cm.meta.nvar, seed=9)
    rho = np.array([0.0, 2.0, 0.0, 1.0, 0.0])
    B1 = fpsb200.BatchFletcherPenaltyNLP(dcm, sigma, rho, delta, 1, qds=fpsb200.LDLtSolver(dcm, 0.0, ordering="amd"))
    B2 = fpsb200.BatchFletcherPenaltyNLP(dcm, sigma, rho, delta, 2, qds=B1.qdsolver)
    H1 = B1.hprod(X, V, obj_weight=0.5)
    H2 = B2.hprod(X, V, obj_weight=0.5)
    qs = fpsb200.LDLtSolver(dcm, 0.0, ordering="amd")
    rel = lambda a, b: float(torch.linalg.norm(a - b) / max(float(torch.linalg.norm(b)), 1e-300))
    for i in range(K):
        S = fpsb200.DeviceFletcherPenaltyNLP(dcm, float(sigma[i]), float(rho[i]), float(delta[i]), 1, qds=qs)
        ref = S.hprod(X[i], V[i], obj_weight=0.5)
        assert rel(H1[i], ref) < 1e-7, i
        assert rel(H2[i], ref) > 1e-4, i


def test_instances_do_not_depend_on_the_batch():
    """An instance's obj, grad, both hprods and CG result are bitwise the same alone, in a batch of 300, at another
    position after a permutation, and on a repeated call."""
    import torch
    import fpsb200
    from fpsb200.fps_solve import _steihaug_batch
    cm = _curved()
    dcm = fpsb200.DeviceCurvedQP(cm)
    K = 300
    X, V, sigma, delta = _inputs(K, cm.meta.nvar, seed=11)
    rho = np.where(np.arange(K) % 3 == 0, 1.5, 0.0)

    def run(idx):
        qs = fpsb200.LDLtSolver(dcm, 0.0, ordering="amd")
        out = {}
        for approx in (1, 2):
            B = fpsb200.BatchFletcherPenaltyNLP(dcm, sigma[idx], rho[idx], delta[idx], approx, qds=qs)
            Xi, Vi = X[idx].contiguous(), V[idx].contiguous()
            phi, g = B.objgrad(Xi)
            out[f"obj"], out["grad"] = phi, g
            out[f"hprod{approx}"] = B.hprod(Xi, Vi)
            out[f"hprod{approx}_again"] = B.hprod(Xi, Vi)
            if approx == 2:
                S, pred, nprod, flags = _steihaug_batch(B.handle, lambda D: B.hprod(Xi, D), g, 0.5, 1e-8, 30)
                out["cg_s"], out["cg_pred"], out["cg_nprod"] = S, pred, nprod
        return out

    full = run(np.arange(K))
    perm = np.random.default_rng(2).permutation(K)
    permuted = run(perm)
    where = {int(p): k for k, p in enumerate(perm)}
    for i in (0, 1, 2, 150, 299):
        alone = run(np.array([i]))
        for key in full:
            assert _same(full[key][i], alone[key][0]), (key, i)
            assert _same(full[key][i], permuted[key][where[i]]), (key, i)
    for key in ("hprod1", "hprod2"):
        assert _same(full[key], full[key + "_again"])


def test_memo_keys_and_resolves():
    import torch
    import fpsb200
    qp = _qp()
    dm = fpsb200.DeviceSparseQP(qp)
    K = 6
    X, V, sigma, delta = _inputs(K, qp.meta.nvar, seed=13)
    B = fpsb200.BatchFletcherPenaltyNLP(dm, sigma, 0.0, delta, 2, qds=fpsb200.LDLtSolver(dm, 0.0, ordering="amd"))
    phi = B.obj(X)
    L = fpsb200._lib.lib()
    for i in range(K):
        k = C.c_uint64()
        assert L.fpsb_fp_hash(B.handle.h, C.c_void_p(X[i].data_ptr()), C.byref(k)) == 0
        assert int(B.keys[i]) & (2 ** 64 - 1) == k.value
    n0 = B.handle.launch_count()
    phi2 = B.obj(X)
    assert B.handle.launch_count() - n0 <= 2                 # the batched hash and the batched obj, no solve
    assert _same(phi, phi2)
    g, Hv = B.grad(X), B.hprod(X, V)
    ys = B.ys.clone()
    X2 = X.clone()
    X2[3] += 0.25
    phi3, g3, Hv3 = B.obj(X2), B.grad(X2), B.hprod(X2, V)
    assert not _same(phi3[3], phi[3])
    for i in (0, 1, 2, 4, 5):
        assert _same(phi3[i], phi[i]) and _same(g3[i], g[i]) and _same(Hv3[i], Hv[i]) and _same(B.ys[i], ys[i])


def test_failing_factorisation_warns_per_instance():
    import torch
    import fpsb200

    class ZeroJac(fpsb200.DeviceSparseQP):
        """rows whose first entry is 123 get a zero Jacobian: with delta = 0 and no regularisation the factorisation
        meets exact zero pivots"""
        def jac_coord_batch(self, X):
            return self._vals * (X[:, :1] != 123.0)

    qp = _qp()
    dm = ZeroJac(qp)
    K = 5
    X, V, sigma, _ = _inputs(K, qp.meta.nvar, seed=17)
    mk = lambda: fpsb200.LDLtSolver(dm, 0.0, ordering="amd", ldlt_tol=0.0, ldlt_r1=0.0, ldlt_r2=0.0)
    B = fpsb200.BatchFletcherPenaltyNLP(dm, sigma, 0.0, 0.0, 2, qds=mk())
    g0 = B.grad(X)
    Xf = X.clone()
    Xf[1, 0] = 123.0
    Xf[3, 0] = 123.0
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        g1 = B.grad(Xf)
    assert sum("failed _factorization" in str(x.message) for x in w) == 2
    for i in (0, 2, 4):
        assert _same(g1[i], g0[i])


def test_batch_jacobian_products():
    import torch
    import fpsb200
    qp = _qp(300, 120)
    A = sp.csr_matrix(qp.A)
    rows, cols = qp.jac_structure()
    H = fpsb200.B200Handle(300, 120, rows, cols)
    rng = np.random.default_rng(21)
    K = 9
    J = qp._vals[None, :] * (1.0 + 0.1 * rng.standard_normal((K, len(rows))))
    Vn, Un = rng.standard_normal((K, 300)), rng.standard_normal((K, 120))
    Jd, Vd, Ud = (torch.tensor(a, device="cuda") for a in (J, Vn, Un))
    # state of the handle before: single values, batched factors
    H.set_jac_values(qp._vals)
    H.ldlt_analyze()
    H.ldlt_batch_solve_two_mixed(1e-2, Jd, Vd, Ud)
    before_j = H.jprod(Vd[0]).clone()
    before_ls = H.ldlt_batch_solve_two_least_squares(Vd, Vd)
    AV, ATU = H.batch_jprod(Jd, Vd), H.batch_jtprod(Jd, Ud)
    for i in range(K):
        Ai = sp.csr_matrix((J[i], (rows, cols)), shape=(120, 300))
        assert np.linalg.norm(AV[i].cpu().numpy() - Ai @ Vn[i]) <= 1e-14 * np.linalg.norm(Ai @ Vn[i])
        assert np.linalg.norm(ATU[i].cpu().numpy() - Ai.T @ Un[i]) <= 1e-14 * np.linalg.norm(Ai.T @ Un[i])
    H2 = fpsb200.B200Handle(300, 120, rows, cols)
    H2.set_jac_values(J[2])
    assert torch.linalg.norm(AV[2] - H2.jprod(Vd[2])) <= 1e-14 * torch.linalg.norm(AV[2])
    assert torch.linalg.norm(ATU[2] - H2.jtprod(Ud[2])) <= 1e-14 * torch.linalg.norm(ATU[2])
    # shared values (stride 0) are bitwise the replicated ones
    shared = torch.tensor(qp._vals, device="cuda")
    assert _same(H.batch_jprod(shared, Vd), H.batch_jprod(shared.expand(K, -1).contiguous(), Vd))
    assert _same(H.batch_jtprod(shared, Ud), H.batch_jtprod(shared.expand(K, -1).contiguous(), Ud))
    # the single values and the batched factors are untouched
    assert _same(H.jprod(Vd[0]), before_j)
    after_ls = H.ldlt_batch_solve_two_least_squares(Vd, Vd)
    for a, b in zip(before_ls[:4], after_ls[:4]):
        assert _same(a, b)
    # shapes
    with pytest.raises(ValueError):
        H.batch_jprod(Jd, Ud)
    with pytest.raises(ValueError):
        H.batch_jtprod(Jd[:2], Ud)
    assert H.batch_jprod(Jd[:0], Vd[:0]).shape == (0, 120)


def _quadratics(K, n, seed):
    """diag + low-rank quadratics, one per instance; some with negative diagonal entries"""
    rng = np.random.default_rng(seed)
    diag = 1.0 + 9.0 * rng.random((K, n))
    U = rng.standard_normal((K, n, 3)) / np.sqrt(n)
    G = rng.standard_normal((K, n))
    return diag, U, G


@pytest.mark.parametrize("masked", [False, True])
def test_batched_cg_against_the_host_loop(masked):
    import torch
    import fpsb200
    from fpsb200.fps_solve import _steihaug, _steihaug_batch
    K, n = 8, 2000
    diag, U, G = _quadratics(K, n, 31)
    diag[2, ::7] = -0.5                   # negative curvature
    diag[5, ::11] = -0.5
    G[6] = 0.0                            # zero gradient
    radius = np.array([1e6, 0.5, 50.0, 1e6, 0.3, 40.0, 1.0, 1e6])
    free = (np.random.default_rng(3).random((K, n)) > 0.3) * 1.0 if masked else None
    tol = 1e-8 * np.maximum(np.linalg.norm(G, axis=1), 1.0)
    dd, dU = torch.tensor(diag, device="cuda"), torch.tensor(U, device="cuda")
    hv = lambda D: dd * D + torch.einsum("kij,kj->ki", dU, torch.einsum("kij,ki->kj", dU, D))
    H = fpsb200.B200Handle(n, 1, np.array([0]), np.array([0]))
    fd = None if free is None else torch.tensor(free, device="cuda")
    S, pred, nprod, flags = _steihaug_batch(H, hv, torch.tensor(G, device="cuda"), torch.tensor(radius, device="cuda"),
                                            torch.tensor(tol, device="cuda"), 200, fd)
    S, pred, nprod, flags = S.cpu().numpy(), pred.cpu().numpy(), nprod.cpu().numpy(), flags.cpu().numpy()
    kinds = set()
    for i in range(K):
        hv_h = lambda v, i=i: diag[i] * v + U[i] @ (U[i].T @ v)
        s0, pred0, np0 = _steihaug(hv_h, G[i], radius[i], tol[i], 200, None if free is None else free[i])
        assert nprod[i] == np0, i
        on_sphere = abs(np.linalg.norm(s0) - radius[i]) <= 1e-8 * radius[i]
        kind = 2 if np0 == 0 else (1 if on_sphere else 2)
        assert flags[i] == kind, i
        kinds.add((kind, np0 == 0))
        if np0 == 0:
            assert not S[i].any() and pred[i] == 0.0
            continue
        assert np.linalg.norm(S[i] - s0) <= 1e-10 * np.linalg.norm(s0), i
        assert abs(pred[i] - pred0) <= 1e-10 * abs(pred0), i
        if kind == 1:
            assert abs(np.linalg.norm(S[i]) - radius[i]) <= 1e-10 * radius[i], i
        if free is not None:
            assert not S[i][free[i] == 0.0].any()
    assert kinds == {(1, False), (2, False), (2, True)}


def test_batched_cg_freezes_finished_instances():
    """Through the C ABI: the count returned by every step equals the instances with flag 0, and an instance's s, st
    and nprod stay bitwise unchanged from the step it finishes on."""
    import torch
    import fpsb200
    K, n = 6, 1000
    diag, U, G = _quadratics(K, n, 41)
    diag[1, ::5] = -1.0
    radius = torch.tensor([1e6, 30.0, 0.2, 1e6, 0.5, 1e6], device="cuda")
    tol = torch.full((K,), 1e-9, device="cuda", dtype=torch.float64)
    dd, dU = torch.tensor(diag, device="cuda"), torch.tensor(U, device="cuda")
    hv = lambda D: dd * D + torch.einsum("kij,kj->ki", dU, torch.einsum("kij,ki->kj", dU, D))
    H = fpsb200.B200Handle(n, 1, np.array([0]), np.array([0]))
    L = fpsb200._lib.lib()
    Gd = torch.tensor(G, device="cuda")
    S, R, D = torch.empty_like(Gd), torch.empty_like(Gd), torch.empty_like(Gd)
    st = torch.zeros((K, 5), dtype=torch.float64, device="cuda")
    nprod = torch.zeros(K, dtype=torch.int32, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    nact = C.c_int32()
    assert L.fpsb_trcg_batch_init(H.h, C.c_int64(K), p(Gd), None, p(tol), p(S), p(R), p(D), p(st), p(nprod),
                                  C.byref(nact)) == 0
    assert nact.value == K
    frozen = {}
    for _ in range(100):
        Hd = hv(D)
        assert L.fpsb_trcg_batch_step(H.h, C.c_int64(K), p(Hd), None, p(radius), p(tol), p(S), p(R), p(D), p(st),
                                      p(nprod), C.byref(nact)) == 0
        flags = st[:, 4].cpu().numpy()
        assert nact.value == int((flags == 0).sum())
        for i, (a, b, c) in frozen.items():
            assert _same(S[i], a) and _same(st[i], b) and int(nprod[i]) == c
        for i in np.nonzero(flags)[0]:
            if i not in frozen:
                frozen[int(i)] = (S[i].clone(), st[i].clone(), int(nprod[i]))
        if nact.value == 0:
            break
    assert nact.value == 0 and len(frozen) == K
    assert len({v[2] for v in frozen.values()}) > 1              # the instances finished at different steps
    assert L.fpsb_trcg_batch_step(H.h, C.c_int64(-1), None, None, None, None, None, None, None, None, None,
                                  C.byref(nact)) == -1


def test_batched_cg_drives_the_batched_evaluator():
    """_steihaug_batch with hv = BatchFletcherPenaltyNLP.hprod (Val(2), rho = 0) against _steihaug_device driving the
    single evaluator per instance: same product counts, steps to 1e-10."""
    import torch
    import fpsb200
    from fpsb200.fps_solve import _steihaug_batch, _steihaug_device
    qp = _qp()
    dm = fpsb200.DeviceSparseQP(qp)
    K = 4
    X, _, sigma, delta = _inputs(K, qp.meta.nvar, seed=23)
    radius = np.array([1e3, 0.05, 1.0, 1e3])
    B = fpsb200.BatchFletcherPenaltyNLP(dm, sigma, 0.0, delta, 2, qds=fpsb200.LDLtSolver(dm, 0.0, ordering="amd"))
    G = B.grad(X)
    tol = 1e-8 * torch.linalg.norm(G, dim=1)
    S, pred, nprod, _ = _steihaug_batch(B.handle, lambda D: B.hprod(X, D), G, torch.tensor(radius, device="cuda"), tol, 60)
    qs = fpsb200.LDLtSolver(dm, 0.0, ordering="amd")
    for i in range(K):
        Sg = fpsb200.DeviceFletcherPenaltyNLP(dm, float(sigma[i]), 0.0, float(delta[i]), 2, qds=qs)
        gi = Sg.grad(X[i])
        s0, pred0, np0 = _steihaug_device(qs.handle, lambda d: Sg.hprod(X[i], d), gi, float(radius[i]), float(tol[i]), 60)
        assert int(nprod[i]) == np0, i
        assert float(torch.linalg.norm(S[i] - s0)) <= 1e-10 * float(torch.linalg.norm(s0)), i
        assert abs(float(pred[i]) - pred0) <= 1e-10 * abs(pred0), i


def test_misuse_and_edges():
    import torch
    import fpsb200
    qp = _qp()
    dm = fpsb200.DeviceSparseQP(qp)
    n = qp.meta.nvar
    B = fpsb200.BatchFletcherPenaltyNLP(dm, 1.0, 0.0, 0.0, 2)
    H = B.handle
    n0 = H.launch_count()
    E = torch.empty((0, n), dtype=torch.float64, device="cuda")
    assert B.obj(E).shape == (0,) and B.grad(E).shape == (0, n) and B.hprod(E, E).shape == (0, n)
    assert H.launch_count() == n0
    L = fpsb200._lib.lib()
    assert L.fpsb_fp_batch_ptv(H.h, C.c_int64(-1), None, None, None) == -1
    assert L.fpsb_batch_jprod(H.h, C.c_int64(-1), None, C.c_int64(0), None, None) == -1
    assert L.fpsb_fp_batch_ptv(H.h, C.c_int64(0), None, None, None) == 0
    X = torch.zeros((3, n), dtype=torch.float64, device="cuda")
    d = C.c_void_p(X.data_ptr())
    # rho without J'c / Hcv and J'Jv
    assert L.fpsb_fp_batch_grad(H.h, C.c_int64(3), d, d, None, d, d, d, d, None, None, None, d) == -1
    assert L.fpsb_fp_batch_hprod2(H.h, C.c_int64(3), d, d, None, None, d, d, d, None, None, d, d) == -1
    with pytest.raises(ValueError):
        B.obj(torch.zeros((3, n + 1), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        B.hprod(X, torch.zeros((2, n), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        fpsb200.BatchFletcherPenaltyNLP(dm, np.ones(2), 0.0, 0.0).obj(X)
    with pytest.raises(TypeError):
        fpsb200.BatchFletcherPenaltyNLP(dm, qds=fpsb200.IterativeSolver(dm, 0.0))
    with pytest.raises(NotImplementedError):
        fpsb200.BatchFletcherPenaltyNLP(dm, explicit_linear_constraints=True)


def test_models_without_batched_methods_use_the_single_ones():
    """A model with only the single methods (the row loop) against the vectorised DeviceCurvedQP: 1e-13 (its cons
    uses the single SELL product)."""
    import torch
    import fpsb200
    cm = _curved()
    dcm = fpsb200.DeviceCurvedQP(cm)

    class Single:
        meta = dcm.meta
        def __getattr__(self, name):
            if name.endswith("_batch"):
                raise AttributeError(name)
            return getattr(dcm, name)

    K = 4
    X, V, sigma, delta = _inputs(K, cm.meta.nvar, seed=29)
    rel = lambda a, b: float(torch.linalg.norm(a - b) / max(float(torch.linalg.norm(b)), 1e-300))
    for approx in (1, 2):
        Bv = fpsb200.BatchFletcherPenaltyNLP(dcm, sigma, 1.0, delta, approx, qds=fpsb200.LDLtSolver(dcm, 0.0, ordering="amd"))
        Bs = fpsb200.BatchFletcherPenaltyNLP(Single(), sigma, 1.0, delta, approx,
                                             qds=fpsb200.LDLtSolver(dcm, 0.0, ordering="amd"))
        pv, gv = Bv.objgrad(X)
        ps, gs = Bs.objgrad(X)
        assert rel(pv, ps) <= 1e-13 and rel(gv, gs) <= 1e-13
        tol = 1e-13 if approx == 2 else 1e-7      # Val(1): iterative extras solves from inputs that differ in the last bits
        assert rel(Bv.hprod(X, V), Bs.hprod(X, V)) <= tol
