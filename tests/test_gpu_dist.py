"""GPU: the row-partitioned Krylov path (fpsb_dist_*, NCCL) against the single-GPU path and the
oracle.  world_size 1 runs on any box (NCCL with one rank); world_size 2 needs two GPUs
and is skipped otherwise."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _problem(m=3000, n=6000, k=9, w=32, seed=11):
    from fpsb200 import models
    A = models.window_random_jacobian(m, n, k, w=w, seed=seed).tocsr()
    coo = A.tocoo()
    rng = np.random.default_rng(seed)
    return A, coo.row.astype(np.int64), coo.col.astype(np.int64), coo.data, rng.standard_normal(n), rng.standard_normal(m), rng.standard_normal(n)


def _rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def test_dist_world1_matches_oracle(oracle):
    from fpsb200.partition import RowPartition, DistHandle
    A, jr, jc, vals, r1, r2, r3 = _problem()
    m, n = A.shape
    part = RowPartition(n, m, jr, jc, 1)
    D = DistHandle(part, 0, device=0)
    D.set_jac_values(vals)
    assert _rel(D.jprod(r1), A @ r1) < 1e-13
    assert _rel(D.jtprod(r2), A.T @ r2) < 1e-13
    import fpsb200
    H = fpsb200.B200Handle(n, m, jr, jc)
    H.set_jac_values(vals)
    for delta in (0.0, 1e-2):
        # reference tolerances (sqrt(eps)): same status / iterations within 1 of the oracle; the
        # iterates themselves agree to the solve tolerance
        p1, q1, p2, q2, st = D.solve_two_mixed(delta, r1, r2)
        ref = oracle.IterativeOracle(A).solve_two_mixed(delta, r1, r2)
        for a, b in zip((p1, q1, p2, q2), ref[:4]):
            assert _rel(a, b) < 1e-6
        assert st[0]["solved"] and st[1]["solved"]
        assert abs(st[0]["niter"] - ref[4][0]["niter"]) <= 1 and abs(st[1]["niter"] - ref[4][1]["niter"]) <= 1
        one = H.iter_solve_two_mixed(delta, r1, r2)
        for a, b in zip((p1, q1, p2, q2), one[:4]):
            assert _rel(a, b) < 1e-6
    # fixed iteration count: the un-fused distributed recurrences reproduce the fused single-GPU ones
    o = fpsb200.IterOpts()
    import ctypes
    assert fpsb200._lib.lib().fpsb_iter_default_opts(ctypes.c_int64(n), ctypes.c_int64(m), ctypes.byref(o)) == 0
    o.ls_itmax = 25; o.ln_itmax = 25
    D.H.iter_setup(o); H.iter_setup(o)
    a4 = D.solve_two_mixed(1e-2, r1, r2)
    b4 = H.iter_solve_two_mixed(1e-2, r1, r2)
    assert [s["niter"] for s in a4[4]] == [25, 25] == [s["niter"] for s in b4[4]]
    for a, b in zip(a4[:4], b4[:4]):
        assert _rel(a, b) < 1e-11
    a4 = D.solve_two_least_squares(1e-2, r1, r3)
    b4 = H.iter_solve_two_least_squares(1e-2, r1, r3)
    for a, b in zip(a4[:4], b4[:4]):
        assert _rel(a, b) < 1e-11
    # solve_two_extras (LSQR + MINRES on A A' + tau I) at a fixed iteration count: distributed == single GPU
    o.ne_itmax = 25
    D.H.iter_setup(o); H.iter_setup(o)
    u1, u2, stx = D.solve_two_extras(1e-2, r1, r2)
    v1, v2, sty = H.iter_solve_two_extras(1e-2, r1, r2)
    assert [s["niter"] for s in stx] == [s["niter"] for s in sty]
    assert _rel(u1, v1) < 1e-11 and _rel(u2, v2) < 1e-10


def test_dist_world1_extras_match_oracle(oracle):
    """src/solve_linear_system.jl:45-77 through the row-partitioned handle at the reference tolerances."""
    from fpsb200.partition import RowPartition, DistHandle
    A, jr, jc, vals, r1, r2, r3 = _problem()
    m, n = A.shape
    D = DistHandle(RowPartition(n, m, jr, jc, 1), 0, device=0)
    D.set_jac_values(vals)
    for delta in (0.0, 1e-2):
        u1, u2, st = D.solve_two_extras(delta, r1, r2)
        ref = oracle.IterativeOracle(A).solve_two_extras(delta, r1, r2)
        assert _rel(u1, ref[0]) < 1e-6 and _rel(u2, ref[1]) < 2e-4        # MINRES at convergence: see test_gpu_krylov.py
        tau = max(delta, 1e-14)
        if delta > 0:       # the normal equations both solve: (A A' + tau I) u2 = rhs2
            assert _rel(A @ (A.T @ u2) + tau * u2, r2) < 1e-3             # MINRES stops on its own sqrt(eps)-level tests


def _worker(rank, world, port, q, peer=True):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from fpsb200.partition import RowPartition, DistHandle
    A, jr, jc, vals, r1, r2, r3 = _problem()
    m, n = A.shape
    part = RowPartition(n, m, jr, jc, world)
    D = DistHandle(part, rank, device=rank, dist=dist, peer=peer)
    assert D.peer == peer                      # the requested transport is the one that runs (no silent fallback)
    D.set_jac_values(vals)
    L = D.loc
    own = slice(L.col0, L.col0 + L.n_own)
    rows = slice(L.row0, L.row0 + L.m_loc)
    y = D.jprod(r1[own])
    z = D.jtprod(r2[rows])
    p1, q1, p2, q2, st = D.solve_two_mixed(1e-2, r1[own], r2[rows])
    P1, Q1, P2, Q2, st2 = D.solve_two_least_squares(0.0, r1[own], r3[own])
    u1, u2, st3 = D.solve_two_extras(1e-2, r1[own], r2[rows])
    q.put((rank, L.row0, L.col0, y, z, p1, q1, p2, q2, st, P1, Q1, P2, Q2, st2, u1, u2, st3))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("transport", ["peer-memory", "nccl"])
def test_dist_world2_matches_single_gpu(oracle, transport):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    import fpsb200
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 32500 + (os.getpid() % 2000) + (0 if transport == "nccl" else 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, transport == "peer-memory")) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=600) for _ in range(2)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    A, jr, jc, vals, r1, r2, r3 = _problem()
    m, n = A.shape
    cat = lambda i: np.concatenate([r[i] for r in res])
    assert _rel(cat(3), A @ r1) < 1e-13 and _rel(cat(4), A.T @ r2) < 1e-13
    H = fpsb200.B200Handle(n, m, jr, jc)
    H.set_jac_values(vals)
    one = H.iter_solve_two_mixed(1e-2, r1, r2)
    for i, b in zip((5, 6, 7, 8), one[:4]):
        assert _rel(cat(i), b) < 1e-6
    for r in res:       # replicated scalar recurrences: identical iteration counts on every rank
        assert [s["niter"] for s in r[9]] == [s["niter"] for s in res[0][9]]
        assert abs(r[9][0]["niter"] - one[4][0]["niter"]) <= 1 and abs(r[9][1]["niter"] - one[4][1]["niter"]) <= 1
    two = H.iter_solve_two_least_squares(0.0, r1, r3)
    for i, b in zip((10, 11, 12, 13), two[:4]):
        assert _rel(cat(i), b) < 1e-6
    ex = H.iter_solve_two_extras(1e-2, r1, r2)
    assert _rel(cat(15), ex[0]) < 1e-6 and _rel(cat(16), ex[1]) < 1e-6
    for r in res:
        assert [s["niter"] for s in r[17]] == [s["niter"] for s in res[0][17]]
        assert abs(r[17][1]["niter"] - ex[2][1]["niter"]) <= 1


def _stencil_problem(nx=1100, ny=64):
    """Interleaved 5-point-stencil operator [L -I] (BASELINE config C3 shape), wide enough for a strip boundary of
    ~3 300 rows: multi-segment gather windows and the helper-CTA path of the in-kernel exchange (>= 1 536 boundary rows)."""
    import scipy.sparse as sp
    Tx = sp.diags([-1.0, 2.0, -1.0], [-1, 0, 1], shape=(nx, nx))
    Ty = sp.diags([-1.0, 2.0, -1.0], [-1, 0, 1], shape=(ny, ny))
    L = sp.kron(Ty, sp.identity(nx)) + sp.kron(sp.identity(ny), Tx)
    m = nx * ny
    A = sp.hstack([L, -sp.identity(m)]).tocoo()
    rng = np.random.default_rng(21)
    vals = A.data * (1.0 + 0.1 * rng.standard_normal(A.nnz))
    perm = np.empty(2 * m, dtype=np.int64)
    perm[:m] = 2 * np.arange(m)
    perm[m:] = 2 * np.arange(m) + 1
    jr, jc = A.row.astype(np.int64), perm[A.col]
    return m, 2 * m, jr, jc, vals, rng.standard_normal(2 * m), rng.standard_normal(m)


def _stencil_worker(rank, world, port, q):
    import ctypes
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import fpsb200
    from fpsb200.partition import RowPartition, DistHandle
    m, n, jr, jc, vals, r1, r2 = _stencil_problem()
    o = fpsb200.IterOpts()
    fpsb200._lib.lib().fpsb_iter_default_opts(ctypes.c_int64(n), ctypes.c_int64(m), ctypes.byref(o))
    o.ls_itmax = o.ln_itmax = 30
    D = DistHandle(RowPartition(n, m, jr, jc, world), rank, device=rank, dist=dist, opts=o, peer=True)
    D.set_jac_values(vals)
    L = D.loc
    own, rows = slice(L.col0, L.col0 + L.n_own), slice(L.row0, L.row0 + L.m_loc)
    a = D.solve_two_mixed(1e-2, r1[own], r2[rows])
    b = D.solve_two_mixed(1e-2, r1[own], r2[rows])                 # again: bitwise reproducible
    q.put((rank, int(L.n_ext - L.n_own), a[:4], [s["niter"] for s in a[4]], all(np.array_equal(x, y) for x, y in zip(a[:4], b[:4]))))
    dist.barrier()
    dist.destroy_process_group()


def test_dist_world2_long_boundary_helper_ctas(oracle):
    import ctypes
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    import fpsb200
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 36500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_stencil_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=600) for _ in range(2)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    m, n, jr, jc, vals, r1, r2 = _stencil_problem()
    assert max(r[1] for r in res) >= 1536                           # long enough for the helper CTAs
    assert all(r[4] for r in res)
    o = fpsb200.IterOpts()
    fpsb200._lib.lib().fpsb_iter_default_opts(ctypes.c_int64(n), ctypes.c_int64(m), ctypes.byref(o))
    o.ls_itmax = o.ln_itmax = 30
    H = fpsb200.B200Handle(n, m, jr, jc)
    H.iter_setup(o)
    H.set_jac_values(vals)
    one = H.iter_solve_two_mixed(1e-2, r1, r2)
    assert res[0][3] == res[1][3] == [s["niter"] for s in one[4]]
    for i in range(4):
        assert _rel(np.concatenate([r[2][i] for r in res]), one[i]) < 1e-9
