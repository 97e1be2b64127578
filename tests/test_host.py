"""CPU: the C ABI loads and exports every declared symbol; the host-only symbolic analysis is
bit-exact against the oracle; the multi-rank plumbing works under gloo (world_size 2)."""
import ctypes
import os
import re

import numpy as np
import pytest

import fpsb200
from fpsb200 import _lib, models, sharding
from fpsb200.symbolic import SymbolicAnalysis, order_dissection

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "fpsb.h")).read()
    declared = set(re.findall(r"\b(fpsb_[a-z0-9_]+)\s*\(", header))
    L = _lib.lib()
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in include/fpsb.h but not exported"
    assert declared == set(_lib.EXPORTS)
    assert L.fpsb_version() == 100
    o = fpsb200.IterOpts()
    assert L.fpsb_iter_default_opts(ctypes.c_int64(10), ctypes.c_int64(3), ctypes.byref(o)) == 0
    assert o.ls_itmax == 65 and o.ne_itmax == 0 and abs(o.ls_atol - np.sqrt(np.finfo(float).eps)) < 1e-20
    lo = fpsb200.LdltOpts()
    assert L.fpsb_ldlt_default_opts(ctypes.byref(lo)) == 0 and lo.ldlt_r2 == -lo.ldlt_r1


def test_no_cpu_fallback_without_gpu():
    L = _lib.lib()
    if L.fpsb_device_count() > 0:
        pytest.skip("a GPU is visible")
    with pytest.raises(fpsb200.FpsbError, match="no CUDA device"):
        fpsb200.B200Handle(4, 2, [0, 1], [0, 1])


def test_argument_validation():
    L = _lib.lib()
    bad = np.array([5], dtype=np.int64)
    h = ctypes.c_void_p()
    rc = L.fpsb_symbolic_create(ctypes.c_int64(3), ctypes.c_int64(2), ctypes.c_int64(1),
                                bad.ctypes.data_as(ctypes.c_void_p), bad.ctypes.data_as(ctypes.c_void_p),
                                ctypes.c_int(0), None, ctypes.byref(h))
    assert rc == -1 and b"out of range" in L.fpsb_last_error()
    with pytest.raises(fpsb200.FpsbError, match="not a permutation"):
        SymbolicAnalysis(3, 2, [0, 1], [0, 2], P=[0, 0, 1, 2, 3])


def test_tile_layout_and_create_validation():
    """fpsb_tile_layout and fpsb_tile_segments reject a NULL handle and a NULL output; fpsb_create rejects an
    out-of-range index before it looks for a device."""
    L = _lib.lib()
    out = (ctypes.c_int64 * 16)()
    assert L.fpsb_tile_layout(None, out) == -1 and b"NULL" in L.fpsb_last_error()
    fake = ctypes.create_string_buffer(64)
    assert L.fpsb_tile_layout(ctypes.cast(fake, ctypes.c_void_p), None) == -1
    seg = (ctypes.c_int64 * 8)()
    assert L.fpsb_tile_segments(None, 0, ctypes.c_int64(0), seg) == -1
    assert L.fpsb_tile_segments(ctypes.cast(fake, ctypes.c_void_p), 0, ctypes.c_int64(0), None) == -1
    h = ctypes.c_void_p()
    for r, c in (([2], [0]), ([0], [4]), ([-1], [0])):
        jr, jc = np.array(r, dtype=np.int64), np.array(c, dtype=np.int64)
        rc = L.fpsb_create(ctypes.c_int64(4), ctypes.c_int64(2), ctypes.c_int64(1), jr.ctypes.data_as(ctypes.c_void_p),
                           jc.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(0), ctypes.c_int(0), ctypes.byref(h))
        assert rc == -1 and b"out of range" in L.fpsb_last_error() and not h.value
    jr = np.array([0], dtype=np.int64)           # one-based: 0 is out of range
    rc = L.fpsb_create(ctypes.c_int64(4), ctypes.c_int64(2), ctypes.c_int64(1), jr.ctypes.data_as(ctypes.c_void_p),
                       jr.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(1), ctypes.c_int(0), ctypes.byref(h))
    assert rc == -1 and b"out of range" in L.fpsb_last_error()


def test_ldlt_routes_validation():
    """fpsb_symbolic_ldlt_routes and fpsb_ldlt_routes reject a NULL analysis / handle and a NULL output."""
    L = _lib.lib()
    out = (ctypes.c_int64 * len(_lib.LDLT_ROUTE_KEYS))()
    assert L.fpsb_symbolic_ldlt_routes(None, out) == -1 and b"NULL" in L.fpsb_last_error()
    assert L.fpsb_ldlt_routes(None, out) == -1 and b"NULL" in L.fpsb_last_error()
    S = SymbolicAnalysis(3, 2, [0, 1], [0, 2])
    assert L.fpsb_symbolic_ldlt_routes(S.h, None) == -1
    rt = S.routes()
    assert rt["nsuper"] >= 1 and rt["leaf1"] + rt["leaf_wide"] >= 1


@pytest.mark.parametrize("m,n,k,w", [(1, 10, 9, 4), (30, 60, 5, 8), (500, 1000, 10, 32), (4000, 8000, 10, 64)])
@pytest.mark.parametrize("pk", ["amd", "id", "rand"])
def test_symbolic_bit_exact_vs_oracle(oracle, m, n, k, w, pk):
    """north_star: "the symbolic analysis must be bit-exact" — (parent, Lnz, Lp, Li) of the
    product's child-merge analysis == the oracle's Davis row-subtree walk, for the same P."""
    if pk == "rand" and m > 1000:
        pytest.skip("random ordering of a large problem: dense fill, slow on the CPU oracle")
    A = models.window_random_jacobian(m, n, k, w=w, seed=m)
    coo = A.tocoo()
    P = None if pk == "amd" else (np.arange(n + m) if pk == "id" else np.random.default_rng(1).permutation(n + m))
    S = SymbolicAnalysis(n, m, coo.row, coo.col, P)
    g = S.get()
    assert sorted(g["P"].tolist()) == list(range(n + m))
    lo = oracle.LDLtOracle(n, m, coo.row, coo.col, g["P"])
    assert lo.solve_two_mixed(coo.data, 1e-2, np.ones(n), np.ones(m))[4]
    s = lo.symbolic()
    for key in ("P", "parent", "Lnz", "Lp", "Li"):
        assert np.array_equal(g[key], s[key]), key
    info = S.plan_info()
    assert info["panel_nnz"] >= S.lnz + n + m and info["nsuper"] <= n + m


def test_amd_reduces_fill_on_grid_and_defers_dense_row():
    """Ordering sanity: on a 2-D Poisson control problem AMD must beat the natural order by a wide
    margin, and a constraint touching every variable must be eliminated last."""
    mdl = models.poisson_control(48)
    r, c = mdl.jac_structure()
    n, m = mdl.meta.nvar, mdl.meta.ncon
    amd = SymbolicAnalysis(n, m, r, c).lnz
    nat = SymbolicAnalysis(n, m, r, c, np.arange(n + m)).lnz
    assert amd < 0.6 * nat
    rows = np.r_[np.zeros(200, dtype=np.int64), np.arange(1, 51)]
    cols = np.r_[np.arange(200), np.arange(50)]
    S = SymbolicAnalysis(200, 51, rows, cols)
    assert S.get()["P"][-1] == 200
    assert S.lnz < 600


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mine = sharding.shard_instances(7, rank, world)
    local = {i: np.full(3, float(i)) for i in mine}
    allr = sharding.gather_results(local, 7, dist)
    t = sharding.max_over_ranks(10.0 + rank, dist)
    q.put((rank, mine, [a.tolist() for a in allr], t))
    dist.barrier()
    dist.destroy_process_group()


def test_instance_sharding_gloo_world2():
    """N>1 path of bench.py / config C5: static sharding, no data-path collective; the control
    plane (barrier, MAX of times, result gather) over gloo with world_size 2."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res[0][1] == [0, 2, 4, 6] and res[1][1] == [1, 3, 5]
    for r in res:
        assert r[2] == [[float(i)] * 3 for i in range(7)]
        assert r[3] == 11.0


def test_dissection_ordering_cuts_dependency_depth(oracle):
    """fpsb_order_dissection: a valid permutation whose supernodal dependency depth is far below
    minimum degree's on band-like KKT structure, at comparable fill; the analysis stays bit-exact
    against the oracle for this P as for any other."""
    m, n = 30000, 60000
    A = models.window_random_jacobian(m, n, 10, w=32, seed=5)
    coo = A.tocoo()
    P = order_dissection(n, m, coo.row, coo.col, nparts=32)
    assert sorted(P.tolist()) == list(range(n + m))
    Sd = SymbolicAnalysis(n, m, coo.row, coo.col, P)
    Sa = SymbolicAnalysis(n, m, coo.row, coo.col)
    d, a = Sd.plan_info(), Sa.plan_info()
    assert d["nlevels"] * 4 < a["nlevels"]
    assert Sd.lnz < 2.5 * Sa.lnz
    g = Sd.get()
    lo = oracle.LDLtOracle(n, m, coo.row, coo.col, g["P"])
    assert lo.solve_two_mixed(coo.data, 1e-2, np.ones(n), np.ones(m))[4]
    s = lo.symbolic()
    for key in ("parent", "Lnz", "Lp", "Li"):
        assert np.array_equal(g[key], s[key]), key
    # small / disconnected graphs fall back gracefully
    P = order_dissection(6, 2, [0, 1], [0, 3])
    assert sorted(P.tolist()) == list(range(8))
