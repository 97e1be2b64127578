"""BatchFletcherPenaltyNLP and _steihaug_batch against a loop of DeviceFletcherPenaltyNLP / _steihaug_device over the
same instances.

Workloads (seeded; DeviceCurvedQP, so Val(1) has real terms; per-instance sigma in [1, 10], delta cycling over
{0, 1e-2}, rho = 0):
  cutest    sparse_qp n = 100, m = 50, 5 nnz per row (CUTEst-sized: the reference's benchmark set is <= 100 variables)
  poisson   models.poisson_control(20) (the docs' example: n = 800, m = 400)
  n4000     sparse_qp n = 4000, m = 2000, 5 nnz per row
K in {1, 64, 1024, 4096}.  Per (workload, K), each timed after a warm-up call, with CUDA events on torch's stream
around a window that ends in a synchronise:
  objgrad   objgrad at a point that differs from the last one (the memo misses: model, batched mixed solve, obj, grad)
  hprod2    one Val(2) hprod at the memoised point
  hprod1    one Val(1) hprod at the memoised point
  cg        one whole _steihaug_batch subproblem (Val(2) hprod, radius 1e3, tol 1e-8 |g|, at most 10 products)
and the same through a loop of the single evaluator over the first `--loop` instances (its per-instance time is
extrapolated to K).  Launches per call count the kernels of libfpsb200 only (the model's torch kernels are not
counted).  One JSON line per (workload, K), and a header line with the card, on stdout and in --out.

  python tools/fp_batch_bench.py --out profiles/r3_fp_batch_bench.jsonl
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def model(name):
    from fpsb200 import models
    if name == "cutest":
        qp = models.sparse_qp(100, 50, nnz_per_row=5, w=8, seed=21)
    elif name == "poisson":
        qp = models.poisson_control(20)
    elif name == "n4000":
        qp = models.sparse_qp(4000, 2000, nnz_per_row=5, w=32, seed=22)
    else:
        raise KeyError(name)
    d = 0.3 * np.random.default_rng(5).standard_normal(qp.meta.ncon)
    return models.CurvedQPModel(qp.Q, qp.q, qp.A, qp.b, d, name=name)


def timed(fn, reps=3):
    """mean ms of fn() over `reps` calls, CUDA events on torch's current stream, after one warm-up call"""
    import torch
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def run(name, K, nloop):
    import torch
    import fpsb200
    from fpsb200.fps_solve import _steihaug_batch, _steihaug_device
    cm = model(name)
    dm = fpsb200.DeviceCurvedQP(cm)
    n, m = cm.meta.nvar, cm.meta.ncon
    rng = np.random.default_rng(7)
    X = torch.tensor(0.5 * rng.standard_normal((K, n)), device="cuda")
    Xs = [X, X + 1e-3]
    V = torch.tensor(rng.standard_normal((K, n)), device="cuda")
    sigma = 1.0 + 9.0 * rng.random(K)
    delta = np.array([(0.0, 1e-2)[i % 2] for i in range(K)])
    qs = fpsb200.LDLtSolver(dm, 0.0, ordering="amd")
    B2 = fpsb200.BatchFletcherPenaltyNLP(dm, sigma, 0.0, delta, 2, qds=qs)
    B1 = fpsb200.BatchFletcherPenaltyNLP(dm, sigma, 0.0, delta, 1, qds=qs)
    H = qs.handle
    out = dict(workload=name, nvar=n, ncon=m, nnzj=int(cm.meta.nnzj), K=K)
    it = [0]

    def objgrad():
        it[0] += 1
        return B2.objgrad(Xs[it[0] % 2])

    def launches(fn):
        l0 = H.launch_count(); fn(); return H.launch_count() - l0

    res = {}
    out["batch_objgrad_ms"] = timed(objgrad)
    out["batch_objgrad_launches"] = launches(objgrad)
    Xc = Xs[it[0] % 2]
    B1.objgrad(Xc)
    out["batch_hprod2_ms"] = timed(lambda: B2.hprod(Xc, V))
    out["batch_hprod2_launches"] = launches(lambda: B2.hprod(Xc, V))
    out["batch_hprod1_ms"] = timed(lambda: B1.hprod(Xc, V))
    out["batch_hprod1_launches"] = launches(lambda: B1.hprod(Xc, V))
    G = B2.grad(Xc)
    tol = 1e-8 * torch.linalg.norm(G, dim=1)

    def cg():
        res["cg"] = _steihaug_batch(H, lambda D: B2.hprod(Xc, D), G, 1e3, tol, 10)
    out["batch_cg_ms"] = timed(cg, reps=1)
    out["batch_cg_launches"] = launches(cg)
    out["batch_cg_products_max"] = int(res["cg"][2].max())
    # the single evaluator over the first k instances
    k = min(nloop, K)
    qs1 = fpsb200.LDLtSolver(dm, 0.0, ordering="amd")
    S2 = [fpsb200.DeviceFletcherPenaltyNLP(dm, float(sigma[i]), 0.0, float(delta[i]), 2, qds=qs1) for i in range(k)]
    S1 = [fpsb200.DeviceFletcherPenaltyNLP(dm, float(sigma[i]), 0.0, float(delta[i]), 1, qds=qs1) for i in range(k)]
    H1 = qs1.handle

    def loop_objgrad():
        it[0] += 1
        Xl = Xs[it[0] % 2]
        for i in range(k):
            S2[i].objgrad(Xl[i])

    def loop_hprod(S):
        for i in range(k):
            S[i].hprod(Xc[i], V[i])

    def loop_cg():
        for i in range(k):
            gi = S2[i].grad(Xc[i])
            _steihaug_device(H1, lambda d, i=i: S2[i].hprod(Xc[i], d), gi, 1e3, float(tol[i]), 10)

    per = lambda ms: ms / k
    out["loop_instances"] = k
    out["loop_objgrad_ms_per_inst"] = per(timed(loop_objgrad, reps=1))
    for i in range(k):
        S2[i].objgrad(Xc[i]); S1[i].objgrad(Xc[i])
    out["loop_hprod2_ms_per_inst"] = per(timed(lambda: loop_hprod(S2), reps=1))
    out["loop_hprod1_ms_per_inst"] = per(timed(lambda: loop_hprod(S1), reps=1))
    out["loop_cg_ms_per_inst"] = per(timed(loop_cg, reps=1))
    l0 = H1.launch_count(); S2[0].hprod(Xc[0], V[0]); out["single_hprod2_launches"] = H1.launch_count() - l0
    for key in ("objgrad", "hprod2", "hprod1", "cg"):
        out[f"{key}_batch_over_loop"] = out[f"loop_{key}_ms_per_inst"] * K / out[f"batch_{key}_ms"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cutest,poisson,n4000")
    ap.add_argument("--ks", default="1,64,1024,4096")
    ap.add_argument("--loop", type=int, default=16, help="instances of the single-evaluator loop")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    lines = [dict(card=card[0] if card else "unknown")]
    print(json.dumps(lines[0]), flush=True)
    for w in a.workloads.split(","):
        for K in (int(k) for k in a.ks.split(",")):
            r = run(w, K, a.loop)
            print(json.dumps(r), flush=True)
            lines.append(r)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
