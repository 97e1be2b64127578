"""Batched LDLt path (fpsb_ldlt_batch_solve_two_mixed) against a loop over the single-instance entry and the CPU oracle.

Workloads (seeded; instances share the pattern, their Jacobian values are the base values times 1 + 0.1 N(0,1), delta
cycles over {0, sqrt(eps), 0.25, 1e-2}):
  c5        n = 10,  m = 3, dense (BASELINE config C5), beside fpsb_batch_solve_two on the same instances
  cutest    window-random n = 100, m = 50, 5 nnz per row (CUTEst-sized: the reference's benchmark set is <= 100 variables)
  poisson   models.poisson_control(20) (the docs' example: n = 800, m = 400)
  n4000     window-random n = 4000, m = 2000, 5 nnz per row
The instance counts make the factor store larger than the B200's 126 MB L2 where the shape allows it, so the timed
calls stream their factors from HBM.  One JSON line per workload (and a header line with the card) on stdout and in
--out.

  python tools/ldlt_batch_bench.py --out profiles/ldlt_batch_bench.jsonl
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SQRT_EPS = float(np.sqrt(np.finfo(float).eps))
DELTAS = (0.0, SQRT_EPS, 0.25, 1e-2)


def workload(name):
    from fpsb200 import models
    if name == "c5":
        rows, cols = np.meshgrid(np.arange(3), np.arange(10), indexing="ij")
        A = sp.csr_matrix((np.random.default_rng(1).standard_normal(30), (rows.ravel(), cols.ravel())), shape=(3, 10))
        return A, 4096
    if name == "cutest":
        return models.window_random_jacobian(50, 100, 5, w=8, seed=21), 20000
    if name == "poisson":
        return models.poisson_control(20).A, 2000
    if name == "n4000":
        return models.window_random_jacobian(2000, 4000, 5, w=32, seed=22), 1000
    raise KeyError(name)


def residual(coo, m, n, J, delta, r1, r2, p1, q1, p2, q2):
    """max over instances of the relative K-residuals of both systems (same pattern: products through 0/1 maps)."""
    nnz = coo.nnz
    Sr = sp.csr_matrix((np.ones(nnz), (np.arange(nnz), coo.row)), shape=(nnz, m))
    Sc = sp.csr_matrix((np.ones(nnz), (np.arange(nnz), coo.col)), shape=(nnz, n))
    Ax = lambda x: np.asarray((J * x[:, coo.col]) @ Sr)
    Aty = lambda y: np.asarray((J * y[:, coo.row]) @ Sc)
    d = delta[:, None]
    e1 = np.hstack([p1 + Aty(q1) - r1, Ax(p1) - d * q1])
    e2 = np.hstack([p2 + Aty(q2), Ax(p2) - d * q2 - r2])
    return float(max((np.linalg.norm(e1, axis=1) / np.linalg.norm(r1, axis=1)).max(),
                     (np.linalg.norm(e2, axis=1) / np.linalg.norm(r2, axis=1)).max()))


def timed(fn, min_s=0.5):
    fn()                                             # warm-up (module load, buffers)
    t0 = time.perf_counter(); fn(); t1 = time.perf_counter()
    reps = max(3, int(math.ceil(min_s / max(t1 - t0, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) / reps


def run(name, nloop, noracle):
    import torch
    import fpsb200
    from oracle import oracle as O
    A, ninst = workload(name)
    coo = sp.coo_matrix(A)
    m, n = A.shape
    rng = np.random.default_rng(7)
    J = coo.data[None, :] * (1.0 + 0.1 * rng.standard_normal((ninst, coo.nnz)))
    delta = np.array([DELTAS[i % 4] for i in range(ninst)])
    r1, r2 = rng.standard_normal((ninst, n)), rng.standard_normal((ninst, m))
    H = fpsb200.B200Handle(n, m, coo.row, coo.col)
    H.ldlt_analyze(np.arange(n + m) if name == "c5" else None)
    info = H.ldlt_plan_info()
    out = dict(workload=name, nvar=n, ncon=m, nnzj=int(coo.nnz), ninst=ninst, plan=info,
               factor_store_mb=round(ninst * (info["panel_nnz"] + n + m) * 8 / 1e6, 1))
    # batched, host buffers
    res = [None]
    def host_call():
        res[0] = H.ldlt_batch_solve_two_mixed(delta, J, r1, r2)
    t_host = timed(host_call)
    p1, q1, p2, q2, ok = res[0]
    out["batch_host_inst_per_s"] = ninst / t_host
    out["factorized_all"] = bool(ok.all())
    out["max_k_residual"] = residual(coo, m, n, J, delta, r1, r2, p1, q1, p2, q2)
    l0 = H.launch_count(); host_call(); out["batch_launches_per_call"] = H.launch_count() - l0
    # batched, device buffers: device events on the handle's stream
    dev = torch.device("cuda", 0)
    tJ, td, t1, t2 = (torch.as_tensor(a, device=dev) for a in (J, delta, r1, r2))
    H.ldlt_batch_solve_two_mixed(td, tJ, t1, t2)
    torch.cuda.synchronize()
    reps = max(3, int(math.ceil(0.5 * out["batch_host_inst_per_s"] / ninst)))
    H.timer_start()
    for _ in range(reps):
        got = H.ldlt_batch_solve_two_mixed(td, tJ, t1, t2)
    ms = H.timer_stop()
    torch.cuda.synchronize()
    out["batch_device_inst_per_s"] = ninst * reps / (ms * 1e-3)
    out["device_equals_host"] = all(np.array_equal(a, b.cpu().numpy()) for a, b in zip(res[0], got))
    # loop over the single-instance entry on one handle (host buffers, as a caller of fpsb_ldlt_solve_two_mixed would)
    k = min(nloop, ninst)
    H.set_jac_values(J[0]); H.ldlt_solve_two_mixed(delta[0], r1[0], r2[0])
    l0 = H.launch_count(); H.ldlt_solve_two_mixed(delta[0], r1[0], r2[0])
    out["single_launches_per_call"] = H.launch_count() - l0
    same = True
    t0 = time.perf_counter()
    for i in range(k):
        H.set_jac_values(J[i])
        s = H.ldlt_solve_two_mixed(delta[i], r1[i], r2[i])
        same = same and np.array_equal(s[0], p1[i]) and np.array_equal(s[3], q2[i])
    out["single_loop_inst_per_s"] = k / (time.perf_counter() - t0)
    out["single_loop_instances"] = k
    out["batch_equals_single_bitwise"] = bool(same)
    out["batch_over_single_loop_device"] = out["batch_device_inst_per_s"] / out["single_loop_inst_per_s"]
    out["batch_over_single_loop_host"] = out["batch_host_inst_per_s"] / out["single_loop_inst_per_s"]
    # single-threaded CPU oracle (same ordering)
    lo = O.LDLtOracle(n, m, coo.row, coo.col, H.ldlt_symbolic()["P"])
    k = min(noracle, ninst)
    lo.solve_two_mixed(J[0], delta[0], r1[0], r2[0])
    t0 = time.perf_counter()
    for i in range(k):
        lo.solve_two_mixed(J[i], delta[i], r1[i], r2[i])
    out["cpu_oracle_inst_per_s"] = k / (time.perf_counter() - t0)
    out["cpu_oracle_instances"] = k
    if name == "c5":
        Ad = np.zeros((ninst, m, n))
        Ad[:, coo.row, coo.col] = J
        dres = [None]
        def dense_call():
            dres[0] = fpsb200.batch_solve_two(Ad, 1e-2, r1, r2)
        # the dense batch takes one delta for all instances: both run with 1e-2 here
        d1 = np.full(ninst, 1e-2)
        ours = [None]
        def ours_call():
            ours[0] = H.ldlt_batch_solve_two_mixed(d1, J, r1, r2)
        out["dense_batch_host_inst_per_s"] = ninst / timed(dense_call)
        out["batch_host_inst_per_s_delta_1e-2"] = ninst / timed(ours_call)
        out["max_rel_diff_vs_dense_batch"] = float(max(
            (np.linalg.norm(a - b, axis=1) / np.linalg.norm(b, axis=1)).max() for a, b in zip(ours[0][:4], dres[0][:4])))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c5,cutest,poisson,n4000")
    ap.add_argument("--loop", type=int, default=300, help="instances of the single-instance loop")
    ap.add_argument("--oracle", type=int, default=50, help="instances of the CPU oracle loop")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    lines = [dict(card=card[0] if card else "unknown", ldlt_mode=os.environ.get("FPSB_LDLT_MODE", "1"))]
    print(json.dumps(lines[0]), flush=True)
    for w in a.workloads.split(","):
        r = run(w, a.loop, a.oracle)
        print(json.dumps(r), flush=True)
        lines.append(r)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
