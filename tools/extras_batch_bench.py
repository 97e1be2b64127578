"""Batched LDLt solve_two_extras (fpsb_ldlt_batch_solve_two_extras) against a loop over the single-instance entry and the
CPU oracle.

Workloads (seeded; instances share the pattern, their Jacobian values are the base values times 1 + 0.1 N(0,1), delta
cycles over {0, sqrt(eps), 0.25, 1e-2}, reference tolerances):
  cutest    window-random n = 100, m = 50, 5 nnz per row (CUTEst-sized: the reference's benchmark set is <= 100 variables)
  poisson   models.poisson_control(20) (the docs' example: n = 800, m = 400)
  n4000     window-random n = 4000, m = 2000, 5 nnz per row (working set beyond shared memory: global workspace)
Per workload: instances/s of the batch through device buffers (CUDA events on the handle's stream) and host buffers,
of a loop over fpsb_ldlt_solve_two_extras on one handle (a subset, host buffers) and of the single-threaded CPU oracle
(a subset); mean / max iterations per method; the largest relative true residual of both systems over all instances:
  CGLS    ||A (rhs1 - A' u1) - tau u1|| / ||A rhs1||      (normal equations of min ||rhs1 - A' u||^2 + tau ||u||^2)
  MINRES  ||A A' u2 + tau u2 - rhs2|| / ||rhs2||
One JSON line per workload (and a header line with the card) on stdout and in --out.

  python tools/extras_batch_bench.py --out profiles/extras_batch_bench.jsonl
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
    if name == "cutest":
        return models.window_random_jacobian(50, 100, 5, w=8, seed=21), 20000
    if name == "poisson":
        return models.poisson_control(20).A, 4000
    if name == "n4000":
        return models.window_random_jacobian(2000, 4000, 5, w=32, seed=22), 1000
    raise KeyError(name)


def residuals(coo, m, n, J, delta, r1, r2, u1, u2):
    """largest relative true residual of the CGLS and of the MINRES system over the instances"""
    nnz = coo.nnz
    Sr = sp.csr_matrix((np.ones(nnz), (np.arange(nnz), coo.row)), shape=(nnz, m))
    Sc = sp.csr_matrix((np.ones(nnz), (np.arange(nnz), coo.col)), shape=(nnz, n))
    Ax = lambda x: np.asarray((J * x[:, coo.col]) @ Sr)
    Aty = lambda y: np.asarray((J * y[:, coo.row]) @ Sc)
    tau = np.maximum(delta, 1e-14)[:, None]
    e1 = Ax(r1 - Aty(u1)) - tau * u1
    e2 = Ax(Aty(u2)) + tau * u2 - r2
    return (float((np.linalg.norm(e1, axis=1) / np.linalg.norm(Ax(r1), axis=1)).max()),
            float((np.linalg.norm(e2, axis=1) / np.linalg.norm(r2, axis=1)).max()))


def timed(fn, min_s=0.5):
    fn()                                             # warm-up (module load, buffers, CSR patterns)
    t0 = time.perf_counter(); fn(); t1 = time.perf_counter()
    reps = max(3, int(math.ceil(min_s / max(t1 - t0, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) / reps


def rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


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
    ws = 2 * coo.nnz + max(2 * n + 3 * m, n + 6 * m)
    out = dict(workload=name, nvar=n, ncon=m, nnzj=int(coo.nnz), ninst=ninst, item_working_set_kb=round(ws * 8 / 1024, 1))
    # batched, host buffers
    res = [None]
    def host_call():
        res[0] = H.ldlt_batch_solve_two_extras(delta, J, r1, r2)
    t_host = timed(host_call)
    u1, u2, st = res[0]
    out["batch_host_inst_per_s"] = ninst / t_host
    for j, meth in enumerate(("cgls", "minres")):
        out[f"{meth}_iter_mean"] = float(st["niter"][:, j].mean())
        out[f"{meth}_iter_max"] = int(st["niter"][:, j].max())
        out[f"{meth}_solved_all"] = bool(st["solved"][:, j].all())
    out["max_rel_residual_cgls"], out["max_rel_residual_minres"] = residuals(coo, m, n, J, delta, r1, r2, u1, u2)
    l0 = H.launch_count(); host_call(); out["batch_launches_per_call"] = H.launch_count() - l0
    # batched, device buffers: device events on the handle's stream
    dev = torch.device("cuda", 0)
    tJ, td, t1, t2 = (torch.as_tensor(a, device=dev) for a in (J, delta, r1, r2))
    H.ldlt_batch_solve_two_extras(td, tJ, t1, t2)
    torch.cuda.synchronize()
    reps = max(3, int(math.ceil(0.5 * out["batch_host_inst_per_s"] / ninst)))
    H.timer_start()
    for _ in range(reps):
        got = H.ldlt_batch_solve_two_extras(td, tJ, t1, t2)
    ms = H.timer_stop()
    torch.cuda.synchronize()
    out["batch_device_inst_per_s"] = ninst * reps / (ms * 1e-3)
    out["device_equals_host"] = bool(np.array_equal(u1, got[0].cpu().numpy()) and np.array_equal(u2, got[1].cpu().numpy()))
    # loop over the single-instance entry on one handle (host buffers, as a caller of fpsb_ldlt_solve_two_extras would)
    k = min(nloop, ninst)
    H.set_jac_values(J[0]); H.ldlt_solve_two_extras(delta[0], r1[0], r2[0])
    l0 = H.launch_count(); H.ldlt_solve_two_extras(delta[0], r1[0], r2[0])
    out["single_launches_per_call"] = H.launch_count() - l0
    d1 = d2 = 0.0
    dit = 0
    t0 = time.perf_counter()
    for i in range(k):
        H.set_jac_values(J[i])
        s1, s2, sst = H.ldlt_solve_two_extras(delta[i], r1[i], r2[i])
        d1, d2 = max(d1, rel(u1[i], s1)), max(d2, rel(u2[i], s2))
        dit = max(dit, abs(sst[0]["niter"] - int(st["niter"][i, 0])), abs(sst[1]["niter"] - int(st["niter"][i, 1])))
    out["single_loop_inst_per_s"] = k / (time.perf_counter() - t0)
    out["single_loop_instances"] = k
    out["batch_vs_single_max_rel_u1"], out["batch_vs_single_max_rel_u2"] = d1, d2
    out["batch_vs_single_max_iter_diff"] = dit
    out["batch_over_single_loop_device"] = out["batch_device_inst_per_s"] / out["single_loop_inst_per_s"]
    out["batch_over_single_loop_host"] = out["batch_host_inst_per_s"] / out["single_loop_inst_per_s"]
    # single-threaded CPU oracle
    lo = O.LDLtOracle(n, m, coo.row, coo.col, np.arange(n + m))
    k = min(noracle, ninst)
    lo.jvals = J[0]; lo.solve_two_extras(delta[0], r1[0], r2[0])
    t0 = time.perf_counter()
    for i in range(k):
        lo.jvals = J[i]
        lo.solve_two_extras(delta[i], r1[i], r2[i])
    out["cpu_oracle_inst_per_s"] = k / (time.perf_counter() - t0)
    out["cpu_oracle_instances"] = k
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cutest,poisson,n4000")
    ap.add_argument("--loop", type=int, default=100, help="instances of the single-instance loop")
    ap.add_argument("--oracle", type=int, default=50, help="instances of the CPU oracle loop")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    lines = [dict(card=card[0] if card else "unknown")]
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
