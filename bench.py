#!/usr/bin/env python
"""bench.py — 2-RHS KKT solves/s at n=1M, nnz(A)=10M (BASELINE.json metric).

A step = one `solve_two_mixed`: refresh the device-resident Jacobian values + the two
quasi-definite solves K [p1 p2; q1 q2] = [g 0; 0 c] on the Krylov (IterativeSolver) path,
LSQR and CRAIG advanced in lock-step by the fused two-column SpMM kernels.

    python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU)
    python bench.py --impl reference --steps K --warmup W    # CPU arm: the oracle port on host cores
    python bench.py --steps K --warmup W --dump-outputs DIR  # also writes the last timed step's outputs as .npy

value : whole-job solves/s with rhs / Jacobian values already resident in HBM (FPSB_DEVICE)
e2e   : the same step through the C ABI with HOST buffers (FPSB_HOST: jac values + both rhs
        copied H2D and the four result vectors copied D2H inside the timed region)
N > 1 : `value` = independent instances sharded across GPUs, no data-path collective ("weak"); the line also
        carries `partitioned`: the row-partitioned Krylov path (halo exchange + all-reduced inner products over
        NVLink peer memory) STRONG-scaled over the N GPUs on BASELINE config C3 and on the headline matrix, with
        the single-GPU time of the same operator and the parity of the two results measured in the same run.
The reference (Julia) cannot run here: the CPU arm is the oracle's C port of the same algorithms
(kind "port", 1 thread — the reference path is single-threaded).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SQRT_EPS = float(np.sqrt(np.finfo(np.float64).eps))

OUTPUT_NAMES = ("p1", "q1", "p2", "q2")
STAT_FIELDS = ("niter", "solved", "inconsistent", "status", "rnorm", "arnorm", "anorm", "acond", "xnorm")
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(d, out):
    """--dump-outputs: what one solve_two_mixed call returns, as DIR/<name>.npy in float64 — the four solution
    vectors p1, q1, p2, q2 and stats.npy, the LSQR and CRAIG stats as a (2, 9) array in STAT_FIELDS order.  At the
    default size the vectors take 24 MB and are written whole; past 64 MB every vector is cut to the same share of
    its entries at positions drawn from a fixed seed, so two runs of the same arguments write the same positions."""
    vecs = [x.cpu().numpy().astype(np.float64) for x in out[:4]]
    total = sum(v.nbytes for v in vecs)
    os.makedirs(d, exist_ok=True)
    for name, v in zip(OUTPUT_NAMES, vecs):
        if total > DUMP_LIMIT_BYTES:
            keep = len(v) * (DUMP_LIMIT_BYTES - 4096) // total
            v = v[np.sort(np.random.default_rng(0).choice(len(v), keep, replace=False))]
        np.save(os.path.join(d, name + ".npy"), v)
    np.save(os.path.join(d, "stats.npy"), np.array([[float(s[f]) for f in STAT_FIELDS] for s in out[4]]))


def make_workload(n, m, k, w, seed):
    from fpsb200 import models
    A = models.window_random_jacobian(m, n, k, w=w, seed=seed)
    coo = A.tocoo()
    rng = np.random.default_rng(seed)
    rhs1 = rng.standard_normal(n)
    rhs2 = rng.standard_normal(m)
    return A, coo.row.astype(np.int64), coo.col.astype(np.int64), coo.data.astype(np.float64), rhs1, rhs2


def algorithmic_bytes(n, m, nnz, it0, it1, delta):
    """SURVEY §8(d) ideal-fusion bytes of one fused LSQR(A') + CRAIG(A) solve: every launch of the
    step kernel streams the matrix once (12 B/nnz + row pointers); LSQR touches u (n) r/w in the
    n-space kernel and v, w, x (m) r/w in the m-space kernel; CRAIG touches v, x (+w2 if delta != 0)
    in n-space and Mu, w, y in m-space.  Gathers (L2/L1 hits) are not counted."""
    both = min(it0, it1)
    only0 = max(it0 - it1, 0)
    only1 = max(it1 - it0, 0)
    mat_n = 12 * nnz + 4 * (n + 1)     # rows of A' (n-space kernel)
    mat_m = 12 * nnz + 4 * (m + 1)     # rows of A  (m-space kernel)
    lsqr_n, lsqr_m = 16 * n, 48 * m
    craig_n, craig_m = (48 if delta != 0 else 32) * n, 48 * m
    launches = 1 + 2 * max(it0, it1)
    total = mat_m + 16 * m             # LSQR init: v1 = A u1 (write v), read u via gather
    total += both * (mat_n + mat_m + lsqr_n + lsqr_m + craig_n + craig_m)
    total += only0 * (mat_n + mat_m + lsqr_n + lsqr_m)
    total += only1 * (mat_n + mat_m + craig_n + craig_m)
    return total, launches


class NvmlClockSampler:
    """In-process NVML sampler (pynvml): SM clock, max SM clock and the clock-event reasons every 10 ms while the timed
    region runs.  nvidia-smi takes longer to start than a short timed region lasts (0 samples at 8 GPUs); NVML does not."""
    _REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index, uuid=None):
        import pynvml
        self.nv = pynvml
        pynvml.nvmlInit()
        self.h = None
        if uuid:
            for cand in (f"GPU-{uuid}", str(uuid)):
                try:
                    self.h = pynvml.nvmlDeviceGetHandleByUUID(cand.encode())
                    break
                except Exception:      # noqa: BLE001
                    try:
                        self.h = pynvml.nvmlDeviceGetHandleByUUID(cand)
                        break
                    except Exception:  # noqa: BLE001
                        pass
        if self.h is None:
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        self._reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons")
        self.sm, self.bits, self.run = [], 0, False

    def _sample(self):
        self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
        self.bits |= int(self._reasons_fn(self.h))

    def _loop(self):
        while self.run:
            try:
                self._sample()
            except Exception:          # noqa: BLE001
                pass
            time.sleep(0.01)

    def start(self):
        self.run = True
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()

    def stop(self):
        self.run = False
        self.th.join(timeout=1.0)
        reasons = sorted(name for bit, name in self._REASONS.items() if self.bits & bit)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx,
                "samples": len(self.sm), "reasons": reasons, "source": "nvml"}


def make_clock_sampler(torch, gpu_index):
    try:
        uuid = str(torch.cuda.get_device_properties(gpu_index).uuid)
        return NvmlClockSampler(gpu_index, uuid)
    except Exception:                  # noqa: BLE001
        return ClockSampler(gpu_index)


class ClockSampler:
    """nvidia-smi clock/throttle sampler running during the timed region (fallback when NVML is not importable)."""

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def oracle_solve_timer(A, rhs1, rhs2, delta):
    """Returns a closure running one full solve_two_mixed on the CPU oracle (1 thread)."""
    from oracle import oracle as O
    O.build()
    it = O.IterativeOracle(A)

    def run():
        t = time.perf_counter()
        out = it.solve_two_mixed(delta, rhs1, rhs2)
        return time.perf_counter() - t, out[4]
    return run


def run_reference(args, cfg):
    """CPU arm: the oracle's C port of LSQR + CRAIG (Krylov.jl restated) on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # all the host threads the path can use: the OpenMP build of the port (row loops of the two SpMVs and the
    # element-wise / reduction loops of LSQR and CRAIG); the sequential build stays the checker of the tests.
    # torchrun exports OMP_NUM_THREADS=1 to every rank: only rank 0 works here (the others returned above), so it
    # takes the whole box — the same baseline at every N
    os.environ.setdefault("FPS_ORACLE_OMP", "1")
    ncores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    os.environ["OMP_NUM_THREADS"] = str(ncores)
    n, m, k, w = cfg["n"], cfg["m"], cfg["nnz_per_row"], cfg["window"]
    A, jrow, jcol, vals, rhs1, rhs2 = make_workload(n, m, k, w, args.seed)
    run = oracle_solve_timer(A, rhs1, rhs2, args.delta)
    from oracle import oracle as _O
    _O.lib()
    threads = 1
    if _O.THREADED:
        gomp = ctypes.CDLL("libgomp.so.1")
        gomp.omp_set_num_threads(ncores)
        threads = int(gomp.omp_get_max_threads())
    for _ in range(args.warmup):
        run()
    times, st = [], None
    for _ in range(args.steps):
        t, st = run()
        times.append(t)
    tot = sum(times)
    val = args.steps / tot
    line = {
        "impl": "reference", "metric": "2-RHS KKT solves/s", "value": val, "unit": "solves/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": val, "unit": "solves/s", "cores": threads, "kind": "port",
                         "sample": f"{args.steps} full-size solve_two_mixed calls (LSQR {st[0]['niter']} it + "
                                   f"CRAIG {st[1]['niter']} it), oracle/fps_oracle.c"
                                   + (f" built with OpenMP, {threads} threads" if threads > 1 else ", 1 thread")
                                   + f" of {os.cpu_count()} host cores; the Julia reference is not runnable here "
                                     "(its own path is single-threaded apart from BLAS-1)"},
        "e2e": {"value": val, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def bind_to_gpu_numa_node(torch, local_rank):
    """Run this rank's host threads on the CPUs of the NUMA node its GPU hangs off (sysfs: the PCI device's
    local_cpulist), BEFORE any host buffer is allocated: first-touch then places the pinned e2e buffers on that node,
    so that at N > 1 the H2D / D2H copies of the ranks do not all cross one socket's memory controller.
    Returns what was done for the JSON line; never fatal (containers may hide sysfs or restrict the cpuset)."""
    info = {"bound": False}
    try:
        p = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        base = "/sys/bus/pci/devices/" + bdf
        node = int(open(base + "/numa_node").read().strip())
        cpulist = open(base + "/local_cpulist").read().strip()
        cpus = set()
        for part in cpulist.split(","):
            if not part:
                continue
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        info.update({"pci": bdf, "numa_node": node, "local_cpus": len(cpus), "allowed_cpus": len(allowed)})
        if node >= 0 and len(use) >= 4 and use != allowed:
            os.sched_setaffinity(0, use)
            info["bound"] = True
            info["cpus_used"] = len(use)
    except Exception as e:      # noqa: BLE001
        info["error"] = repr(e)[:120]
    return info


def partitioned_operators(args):
    """The two operators of the strong-scaled row-partitioned record (SURVEY 8 e1): BASELINE config C3
    (Poisson-constrained control, state / control interleaved -> banded Jacobian) and the headline matrix."""
    from fpsb200 import models

    def c3():
        N = args.part_grid
        A = models.poisson_control(N).A.tocsr()
        m, n = A.shape
        perm = np.empty(n, dtype=np.int64)
        perm[:m] = 2 * np.arange(m)
        perm[m:] = 2 * np.arange(m) + 1
        coo = A.tocoo()
        return (f"C3 poisson-control grid {N}x{N}: n={n} m={m} nnz={A.nnz}", n, m, coo.row.astype(np.int64), perm[coo.col],
                coo.data.astype(np.float64), 1e-2, args.part_iters)

    def headline():
        n, m, k, w = args.n, args.m, args.nnz_per_row, args.window
        A, jr, jc, vals, _, _ = make_workload(n, m, k, w, args.seed)
        return (f"headline window-random Jacobian n={n} m={m} nnz={m * k}", n, m, jr, jc, vals, args.delta, 0)
    return [c3, headline]


def run_partitioned(args, dist, rank, world, local_rank, make):
    """One strong-scaled solve_two_mixed of the row-partitioned Krylov path on `world` GPUs (peer-memory halo
    exchange + all-reduced inner products), the same operator on ONE GPU (rank 0, the plain single-GPU handle),
    and the parity of the two results, all inside this torchrun.  itmax > 0: fixed iteration count (timing of
    an operator the reference tolerances do not converge on in a bench-sized run); 0: reference tolerances."""
    import torch
    import fpsb200
    from fpsb200 import _lib
    from fpsb200.partition import RowPartition, DistHandle
    name, n, m, jr, jc, vals, delta, itmax = make()
    dev = torch.device("cuda", local_rank)
    lib = _lib.lib()
    o = _lib.IterOpts()
    _lib.check(lib.fpsb_iter_default_opts(ctypes.c_int64(n), ctypes.c_int64(m), ctypes.byref(o)), "fpsb_iter_default_opts")
    if itmax > 0:       # timing run of exactly itmax iterations with BOTH slots alive: no early exit of either method
        o.ls_itmax = itmax
        o.ln_itmax = itmax
        o.ls_atol = o.ls_rtol = 0.0
        o.ln_atol = o.ln_rtol = o.ln_btol = 0.0
        o.ln_conlim = 1e300
    rng = np.random.default_rng(args.seed)
    g1, g2 = rng.standard_normal(n), rng.standard_normal(m)
    part = RowPartition(n, m, jr, jc, world)
    D = DistHandle(part, rank, device=local_rank, dist=dist, opts=o, peer=True)
    D.set_jac_values(vals)
    L = D.loc
    r1, r2 = g1[L.col0:L.col0 + L.n_own], g2[L.row0:L.row0 + L.m_loc]
    D.solve_two_mixed(delta, r1, r2)
    ts = []
    for _ in range(3):
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        out = D.solve_two_mixed(delta, r1, r2)
        ts.append(D.H.iter_last_profile()[0])
    t = torch.tensor([min(ts)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    loop_ms = float(t.item())
    iters = [out[4][0]["niter"], out[4][1]["niter"]]
    # per-launch shares (one extra solve with an event after every launch; max over ranks)
    lib.fpsb_dist_profile(1)
    torch.cuda.synchronize(); dist.barrier()
    D.solve_two_mixed(delta, r1, r2)
    fallback_ms = torch.tensor([D.H.iter_last_profile()[0]], dtype=torch.float64, device=dev)
    dist.all_reduce(fallback_ms, op=dist.ReduceOp.MAX)
    lib.fpsb_dist_profile(0)
    us4 = (ctypes.c_double * 4)(); c4 = (ctypes.c_int64 * 4)()
    lib.fpsb_dist_last_profile(us4, c4)
    t4 = torch.tensor(list(us4), dtype=torch.float64, device=dev)
    dist.all_reduce(t4, op=dist.ReduceOp.MAX)
    shares = dict(zip(["step_n_us", "xchg_after_n_us", "step_m_us", "xchg_after_m_us"], [float(x) for x in t4.tolist()]))
    transport = "peer-memory (CUDA IPC mailboxes over NVLink)" if D.peer else "nccl"
    halo = int(L.n_ext - L.n_own)
    # ---- the same operator on one GPU (rank 0), then its solution to everybody for the parity check
    full = [torch.empty(k, dtype=torch.float64, device=dev) for k in (n, m, n, m)]
    single = torch.zeros(3, dtype=torch.float64, device=dev)
    if rank == 0:
        H1 = fpsb200.B200Handle(n, m, jr, jc, device=local_rank)
        H1.iter_setup(o)
        H1.set_jac_values(vals)
        d1, d2 = torch.tensor(g1, device=dev), torch.tensor(g2, device=dev)
        o1 = H1.iter_solve_two_mixed(delta, d1, d2)
        t1 = []
        for _ in range(3):
            torch.cuda.synchronize()
            o1 = H1.iter_solve_two_mixed(delta, d1, d2)
            t1.append(H1.iter_last_profile()[0])
        for k in range(4):
            full[k].copy_(o1[k])
        single[0], single[1], single[2] = min(t1), o1[4][0]["niter"], o1[4][1]["niter"]
        H1.synchronize()
        del H1
    torch.cuda.synchronize()
    dist.broadcast(single, src=0)
    err = torch.zeros(8, dtype=torch.float64, device=dev)
    sl = [(L.col0, L.n_own), (L.row0, L.m_loc), (L.col0, L.n_own), (L.row0, L.m_loc)]
    for k in range(4):
        dist.broadcast(full[k], src=0)
        ref = full[k][sl[k][0]:sl[k][0] + sl[k][1]]
        mine = torch.tensor(out[k], device=dev)
        err[2 * k] = torch.sum((mine - ref) ** 2)
        err[2 * k + 1] = torch.sum(ref ** 2)
    dist.all_reduce(err, op=dist.ReduceOp.SUM)
    e = err.tolist()
    rel = [float(np.sqrt(e[2 * k] / e[2 * k + 1])) if e[2 * k + 1] > 0 else float(np.sqrt(e[2 * k])) for k in range(4)]
    it1 = [int(single[1].item()), int(single[2].item())]
    nit, nit1 = max(iters), max(it1)
    in_kernel = bool(D.peer) and os.environ.get("FPSB_DIST_LOOP", "1") != "0"
    del D
    torch.cuda.synchronize(); dist.barrier()
    us, us1 = 1e3 * loop_ms / max(nit, 1), 1e3 * float(single[0].item()) / max(nit1, 1)
    xs = shares["xchg_after_n_us"] + shares["xchg_after_m_us"]
    return {
        "workload": name, "path": "row-partitioned solve_two_mixed (LSQR(A') + CRAIG(A) in lock step), strong scaling",
        "n_gpus": world, "transport": transport, "halo_entries_rank0": halo,
        "stopping": f"fixed {itmax} iterations (tolerances 0, conlim off: both methods run every iteration)" if itmax > 0 else "reference tolerances sqrt(eps)",
        "iterations": iters, "krylov_loop_ms": loop_ms, "us_per_iteration": us,
        "single_gpu": {"iterations": it1, "krylov_loop_ms": float(single[0].item()), "us_per_iteration": us1,
                       "what": "the same operator on rank 0's GPU through the plain (unpartitioned) handle"},
        "speedup_vs_single_gpu": us1 / us if us > 0 else None,
        "kernel": "one persistent kernel per chunk of 24 iterations on every rank; its CTA 0 does the halo scatter-add, the halo "
                  "gather and the all-reduce of the four inner products through the peers' mailboxes (NVLink), the boundary rows "
                  "are shared out over 16 helper CTAs (long boundaries only), the other CTAs wait for CTA 0's release instead of "
                  "the grid barrier" if in_kernel
                  else "launch per half iteration (step kernel + exchange kernel)",
        "launch_per_half_iteration_path": {"us_per_iteration": 1e3 * float(fallback_ms.item()) / max(nit, 1),
                                           "per_launch_us_max_over_ranks": shares,
                                           "what": "the same solve with a kernel launch per half iteration and a separate exchange kernel "
                                                   "(round 1's path, still the fallback for operators with long rows): one profiled run"},
        "per_launch_us_max_over_ranks": shares,
        "exchange_share": xs / max(xs + shares["step_n_us"] + shares["step_m_us"], 1e-30),
        "parity": {"rel_err_p1_q1_p2_q2_vs_single_gpu": rel, "max_rel_err": max(rel), "tol": 1e-6,
                   "iterations_equal": iters == it1, "ok": bool(max(rel) <= 1e-6 and iters == it1)},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--m", type=int, default=500_000)
    ap.add_argument("--nnz-per-row", type=int, default=20)
    ap.add_argument("--window", type=int, default=64)
    ap.add_argument("--delta", type=float, default=0.0)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--cpu-baseline-solves", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ldlt", action="store_true", help="skip the LDLt-path extra measurements")
    ap.add_argument("--ldlt-amd", action="store_true", help="also time the LDLt path with the AMD ordering")
    ap.add_argument("--e2e-serial", action="store_true", help="e2e with one solve in flight only")
    ap.add_argument("--no-partitioned", action="store_true", help="N>1: skip the strong-scaled row-partitioned record")
    ap.add_argument("--part-grid", type=int, default=2048, help="grid of the C3 operator of the partitioned record")
    ap.add_argument("--part-iters", type=int, default=100, help="fixed Krylov iterations of the C3 partitioned run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) to DIR/<name>.npy, to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")

    n, m, k, w = args.n, args.m, args.nnz_per_row, args.window
    cfg = {"workload": "C4-shape synthetic sparse equality-constrained problem: window-random Jacobian "
                       f"n={n} m={m} nnz={m * k} ({k}/row, |j-2i|<={w}), N(0,1) values, seed {args.seed}; "
                       "step = solve_two_mixed (Jacobian refresh + LSQR/CRAIG 2-RHS solve), Krylov path, "
                       f"reference tolerances sqrt(eps), delta={args.delta}",
           "n": n, "m": m, "nnz": m * k, "nnz_per_row": k, "window": w, "delta": args.delta,
           "l2_policy": "inputs larger than L2 (tile blocks of A and A' = 200 MB + 100 MB of Krylov vectors streamed every iteration vs 126 MB L2)",
           "parallelism": f"{args.gpus} independent instance(s), one per GPU, no collective"}
    if args.impl == "reference":
        run_reference(args, cfg)
        return

    import torch
    import fpsb200
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(torch, local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    A, jrow, jcol, vals, rhs1, rhs2 = make_workload(n, m, k, w, args.seed + rank)
    nnz = len(vals)
    H = fpsb200.B200Handle(n, m, jrow, jcol, device=local_rank)
    H.iter_setup(None)
    dev = torch.device("cuda", local_rank)
    d_vals = torch.tensor(vals, device=dev)
    d_r1 = torch.tensor(rhs1, device=dev)
    d_r2 = torch.tensor(rhs2, device=dev)
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        H.set_jac_values(d_vals)
        return H.iter_solve_two_mixed(args.delta, d_r1, d_r2)

    # e2e buffers: long-lived host arrays, page-locked once (what the Julia shim does with its
    # solver-owned vectors) so the copies inside the timed region are plain DMA
    h_out = [np.empty(n), np.empty(m), np.empty(n), np.empty(m)]
    for a in [vals, rhs1, rhs2] + h_out:
        H.pin_host(a)

    def step_host():
        H.set_jac_values(vals)
        return H.iter_solve_two_mixed(args.delta, rhs1, rhs2, out=h_out)

    # ---- resident (value) -------------------------------------------------------------------
    import gc
    for _ in range(max(args.warmup, 3)):
        out = step_resident()
    gc.collect()
    gc.disable()          # no collector pause inside the timed regions (re-enabled after the e2e measurement)
    sampler = make_clock_sampler(torch, local_rank)
    barrier()
    sampler.start()
    l0 = H.launch_count()
    loop_ms, step_launches = 0.0, 0
    H.timer_start()
    for _ in range(args.steps):
        out = step_resident()
        ms, nl = H.iter_last_profile()
        loop_ms += ms
        step_launches += nl
    dev_ms = H.timer_stop()
    barrier()
    clocks = sampler.stop()
    launches = H.launch_count() - l0
    last_out = out
    st = out[4]
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    max_ms = float(t.item())

    # ---- end to end through the C ABI with host buffers ----------------------------------------
    # (a) one solve at a time: H2D -> solve -> D2H strictly serial on the handle's stream (the latency a single
    #     caller sees);  (b) the throughput figure: two handles on the same sparsity pattern, each driven by its own
    #     host thread (ctypes releases the GIL), so the PCIe copies of one step overlap the Krylov loop of the
    #     other.  Every step still copies its own inputs H2D and its own results D2H inside the timed region.
    for _ in range(2):
        step_host()
    barrier()
    t0 = time.perf_counter()
    H.timer_start()
    for _ in range(args.steps):
        step_host()
    e2e1_dev_ms = H.timer_stop()
    e2e1_wall_ms = 1e3 * (time.perf_counter() - t0)
    barrier()
    e2e_serial_ms = max(e2e1_dev_ms, e2e1_wall_ms)
    in_flight = 1 if args.e2e_serial else 2
    if in_flight == 2:
        # two fresh handles on the same sparsity pattern (H itself stays the single-caller handle of the other measurements)
        H2 = fpsb200.B200Handle(n, m, jrow, jcol, device=local_rank)
        H3 = fpsb200.B200Handle(n, m, jrow, jcol, device=local_rank)
        H2.iter_setup(None)
        H3.iter_setup(None)
        h_out2 = [np.empty(n), np.empty(m), np.empty(n), np.empty(m)]
        h_out3 = [np.empty(n), np.empty(m), np.empty(n), np.empty(m)]
        for a in h_out2 + h_out3:
            H.pin_host(a)
        lanes = [(H3, h_out3), (H2, h_out2)]
        errs = []
        # fpsb_pipeline_gate: one solve computes at a time, the copies of the other lane ride on the copy engines under it.
        # Without the turn-taking both loops interleave chunk by chunk, finish together and copy together: how much overlap
        # is left is luck (measured box to box: 148-182 solves/s for the same build).
        fpsb200._lib.lib().fpsb_pipeline_gate(0 if os.environ.get("FPSB_BENCH_NO_GATE") else 1)

        def lane(i, count):
            try:
                torch.cuda.set_device(local_rank)
                Hi, oi = lanes[i]
                for _ in range(count):
                    Hi.set_jac_values(vals)
                    Hi.iter_solve_two_mixed(args.delta, rhs1, rhs2, out=oi)
            except Exception as e:      # noqa: BLE001
                errs.append(repr(e))

        def run_lanes(total):
            ths = [threading.Thread(target=lane, args=(i, (total + 1 - i) // 2)) for i in range(2)]
            for th in ths:
                th.start()
            for th in ths:
                th.join()
        run_lanes(4)
        barrier()
        t0 = time.perf_counter()
        run_lanes(args.steps)
        torch.cuda.synchronize()
        e2e_ms = 1e3 * (time.perf_counter() - t0)
        barrier()
        if errs or not all(np.array_equal(a, b) and np.array_equal(a, c) for a, b, c in zip(h_out, h_out2, h_out3)):
            raise SystemExit(f"bench.py: pipelined e2e lanes failed or disagree: {errs}")
        lanes.clear()
        fpsb200._lib.lib().fpsb_pipeline_gate(0)
        for a in h_out2 + h_out3:
            H.unpin_host(a)
        H2.close()          # (their L2 persistence windows must not shrink the cache of the measurements that follow)
        H3.close()
        del H2, H3
    else:
        e2e_ms = e2e_serial_ms
    gc.enable()
    t = torch.tensor([e2e_ms, e2e_serial_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms, e2e_serial_ms = float(t[0].item()), float(t[1].item())

    # ---- N > 1: the path that needs collectives (row-partitioned Krylov, strong scaling), next to the replicas
    partitioned = None
    if dist is not None and not args.no_partitioned:
        partitioned = []
        for make in partitioned_operators(args):
            try:
                partitioned.append(run_partitioned(args, dist, rank, world, local_rank, make))
            except Exception as e:       # never take the headline line down
                partitioned.append({"error": repr(e)})
                break
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
        dist = None
    if rank != 0:
        return

    # ---- roofline of the dominant kernel (fused SpMM step) ---------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    traffic, traffic_src = None, None
    try:        # DRAM bytes per half iteration of the same kernel from the committed ncu --set full capture (headline shape only)
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if (n, m, k) == (1_000_000, 500_000, 20):
            traffic = float(tj["dram_bytes_per_launch"])
            traffic_src = "static: " + tj.get("source", "profiles/traffic.json (ncu --set full capture of this kernel, not measured in this run)")
    except Exception:
        pass
    tot_bytes, eff_launches = algorithmic_bytes(n, m, nnz, st[0]["niter"], st[1]["niter"], args.delta)
    loop_ms_per_solve = loop_ms / args.steps
    achieved = tot_bytes / (loop_ms_per_solve * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": "gk_loop_kernel (persistent Krylov loop: fused 2-column SpMM + Krylov row epilogue + scalar recurrences, "
                                  "one launch per chunk of 24 iterations; a 'launch' below is one half iteration = one pass over A or A')",
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "frac_of_nominal_8000": achieved / 8000.0, "peak_source": peak_src,
        "traffic": traffic, "traffic_static": traffic is not None, "traffic_source": traffic_src,
        "bytes_per_launch": tot_bytes / eff_launches,
        "avg_launch_us": 1e3 * loop_ms_per_solve / eff_launches,
        "launches_per_solve": eff_launches,
        "launched_incl_post_convergence_noops": step_launches / args.steps,
        "iters": {"lsqr": st[0]["niter"], "craig": st[1]["niter"]},
        "note": "achieved = SURVEY 8(d) algorithmic bytes of the whole Krylov loop / CUDA-event time of "
                "that loop on the handle's stream (includes host polling gaps and the no-op launches "
                "queued after convergence)",
    }

    # ---- extras: SpMV and the LDLt path on the same matrix ------------------------------------------
    extra = {}
    if args.gpus > 1:            # scaling runs: headline only (extras / CPU baseline are N=1 work)
        args.no_ldlt = True
        args.no_cpu_baseline = True
    try:
        if args.gpus > 1:
            raise RuntimeError("skipped at N>1")
        gc.collect()                           # the e2e lanes' handles and buffers go now, not inside a timed extra
        gc.disable()                           # (a generation-2 pass between two launches reads as 25 ms of 'kernel' time)
        torch.cuda.synchronize()
        t_warm = time.perf_counter()           # the e2e phase above is PCIe-bound: let the SM clocks ramp up again
        while time.perf_counter() - t_warm < 0.5:
            step_resident()
        reps = 100                             # (20 left 1-2 us of event / launch-pipeline start-up in every figure)
        for _ in range(5):
            H.jprod(d_r1); H.jtprod(d_r2)
        H.timer_start()
        for _ in range(reps):
            y = H.jprod(d_r1)
        ms = H.timer_stop() / reps
        b = 12 * nnz + 4 * (m + 1) + 8 * n + 8 * m
        extra["spmv_A"] = {"us": 1e3 * ms, "GB/s": b / ms / 1e6, "frac_of_measured_peak": b / ms / 1e6 / peak}
        H.timer_start()
        for _ in range(reps):
            y = H.jtprod(d_r2)
        ms = H.timer_stop() / reps
        b = 12 * nnz + 4 * (n + 1) + 8 * n + 8 * m
        extra["spmv_At"] = {"us": 1e3 * ms, "GB/s": b / ms / 1e6, "frac_of_measured_peak": b / ms / 1e6 / peak}
        d_r3 = torch.tensor(np.random.default_rng(7).standard_normal(n), device=dev)
        for _ in range(3):
            H.iter_solve_two_least_squares(args.delta, d_r1, d_r3)
        per_call = []
        for _ in range(7):            # per-call device times: one host hiccup (allocator, GC) must not pass for kernel time
            H.timer_start()
            o2 = H.iter_solve_two_least_squares(args.delta, d_r1, d_r3)
            per_call.append(H.timer_stop())
        ms = float(np.median(per_call))
        extra["iter_solve_two_least_squares"] = {"ms": ms, "solves/s": 1e3 / ms, "ms_max_of_7": max(per_call),
                                                 "krylov_loop_ms_last": H.iter_last_profile()[0],
                                                 "iters": [o2[4][0]["niter"], o2[4][1]["niter"]]}
    except Exception as e:   # extras must never take the headline down
        extra["error_spmv"] = repr(e)
    if not args.no_ldlt:
        try:
            from fpsb200.symbolic import SymbolicAnalysis, order_dissection
            sym_N = n + m
            t0 = time.perf_counter()
            Pd = order_dissection(n, m, jrow, jcol)
            extra["ldlt_order_dissection_host_s"] = time.perf_counter() - t0
            t0 = time.perf_counter()
            H.ldlt_analyze(Pd)
            extra["ldlt_analyze_host_s"] = time.perf_counter() - t0
            lnz = int(H.ldlt_symbolic()["Lp"][-1])
            extra["ldlt_plan_dissection"] = dict(H.ldlt_plan_info(), lnz=lnz)
            for _ in range(2):
                H.ldlt_solve_two_mixed(SQRT_EPS, d_r1, d_r2)
            per_call = []
            for _ in range(5):        # per-call device times, median (see the two-LSQR extra)
                H.timer_start()
                H.set_jac_values(d_vals)
                o3 = H.ldlt_solve_two_mixed(SQRT_EPS, d_r1, d_r2)
                per_call.append(H.timer_stop())
            ms = float(np.median(per_call))
            extra["ldlt_solve_two_mixed"] = {"ms": ms, "solves/s": 1e3 / ms, "ms_all": [round(x, 2) for x in per_call],
                                             "factorized": bool(o3[4]),
                                             "delta": SQRT_EPS, "ordering": "dissection",
                                             "GFLOP/s": extra["ldlt_plan_dissection"]["flops"] / ms / 1e6}
            per_call = []
            for _ in range(7):
                H.timer_start()
                o3 = H.ldlt_solve_two_least_squares(d_r1, d_r3)
                per_call.append(H.timer_stop())
            ms = float(np.median(per_call))
            sb = 24 * lnz + 88 * sym_N
            extra["ldlt_solve_two_least_squares"] = {"ms": ms, "solves/s": 1e3 / ms, "ms_max_of_7": max(per_call), "GB/s": sb / ms / 1e6,
                                                     "frac_of_measured_peak": sb / ms / 1e6 / peak,
                                                     "ordering": "dissection"}
            res = o3[0] + H.jtprod(o3[1]) - d_r1          # K-residual of the first system, on the device
            extra["ldlt_residual_rel"] = float(torch.linalg.norm(res) / torch.linalg.norm(d_r1))
            if args.ldlt_amd:
                H.ldlt_analyze()
                extra["ldlt_plan_amd"] = dict(H.ldlt_plan_info(), lnz=int(H.ldlt_symbolic()["Lp"][-1]))
                H.timer_start()
                o3 = H.ldlt_solve_two_mixed(SQRT_EPS, d_r1, d_r2)
                extra["ldlt_solve_two_mixed_amd_ms"] = H.timer_stop()
        except Exception as e:
            extra["error_ldlt"] = repr(e)

    gc.enable()
    # ---- CPU baseline (oracle port, bounded sample) -------------------------------------------------
    cpu = None
    if not args.no_cpu_baseline:
        # the OpenMP build of the port with every host thread (what --impl reference times), plus one solve on a
        # single thread: the reference's own path is single-threaded apart from BLAS-1
        os.environ.setdefault("FPS_ORACLE_OMP", "1")
        run = oracle_solve_timer(A, rhs1, rhs2, args.delta)
        from oracle import oracle as _O
        _O.lib()
        threads, t1 = 1, None
        if _O.THREADED:
            import ctypes
            gomp = ctypes.CDLL("libgomp.so.1")
            threads = int(gomp.omp_get_max_threads())
            gomp.omp_set_num_threads(1)
            t1, _ = run()
            gomp.omp_set_num_threads(threads)
            run()                                    # warm the thread pool
        ts, ost = [], None
        for _ in range(args.cpu_baseline_solves):
            tt, ost = run()
            ts.append(tt)
        cpu = {"value": len(ts) / sum(ts), "unit": "solves/s", "cores": threads, "kind": "port",
               "sample": f"{len(ts)} full-size solve_two_mixed calls ({sum(ts):.1f} s; LSQR {ost[0]['niter']} it + "
                         f"CRAIG {ost[1]['niter']} it) with oracle/fps_oracle.c, gcc -O3"
                         + (f" -fopenmp, {threads} threads" if threads > 1 else ", 1 thread")
                         + f" of {os.cpu_count()} host cores (Julia absent)"}
        if t1 is not None:
            cpu["single_thread_value"] = 1.0 / t1

    value = args.gpus * args.steps / (max_ms * 1e-3)
    e2e_value = args.gpus * args.steps / (e2e_ms * 1e-3)
    line = {
        "metric": "2-RHS KKT solves/s", "value": value, "unit": "solves/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": max_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": cfg, "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "solves/s",
                "h2d_bytes_per_step": 8 * (nnz + n + m), "d2h_bytes_per_step": 16 * (n + m),
                "ms_per_step": e2e_ms / args.steps, "solves_in_flight": in_flight,
                "one_at_a_time": {"value": args.gpus * args.steps / (e2e_serial_ms * 1e-3), "ms_per_step": e2e_serial_ms / args.steps},
                "host_numa": numa,
                "note": "host buffers through the C ABI; every step copies its Jacobian values + both rhs H2D and its four "
                        "result vectors D2H inside the timed region; value = two independent solves in flight per GPU (two "
                        "handles, two host threads, fpsb_pipeline_gate on: one solve computes at a time) so that the copies of "
                        "one overlap the Krylov loop of the other; one_at_a_time = the strictly serial figure"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "solver_stats": {"lsqr": st[0], "craig": st[1]},
        "extra": extra,
    }
    if partitioned is not None:
        line["partitioned"] = partitioned
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_out)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
