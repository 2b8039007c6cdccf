"""The multi-column set on slab-sharded handles (run under torchrun, one rank per GPU).

For C5 (weak: 2^24 DG p=3 elements per GPU) and C4 (strong: one 2^26-element CG-first problem over all ranks) and each
column count k, on one sharded handle:
  - ms per V-cycle and column of the set (dev_vcycle_multi / k; slab edges through NCCL), next to the resident
    single-column cycle (dev_vcycle; slab edges through peer memory where the ranks could map each other's arenas);
  - seconds to tol = 1e-10 for the k columns through one dev_pcg_multi call, next to k sequential dev_pcg calls,
    alternated, with a check that every column's iteration count and residual history are bit-identical.
With --t-k8 also T (2^26 DG p=3 elements over all ranks) with k = 8 through dev_pcg_multi: device_bytes per rank and
time, or the error when the storage does not fit.  A set or CG storage that does not fit on one rank makes every rank
return AMG1D_ERR_NOMEM (the library agrees on the outcome), so all ranks skip that k together.

Times: host clock from a barrier of all ranks to the end of the work on this rank (a stream synchronisation); the
slowest rank counts.  The columns are seeded host vectors, every rank its own slab.  The card's name and power limit
are read in the same run.

    torchrun --nproc-per-node=2 tools/bench_dist_multi.py --t-k8        (writes profiles/r06_bench_dist_multi_w2.json)
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload definitions)
from agglomerationmultigrid1d_b200 import _capi as capi  # noqa: E402

SEED = 4321
TOL = 1e-10


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        cards = []
        for line in out:
            name, power, clock = [s.strip() for s in line.split(",")]
            cards.append({"name": name, "power_limit": power, "max_sm_clock": clock})
        return cards
    except Exception as e:          # the numbers below are then without their card: say so
        return [{"name": "unknown", "error": str(e)}]


def slowest(t):
    out = [None] * dist.get_world_size()
    dist.all_gather_object(out, t)
    return max(out)


def timed(dev, fn):
    dev.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    r = fn()
    dev.synchronize()
    return slowest(time.perf_counter() - t0), r


def nccl_id():
    ids = [None]
    if dist.get_rank() == 0:
        buf = C.create_string_buffer(128)
        capi.check(None, capi.load().amg1d_nccl_unique_id(C.cast(buf, C.c_void_p)))
        ids[0] = buf.raw
    dist.broadcast_object_list(ids, src=0)
    return ids[0]


def upload(name, n):
    rank, world = dist.get_rank(), dist.get_world_size()
    U = bench.build_hierarchy(name, n)
    dev = U.upload(device=rank, dist=(rank, world, nccl_id()))
    dev.synchronize()
    return dev


def columns(dev, k):
    rank = dist.get_rank()
    B = np.empty((dev.n_dof[0], k), order="F")
    for c in range(k):
        B[:, c] = np.random.default_rng([SEED + c, rank]).standard_normal(dev.n_dof[0])
    return B


def pcg_pair(dev, B, maxiter):
    k = B.shape[1]

    def multi():
        dev.dev_set_problems(None, B)
        return timed(dev, lambda: dev.dev_pcg_multi(maxiter, TOL))

    def sequential():
        t, its, rs = 0.0, [], []
        for c in range(k):
            dev.dev_set_problem(None, B[:, c])
            dt, (it, r) = timed(dev, lambda: dev.dev_pcg(maxiter, TOL))
            t += dt
            its.append(it)
            rs.append(r)
        return t, (its, rs)
    return multi, sequential


def bench_workload(name, ks, reps, maxiter, cycles):
    world = dist.get_world_size()
    log2n = bench.WORKLOADS[name][0]
    n = 1 << (log2n if name in bench.STRONG else log2n + world.bit_length() - 1)
    t0 = time.perf_counter()
    dev = upload(name, n)
    rec = {"workload": bench.WORKLOADS[name][3], "n_elements": n, "ranks": world,
           "scaling": "strong" if name in bench.STRONG else "weak", "local_dofs": dev.info("local_dofs"),
           "sharded_levels": dev.info("sharded_levels"), "gather_level": dev.info("gather_level"),
           "p2p_halo_resident": dev.info("p2p_halo"), "setup_s": round(time.perf_counter() - t0, 1), "k": {}}
    B1 = columns(dev, 1)
    dev.dev_set_problem(None, B1[:, 0])
    dev.dev_vcycle()
    t, _ = timed(dev, lambda: [dev.dev_vcycle() for _ in range(cycles)])
    rec["resident_vcycle_ms"] = t / cycles * 1e3
    for k in ks:
        B = columns(dev, k)
        r = {}
        try:
            dev.dev_set_problems(None, B)
            dev.dev_vcycle_multi()
            t, _ = timed(dev, lambda: [dev.dev_vcycle_multi() for _ in range(cycles)])
            r["set_vcycle_ms_per_column"] = t / cycles * 1e3 / k
            r["set_vs_resident_cycle"] = r["set_vcycle_ms_per_column"] / rec["resident_vcycle_ms"]
            r["multi_launches_per_cycle"] = dev.info("multi_launches_per_cycle")
            multi, sequential = pcg_pair(dev, B, maxiter)
            multi()                                   # warm-up: the graphs of this k, the CG vectors
            sequential()
        except capi.Amg1dError as e:
            if e.code != capi.ERR_NOMEM:
                raise
            rec["k"][str(k)] = {"skipped": "ERR_NOMEM: column storage does not fit", "message": str(e)}
            continue
        tm, ts = [], []
        for _ in range(reps):                         # alternate the two on the same handle
            t, (iters_m, res_m) = multi()
            tm.append(t)
            t, (iters_s, res_s) = sequential()
            ts.append(t)
        t_m, t_s = float(np.median(tm)), float(np.median(ts))
        r.update({"iters": iters_m, "pcg_multi_s": t_m, "pcg_multi_s_all": tm, "pcg_sequential_s": t_s,
                  "pcg_sequential_s_all": ts, "pcg_per_column_speedup": t_s / t_m,
                  "check_iters_and_res_bit_identical": bool(
                      iters_m == iters_s and all(np.array_equal(a, b) for a, b in zip(res_m, res_s)))})
        rec["k"][str(k)] = r
        if dist.get_rank() == 0:
            print(json.dumps({"workload": name, "ranks": world, "k": k,
                              "set_ms_per_column": round(r["set_vcycle_ms_per_column"], 3),
                              "resident_ms": round(rec["resident_vcycle_ms"], 3), "pcg_multi_s": round(t_m, 4),
                              "pcg_sequential_s": round(t_s, 4), "check": r["check_iters_and_res_bit_identical"]}),
                  flush=True)
    rec["device_bytes_rank0"] = dev.info("device_bytes")
    dev.close()
    return rec


def t_k8(maxiter):
    """T, one 2^26-element problem over all ranks, 8 columns through dev_pcg_multi."""
    world = dist.get_world_size()
    dev = upload("T", 1 << bench.WORKLOADS["T"][0])
    rec = {"workload": bench.WORKLOADS["T"][3], "ranks": world, "k": 8, "local_dofs": dev.info("local_dofs")}
    B = columns(dev, 8)
    try:
        multi, sequential = pcg_pair(dev, B, maxiter)
        t, (iters, _) = multi()
        rec.update(iters=iters, pcg_multi_s_first_call=t)
        t, (iters, _) = multi()
        rec.update(pcg_multi_s=t)
        t, (iters_s, _) = sequential()
        rec.update(pcg_sequential_s=t, check_iters_equal=iters == iters_s)
    except capi.Amg1dError as e:
        rec.update(error=str(e), code=e.code)
    bytes_all = [None] * world
    dist.all_gather_object(bytes_all, dev.info("device_bytes"))
    rec["device_bytes_per_rank"] = bytes_all
    dev.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="C5,C4")
    ap.add_argument("--ks", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--cycles", type=int, default=20)
    ap.add_argument("--maxiter", type=int, default=200)
    ap.add_argument("--t-k8", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_bench_dist_multi_w{ranks}.json"))
    a = ap.parse_args()
    dist.init_process_group("gloo")
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    out = {"card": card() if dist.get_rank() == 0 else None, "ranks": dist.get_world_size(), "tol": TOL,
           "nPre": 3, "nPost": 3,
           "timing": f"host clock from a barrier of all ranks to a stream synchronisation, slowest rank; V-cycles: "
                     f"{a.cycles} in a row after one warm-up; PCG: median of {a.reps} alternations multi / sequential "
                     f"after one warm-up of each, right-hand side installs outside the clock", "workloads": {}}
    for w in a.workloads.split(","):
        if w:
            out["workloads"][w] = bench_workload(w, [int(k) for k in a.ks.split(",")], a.reps, a.maxiter, a.cycles)
    if a.t_k8:
        out["T_k8"] = t_k8(a.maxiter)
    if dist.get_rank() == 0:
        text = json.dumps(out, indent=1)
        path = a.out.format(ranks=dist.get_world_size())
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:
            f.write(text + "\n")
        print(text)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
