"""Multi-column PCG (amg1d_dev_pcg_multi) against k sequential single-column solves (amg1d_dev_pcg) on the same handle.

For each workload (bench.py's WORKLOADS, one GPU, each at its own size) and each column count k: seconds to
tol = 1e-10 for the k columns through one amg1d_dev_pcg_multi call, next to k sequential amg1d_dev_pcg calls -
alternated in the same process, host clock around calls that end in a stream synchronisation (the right-hand side
uploads and fills are outside the clock).  Beside them the time of one V-cycle for the same k (multi-column and single
column, from the resident iterate), so that the part of a PCG iteration outside the V-cycle can be read off; the launches of one PCG
iteration outside the V-cycle; and an output check: every column's iteration count and residual history, and column
0's solution, bit-identical to the sequential run.  T, C3 and C2 fill their columns on the device
(dev_fill_rhs_random_multi, column c = dev_fill_rhs_random(seed + c)); C4's CG-first level 0 is not supported there,
so its columns are seeded host vectors, uploaded.  A k whose storage does not fit (AMG1D_ERR_NOMEM) is reported as
skipped.

    python tools/bench_pcg_multi.py --workloads T,C3,C2,C4 --ks 1,2,4,8 --out DIR/bench_pcg_multi.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload definitions)
from agglomerationmultigrid1d_b200 import _capi as capi  # noqa: E402

SEED = 4321
TOL = 1e-10


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:          # the numbers below are then without their card: say so
        return {"name": "unknown", "error": str(e)}


class Columns:
    """The k right-hand sides of one workload: filled on the device, or seeded host vectors (CG-first level 0)."""

    def __init__(self, dev, k, host):
        self.dev, self.k, self.host = dev, k, host
        self.B = None
        if host:
            self.B = np.empty((dev.n_dof[0], k), order="F")
            for c in range(k):
                self.B[:, c] = np.random.default_rng(SEED + c).standard_normal(dev.n_dof[0])

    def install_set(self):
        if self.host:
            self.dev.dev_set_problems(None, self.B)
        else:
            self.dev.dev_fill_rhs_random_multi(self.k, SEED)

    def install_single(self, c):
        if self.host:
            self.dev.dev_set_problem(None, self.B[:, c])
        else:
            self.dev.dev_fill_rhs_random(SEED + c)


def timed(fn, dev):
    dev.synchronize()
    t0 = time.perf_counter()
    out = fn()
    dev.synchronize()
    return time.perf_counter() - t0, out


def run_multi(cols, maxiter):
    cols.install_set()
    dev = cols.dev
    t, (iters, res) = timed(lambda: dev.dev_pcg_multi(maxiter, TOL), dev)
    return t, iters, res


def run_sequential(cols, maxiter):
    t, iters, res = 0.0, [], []
    for c in range(cols.k):
        cols.install_single(c)
        dt, (it, r) = timed(lambda: cols.dev.dev_pcg(maxiter, TOL), cols.dev)
        t += dt
        iters.append(it)
        res.append(r)
    return t, iters, res


def vcycle_ms(cols, multi, cycles=10):
    dev = cols.dev
    if multi:
        cols.install_set()
        run = lambda: dev.dev_vcycle_multi()                            # noqa: E731
    else:
        cols.install_single(0)
        run = lambda: dev.dev_vcycle()                                  # noqa: E731
    run()
    t, _ = timed(lambda: [run() for _ in range(cycles)], dev)
    return t / cycles * 1e3


def bench_workload(name, ks, reps, maxiter):
    n = 1 << bench.WORKLOADS[name][0]
    t_setup = time.perf_counter()
    U = bench.build_hierarchy(name, n)
    dev = U.upload()
    host = bool(bench.WORKLOADS[name][1])          # CG-first level 0: columns uploaded from the host
    rec = {"workload": bench.WORKLOADS[name][3], "n_elements": n, "n_dof": dev.n_dof[0],
           "columns": "seeded host vectors, uploaded" if host else "dev_fill_rhs_random_multi",
           "setup_s": round(time.perf_counter() - t_setup, 1), "k": {}}
    for k in ks:
        r = {}
        try:
            cols = Columns(dev, k, host)
            run_multi(cols, maxiter)               # warm-up: the multi-column graphs of this k, the CG vectors
            run_sequential(cols, maxiter)
        except capi.Amg1dError as e:
            if e.code != capi.ERR_NOMEM:
                raise
            rec["k"][str(k)] = {"skipped": "ERR_NOMEM: column storage does not fit", "message": str(e)}
            continue
        tm, ts = [], []
        for _ in range(reps):                      # alternate the two on the same handle
            t, iters_m, res_m = run_multi(cols, maxiter)
            tm.append(t)
            x0_multi = dev.dev_get_solutions()[:, 0].copy()
            t, iters_s, res_s = run_sequential(cols, maxiter)
            ts.append(t)
        launches = dev.info("multi_pcg_launches_per_iteration")   # of the last multi run above
        t_m, t_s = float(np.median(tm)), float(np.median(ts))
        it_sum = sum(iters_s)
        r.update({
            "iters": iters_m,
            "multi_s": t_m, "multi_s_all": tm, "sequential_s": t_s, "sequential_s_all": ts,
            "per_column_s_multi": t_m / k, "per_column_s_sequential": t_s / k,
            "per_column_speedup": t_s / t_m,
            "ms_per_column_iteration_multi": t_m * 1e3 / it_sum if it_sum else None,
            "ms_per_column_iteration_sequential": t_s * 1e3 / it_sum if it_sum else None,
            "vcycle_ms_multi_per_column": vcycle_ms(cols, True) / k,
            "vcycle_ms_single": vcycle_ms(cols, False),
            "multi_pcg_launches_per_iteration": launches,
            "check_iters_and_res_bit_identical": bool(iters_m == iters_s and
                                                      all(np.array_equal(a, b) for a, b in zip(res_m, res_s))),
        })
        cols.install_single(0)
        dev.dev_pcg(maxiter, TOL)
        r["check_column0_solution_bit_identical"] = bool(np.array_equal(x0_multi, dev.dev_get_solution()))
        rec["k"][str(k)] = r
        print(json.dumps({"workload": name, "k": k, "iters": iters_m, "multi_s": round(t_m, 4),
                          "sequential_s": round(t_s, 4), "speedup": round(t_s / t_m, 3),
                          "check": [r["check_iters_and_res_bit_identical"],
                                    r["check_column0_solution_bit_identical"]]}), flush=True)
        del cols
    rec["device_bytes"] = dev.info("device_bytes")
    dev.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="T,C3,C2,C4")
    ap.add_argument("--ks", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--maxiter", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"card": card(), "tol": TOL, "nPre": 3, "nPost": 3,
           "timing": f"host clock around one dev_pcg_multi call / k dev_pcg calls (each ending in a stream "
                     f"synchronisation, right-hand side installs outside the clock), median of {a.reps} alternations "
                     f"multi / sequential on one handle after one warm-up of each", "workloads": {}}
    for w in a.workloads.split(","):
        out["workloads"][w] = bench_workload(w, [int(k) for k in a.ks.split(",")], a.reps, a.maxiter)
    text = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
