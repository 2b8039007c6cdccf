"""Multi-column V-cycle (amg1d_dev_vcycle_multi) against the single-column cycle on the same handle.

For each workload (bench.py's WORKLOADS, one GPU) and each column count k: the time of one V-cycle on k device-resident
right-hand sides, per column, next to the single-column amg1d_dev_vcycle - alternated in the same process, host clock
around graph-replayed cycles that end in a stream synchronisation; the level-0 / level-1 leg times of option "profile"
(a separate pass); the byte model of the levels whose legs read their operator once for all columns; and an output
check: column 0 (and every column's residual norm) bit-identical to the single-column cycle.  A k whose column storage
does not fit (AMG1D_ERR_NOMEM) is reported as skipped.

    python tools/bench_multi.py --workloads T,C3,C2 --ks 1,2,4,8 --cycles 20 --out DIR/bench_multi.json
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

import bench  # noqa: E402  (workload definitions, measured_peak)
from agglomerationmultigrid1d_b200 import _capi as capi  # noqa: E402

SEED = 1234


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:          # the numbers below are then without their card: say so
        return {"name": "unknown", "error": str(e)}


def byte_model(U, dev, k):
    """Algorithmic HBM bytes per column of one V-cycle on the levels with multi-column legs (kernels_multi.cuh):
    per element and leg 8 (Kop / k + 3 m + mc / ratio), Kop = operator doubles the leg reads (the stored inverse
    not counted where it is recomputed in registers).  The other levels (tail, coarse solve) are not modelled."""
    total, per_level = 0.0, {}
    for l in range(len(U.levels) - 1):
        if dev.info(f"multi_legs:{l}") != 1:
            continue
        lv, (_, ratio) = U.levels[l], U.transfers[l]
        mc = U.levels[l + 1].m
        kop = dev.info(f"tile_rows:{l}") - (lv.m * lv.m if dev.info(f"dinv_recompute:{l}") else 0)
        b = 2 * lv.n * 8 * (kop / k + 3 * lv.m + mc / ratio)
        per_level[l] = b
        total += b
    return total, per_level


def time_cycles(run, cycles, dev):
    dev.synchronize()
    t0 = time.perf_counter()
    for _ in range(cycles):
        run()
    dev.synchronize()
    return (time.perf_counter() - t0) / cycles * 1e3


def leg_profile(dev, run, cycles=5):
    dev.set_option("profile", 1)
    for _ in range(cycles):
        run()
    dev.synchronize()
    out = {f"L{l}_{'down' if leg == 0 else 'up'}_ms": dev.profile(l, leg)[0] / cycles for l in (0, 1) for leg in (0, 1)}
    dev.set_option("profile", 0)
    return out


def bench_workload(name, ks, cycles, warmup, reps, peak_gbs):
    log2n = bench.WORKLOADS[name][0]
    n = 1 << log2n
    t_setup = time.perf_counter()
    U = bench.build_hierarchy(name, n)
    dev = U.upload()
    rec = {"workload": bench.WORKLOADS[name][3], "n_elements": n, "setup_s": round(time.perf_counter() - t_setup, 1)}
    single = lambda: dev.dev_vcycle()                                   # noqa: E731
    multi = lambda: dev.dev_vcycle_multi()                              # noqa: E731
    dev.dev_fill_rhs_random(SEED)
    for _ in range(warmup):
        single()
    b1, _ = byte_model(U, dev, 1)
    rec["single"] = {"bytes_model_per_cycle": b1, "legs": leg_profile(dev, single)}
    rec["multi_legs"] = [dev.info(f"multi_legs:{l}") for l in range(len(U.levels))]
    rec["k"] = {}
    for k in ks:
        r = {}
        try:
            dev.dev_fill_rhs_random_multi(k, SEED)
        except capi.Amg1dError as e:
            if e.code != capi.ERR_NOMEM:
                raise
            rec["k"][str(k)] = {"skipped": "ERR_NOMEM: column storage does not fit", "message": str(e)}
            continue
        # output check at the timed size: one cycle from the filled state, every column's norm and column 0's iterate
        dev.dev_vcycle_multi(with_residual_norms=True)
        norms = dev.dev_residual_norms()
        same_norms = True
        for c in range(k):
            dev.dev_fill_rhs_random(SEED + c)
            dev.dev_vcycle(with_residual_norm=True)
            same_norms &= bool(dev.dev_residual_norm() == norms[c])
        r["residual_norms_bit_identical"] = same_norms
        if k <= 2 or name != "T":                # (the k-column download is n_dof * k doubles of host memory)
            x0 = dev.dev_get_solutions()[:, 0].copy()
            dev.dev_fill_rhs_random(SEED)
            dev.dev_vcycle()
            r["column0_bit_identical"] = bool(np.array_equal(x0, dev.dev_get_solution()))
        else:
            r["column0_bit_identical"] = "not measured at this k (host memory); see the residual norms"
        dev.dev_fill_rhs_random(SEED)
        dev.dev_fill_rhs_random_multi(k, SEED)
        for _ in range(warmup):
            single()
            multi()
        ts, tm = [], []
        for _ in range(reps):                    # alternate the two on the same handle
            ts.append(time_cycles(single, cycles, dev))
            tm.append(time_cycles(multi, cycles, dev))
        t1, tk = float(np.median(ts)), float(np.median(tm))
        bk, per_level = byte_model(U, dev, k)
        r.update({
            "single_cycle_ms": t1, "single_cycle_ms_all": ts,
            "multi_cycle_ms": tk, "multi_cycle_ms_all": tm,
            "per_column_ms": tk / k, "per_column_speedup_vs_single": t1 / (tk / k),
            "bytes_model_per_column": bk, "bytes_model_per_column_single": b1,
            "bytes_model_level0_per_column": per_level.get(0), "bytes_model_level1_per_column": per_level.get(1),
            "achieved_fraction_of_peak_multi": bk * k / (tk * 1e-3) / (peak_gbs * 1e9),
            "achieved_fraction_of_peak_single": b1 / (t1 * 1e-3) / (peak_gbs * 1e9),
            "multi_launches_per_cycle": dev.info("multi_launches_per_cycle"),
            "single_launches_per_cycle": dev.info("launches_per_cycle"),
        })
        r["legs"] = leg_profile(dev, multi)
        rec["k"][str(k)] = r
        print(json.dumps({"workload": name, "k": k, "single_ms": round(t1, 3), "multi_ms": round(tk, 3),
                          "per_column_ms": round(tk / k, 3), "check": r["residual_norms_bit_identical"]}), flush=True)
    rec["device_bytes"] = dev.info("device_bytes")
    dev.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="T,C3,C2")
    ap.add_argument("--ks", default="1,2,4,8")
    ap.add_argument("--cycles", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    peak, peak_src = bench.measured_peak()
    out = {"card": card(), "timing": f"host clock around {a.cycles} graph-replayed cycles ending in a stream "
           f"synchronisation, median of {a.reps} alternations single / multi on one handle",
           "peak_gbs": peak, "peak_source": peak_src, "nPre": 3, "nPost": 3, "workloads": {}}
    for w in a.workloads.split(","):
        out["workloads"][w] = bench_workload(w, [int(k) for k in a.ks.split(",")], a.cycles, a.warmup, a.reps, peak)
    text = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
