"""Worker for the multi-GPU multi-column test (run under torch.distributed.run, one rank per GPU).

Every rank uploads its slab of the same uniform hierarchy through amg1d_create_dist and runs the multi-column calls on
its slabs of the columns.  Each column must be BIT-IDENTICAL to the single-column call on the same sharded handle
(compared with np.array_equal / ==, never with a tolerance); the gathered slabs of dev_vcycle_multi must equal a
single-GPU handle's dev_vcycle_multi.  Rank 0 collects every rank's findings and writes one JSON report per kind."""
import ctypes as C
import json
import math
import os
import sys
import types

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from agglomerationmultigrid1d_b200 import _capi as capi, solvers, uniform   # noqa: E402

CYCLES = {"v312": (3, 1, 0.5), "v023": (0, 2, 2.0 / 3.0), "v330": (3, 3, 0.8)}
KS = (1, 3, 8)
TOL = 1e-10


def main():
    out = sys.argv[1]
    log2n = int(sys.argv[2])
    kinds = sys.argv[3].split(",")
    dist.init_process_group("gloo")
    rank = dist.get_rank()
    torch.cuda.set_device(rank)
    reports = {}
    for kind in kinds:                      # one rendezvous, one NCCL communicator per kind
        reports[kind] = run_kind(kind, log2n)
        dist.barrier()
    if rank == 0:
        json.dump(reports, open(out, "w"))
    dist.barrier()
    dist.destroy_process_group()


def nccl_id():
    ids = [None]
    if dist.get_rank() == 0:
        buf = C.create_string_buffer(128)
        capi.check(None, capi.load().amg1d_nccl_unique_id(C.cast(buf, C.c_void_p)))
        ids[0] = buf.raw
    dist.broadcast_object_list(ids, src=0)
    return ids[0]


def build(kind, n, log2n):
    if kind == "cg":        # BASELINE C4 shape: CG 3 -> 1 -> DG 1 -> agglomerated levels (two-parent transfers)
        return uniform.UniformCgHierarchy(n, [3, 1], [1], [2] * log2n, xin=0.0, xout=float(n), CDir=1000.0)
    if kind == "dg8":       # 9 x 9 blocks: row-per-thread legs, run once per column
        return uniform.UniformDgHierarchy(n, [8, 4, 2, 1], [2] * log2n, xin=0.0, xout=float(n), CDir=1000.0)
    return uniform.UniformDgHierarchy(n, [3, 1], [2] * log2n, xin=0.0, xout=float(n), CDir=1000.0)


class Checker:
    def __init__(self):
        self.msgs = []

    def eq(self, a, b, what):
        if not np.array_equal(np.asarray(a), np.asarray(b)):
            d = np.abs(np.asarray(a, dtype=float) - np.asarray(b, dtype=float)).max() if np.shape(a) == np.shape(b) else None
            self.msgs.append(f"{what}: differs (max diff {d})")

    def true(self, cond, what):
        if not cond:
            self.msgs.append(what)


def run_kind(kind, log2n):
    pattern_resident = 1 if kind.endswith("_pat") else 0
    kind = kind[:-4] if pattern_resident else kind
    p2p = 0 if kind.endswith("_nccl") else 1
    kind = kind[:-5] if not p2p else kind
    rank, world = dist.get_rank(), dist.get_world_size()
    nid = nccl_id()
    n = 2 ** log2n
    U = build(kind, n, log2n)
    dev = U.upload(device=rank, dist=(rank, world, nid), options={"shard_min": 512, "p2p_halo": p2p,
                                                                  "leg_pipeline_min": 0})
    if pattern_resident:
        dev.set_option("pattern_resident", pattern_resident)
    nl = dev.n_levels
    m0 = U.levels[0].m
    nloc = n // world
    is_cg = kind == "cg"
    lo = rank * nloc
    hi = (rank + 1) * nloc + (1 if is_cg and rank == world - 1 else 0)     # the last rank holds the closing group
    n_blocks = n + 1 if is_cg else n
    sl = slice(lo * m0, hi * m0)
    w = 2.0 * math.pi / 64.0
    vals = [0.0, math.cos(w * n)]
    smooth = U.rhs(lambda x: w * w * np.cos(w * x), vals)                   # the global right-hand side
    ck = Checker()

    def columns(k, seed):
        """Global X0, B (n_dof x k): column 0 the smooth rhs, column 2 zero, the others random."""
        rng = np.random.default_rng(seed)
        X0 = rng.standard_normal((n_blocks * m0, k))
        B = rng.standard_normal((n_blocks * m0, k))
        B[:, 0] = smooth
        if k > 2:
            B[:, 2] = 0.0
        if is_cg:                                                            # padding slots of the closing group
            X0.reshape(n_blocks, m0, k)[n, 1:] = 0.0
            B.reshape(n_blocks, m0, k)[n, 1:] = 0.0
        return X0, B

    sharded = [dev.info(f"multi_legs:{l}") for l in range(nl)]
    report = {"rank": rank, "gather_level": dev.info("gather_level"), "sharded_levels": dev.info("sharded_levels"),
              "p2p_halo": dev.info("p2p_halo"), "p2p_requested": p2p, "multi_legs": sharded}
    gathered_v = {}
    for k in KS:
        X0g, Bg = columns(k, 100 + k)
        X0, B = X0g[sl], Bg[sl]
        # V-cycles: incoming iterate and zero guess, against dev_vcycle / ldiv on the same handle
        for key, cyc in CYCLES.items():
            for zg in (False, True):
                dev.dev_set_problems(X0, B)
                dev.dev_vcycle_multi(*cyc, zero_guess=zg)
                Y = dev.dev_get_solutions()
                gathered_v[(k, key, zg)] = Y
                for c in range(k):
                    if zg:
                        ref = dev.ldiv(B[:, c], *cyc)
                    else:
                        dev.dev_set_problem(X0[:, c], B[:, c])
                        dev.dev_vcycle(*cyc)
                        ref = dev.dev_get_solution()
                    ck.eq(Y[:, c], ref, f"k={k} {key} zero_guess={zg} column {c}")
            # residual norms: fused into the cycle, and computed afterwards
            dev.dev_set_problems(X0, B)
            r0 = dev.dev_residual_norms()
            dev.dev_vcycle_multi(*cyc, with_residual_norms=True)
            r1 = dev.dev_residual_norms()
            for c in range(k):
                dev.dev_set_problem(X0[:, c], B[:, c])
                ck.true(dev.dev_residual_norm() == r0[c], f"k={k} {key} residual norm before the cycle, column {c}")
                dev.dev_vcycle(*cyc, with_residual_norm=True)
                ck.true(dev.dev_residual_norm() == r1[c], f"k={k} {key} fused residual norm, column {c}")
        # multigrid(): columns stop at different cycles, the zero column runs to maxiter
        dev.dev_set_problems(X0, B)
        iters, res = dev.dev_solve_multi(25, TOL)
        X = dev.dev_get_solutions()
        for c in range(k):
            dev.dev_set_problem(X0[:, c], B[:, c])
            it, r = dev.dev_solve(25, TOL)
            ck.true(iters[c] == it, f"k={k} solve iters column {c}: {iters[c]} vs {it}")
            ck.eq(res[c], r, f"k={k} solve history column {c}")
            ck.eq(X[:, c], dev.dev_get_solution(), f"k={k} solve x column {c}")
        # PCG: the zero column never iterates; the state rules after the call
        dev.dev_set_problems(X0, B)
        iters, res = dev.dev_pcg_multi(40, TOL)
        X = dev.dev_get_solutions()
        try:
            dev.dev_vcycle_multi()
            ck.true(False, "dev_vcycle_multi after dev_pcg_multi did not fail")
        except capi.Amg1dError as e:
            ck.true(e.code == capi.ERR_STATE, f"dev_vcycle_multi after dev_pcg_multi: code {e.code}")
        for c in range(k):
            dev.dev_set_problem(X0[:, c], B[:, c])
            it, r = dev.dev_pcg(40, TOL)
            ck.true(iters[c] == it, f"k={k} pcg iters column {c}: {iters[c]} vs {it}")
            ck.eq(res[c], r, f"k={k} pcg history column {c}")
            ck.eq(X[:, c], dev.dev_get_solution(), f"k={k} pcg x column {c}")
        if k > 2:
            ck.true(iters[2] == 0, f"k={k} zero column iterated {iters[2]} times")
            ck.true(len(set(iters)) > 1, f"k={k} pcg columns all stop together: {iters}")
            report[f"pcg_iters_k{k}"] = iters
        # launches of a norm-free cycle: on a rank that runs no coarse level every exchange is one group for all columns
        # (the calls are collective: every rank makes them)
        dev.dev_set_problems(X0, B)
        dev.dev_vcycle_multi(3, 3, 2.0 / 3.0)
        if rank > 0 and all(sharded[l] for l in range(report["gather_level"])):
            report[f"launches_k{k}"] = dev.info("multi_launches_per_cycle")
        # device-filled columns (DG-first level 0): column c is the slab of dev_fill_rhs_random(seed + c), ghosts included
        if not is_cg:
            dev.dev_fill_rhs_random_multi(k, 50 + k)
            dev.dev_vcycle_multi(3, 1, 0.5)
            dev.dev_vcycle_multi(3, 1, 0.5)
            Y = dev.dev_get_solutions()
            for c in range(k):
                dev.dev_fill_rhs_random(50 + k + c)
                dev.dev_vcycle(3, 1, 0.5)
                dev.dev_vcycle(3, 1, 0.5)
                ck.eq(Y[:, c], dev.dev_get_solution(), f"k={k} fill_rhs_random_multi column {c}")
    # the resident problem (peer memory when on) and the set interleaved: neither disturbs the other
    X0g, Bg = columns(3, 7)
    X0, B = X0g[sl], Bg[sl]
    xr, br = X0g[sl, 1].copy(), Bg[sl, 0].copy()
    dev.dev_set_problem(xr, br)
    dev.dev_vcycle(); dev.dev_vcycle()
    x_ref = dev.dev_get_solution()
    dev.dev_set_problems(X0, B)
    dev.dev_vcycle_multi(); dev.dev_vcycle_multi()
    Y_ref = dev.dev_get_solutions()
    dev.dev_set_problem(xr, br)
    dev.dev_set_problems(X0, B)
    for _ in range(2):
        dev.dev_vcycle()
        dev.dev_vcycle_multi()
    ck.eq(dev.dev_get_solution(), x_ref, "interleaved resident problem")
    ck.eq(dev.dev_get_solutions(), Y_ref, "interleaved set")
    report["p2p_halo_after"] = dev.info("p2p_halo")
    # solvers.ldiv / solvers.pcg with 11 columns (two sets) against the 1-D calls
    H = types.SimpleNamespace(device=dev)
    X0g, Bg = columns(11, 11)
    X0, B = X0g[sl], Bg[sl]
    Y = np.zeros_like(B)
    solvers.ldiv(Y, H, B)
    for c in range(11):
        y = np.zeros(B.shape[0])
        solvers.ldiv(y, H, B[:, c])
        ck.eq(Y[:, c], y, f"solvers.ldiv column {c}")
    X, iters, res = solvers.pcg(H, X0, B, 30, TOL)
    for c in range(11):
        x, it, r = solvers.pcg(H, X0[:, c], B[:, c], 30, TOL)
        ck.true(iters[c] == it, f"solvers.pcg iters column {c}: {iters[c]} vs {it}")
        ck.eq(res[c], r, f"solvers.pcg history column {c}")
        ck.eq(X[:, c], x, f"solvers.pcg x column {c}")
    report["msgs"] = ck.msgs
    allrep = [None] * world
    dist.gather_object((report, {key: v for key, v in gathered_v.items() if key[0] != 8 or key[1] == "v312"}),
                       allrep if rank == 0 else None, dst=0)
    if rank == 0:
        # the gathered slabs against a single-GPU handle's multi-column cycle
        U1 = build(kind, n, log2n)
        d1 = U1.upload(device=0)
        msgs = [f"rank {r}: {m}" for r, (rep, _) in enumerate(allrep) for m in rep["msgs"]]
        for (k, key, zg) in allrep[0][1]:
            X0g, Bg = columns(k, 100 + k)
            d1.dev_set_problems(X0g, Bg)
            d1.dev_vcycle_multi(*CYCLES[key], zero_guess=zg)
            got = np.concatenate([g[(k, key, zg)] for _, g in allrep], axis=0)
            if not np.array_equal(got, d1.dev_get_solutions()):
                msgs.append(f"k={k} {key} zero_guess={zg}: gathered slabs differ from the single-GPU set")
        d1.close()
        report = {"ok": not msgs, "msgs": msgs[:40], "world": world, "ranks": [rep for rep, _ in allrep]}
    dev.close()
    return report


if __name__ == "__main__":
    main()
