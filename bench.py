#!/usr/bin/env python
"""bench.py - headline benchmark of the B200 V-cycle (contract: see the task statement / DESIGN.md).

A "step" is one pass of the hot path over one batch: ONE V-cycle (nPre = nPost = 3, alpha = 2/3)
plus the convergence check ||A x - b||_2 that ``multigrid`` performs after every cycle
(src/solvers.jl:124-131).  `value` = smoother DOF-updates per second with x, b and the hierarchy
resident in HBM; `e2e` = the same metric through the reference-facing call
``multigrid_v_cycle(H, x0, b)`` (amg1d_vcycle) with pinned HOST vectors, copies inside the timing.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload T|C2|C3|C4|C5|P8|S] [--impl reference]
                  [--dump-outputs DIR]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True      # no __pycache__ in the tree: the benchmark may run from a read-only checkout
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "FP64 V-cycle DOF-updates/s"
UNIT = "DOF-updates/s"

# name -> (log2 n per GPU, CG orders, DG orders, description); pAgg = 1, factor-2 agglomeration down to
# one element in every workload (SURVEY 8d).  Every workload scales weakly (2^log2n elements per GPU)
# except C4, which BASELINE.json defines as ONE 2^26-element problem sliced over 1/2/4/8 GPUs (strong).
WORKLOADS = {
    "T": (26, [], [3, 1], "DG p=3, 2^26 elements, DG 3->1 then pAgg=1 factor-2 agglomeration to one element (28 levels)"),
    "C2": (20, [], [3, 1], "DG p=3, 2^20 elements, full hierarchy (22 levels)"),
    "C3": (24, [], [4, 2, 1], "DG p=4, 2^24 elements, DG 4->2->1 then factor-2 agglomeration (27 levels)"),
    "C4": (26, [3, 1], [1], "CG p=3 -> CG 1 -> DG 1 -> factor-2 agglomeration, 2^26 elements (dg_cg_heirarchy shape, 29 levels)"),
    "C5": (24, [], [3, 1], "DG p=3, 2^24 elements per GPU, full hierarchy"),
    "S": (14, [], [3, 1], "DG p=3, 2^14 elements (smoke-sized)"),
    # the order the reference's own hierarchy scripts start from (tests/dg_heirarchy_test.jl: p = 8, 4, 2, 1):
    # 9x9 element blocks on level 0, handled by the row-per-thread fused legs (csrc/kernels_rows.cuh)
    "P8": (23, [], [8, 4, 2, 1], "DG p=8, 2^23 elements, DG 8->4->2->1 then factor-2 agglomeration (27 levels)"),
}


STRONG = {"C4"}


def build_hierarchy(workload, n):
    """The uniform-mesh pattern set-up of one workload at n elements (host side, seconds)."""
    from agglomerationmultigrid1d_b200 import uniform
    _, cg, dg, _ = WORKLOADS[workload]
    pr = problem(n)
    k = n.bit_length() - 1
    if cg:
        return uniform.UniformCgHierarchy(n, cg, dg, [2] * k, pAgg=1, xin=pr["xin"], xout=pr["xout"],
                                          CDir=pr["CDir"])
    return uniform.UniformDgHierarchy(n, dg, [2] * k, pAgg=1, xin=pr["xin"], xout=pr["xout"], CDir=pr["CDir"])


def rhs_slab(U, pr, rank, world):
    """This rank's slab of the right-hand side (elements for DG-first, vertex groups for CG-first)."""
    nloc = U.n // world
    if hasattr(U, "cg_orders"):
        return U.rhs(pr["func"], pr["bc_values"],
                     group_range=(rank * nloc, (rank + 1) * nloc + (1 if rank == world - 1 else 0)))
    return U.rhs(pr["func"], pr["bc_values"], elem_range=(rank * nloc, (rank + 1) * nloc))


def problem(n):
    """Domain [0, n] (h = 1), CDir = 1000, u = cos(2 pi x / 64): FP64 can reach 1e-10 at any n
    (SURVEY section 7); Neumann left, Dirichlet right as in the reference's hierarchy scripts."""
    w = 2.0 * math.pi / 64.0
    return dict(xin=0.0, xout=float(n), CDir=1000.0,
                func=lambda x: w * w * np.cos(w * x),
                bc_values=[-w * math.sin(0.0), math.cos(w * n)])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.lines = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        rows = [l.split(", ") for (t, l) in self.lines if t0 <= t <= t1 + 0.2] or \
               [l.split(", ") for (t, l) in self.lines[-3:]]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                    "sw_power_cap"), r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_MAX_ENTRIES = 2 ** 21      # 16 MB of x values + 16 MB of their indices


def dump_outputs(out_dir, dev, res_norm):
    """What the last timed step left for its caller, as DIR/<name>.npy (float64): x, the iterate after the last
    V-cycle (this rank's slab; longer than DUMP_MAX_ENTRIES, a fixed seeded sample of it, positions in x_index),
    and residual_norm, the ||b - A x|| of that cycle's convergence check."""
    x = dev.dev_get_solution()
    idx = np.arange(len(x))
    if len(x) > DUMP_MAX_ENTRIES:
        idx = np.sort(np.random.default_rng(0).choice(len(x), DUMP_MAX_ENTRIES, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "x.npy"), x[idx])
    np.save(os.path.join(out_dir, "x_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "residual_norm.npy"), np.array([res_norm]))


# ---- CPU reference arm: the oracle's restatement of multigrid_v_cycle on the host cores ------------
REF_LOG2N = 24          # bounded sample of the reference arm: the same hierarchy shape at 2^24 elements (64 x round 1's)


def host_ram_gb():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                return int(line.split()[1]) / 2 ** 20
    except OSError:
        pass
    return 0.0


def _oracle_pattern(workload, n):
    """oracle/vcycle_ref.c in block-pattern storage, fed with the arrays the GPU upload uses."""
    from oracle import cref
    U = build_hierarchy(workload, n)
    pr = problem(n)
    b = U.rhs(pr["func"], pr["bc_values"])
    return U, b, cref.CRefPattern(*cref.pattern_arrays(U))


def _time_cycles(c, b, nsteps, warmup):
    x = np.zeros(len(b))
    for _ in range(warmup):
        x = c.vcycle(x, b)
    t0 = time.perf_counter()
    for _ in range(nsteps):
        x = c.vcycle(x, b)
        c.residual_norm(x, b)
    return (time.perf_counter() - t0) / nsteps


def literal_scipy_figure(log2n=10):
    """BASELINE.md figure (i): the literal single-thread path (oracle/solvers.py: scipy CSC SpMV, one LAPACK LU
    solve per element in a Python loop, SuperLU coarse solve, fresh temporaries) on the DG p=3 shape at a size
    it finishes in seconds."""
    from oracle import drivers, solvers
    n = 2 ** log2n
    H, x0, b, _ = drivers.dg_agg_problem(n, p=3, unit_h=True)
    upd = 6 * sum(A.shape[0] for A in H.mStiffness[:-1])
    x = solvers.multigrid_v_cycle(H, x0, b)
    t0 = time.perf_counter()
    x = solvers.multigrid_v_cycle(H, x, b)
    dt = time.perf_counter() - t0
    return {"value": upd / dt, "unit": UNIT, "cores": 1, "n_elements": n, "seconds_per_cycle": dt,
            "what": "literal numpy/scipy restatement (oracle/solvers.py), DG p=3 -> 1 -> agglomerated, one V-cycle"}


def cpu_reference(workload, nsteps, warmup=1, log2n_sample=None, threads=0, with_single=True, with_literal=True):
    """Times the oracle's plain-C restatement of the reference algorithm (oracle/vcycle_ref.c: sparse row
    walks for A*u, one partial-pivoting LU solve per element for block Jacobi, sparse L' / L products, direct
    coarse solve, fresh temporaries per expression as in src/solvers.jl:19-50) with all host threads on a
    bounded sample of the same hierarchy shape: 2^REF_LOG2N elements (or the workload's own size if that is
    smaller, or less if the host's RAM does not hold it).  The method is O(N): DOF-updates/s at 2^24 elements is
    memory-bound like the full size.  Also reported: the same port on ONE thread (at 2^20 elements) and
    BASELINE.md's figure (i), the literal scipy loop."""
    log2n = min(WORKLOADS[workload][0], log2n_sample or REF_LOG2N)
    ram = host_ram_gb()
    while log2n > 18 and (2 ** log2n) * 5 * 8 * 12 / 2 ** 30 > 0.5 * max(ram, 8.0):    # ~12 fine vectors live
        log2n -= 1
    n = 2 ** log2n
    U, b, c = _oracle_pattern(workload, n)
    upd = U.dof_updates_per_cycle()
    used = c.set_threads(threads or (os.cpu_count() or 1))
    dt = _time_cycles(c, b, nsteps, warmup)
    c.close()
    out = {"value": upd / dt, "seconds_per_step": dt, "cores": used, "log2n": log2n, "upd": upd,
           "host_ram_gb": round(ram, 1)}
    if with_single:
        n1 = 2 ** min(log2n, 20)
        U1, b1, c1 = _oracle_pattern(workload, n1)
        c1.set_threads(1)
        dt1 = _time_cycles(c1, b1, 1, 1)
        c1.set_threads(used)
        c1.close()
        out["single_thread_value"] = U1.dof_updates_per_cycle() / dt1
        out["single_thread_log2n"] = min(log2n, 20)
    if with_literal:
        try:
            out["literal_scipy"] = literal_scipy_figure()
        except Exception as exc:                     # never lose the line over the auxiliary figure
            out["literal_scipy"] = {"error": f"{type(exc).__name__}: {exc}"}
    out["sample"] = (f"{nsteps} V-cycles (+ residual check) after {warmup} warm-up, same hierarchy shape at n = 2^{log2n} "
                     f"elements ({upd} DOF-updates per cycle; host RAM {ram:.0f} GB); oracle/vcycle_ref.c (C port of the "
                     f"reference algorithm, block-pattern storage, OpenMP over rows / elements, {used} threads)"
                     + (f"; single thread at 2^{out['single_thread_log2n']}: {out['single_thread_value']:.3e} DOF-updates/s"
                        if with_single else ""))
    return out


def default_workload(world):
    """N = 1: T, the north-star's headline configuration (DG p=3, 2^26 elements on one B200).  N > 1: C5,
    BASELINE's weak-scaling configuration (2^24 elements per GPU) - T x 4 / T x 8 would be 2^28 / 2^29
    elements, where cond(A) ~ (2n / pi)^2 exceeds 1 / eps and no FP64 iteration reaches 1e-10 (DESIGN.md 6)."""
    return "T" if world == 1 else "C5"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    workload = args.workload or default_workload(world)
    log2n, _, _, desc = WORKLOADS[workload]
    r = cpu_reference(workload, max(1, args.steps), warmup=max(0, args.warmup))
    val, dt = r["value"], r["seconds_per_step"]
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong" if workload in STRONG else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{workload}: {desc}", "sample_log2n": r["log2n"], "note": "Julia is not installed "
                   "here; this is the C port of the reference algorithm (oracle/vcycle_ref.c) on all host threads, on "
                   "a bounded sample of the workload (DOF-updates/s is size-independent for this O(N) method)"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"],
                         "single_thread_value": r.get("single_thread_value"),
                         "literal_scipy": r.get("literal_scipy"), "host_cores_available": os.cpu_count()},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- GPU arm ----------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(torch, local):
    """Run this rank on the CPUs of the NUMA node its GPU hangs off, so that the pinned host vectors it allocates
    afterwards (cudaMallocHost, first touch) and its PCIe copies stay node-local - with all ranks of a box on node 0
    the end-to-end numbers at 4 / 8 GPUs were bound by one node's memory controllers (round 1: e2e weak efficiency
    0.32 at 8 GPUs).  Returns what was done, for the JSON line; never fails the run."""
    info = {"gpu_numa_node": None, "bound": False}
    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
        info["pci"] = bdf
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        info["gpu_numa_node"] = node
        if node < 0:
            return info
        cpus = set()
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        info["node_cpus_allowed"] = len(use)
        if len(use) >= 2 and use != allowed:                 # never squeeze a rank (and its NCCL threads) onto one CPU
            os.sched_setaffinity(0, use)
            info["bound"] = True
    except Exception as e:                                   # no sysfs, no such attribute, cpuset forbids it ...
        info["note"] = f"{type(e).__name__}: {e}"[:120]
    return info


class Ctx:
    """Process-wide plumbing of the GPU arm: torch stream / events, torch.distributed group, libamg1d."""

    def __init__(self):
        import torch
        import agglomerationmultigrid1d_b200 as aggmg          # noqa: F401  raises if libamg1d.so is missing
        from agglomerationmultigrid1d_b200 import _capi as capi
        self.torch, self.capi = torch, capi
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world & (self.world - 1):
            raise SystemExit("the slab-sharded workloads need a power-of-two rank count")
        torch.cuda.set_device(self.local)
        # before any pinned allocation (first touch); a single rank keeps all host cores (its CPU-baseline leg uses them)
        self.numa = bind_to_gpu_numa_node(torch, self.local) if self.world > 1 else {"bound": False, "note": "single rank"}
        self.tdist = None
        if self.world > 1:
            import torch.distributed as tdist
            tdist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.tdist = tdist
        # a non-default stream: its handle is non-zero, so the library runs on exactly the stream that
        # torch.cuda.Event records on (handle 0 would make the library create a stream of its own)
        self.tstream = torch.cuda.Stream(device=self.local)
        torch.cuda.set_stream(self.tstream)
        self.stream = self.tstream.cuda_stream
        assert self.stream != 0
        self.lib = capi.load()

    def dist_arg(self, ranks):
        """(rank, nranks, ncclUniqueId) for a sharded handle over all ranks, None for a single-GPU one."""
        if ranks == 1:
            return None
        import ctypes as C0
        ids = [None]
        if self.rank == 0:
            buf = C0.create_string_buffer(128)
            self.capi.check(None, self.lib.amg1d_nccl_unique_id(C0.cast(buf, C0.c_void_p)))
            ids[0] = buf.raw
        self.tdist.broadcast_object_list(ids, src=0)
        return (self.rank, self.world, ids[0])

    def barrier(self, ranks):
        self.torch.cuda.synchronize()
        if ranks > 1:
            self.tdist.barrier()

    def max_over_ranks(self, v, ranks):
        if ranks == 1:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        self.tdist.all_reduce(t, op=self.tdist.ReduceOp.MAX)
        return float(t.item())


def measure(ctx, args, workload, ranks, full, dump=None):
    """One workload on `ranks` GPUs (ranks == ctx.world: slab-sharded over every rank; ranks == 1: a single-GPU
    handle - the caller runs it on rank 0 only).  full = True: the whole JSON line (roofline, e2e, ldiv, PCG,
    pattern modes, CPU baseline); False: throughput + time-to-1e-10 only (the secondary objects).  dump: a
    directory for rank 0 to write the outputs of the last timed step to (dump_outputs)."""
    import ctypes as C
    torch, capi, lib = ctx.torch, ctx.capi, ctx.lib
    world = ranks
    rank = ctx.rank if ranks > 1 else 0
    barrier = lambda: ctx.barrier(ranks)                          # noqa: E731
    mx = lambda v: ctx.max_over_ranks(v, ranks)                   # noqa: E731
    log2n, _, _, desc = WORKLOADS[workload]
    log2w = world.bit_length() - 1
    strong = workload in STRONG
    n = 2 ** (log2n if strong else log2n + log2w) # weak scaling: 2^log2n elements per GPU; strong: in total
    nloc = n // world
    pr = problem(n)
    t_setup = time.perf_counter()
    U = build_hierarchy(workload, n)
    pre = {kv.split("=")[0]: int(kv.split("=")[1]) for kv in args.pre_opt}
    dev = U.upload(device=ctx.local, stream=ctx.stream, dist=ctx.dist_arg(ranks), options=pre or None)
    dev.synchronize()
    t_setup = time.perf_counter() - t_setup
    for kv in args.opt:
        k, v = kv.split("=")
        dev.set_option(k, int(v))
    N0 = dev.info("local_dofs")                   # DOFs (slots) of this rank's slab of the fine level
    N0_all = U.levels[0].n * U.levels[0].m        # whole fine level
    upd = U.dof_updates_per_cycle()               # whole job

    # ---- value: device-resident steps (random rhs; throughput does not depend on the data) --------
    dev.dev_fill_rhs_random(0)
    for _ in range(args.warmup):
        dev.dev_vcycle(with_residual_norm=True)
    dev.synchronize()
    launches0 = dev.info("kernel_launches")
    sampler = ClockSampler(ctx.local)
    sampler.start()
    time.sleep(0.25)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    tw0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        dev.dev_vcycle(with_residual_norm=True)
    ev1.record()
    barrier()
    tw1 = time.time()
    clocks = sampler.stop(tw0, tw1)
    ms_step = mx(ev0.elapsed_time(ev1)) / args.steps
    launches = dev.info("kernel_launches") - launches0
    value = upd / (ms_step * 1e-3)
    res_after = dev.dev_residual_norm()
    if dump and rank == 0:
        dump_outputs(dump, dev, res_after)

    # ---- host vectors (pinned) with the workload's right-hand side -----------------------------------
    bufs = []
    for _ in range(2):
        p = C.c_void_p()
        capi.check(None, lib.amg1d_host_alloc(C.byref(p), N0 * 8))
        bufs.append(p)
    xh = np.ctypeslib.as_array(C.cast(bufs[0], C.POINTER(C.c_double)), shape=(N0,))
    bh = np.ctypeslib.as_array(C.cast(bufs[1], C.POINTER(C.c_double)), shape=(N0,))
    # the right-hand side assembled ON THE DEVICE (amg1d_dev_assemble_rhs: every rank its slab, nothing but the
    # quadrature tables crosses PCIe) and multigrid() on the device-resident problem
    w = 2.0 * math.pi / 64.0
    barrier()
    t0 = time.perf_counter()
    U.device_rhs([("cos", w * w, 0, w, 0.0)], pr["bc_values"], dev)
    dev.synchronize()
    barrier()
    t_rhs_dev = mx(time.perf_counter() - t0)
    t0 = time.perf_counter()
    it_dev, res_dev = dev.dev_solve(100, 1e-10)
    barrier()
    t_solve_dev = mx(time.perf_counter() - t0)
    nb_dev = dev.dev_rhs_norm()
    dev_solve = {"rhs_assembly_s": t_rhs_dev, "iters": it_dev, "seconds": t_solve_dev,
                 "final_relative_residual": float(res_dev[-1] / nb_dev), "converged": bool(res_dev[-1] < 1e-10 * nb_dev),
                 "call": "amg1d_dev_assemble_rhs + amg1d_dev_solve (multigrid on the device-resident problem)"}
    if not dev_solve["converged"]:
        # plain V-cycle iteration stalls in FP64 at this size (CG-first hierarchy at 2^26 elements: cond ~ 1 / eps; the
        # CPU oracle shows the same history, profiles/r02_hist_*_C4_2p26.json): CG with the same V-cycle as preconditioner
        U.device_rhs([("cos", w * w, 0, w, 0.0)], pr["bc_values"], dev)
        barrier()
        t0 = time.perf_counter()
        it_p, res_p = dev.dev_pcg(100, 1e-10)
        barrier()
        t_p = mx(time.perf_counter() - t0)
        dev_solve["pcg"] = {"iters": it_p, "seconds": t_p, "final_relative_residual": float(res_p[-1] / nb_dev),
                            "converged": bool(res_p[-1] < 1e-10 * nb_dev), "call": "amg1d_dev_pcg"}
        dev_solve["converged_via"] = "pcg" if dev_solve["pcg"]["converged"] else None
        dev_solve["seconds_to_1e-10"] = t_p if dev_solve["pcg"]["converged"] else None
    else:
        dev_solve["converged_via"] = "multigrid"
        dev_solve["seconds_to_1e-10"] = t_solve_dev
    if not full:
        # secondary objects: no host vectors at all; CG as the fall-back where plain cycling stalls in FP64
        line_light = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "scaling": "strong" if strong else "weak",
            "config": {"workload": f"{workload}: {desc}", "n_elements": n, "elements_per_gpu": nloc, "levels": len(U.levels),
                       "gather_level": dev.info("gather_level"), "p2p_halo": dev.info("p2p_halo"), "numa": ctx.numa, "numa": ctx.numa,
                       "sharded_levels": dev.info("sharded_levels"),
                       "halo_bytes_per_cycle_per_rank": dev.info("halo_bytes_per_cycle"),
                       "options": args.opt + args.pre_opt, "setup_s": t_setup, "dof_updates_per_step": upd},
            "clocks": clocks, "gpu_launches": int(launches), "time_to_1e-10": dev_solve}
        for p in bufs:
            lib.amg1d_host_free(p)
        dev.close()
        return line_light
    t_rhs = time.perf_counter()
    bh[:] = rhs_slab(U, pr, rank, world)
    t_rhs = time.perf_counter() - t_rhs

    # ---- time-to-1e-10: full multigrid() solve through the ABI (host vectors in, solution out) ----
    xh[:] = 0.0
    res = np.zeros(100)
    it = C.c_int(0)
    barrier()
    t0 = time.perf_counter()
    capi.check(dev._h, lib.amg1d_solve(dev._h, capi.dptr(xh), capi.dptr(bh), 100, 1e-10, 3, 3, 2.0 / 3.0,
                                        C.byref(it), capi.dptr(res), None, None))
    barrier()
    t_solve = mx(time.perf_counter() - t0)
    nb = dev.dev_rhs_norm()
    rel = float(res[it.value - 1] / nb)
    solve = {"iters": it.value, "seconds_e2e": t_solve, "final_relative_residual": rel, "converged": rel < 1e-10,
             "call": "amg1d_solve (multigrid(H, x0, b, 100, 1e-10)), host b in / host x out"}
    # ---- the same solve with CG, one V-cycle (ldiv!(z, H, r)) as the preconditioner ------------------
    xh[:] = 0.0
    res2 = np.zeros(100)
    it2 = C.c_int(0)
    barrier()
    t0 = time.perf_counter()
    capi.check(dev._h, lib.amg1d_pcg(dev._h, capi.dptr(xh), capi.dptr(bh), 100, 1e-10, 3, 3, 2.0 / 3.0,
                                      C.byref(it2), capi.dptr(res2)))
    barrier()
    t_pcg = mx(time.perf_counter() - t0)
    rel2 = float(res2[max(it2.value, 1) - 1] / nb)
    solve["pcg"] = {"iters": it2.value, "seconds_e2e": t_pcg, "final_relative_residual": rel2,
                    "converged": rel2 < 1e-10,
                    "call": "amg1d_pcg (CG preconditioned with ldiv!(z, H, r)), host b in / host x out"}
    if not solve["converged"]:
        # CG-first hierarchy at 2^26 elements: cond(A) ~ (2n / pi)^2 = 1.8e15 ~ 0.4 / eps.  The CPU oracle shows the
        # same history (profiles/r02_hist_*_C4_2p26.json, DESIGN.md section 6): it is the algorithm in FP64, not the
        # kernels.  CG with the same V-cycle as preconditioner converges; that is this workload's time-to-1e-10.
        solve["note"] = ("plain V-cycle iteration does not reach 1e-10 at this size in FP64 on either the GPU or the CPU "
                         "oracle (cond ~ 1/eps); amg1d_pcg with the same V-cycle as preconditioner does")
        solve["seconds_to_1e-10"] = t_pcg if solve["pcg"]["converged"] else None
        solve["converged_via"] = "pcg" if solve["pcg"]["converged"] else None
    else:
        solve["seconds_to_1e-10"] = t_solve
        solve["converged_via"] = "multigrid"

    config = {"workload": f"{workload}: {desc}" + (
                  "" if world == 1 else f" sliced over {world} GPUs (slab-sharded)" if strong else
                  f" x {world} GPUs (2^{log2n} elements per GPU, slab-sharded)"),
              "n_elements": n, "fine_dofs": N0_all, "elements_per_gpu": nloc,
              "parallelism": f"slab{world}" if world > 1 else "single",
              "levels": len(U.levels), "nPre": 3, "nPost": 3, "alpha": 2.0 / 3.0,
              "dof_updates_per_step": upd, "step": "one V-cycle + ||Ax-b|| check, CUDA graph replay",
              "l2": "inputs larger than L2 (operators + vectors of the fine levels are GBs)"
              if dev.info("device_bytes") > 2 ** 29 else "working set comparable to L2; no flush",
              "structure_classes": [dev.info(f"structure:{l}") for l in range(min(4, len(U.levels)))],
              "tile_rows": [U.tile_rows(l) for l in range(min(4, len(U.levels)))],
              "streamed_operator_doubles": [U.streamed_operator_doubles(l) for l in range(min(4, len(U.levels)))],
              "tail_start": dev.info("tail_start"), "options": args.opt + args.pre_opt,
              "gather_level": dev.info("gather_level"), "p2p_halo": dev.info("p2p_halo"), "numa": ctx.numa,
              "sharded_levels": dev.info("sharded_levels"),
              "halo_bytes_per_cycle_per_rank": dev.info("halo_bytes_per_cycle"),
              "device_bytes": dev.info("device_bytes"), "setup_s": t_setup, "rhs_assembly_s": t_rhs_dev,
              "rhs_assembly_host_numpy_s": t_rhs,
              "residual_after_timed_steps": res_after}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
        "clocks": clocks, "time_to_1e-10": solve, "time_to_1e-10_device_resident": dev_solve, "gpu_launches": int(launches),
        "fine_dof_cycles_per_s": N0_all / (ms_step * 1e-3),
    }
    # ---- roofline of the dominant kernel, CUDA events around each launch (un-graphed pass) --------
    peak, peak_src = measured_peak()
    dev.dev_fill_rhs_random(0)
    dev.set_option("profile", 1)
    for _ in range(args.steps):
        dev.dev_vcycle(with_residual_norm=True)
    dev.synchronize()
    legs = {}
    for l in range(min(3, len(U.levels) - 1)):
        for leg, nm in ((0, "down"), (1, "up")):
            ms, cnt = dev.profile(l, leg)
            legs[f"L{l}_{nm}"] = ms / max(cnt, 1)
    dev.set_option("profile", 0)
    lv0, lv1 = U.levels[0], U.levels[1]
    m, mc = lv0.m, lv1.m
    st0 = dev.info("structure:0")
    # f_up at level 0 (prolongation + 3 sweeps + ||b - A x||^2), this rank's slab: the level's stored
    # operator once (tile_rows doubles per element for its structure class), b, x in, x out, coarse x
    bytes_up = U.bytes_per_leg_fused(0, down=False) // world
    kname = ("f_up_pp<%d,%d,128" if dev.info("leg_pipeline:0") == 1 else "f_up<%d,%d,128") % (m, mc) if m <= 5 \
        else "r_up<%d,%d,%d" % (m, mc, dev.info("rows_window"))
    kern = (f"{kname},st={st0},{'point' if getattr(lv0, 'is_cg', False) else 'block'}-Jacobi> level 0 "
            f"(prolong + 3 sweeps + ||b-Ax||^2; {U.streamed_operator_doubles(0)} operator + {3 * m} vector doubles per "
            f"element streamed; {U.tile_rows(0)} stored" + (", Dinv recomputed in registers" if dev.info("dinv_recompute:0") == 1 else "")
            + ("; persistent CTAs, next window prefetched by TMA bulk copies" if dev.info("leg_pipeline:0") == 1 else "") + ")")
    t_k = legs["L0_up"]
    achieved = bytes_up / (t_k * 1e-3) / 1e9
    cyc_bytes = U.bytes_per_cycle_fused()
    traffic, traffic_src = None, None               # DRAM bytes per launch from the committed ncu capture
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and world == 1:
        tj = json.load(open(tpath)).get(workload, {})
        if tj.get("streamed_doubles") == U.streamed_operator_doubles(0):   # a capture of another layout does not apply
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": traffic, "traffic_source": traffic_src, "kernel": kern, "algorithmic_bytes_per_launch": bytes_up,
        "avg_launch_ms": t_k, "peak_source": peak_src,
        "whole_cycle": {"algorithmic_bytes": cyc_bytes, "GBps": cyc_bytes / (ms_step * 1e-3) / 1e9,
                        "frac": cyc_bytes / (ms_step * 1e-3) / 1e9 / (peak * world),
                        "B_ref_bytes": U.bytes_per_cycle_reference_model(),
                        "B_ref_equiv_GBps": U.bytes_per_cycle_reference_model() / (ms_step * 1e-3) / 1e9},
        "leg_ms": legs,
    }

    # ---- the same legs with the smoother inverse STREAMED from HBM instead of recomputed in registers (option
    # recompute_dinv = 0; same bits): the byte count of round 1, reported beside the default for comparison
    if dev.info("dinv_recompute:0") == 1:
        rec_default = dev.info("recompute_dinv")
        dev.set_option("recompute_dinv", 0)
        dev.dev_fill_rhs_random(0)
        for _ in range(args.warmup):
            dev.dev_vcycle(with_residual_norm=True)
        barrier()
        ev0.record()
        for _ in range(args.steps):
            dev.dev_vcycle(with_residual_norm=True)
        ev1.record()
        barrier()
        ms_s = mx(ev0.elapsed_time(ev1)) / args.steps
        dev.set_option("profile", 1)
        for _ in range(args.steps):
            dev.dev_vcycle(with_residual_norm=True)
        dev.synchronize()
        t_s, c_s = dev.profile(0, 1)
        t_sd, c_sd = dev.profile(0, 0)
        dev.set_option("profile", 0)
        b_s = U.bytes_per_leg_fused(0, down=False) // world
        roofline["streamed_inverse"] = {
            "what": "option recompute_dinv = 0: level 0 streams the stored block-Jacobi inverses (bit-identical results)",
            "algorithmic_bytes_per_launch": b_s, "avg_launch_ms": t_s / max(c_s, 1),
            "achieved": b_s / (t_s / max(c_s, 1) * 1e-3) / 1e9, "frac": b_s / (t_s / max(c_s, 1) * 1e-3) / 1e9 / peak,
            "L0_down_ms": t_sd / max(c_sd, 1), "ms_per_step": ms_s, "value": upd / (ms_s * 1e-3),
            "whole_cycle_bytes": U.bytes_per_cycle_fused()}
        dev.set_option("recompute_dinv", rec_default)

    # ---- e2e: the reference-facing call with pinned host vectors, copies inside the timed region ---
    xh[:] = 0.0
    e2e_steps = max(1, min(args.steps, 5))
    capi.check(dev._h, lib.amg1d_vcycle(dev._h, capi.dptr(xh), capi.dptr(bh), 3, 3, 2.0 / 3.0))  # warm
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        capi.check(dev._h, lib.amg1d_vcycle(dev._h, capi.dptr(xh), capi.dptr(bh), 3, 3, 2.0 / 3.0))
    barrier()
    t_e2e = mx(time.perf_counter() - t0) / e2e_steps
    e2e = {"value": upd / t_e2e, "unit": UNIT, "h2d_bytes_per_step": 2 * N0_all * 8,
           "d2h_bytes_per_step": N0_all * 8, "ms_per_step": t_e2e * 1e3, "steps": e2e_steps,
           "call": "amg1d_vcycle (multigrid_v_cycle(H, x0, b)) with pinned host x0, b"}
    # ---- the same call for a stream of independent problems: amg1d_vcycle_batch pipelines upload / cycle /
    # download over the full-duplex PCIe link.  Every step still moves its own x0 and b up and its own x down.
    pipe_steps = max(4, 2 * e2e_steps)
    pb = []
    for _ in range(4):                       # two (x, b) pairs of pinned host vectors, used alternately
        p = C.c_void_p()
        capi.check(None, lib.amg1d_host_alloc(C.byref(p), N0 * 8))
        pb.append(p)
    hv = [np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), shape=(N0,)) for p in pb]
    hv[0][:] = 0.0; hv[1][:] = 0.0; hv[2][:] = bh; hv[3][:] = bh
    PD = C.POINTER(C.c_double)
    xa = (PD * pipe_steps)(*[hv[k % 2].ctypes.data_as(PD) for k in range(pipe_steps)])
    ba = (PD * pipe_steps)(*[hv[2 + k % 2].ctypes.data_as(PD) for k in range(pipe_steps)])
    capi.check(dev._h, lib.amg1d_vcycle_batch(dev._h, 2, xa, ba, 0, 3, 3, 2.0 / 3.0))            # warm (allocates staging)
    barrier()
    t0 = time.perf_counter()
    capi.check(dev._h, lib.amg1d_vcycle_batch(dev._h, pipe_steps, xa, ba, 0, 3, 3, 2.0 / 3.0))
    barrier()
    t_pipe = mx(time.perf_counter() - t0) / pipe_steps
    barrier()
    t0 = time.perf_counter()
    capi.check(dev._h, lib.amg1d_vcycle_batch(dev._h, pipe_steps, xa, ba, 1, 3, 3, 2.0 / 3.0))
    barrier()
    t_pipe0 = mx(time.perf_counter() - t0) / pipe_steps
    for p in pb:
        lib.amg1d_host_free(p)
    e2e["single_call"] = {"value": e2e["value"], "ms_per_step": e2e["ms_per_step"], "call": e2e["call"]}
    e2e.update(value=upd / t_pipe, ms_per_step=t_pipe * 1e3, steps=pipe_steps,
               call="amg1d_vcycle_batch: multigrid_v_cycle(H, x0_k, b_k) for a stream of independent problems, pinned host "
                    "vectors; upload of problem k + 1, V-cycle of k and download of k - 1 overlap; every step moves its own "
                    "x0, b up and x down (one problem per call: see single_call)")
    e2e["ldiv_pipelined"] = {"value": upd / t_pipe0, "ms_per_step": t_pipe0 * 1e3, "h2d_bytes_per_step": N0_all * 8,
                             "d2h_bytes_per_step": N0_all * 8, "call": "amg1d_vcycle_batch with zero_guess = 1 (ldiv!(y_k, H, b_k))"}
    # ---- ldiv!(y, H, b): one V-cycle from zero, only b travels up ----------------------------------------
    capi.check(dev._h, lib.amg1d_ldiv(dev._h, capi.dptr(xh), capi.dptr(bh), 3, 3, 2.0 / 3.0))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        capi.check(dev._h, lib.amg1d_ldiv(dev._h, capi.dptr(xh), capi.dptr(bh), 3, 3, 2.0 / 3.0))
    barrier()
    t_ldiv = mx(time.perf_counter() - t0) / e2e_steps
    e2e["ldiv"] = {"value": upd / t_ldiv, "ms_per_step": t_ldiv * 1e3, "h2d_bytes_per_step": N0_all * 8,
                   "d2h_bytes_per_step": N0_all * 8, "call": "amg1d_ldiv (ldiv!(y, H, b)) with pinned host b, y"}

    # ---- the same cycle with pattern-resident operators ----------------------------------------------
    # Uniform meshes only (every level was given as a head / interior / tail pattern): the fused legs take
    # an element's block set from the level's pattern table (a few KB, L1) instead of streaming one stored
    # set per element, so HBM carries the vectors only.  Same arithmetic, bit-identical iterates.  Reported
    # beside the headline, which stays on the general per-element layout the north-star prescribes.
    pattern = None
    if not dev.info("pattern_resident") and dev.info("pattern:0") and not args.no_pattern:
        pattern = {"what": "option pattern_resident: operators of the translation-invariant levels are not streamed "
                           "from HBM (uniform meshes only, bit-identical iterates); 1 = every thread fetches its "
                           "block set from the level's pattern table (L1), 2 = CTAs in the interior of a level take "
                           "the interior block set as a by-value kernel parameter (constant-bank operands)"}
        try:
            for mode in (1, 2):
                dev.set_option("pattern_resident", mode)
                dev.dev_fill_rhs_random(0)
                for _ in range(args.warmup):
                    dev.dev_vcycle(with_residual_norm=True)
                barrier()
                ev0.record()
                for _ in range(args.steps):
                    dev.dev_vcycle(with_residual_norm=True)
                ev1.record()
                barrier()
                ms_p = mx(ev0.elapsed_time(ev1)) / args.steps
                res_p = dev.dev_residual_norm()
                dev.set_option("profile", 1)
                for _ in range(args.steps):
                    dev.dev_vcycle(with_residual_norm=True)
                dev.synchronize()
                legs_p = {}
                for l in range(min(3, len(U.levels) - 1)):
                    for leg, nm in ((0, "down"), (1, "up")):
                        ms, cnt = dev.profile(l, leg)
                        legs_p[f"L{l}_{nm}"] = ms / max(cnt, 1)
                dev.set_option("profile", 0)
                cyc_p = U.bytes_per_cycle_fused()
                up_p = U.bytes_per_leg_fused(0, down=False) // world
                xh[:] = 0.0
                res3 = np.zeros(100)
                it3 = C.c_int(0)
                barrier()
                t0 = time.perf_counter()
                capi.check(dev._h, lib.amg1d_solve(dev._h, capi.dptr(xh), capi.dptr(bh), 100, 1e-10, 3, 3, 2.0 / 3.0,
                                                    C.byref(it3), capi.dptr(res3), None, None))
                barrier()
                t_solve_p = mx(time.perf_counter() - t0)
                pattern[f"mode_{mode}"] = {
                    "ms_per_step": ms_p, "value": upd / (ms_p * 1e-3), "unit": UNIT,
                    "residual_identical_to_streamed_operator_run": bool(res_p == res_after),
                    "algorithmic_bytes_per_cycle": cyc_p, "GBps": cyc_p / (ms_p * 1e-3) / 1e9,
                    "frac_of_hbm_peak": cyc_p / (ms_p * 1e-3) / 1e9 / (peak * world),
                    "L0_up": {"algorithmic_bytes": up_p, "ms": legs_p["L0_up"],
                              "GBps": up_p / (legs_p["L0_up"] * 1e-3) / 1e9,
                              "frac_of_hbm_peak": up_p / (legs_p["L0_up"] * 1e-3) / 1e9 / peak},
                    "leg_ms": legs_p,
                    "time_to_1e-10": {"iters": it3.value, "seconds_e2e": t_solve_p,
                                      "iters_and_history_identical": bool(it3.value == it.value and
                                                                          np.array_equal(res3[:it3.value], res[:it.value]))},
                }
        except Exception as exc:      # the headline line must still be printed
            pattern["error"] = f"{type(exc).__name__}: {exc}"
        dev.set_option("pattern_resident", 0)

    for p in bufs:
        lib.amg1d_host_free(p)
    dev.close()

    # ---- CPU baseline beside it (oracle port, bounded sample) ----------------------------------------
    cpu = None
    if not args.no_cpu and world == 1:
        r = cpu_reference(workload, 3, warmup=1, log2n_sample=22)         # ~10-30 s of CPU work
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"],
               "single_thread_value": r.get("single_thread_value"), "literal_scipy": r.get("literal_scipy"),
               "host_cores_available": os.cpu_count()}
    line.update(roofline=roofline, cpu_baseline=cpu, e2e=e2e, pattern_resident=pattern)
    return line


def run_gpu(args):
    ctx = Ctx()
    world = ctx.world
    workload = args.workload or default_workload(world)
    line = measure(ctx, args, workload, world, full=not args.light, dump=args.dump_outputs)
    if not args.workload and not args.no_extra and not args.light:
        # The default run also carries BASELINE's other multi-GPU configuration and the bases its scaling is
        # judged against, measured in this very process group (rank 0 alone for the single-GPU bases).
        light = argparse.Namespace(**vars(args))
        light.steps, light.warmup = max(3, min(args.steps, 10)), 3
        extra = {}
        try:
            if world == 1:
                extra["C5_1gpu"] = measure(ctx, light, "C5", 1, full=False)     # base of the N > 1 weak-scaling line
            else:
                base = [None]
                if ctx.rank == 0:
                    base[0] = measure(ctx, light, "C5", 1, full=False)
                ctx.tdist.barrier()
                ctx.tdist.broadcast_object_list(base, src=0)
                extra["C5_1gpu_same_run"] = base[0]
                extra["weak_efficiency_same_run"] = line["value"] / (world * base[0]["value"])
                c4 = measure(ctx, light, "C4", world, full=False)               # ONE 2^26-element problem, sliced
                b4 = [None]
                if ctx.rank == 0:
                    b4[0] = measure(ctx, light, "C4", 1, full=False)
                ctx.tdist.barrier()
                ctx.tdist.broadcast_object_list(b4, src=0)
                c4["same_run_1gpu"] = b4[0]
                c4["strong_speedup"] = c4["value"] / b4[0]["value"]
                c4["strong_efficiency"] = c4["value"] / b4[0]["value"] / world
                extra["C4_strong"] = c4
        except Exception as exc:          # the headline line must still be printed
            extra["error"] = f"{type(exc).__name__}: {exc}"
        line["baseline_multi_gpu_configs"] = extra
    if ctx.rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        ctx.tdist.barrier()
        ctx.tdist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="default: T on one GPU, C5 (weak, 2^24 elements per GPU) on several")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-pattern", action="store_true", help="skip the pattern-resident variants")
    ap.add_argument("--light", action="store_true",
                    help="throughput + device-resident time-to-1e-10 only (A/B runs; not the contract line)")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the secondary objects of the default run (C5 base, C4 strong)")
    ap.add_argument("--pre-opt", action="append", default=[], metavar="KEY=VALUE",
                    help="amg1d_set_option before the first level is set (e.g. --pre-opt shard_min=65536)")
    ap.add_argument("--opt", action="append", default=[], metavar="KEY=VALUE",
                    help="amg1d_set_option after the upload (A/B experiments, e.g. --opt pdl=0)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (GPU arm; inputs are seeded)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (--impl b200)")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
