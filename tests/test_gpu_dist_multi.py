"""The multi-column set on slab-sharded handles: needs >= 2 GPUs on the box; skipped below the world size.

tests/dist_multi_worker.py runs every multi-column call on each rank's slabs and checks each column bit for bit against
the single-column call on the same sharded handle, and the gathered slabs of the multi-column cycle against a
single-GPU handle."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ngpu():
    import torch
    return torch.cuda.device_count()


# dg: T shape with pipelined level-0 legs; cg: C4 shape (two-parent transfers: coarse elements owned past the right
# slab edge); dg8: 9 x 9 blocks (row-per-thread legs, once per column); dg_pat: pattern-resident operators;
# dg_nccl: the resident problem's slab edges through NCCL as well (option p2p_halo = 0)
KINDS = ["dg", "cg", "dg8", "dg_pat", "dg_nccl"]


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_multi_column_set(world, tmp_path):
    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs")
    out = tmp_path / "dist_multi.json"
    log2n = 15 if world <= 4 else 16                     # several sharded levels at shard_min = 512
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29600 + world),
           os.path.join(ROOT, "tests", "dist_multi_worker.py"), str(out), str(log2n), ",".join(KINDS)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=2400)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    reps = json.load(open(out))
    keep = os.environ.get("AMG1D_DIST_MULTI_LOG")
    if keep:
        json.dump(reps, open(keep.format(world=world), "w"), indent=1)
    assert sorted(reps) == sorted(KINDS)
    for kind, rep in reps.items():
        assert rep["ok"], (kind, rep["msgs"])
        for rr in rep["ranks"]:
            assert rr["gather_level"] > 1 and rr["sharded_levels"] >= 2, (kind, rr)
            assert rr["p2p_halo"] == rr["p2p_requested"] == rr["p2p_halo_after"], (kind, rr)
            # the exchanges are batched: a rank without coarse levels launches as much for 8 columns as for 1
            if "launches_k1" in rr:
                assert rr["launches_k1"] == rr["launches_k3"] == rr["launches_k8"], (kind, rr)
        if kind != "dg8":
            # every sharded level reads its operator once for all columns: on the C4 shape (cg) this includes the
            # two-parent levels whose restriction gathers past the right slab edge (n_cover)
            for rr in rep["ranks"]:
                assert all(rr["multi_legs"][l] == 1 for l in range(rr["gather_level"])), (kind, rr)
            assert all("launches_k8" in rr for rr in rep["ranks"][1:]), (kind, rep["ranks"])
