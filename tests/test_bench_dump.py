"""bench.py --dump-outputs: the outputs of the last timed step, written so that two builds can be compared.

CPU: the seeded sample of a long x is fixed and bounded.  GPU: a small bench run writes x and the residual norm
of exactly warmup + steps V-cycles from the seeded right-hand side, as the library computes them in-process."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _FakeDevice:
    def __init__(self, n):
        self.n = n

    def dev_get_solution(self):
        return np.arange(self.n, dtype=np.float64)


def test_dump_samples_long_outputs_with_a_fixed_seed(tmp_path):
    import bench
    n = 4 * bench.DUMP_MAX_ENTRIES
    runs = []
    for k in range(2):
        d = tmp_path / str(k)
        bench.dump_outputs(str(d), _FakeDevice(n), 1.5)
        runs.append({f: np.load(d / f"{f}.npy") for f in ("x", "x_index", "residual_norm")})
    x, idx = runs[0]["x"], runs[0]["x_index"]
    assert x.dtype == np.float64 and idx.dtype == np.float64
    assert len(x) == bench.DUMP_MAX_ENTRIES and np.all(np.diff(idx) > 0) and idx[-1] < n
    assert np.array_equal(x, idx)                         # x[i] == i: the values are those at the stored positions
    assert np.array_equal(runs[0]["residual_norm"], [1.5])
    for f in runs[0]:
        assert np.array_equal(runs[0][f], runs[1][f])
    small = tmp_path / "small"
    bench.dump_outputs(str(small), _FakeDevice(1000), 0.0)
    assert np.array_equal(np.load(small / "x.npy"), np.arange(1000))


@pytest.mark.gpu
def test_dump_holds_the_last_timed_step(tmp_path):
    import bench
    steps, warmup = 2, 3
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "S", "--light", "--steps", str(steps),
           "--warmup", str(warmup), "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    x, idx, res = (np.load(out / f"{f}.npy") for f in ("x", "x_index", "residual_norm"))

    U = bench.build_hierarchy("S", 2 ** bench.WORKLOADS["S"][0])
    dev = U.upload()
    try:
        dev.dev_fill_rhs_random(0)
        for _ in range(warmup + steps):
            dev.dev_vcycle(with_residual_norm=True)
        x_ref, res_ref = dev.dev_get_solution(), dev.dev_residual_norm()
    finally:
        dev.close()
    assert np.array_equal(idx, np.arange(len(x_ref)))
    assert np.allclose(x, x_ref, rtol=1e-12, atol=1e-14 * np.abs(x_ref).max())
    assert np.isclose(res[0], res_ref, rtol=1e-12)
