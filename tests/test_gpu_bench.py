"""bench.py --dump-outputs: the arrays of the last timed training step, written as .npy files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "4", "--warmup", "3",
                        "--no-phases", "--no-cpu-baseline", "--no-gpu-eager-bar", "--no-per-config", "--no-fp32-line",
                        "--dump-outputs", str(out)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 4
    a = {f[:-len(".npy")]: np.load(out / f) for f in os.listdir(out)}
    assert set(a) == {"node_loc", "virtual_node_loc", "loss", "mse", "params", "grads"}
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64_000_000

    sys.path.insert(0, ROOT)
    import bench
    data, _ = bench.make_workload("water3d", seed=0, nodes=0)
    assert a["node_loc"].shape == tuple(data["loc_0"].shape) and a["virtual_node_loc"].shape == (1, 3, data["C"])
    assert a["loss"].shape == a["mse"].shape == (1,) and a["params"].shape == a["grads"].shape
    assert np.abs(a["grads"]).max() > 0
    # the dumped MSE is the one of the dumped prediction against the workload's targets: one and the same step
    mse = np.mean((a["node_loc"].astype(np.float64) - data["loc_t"].numpy()) ** 2)
    assert abs(mse - float(a["mse"][0])) <= 1e-4 * mse
