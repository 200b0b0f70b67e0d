"""bench.py on the GPU: --dump-outputs writes what the timed path computed in its last step, the same for the same arguments,
so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_are_reproducible(tmp_path):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--warmup", "1", "--no-subrecords", "--no-cpu-baseline", "--clock-ms", "0"]
    lines = {}
    for run, steps in (("a", 3), ("b", 3), ("c", 5)):
        r = subprocess.run(cmd + ["--steps", str(steps)] + (["--dump-outputs", str(tmp_path / run)] if steps == 3 else []),
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        lines[run] = json.loads(r.stdout)
    # --steps sets the timed steps: the launches counted inside the timed region grow with it, by the same count per step
    per_step = lines["a"]["gpu_launches"] / 3
    assert per_step >= 1 and lines["b"]["gpu_launches"] == lines["a"]["gpu_launches"] and lines["c"]["gpu_launches"] == 5 * per_step
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["brick_counters.npy", "occupied_bricks.npy", "tsdf_occupied_bricks.npy", "tsdf_sample.npy", "tsdf_sample_index.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 20
    out = {}
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and a.tobytes() == b.tobytes(), n
        out[n[:-4]] = a
    assert len(out["occupied_bricks"]) > 100 and (out["brick_counters"][out["occupied_bricks"].astype(np.int64)] >= 10).all()
    assert (np.abs(out["tsdf_occupied_bricks"]) < 0.01).sum() > 100000, "the occupied bricks hold the surface band"
    assert (np.abs(out["tsdf_sample"]) < 0.01).sum() > 1000
