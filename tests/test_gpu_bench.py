"""GPU: ``bench.py --dump-outputs`` writes what the timed path computed in its last step -- the same arrays
from run to run with the same workload arguments, whatever the number of timed steps."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
           "--orbits-per-gpu", "6", "--no-verify", "--no-png", "--no-e2e", "--no-api-e2e", "--no-cpu-baseline",
           "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[:2000]
    return json.loads(lines[0])


def test_bench_dump_outputs_repeat_across_runs(tmp_path):
    a = _bench(tmp_path / "a", 2)
    b = _bench(tmp_path / "b", 3)
    assert (a["steps"], b["steps"]) == (2, 3)
    assert a["gpu_launches"] * 3 == b["gpu_launches"] * 2  # every timed step is one whole step
    names = ["extrema.npy", "panel_vmin_vmax.npy", "rgba_sample.npy"]
    assert sorted(os.listdir(tmp_path / "a")) == sorted(os.listdir(tmp_path / "b")) == names
    got = {}
    for name in names:
        x, y = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert x.dtype in (np.float32, np.float64) and x.dtype == y.dtype and x.shape == y.shape, name
        assert np.array_equal(x, y, equal_nan=True), name
        got[name[:-4]] = x
    assert sum(x.nbytes for x in got.values()) <= 64 << 20
    assert got["extrema"].shape == (16,) and np.isfinite(got["extrema"]).any()  # 4 instruments x y/z min/max
    assert got["panel_vmin_vmax"].shape == (a["plan"]["panels_per_gpu"], 2)
    rgba = got["rgba_sample"]
    assert a["plan"]["pixels_per_gpu"] > len(rgba) and rgba.shape[1] == 4  # a sample of a larger raster
    assert rgba.min() >= 0 and rgba.max() <= 255 and np.all(rgba == np.floor(rgba))
