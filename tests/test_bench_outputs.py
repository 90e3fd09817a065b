"""bench.py --dump-outputs on a small workload: the state of the last timed step is written as float64 .npy files,
and two runs with the same workload arguments but different step counts write the same arrays."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--gpus", "1", "--reaches", "3000", "--members", "16", "--gauges", "20", "--days", "0.25",
         "--c4-reaches", "20000", "--no-cpu-baseline", "--no-e2e"]


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), *SMALL, "--steps", str(steps), "--warmup", "1",
           "--dump-outputs", str(out_dir)]
    res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, (res.stdout + res.stderr)[-3000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


def test_dump_outputs_are_the_same_for_any_step_count(libtxh, tmp_path):
    line1 = _bench(tmp_path / "a", 1)
    line3 = _bench(tmp_path / "b", 3)
    assert line1["steps"] == 1 and line3["steps"] == 3
    shapes = {"c3_outflow": (3000, 16), "c3_inflow": (3000, 16), "c4_outflow": (20000,), "c4_inflow": (20000,)}
    assert sorted(os.listdir(tmp_path / "a")) == sorted(k + ".npy" for k in shapes)
    for name, shape in shapes.items():
        a = np.load(tmp_path / "a" / (name + ".npy"))
        b = np.load(tmp_path / "b" / (name + ".npy"))
        assert a.dtype == np.float64 and a.shape == shape and np.isfinite(a).all() and np.abs(a).max() > 0
        assert np.array_equal(a, b), name
