"""bench.py --dump-outputs: the headline path's outputs of its last timed step, for a fixed sample of
series, identical however the batch is cut into launches."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["C", "Q", "R", "S", "a", "f", "m", "s", "status"]


def _bench(out_dir, chunks):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--series", "3000", "--T", "40",
           "--steps", "2", "--warmup", "1", "--chunks", str(chunks), "--no-e2e", "--no-ffbs",
           "--no-cpu", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_do_not_depend_on_the_launch_geometry(tmp_path):
    line1, one = _bench(tmp_path / "one", 1)
    line3, three = _bench(tmp_path / "three", 3)
    assert line1["steps"] == 2 and line1["gpu_launches"] == 2      # --steps timed steps, one launch each
    assert line3["gpu_launches"] == 6 and line1["status_max"] == 0
    assert sorted(one) == FIELDS and sorted(three) == FIELDS
    assert one["m"].shape == (41, 2, 256) and one["S"].shape == (41, 4, 256)
    assert one["f"].shape == (40, 1, 256) and one["Q"].shape == (40, 1, 256)  # T forecasts, no init row
    assert one["status"].shape == (256,) and not one["status"].any()
    assert sum(a.nbytes for a in one.values()) <= 64e6
    for k in FIELDS:
        assert one[k].dtype == np.float64
        assert np.isfinite(one[k]).all(), k
        assert np.array_equal(one[k], three[k]), k
