"""bench.py --dump-outputs on the device: the last timed step's loss and a fixed sample of the updated parameters, next to
the one JSON line on stdout."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_after_the_timed_steps(cuda_device, tmp_path):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--no-cpu-baseline",
           "--dump-outputs", str(tmp_path)]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    assert json.loads(r.stdout)["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["loss.npy", "params.npy"]
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20
    loss, params = np.load(tmp_path / "loss.npy"), np.load(tmp_path / "params.npy")
    assert loss.dtype == np.float32 and loss.shape == () and np.isfinite(loss) and loss > 0
    assert params.dtype == np.float32 and params.shape == (1 << 22,) and np.isfinite(params).all()
