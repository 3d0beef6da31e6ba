"""bench.py --dump-outputs on the GPU at a small size: the final latent of the last timed step, float32, the same bits
from run to run (the inputs are seeded), and --steps is the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _run(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--config", "tiny", "--batch", "2", "--max-objs", "6", "--plms-steps", "4",
           "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--no-kernel-pass", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_outputs_repeatable(tmp_path):
    line1 = _run(tmp_path / "a", 2)
    line2 = _run(tmp_path / "b", 3)
    assert line1["steps"] == 2 and line2["steps"] == 3
    # every step launches the same kernels: the timed window's launch count is proportional to --steps
    assert line1["gpu_launches"] > 0 and 3 * line1["gpu_launches"] == 2 * line2["gpu_launches"]
    assert sorted(os.listdir(tmp_path / "a")) == ["latent.npy"]
    a, b = np.load(tmp_path / "a" / "latent.npy"), np.load(tmp_path / "b" / "latent.npy")
    assert a.dtype == np.float32 and a.shape == (2, 4, 16, 16) and np.isfinite(a).all()
    assert np.array_equal(a, b)
