"""bench.py contract pieces that run without a GPU: the reference arm (the real reference PLMSSampler + UNetModel from
oracle/_ref or a reference checkout on the host cores; the oracle port only when neither exists) prints one JSON line with the
keys the driver reads; the product arm refuses to run without CUDA (no CPU fallback)."""
import json
import os
import subprocess
import sys

import torch

from oracle import build_ref, ref_harness as RH

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "tiny", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["unit"] == "images/s"
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    cb = line["cpu_baseline"]
    have_ref = os.path.isdir(RH.REF_DIR) or build_ref.available()          # what ref_harness.mount() can use
    assert cb["kind"] == ("reference" if have_ref else "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    if have_ref:
        assert "PLMSSampler.sample" in cb["sample"] and line["config"]["reference_batch"] >= 1
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_other_ranks_are_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "tiny", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_needs_cuda():
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_dump_outputs_float32_and_bounded(tmp_path):
    """--dump-outputs: every array as <name>.npy in float32; above the budget, the same seeded sample every time."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    arrays = {"a": torch.randn(4, 4, 8, 8, dtype=torch.bfloat16), "b": torch.arange(1000, dtype=torch.float64)}
    bench.dump_outputs(str(tmp_path / "full"), arrays, budget=1 << 20)
    a = np.load(tmp_path / "full" / "a.npy")
    assert a.dtype == np.float32 and a.shape == (4, 4, 8, 8) and np.array_equal(a, arrays["a"].float().numpy())
    assert np.array_equal(np.load(tmp_path / "full" / "b.npy"), np.arange(1000, dtype=np.float32))
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget=2000)
    sa, sb = np.load(tmp_path / "s1" / "a.npy"), np.load(tmp_path / "s1" / "b.npy")
    assert 4 * (sa.size + sb.size) <= 2000 and sa.size == 1024 * 2000 // 8096 and sb.size == 1000 * 2000 // 8096
    assert set(sb.tolist()) <= set(range(1000)) and np.all(np.diff(sb) > 0)
    assert np.array_equal(sa, np.load(tmp_path / "s2" / "a.npy")) and np.array_equal(sb, np.load(tmp_path / "s2" / "b.npy"))
