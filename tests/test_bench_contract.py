"""bench.py contract: the reference arm prints ONE JSON line with the keys a caller reads; the b200 arm times the
requested steps, dumps what the last one computed (-m gpu) and fails loudly without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True and d["value"] > 0
    for k in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        assert d["metric"] == json.load(f)["metric"]


@pytest.mark.gpu
def test_b200_arm_times_the_requested_steps_and_dumps_the_last_output(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-train", "--no-alt",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    assert json.loads(lines[0])["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["output.npy"]
    y = np.load(tmp_path / "output.npy")
    assert y.shape == (32, 1, 288, 288) and y.dtype == np.float32
    assert np.isfinite(y).all() and np.abs(y).max() > 0


def test_b200_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "{" not in out.stdout      # no silent CPU fallback, no fake bench line
