"""GPU tier: bench.py's command line at a small size. --steps is the number of timed steps of the headline (one launch of the
fused kernel each), and --dump-outputs writes the same features whatever the step count, so that two builds can be compared
output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench(steps, dump_dir, utts=16):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
                        "--utts", str(utts), "--no-e2e", "--no-cpu", "--no-extras", "--dump-outputs", str(dump_dir)],
                       cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_steps_and_dump_outputs(tmp_path):
    a = bench(1, tmp_path / "a")
    b = bench(4, tmp_path / "b")
    assert (a["steps"], b["steps"]) == (1, 4)
    assert a["gpu_launches"] >= 1 and b["gpu_launches"] == 4 * a["gpu_launches"]
    assert os.listdir(tmp_path / "a") == ["features.npy"]
    fa, fb = np.load(tmp_path / "a" / "features.npy"), np.load(tmp_path / "b" / "features.npy")
    assert fa.dtype == np.float32 and fa.shape == (16, 998, 39) and np.isfinite(fa).all()
    np.testing.assert_array_equal(fa, fb)        # same seeded inputs, deterministic kernel
