"""bench.py --dump-outputs on the GPU path: the final output of the last timed step is written, and two runs with the same arguments
write the same values (the inputs are seeded), so two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "1", "--steps", str(steps), "--warmup", "0", "--no-cpu-baseline",
                        "--dump-outputs", str(out_dir)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])


def test_dump_outputs_repeatable(tmp_path):
    lines = [run_bench(tmp_path / d, 3) for d in ("a", "b")]
    assert all(d["steps"] == 3 for d in lines)
    assert os.listdir(tmp_path / "a") == ["shadows.npy"]
    a, b = np.load(tmp_path / "a" / "shadows.npy"), np.load(tmp_path / "b" / "shadows.npy")
    assert a.dtype == np.float64 and a.shape == (64, 32)  # config 1 is not denoised: its final output is the R32_UINT visibility mask (8x4 px per word)
    assert np.array_equal(a, b)
