"""bench.py contract on the CPU: the reference arm (`--impl reference`, the CPU oracle timed on the host cores) prints ONE JSON line
with the keys the driver reads, for every BASELINE config, and — launched as N ranks — only rank 0 prints it.  The GPU arm needs
a B200 and is exercised by the driver; its line carries the same keys plus roofline / clocks / gpu_launches."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
            "impl", "cpu_baseline", "e2e")


def run_reference(config, env=None, steps=1):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", str(config), "--steps", str(steps), "--warmup", "0"],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, env=e, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return [ln for ln in out.stdout.splitlines() if ln.strip()]


@pytest.mark.parametrize("config", [1, 2])
def test_reference_arm_line(config):
    lines = run_reference(config)
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in REQUIRED:
        assert k in d, k
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "frames/s" and d["value"] > 0
    assert d["config"]["baseline_config"] == config and "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert abs(d["ms_per_step"] - 1e3 / d["value"]) <= 1e-6 * d["ms_per_step"] + 1e-9


def test_reference_arm_only_rank0_prints():
    env = {"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29599"}
    assert run_reference(1, env) == []


def test_dump_outputs_bounded_and_repeatable(tmp_path):
    """--dump-outputs: a 4K RGBA16F image is sampled under its share of the 64 MB, a small R32_UINT image is written whole and exactly,
    and the same images give the same files."""
    import numpy as np
    import bench
    rng = np.random.default_rng(3)
    imgs = {"big": rng.standard_normal((2160, 3840, 4)).astype(np.float16), "small": rng.integers(0, 2**32, (48, 64), dtype=np.uint32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), imgs)
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert sorted(os.listdir(tmp_path / "a")) == ["big.npy", "small.npy"] and total <= bench.DUMP_BYTES
    big, small = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "a" / "small.npy")
    assert big.dtype == np.float32 and big.shape[1] == 4 and big.nbytes > 0.99 * bench.DUMP_BYTES / 2  # the sample fills its half of the budget
    assert small.dtype == np.float64 and np.array_equal(small, imgs["small"])
    assert np.array_equal(big, np.load(tmp_path / "b" / "big.npy"))
    px = imgs["big"].reshape(-1, 4).astype(np.float32)
    assert all((px == big[i]).all(1).any() for i in (0, len(big) // 2, -1)), "sampled values are not pixels of the image"
