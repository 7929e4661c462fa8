"""The bench contract on CPU: `bench.py --impl reference` (the CPU arm, the one leg that runs without a GPU) prints exactly ONE JSON
line with the keys its consumers read; the GPU arm's argument surface exists, and (GPU) the arm dumps what it computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from _helpers import ROOT

REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
            "data", "config", "cpu_baseline", "e2e"}


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, FZ_CPU_THREADS="8", FZ_REF_FRAMES="1")  # one frame instead of the clip: the contract, not the number
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0"], env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "frames/s" and d["value"] > 0
    assert d["steps"] == 2 and d["warmup"] == 0  # --steps sets the number of timed passes
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and "workload" in d["config"]


def test_bench_cli_surface():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--shard", "--config", "--graphs", "--dump-outputs"):
        assert flag in r.stdout


def _run_gpu_arm(steps, dump):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "0",
                        "--no-cpu-baseline", "--no-instrument", "--dump-outputs", str(dump)], capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


@pytest.mark.gpu
def test_gpu_arm_dumps_last_step_outputs(tmp_path):
    """--dump-outputs DIR: float32 .npy of what the last timed clip edit returned.  Two runs with different --steps see the same seeded
    inputs, so their dumps agree; --steps is the number of timed clip edits, so the timed region launches twice the kernels for 2 as for 1."""
    d1, d2 = _run_gpu_arm(1, tmp_path / "d1"), _run_gpu_arm(2, tmp_path / "d2")
    assert d1["steps"] == 1 and d2["steps"] == 2
    assert d1["gpu_launches"] > 0 and d2["gpu_launches"] == 2 * d1["gpu_launches"]
    for d in ("d1", "d2"):
        assert sorted(os.listdir(tmp_path / d)) == ["edited_latents.npy", "inverted_latents.npy"]
    for name in ("inverted_latents", "edited_latents"):
        a, b = np.load(tmp_path / "d1" / f"{name}.npy"), np.load(tmp_path / "d2" / f"{name}.npy")
        assert a.dtype == np.float32 and a.shape == (1, 4, 8, 64, 64) and np.isfinite(a).all()
        scale = np.abs(a).max()
        assert scale > 0 and np.abs(a - b).max() <= 1e-3 * scale, (name, np.abs(a - b).max(), scale)
    inv, edit = np.load(tmp_path / "d1" / "inverted_latents.npy"), np.load(tmp_path / "d1" / "edited_latents.npy")
    assert np.abs(edit - inv).max() > 0.1 * np.abs(inv).max()  # the edit moved the latents well away from the inversion's
