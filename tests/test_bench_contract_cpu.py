"""bench.py's driver contract, as far as it can be checked without a GPU: the reference arm prints ONE JSON line with
every key the contract names, on this arm's metric / unit / config; the B200 arm refuses to run without a device (there
is no CPU path) instead of measuring something else."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_json_line():
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "3"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "particle-steps/s" and d["metric"].startswith("particle-steps/sec at 64M")
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert d["value"] > 1e6 and d["steps"] == 2 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_stay_silent():
    """Under torchrun only rank 0 runs the CPU arm; the other ranks exit 0 without output."""
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "3"], capture_output=True, text=True,
                       timeout=300, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_b200_arm_has_no_cpu_path():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "2", "--warmup", "3"], capture_output=True, text=True, timeout=300)
    assert p.returncode != 0
    assert "no CUDA device" in (p.stdout + p.stderr) and "{" not in p.stdout


@pytest.mark.parametrize("args,message", [(["--steps", "0"], "--steps must be at least 1"),
                                          (["--impl", "reference", "--dump-outputs", "out"], "--dump-outputs applies to --impl b200")])
def test_bad_arguments_are_refused(tmp_path, args, message):
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=120, cwd=tmp_path)
    assert p.returncode != 0 and message in p.stderr and "{" not in p.stdout
    assert not any(tmp_path.iterdir())


@pytest.mark.parametrize("particles", [64 << 20, 1 << 20, 1000])
@pytest.mark.parametrize("world", [1, 2, 3, 8, 200])
def test_dump_sample_is_capped_over_the_whole_job(world, particles):
    """--dump-outputs keeps at most DUMP_SAMPLE_ROWS rows over all ranks (64 bytes a row: 32 MiB), the same rows every run."""
    import numpy as np
    import bench
    from bevy_hanabi_b200.sharding import shard_range
    kept = 0
    for rank in range(world):
        first, end = shard_range(particles, rank, world)
        block, starts = bench.dump_sample(end - first, world)
        rows = (starts[:, None] + np.arange(block)).reshape(-1)
        assert np.unique(rows).size == rows.size and 0 <= rows.min() and rows.max() < end - first
        again = bench.dump_sample(end - first, world)
        assert again[0] == block and np.array_equal(again[1], starts)
        kept += rows.size
    assert kept <= bench.DUMP_SAMPLE_ROWS and kept * 64 <= 32 << 20
    if particles <= bench.DUMP_SAMPLE_ROWS:
        assert kept == particles
