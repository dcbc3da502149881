"""bench.py --dump-outputs: the files it writes, the same bytes from two runs with the same arguments, and the state the
CPU oracle reaches after as many frames as the bench simulated (the bench's own CPU arm, bench.CpuC5)."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
N = 1 << 20  # more rows than the dump keeps, so that the sampled path runs


def _bench(out: Path):
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "2", "--warmup", "1", "--particles", str(N), "--no-cpu-baseline",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-6000:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    return line, {f.stem: np.load(f) for f in sorted(out.glob("*.npy"))}


def test_dump_outputs_are_reproducible_and_match_the_oracle(tmp_path):
    line, a = _bench(tmp_path / "a")
    _, b = _bench(tmp_path / "b")
    assert line["steps"] == 2
    assert sorted(a) == ["draw_args", "indirect", "metadata", "particles", "rows"]
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for name, x in a.items():
        assert x.dtype in (np.float32, np.float64), name
        assert x.dtype == b[name].dtype and x.tobytes() == b[name].tobytes(), name
    rows = a["rows"].astype(np.int64)
    assert a["particles"].shape == (rows.size, 8) and a["indirect"].shape == (rows.size, 3)
    assert N // 4 <= rows.size < N and np.unique(rows).size == rows.size and rows.max() < N
    assert a["metadata"][1] == N and a["draw_args"][1] == N  # alive_count, instance_count: nothing dies in C5

    import bench
    arm = bench.CpuC5(N, bench.usable_cpus()[1])
    for _ in range(line["config"]["state_checksum"]["frames"]):
        arm.step()
    np.testing.assert_array_equal(a["particles"].view(np.uint32), arm.particles[rows].view(np.uint32))
    np.testing.assert_array_equal(a["indirect"], arm.indirect[rows].astype(np.float64))
