"""`bench.py --dump-outputs DIR` -- the timed step's outputs as float32 .npy files, whole when they fit the 64 MB budget,
otherwise the same seeded sample in every run (CPU, and one -m gpu run of bench.py itself)."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402


def test_small_output_is_written_whole(tmp_path):
    t = torch.randn(2, 9, 13, dtype=torch.float64)
    bench.dump_outputs(tmp_path / "a", {"disparity": t})
    a = np.load(tmp_path / "a" / "disparity.npy")
    assert a.dtype == np.float32 and a.shape == (2, 9, 13)
    assert np.array_equal(a, t.float().numpy())


def test_large_output_is_a_fixed_sample_within_the_budget(tmp_path):
    t = torch.arange(bench.DUMP_BYTES // 4 + 12345, dtype=torch.float32).reshape(-1, 5)   # value == flat position
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, {"disparity": t})
    a, b = np.load(tmp_path / "a" / "disparity.npy"), np.load(tmp_path / "b" / "disparity.npy")
    assert (tmp_path / "a" / "disparity.npy").stat().st_size <= bench.DUMP_BYTES
    assert a.dtype == np.float32 and a.ndim == 1 and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0) and a[-1] < t.numel()                  # distinct positions, in order


@pytest.mark.gpu
def test_dump_is_what_the_timed_step_computed(tmp_path):
    """bench.py hands the last timed step's result to the dump: the file equals an eager step on the same seeded workload."""
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "tiny", "--batch", "2", "--steps", "3",
                        "--warmup", "1", "--no-extras", "--no-cpu-baseline", "--no-from-images", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])["steps"] == 3
    from decnet_b200.synthetic import build_workload
    model, left, right, _ = build_workload("tiny", 2, seed=17, device="cuda")
    want = model(left, right)[0].cpu().numpy()
    got = np.load(tmp_path / "disparity.npy")
    assert got.dtype == np.float32 and got.shape == want.shape == (2, 108, 162)
    assert np.allclose(got, want, atol=1e-4, rtol=1e-4), float(np.abs(got - want).max())


def test_dump_is_refused_for_the_reference_arm(tmp_path):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=120, cwd=str(ROOT))
    assert r.returncode != 0 and "--dump-outputs" in r.stderr
