"""bench.py --dump-outputs: the written arrays are float64, small enough to keep and compare, and sampled at the same
positions on every run, so that the outputs of two builds can be compared entry for entry."""
import os
import subprocess
import sys

import numpy as np

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_is_float64_bounded_and_reproducible(tmp_path):
    big = np.random.default_rng(5).standard_normal(bench.DUMP_MAX_ENTRIES + 12345)
    arrays = {"objective": np.array([2.5]), "constraint": np.arange(7, dtype=np.float32), "jacobian": big}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    assert sorted(os.listdir(tmp_path / "a")) == ["constraint.npy", "jacobian.npy", "objective.npy"]
    for name in arrays:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float64 and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "constraint.npy"), np.arange(7.0))
    sampled = np.load(tmp_path / "a" / "jacobian.npy")
    assert sampled.size == bench.DUMP_MAX_ENTRIES and np.isin(sampled, big).all()
    assert 5 * 8 * bench.DUMP_MAX_ENTRIES <= 64 << 20  # five outputs at most


def test_bench_rejects_zero_steps():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr
