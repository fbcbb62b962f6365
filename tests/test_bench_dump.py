"""`bench.py --dump-outputs DIR`: the arrays the caller received in the last timed step, as float64
.npy files, the same rows from run to run and within the size budget."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _received(n):
    return {"assignment_v3": np.arange(n, dtype=np.int64) % 7, "logweights": -np.linspace(0.0, 1.0, n)}


def test_dump_writes_every_row_when_it_fits(tmp_path):
    bench.dump_outputs(str(tmp_path), _received(100), 50, 150, 1, lambda m: None)
    rows = np.load(tmp_path / "rows.npy")
    assert rows.dtype == np.float64 and (rows == np.arange(50, 150)).all()
    a = np.load(tmp_path / "assignment_v3.npy")
    w = np.load(tmp_path / "logweights.npy")
    assert a.dtype == np.float64 and (a == np.arange(100) % 7).all()
    assert w.dtype == np.float64 and (w == -np.linspace(0.0, 1.0, 100)).all()


def test_dump_samples_the_same_rows_of_every_array(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 8 * 3 * 40)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), _received(1000), 0, 1000, 7, lambda m: None)
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert len(rows) == 40 and (np.diff(rows) > 0).all()
    assert (np.load(tmp_path / "a" / "assignment_v3.npy") == rows % 7).all()
    assert (np.load(tmp_path / "a" / "logweights.npy") == -np.linspace(0.0, 1.0, 1000)[rows.astype(int)]).all()
    for name in ("rows", "assignment_v3", "logweights"):
        assert (np.load(tmp_path / "a" / f"{name}.npy") == np.load(tmp_path / "b" / f"{name}.npy")).all()
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert total <= 8 * 3 * 40 + 3 * 128


@pytest.mark.gpu
def test_bench_dumps_the_last_step(tmp_path):
    """two runs with the same arguments dump the same arrays: the engine's sweeps are keyed by
    (seed, sweep index), so a difference between two builds is a difference in what they compute"""
    for d in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--rows", "3000", "--hospitals", "32", "--steps", "2",
                              "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / d)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b"))
    assert "rows.npy" in files and "logweights.npy" in files and any(f.startswith("assignment_v") for f in files)
    assert (np.load(tmp_path / "a" / "rows.npy") == np.arange(3000)).all()
    for f in files:
        v = np.load(tmp_path / "a" / f)
        assert v.dtype == np.float64 and v.shape == (3000,) and not np.isnan(v).any(), f
        if f.startswith("assignment_v"):
            assert (v >= -1).all() and (v == np.round(v)).all(), f
        assert np.array_equal(v, np.load(tmp_path / "b" / f)), f
