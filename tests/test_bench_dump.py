"""bench.py's command line and --dump-outputs: the result of the timed path as float64 .npy files of bounded total size."""
import os
import subprocess
import sys

import numpy as np

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_small_result_is_written_whole(tmp_path):
    res = {"revenue": np.array([123456789012, -5], dtype=np.int64), "l_returnflag__lineitem__l_returnflag": np.array([16, 40], dtype=np.int32)}
    bench.dump_outputs(res, str(tmp_path / "d"))
    assert sorted(os.listdir(tmp_path / "d")) == ["l_returnflag__lineitem__l_returnflag.npy", "revenue.npy"]
    for k, v in res.items():
        got = np.load(tmp_path / "d" / f"{k}.npy")
        assert got.dtype == np.float64
        np.testing.assert_array_equal(got, v)


def test_large_result_keeps_the_same_seeded_rows_in_every_column(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096)
    n = 10_000
    res = {"a": np.arange(n, dtype=np.int64), "b": np.arange(n, dtype=np.int32) * 2}
    for d in ("x", "y"):
        bench.dump_outputs(res, str(tmp_path / d))
    assert sum(os.path.getsize(tmp_path / "x" / f) for f in os.listdir(tmp_path / "x")) <= 4096
    a, b = np.load(tmp_path / "x" / "a.npy"), np.load(tmp_path / "x" / "b.npy")
    assert 0 < len(a) < n and np.all(np.diff(a) > 0)
    np.testing.assert_array_equal(b, 2 * a)                                  # the same rows in every column ...
    np.testing.assert_array_equal(np.load(tmp_path / "y" / "a.npy"), a)      # ... and in every run


def test_bad_arguments_are_refused_before_any_work():
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=60)
        assert r.returncode == 2 and "error" in r.stderr, (argv, r.stderr)
