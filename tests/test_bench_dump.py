"""bench.py --dump-outputs: the files it writes (float32 / float64 .npy, one row per stream) and the seeded sample it keeps beyond its
size limit.  CPU only."""
import os

import numpy as np

import bench


def _arrays(n):
    rng = np.random.default_rng(1)
    return {"xy": rng.normal(size=(n, 4, 2)).astype(np.float32), "status": rng.integers(0, 2, (n, 4), dtype=np.uint8),
            "cost": rng.normal(size=n), "row": np.arange(n, dtype=np.float64)}


def test_all_streams_below_the_limit(tmp_path):
    a = _arrays(10)
    bench.write_outputs(str(tmp_path), a)
    assert sorted(os.listdir(tmp_path)) == ["cost.npy", "row.npy", "status.npy", "xy.npy"]
    for k, v in a.items():
        got = np.load(tmp_path / f"{k}.npy")
        assert got.dtype == (np.float64 if v.dtype == np.float64 else np.float32)
        assert np.array_equal(got, v)


def test_same_seeded_sample_in_every_array_beyond_the_limit(tmp_path):
    a = _arrays(1000)
    per_stream = 4 * 2 * 4 + 4 * 4 + 8 + 8  # bytes of one stream once written
    limit = 100 * per_stream
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), a, limit=limit)
    rows = np.load(tmp_path / "a" / "row.npy").astype(int)
    assert len(rows) == 100 and np.all(np.diff(rows) > 0)
    assert sum(np.load(tmp_path / "a" / f).nbytes for f in os.listdir(tmp_path / "a")) <= limit
    for k, v in a.items():
        got = np.load(tmp_path / "a" / f"{k}.npy")
        assert np.array_equal(got, v[rows].astype(got.dtype))
        assert np.array_equal(got, np.load(tmp_path / "b" / f"{k}.npy"))
