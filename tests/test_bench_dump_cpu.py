"""bench.py --dump-outputs: the file format, on a synthetic TopDocs triple (no GPU needed)."""
import os

import numpy as np

import bench
from rucene_b200 import engine


def _result(nq, k, seed=1):
    rng = np.random.default_rng(seed)
    hits = np.zeros((nq, k), engine.HIT_DTYPE)
    hits["doc"] = rng.integers(0, 100_000_000, size=(nq, k))
    hits["score"] = rng.random((nq, k), dtype=np.float32)
    counts = rng.integers(0, k + 1, size=nq).astype(np.uint32)
    total = (counts + rng.integers(0, 1000, size=nq)).astype(np.uint64)
    return hits, counts, total


def _load(d):
    return {n: np.load(os.path.join(d, n + ".npy")) for n in ("docs", "scores", "counts", "total_hits", "query_rows")}


def test_dump_writes_every_row_exactly(tmp_path):
    hits, counts, total = _result(64, 10)
    bench.dump_outputs(str(tmp_path), (hits, counts, total))
    got = _load(str(tmp_path))
    assert {a.dtype for a in got.values()} <= {np.dtype(np.float32), np.dtype(np.float64)}
    assert np.array_equal(got["query_rows"], np.arange(64))
    assert np.array_equal(got["counts"], counts) and np.array_equal(got["total_hits"], total)
    for i in range(64):
        n = int(counts[i])
        assert np.array_equal(got["docs"][i, :n], hits["doc"][i, :n])
        assert np.array_equal(got["scores"][i, :n].view(np.uint32), hits["score"][i, :n].view(np.uint32))
        assert np.all(got["docs"][i, n:] == -1) and np.all(got["scores"][i, n:] == 0)


def test_dump_samples_rows_above_the_size_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 20 * (10 * 12 + 24))
    res = _result(100, 10)
    bench.dump_outputs(str(tmp_path / "a"), res)
    bench.dump_outputs(str(tmp_path / "b"), res)
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    rows = a["query_rows"].astype(np.int64)
    assert len(rows) == 20 and np.all(np.diff(rows) > 0)
    assert all(np.array_equal(a[n], b[n]) for n in a)      # the same sample every time
    assert np.array_equal(a["total_hits"], res[2][rows])
