"""CPU test of bench.py --dump-outputs: the files, their dtypes, the masking of empty slots and the 64 MB cap."""
import os

import numpy as np

import bench
from searchlite_b200.engine import HIT_DTYPE


def _results(n_q, k, seed):
    rng = np.random.default_rng(seed)
    hits = np.zeros((n_q, k), dtype=HIT_DTYPE)
    hits["segment_ord"] = rng.integers(0, 8, size=(n_q, k))
    hits["doc_id"] = rng.integers(0, 2**32, size=(n_q, k), dtype=np.uint64)
    hits["score"] = rng.random((n_q, k), dtype=np.float32)
    return hits, rng.integers(0, k + 1, size=n_q).astype(np.uint32)


def _load(d):
    return {n[:-4]: np.load(os.path.join(d, n)) for n in os.listdir(d)}


def test_dump_writes_every_query_exactly(tmp_path):
    hits, counts = _results(300, 11, 1)
    bench.dump_outputs(str(tmp_path), hits, counts)
    out = _load(tmp_path)
    assert sorted(out) == ["counts", "hits_doc_id", "hits_score", "hits_segment_ord", "query_index"]
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert np.array_equal(out["query_index"], np.arange(300)) and np.array_equal(out["counts"], counts)
    valid = np.arange(11)[None, :] < counts[:, None]
    for name in ("doc_id", "segment_ord", "score"):
        a = out["hits_" + name]
        assert np.array_equal(a[valid], hits[name][valid]) and not a[~valid].any()
    assert out["hits_score"].dtype == np.float32


def test_dump_of_a_large_batch_is_a_fixed_sample_under_64_mb(tmp_path):
    hits, counts = _results(4000, 1001, 2)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), hits, counts)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    rows = a["query_index"].astype(np.int64)
    assert 0 < len(rows) < 4000 and np.all(np.diff(rows) > 0)
    assert all(np.array_equal(a[n], b[n]) for n in a)
    assert np.array_equal(a["counts"], counts[rows]) and np.array_equal(a["hits_doc_id"][:, 0][counts[rows] > 0],
                                                                        hits["doc_id"][rows, 0][counts[rows] > 0])
