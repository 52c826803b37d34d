"""Presence bitmaps with interleaved rank (slg_residency.cuh): a verification takes a bitmap term's held bit and its list
position from one 32-byte unit (a rank word + the bits of 224 docs).  The looked-up posting is the same posting a search
finds, so results must not move by a bit: against the oracle, between bm25 and bmw, and against the same segments loaded
without bitmaps (bitmap_den 0: every look-up searches the list)."""
from __future__ import annotations

import numpy as np
import pytest

from searchlite_b200 import GpuIndex, QueryBatch
from tests.helpers import canonical_batch, segment_from_postings

pytestmark = pytest.mark.gpu

UNIT = 224
DEN = 64  # bitmap_den: a term without a column gets a bitmap at df * 64 >= doc_count (and df >= 64)
OPTIONS = {"dense_den": 6, "dense_min_df": 64, "bitmap_den": DEN}


def _segment(doc_count: int, ord_: int, seed: int, threshold_term: bool):
    """terms 0..3 are the edge cases, then mid-dense terms (bitmaps), rare terms (searched) and dense ones (columns)"""
    rng = np.random.default_rng(seed)
    edges = [0, UNIT - 1, UNIT, 2 * UNIT - 1, doc_count - 1]

    def some(df, must=()):
        pick = set(int(x) for x in rng.choice(doc_count, size=df, replace=False))
        pick.update(must)
        return sorted(pick)

    thr = (doc_count + DEN - 1) // DEN  # the smallest df that gets a bitmap
    lists = []
    if threshold_term:
        assert thr * DEN == doc_count
        base = some(thr - len(edges), edges)
        while len(base) < thr:  # (the random part may have hit an edge doc)
            base = sorted(set(base) | {int(rng.integers(doc_count))})
        lists.append(base)                                    # 0: df exactly at the threshold, holds every edge doc
        lists.append(some(thr - 1 - len(edges), edges))       # 1: one below: no bitmap, searched
    else:
        lists.append(some(thr + 40, edges))
        lists.append(some(max(thr - 30, 70), edges))
    full = 5 * UNIT
    lists.append(sorted(set(range(full, full + UNIT)) | set(some(300))))  # 2: every doc of unit 5
    lists.append(some(400, edges))                                          # 3: edge docs again, mid density
    for _ in range(24):
        lists.append(some(int(rng.integers(thr, doc_count // 8))))          # mid-dense: bitmaps
    for _ in range(12):
        lists.append(some(int(rng.integers(8, 60))))                        # rare: searched
    for _ in range(6):
        lists.append(some(int(rng.integers(doc_count // 5, doc_count // 2))))  # dense: columns
    postings = [(d, rng.integers(1, 6, size=len(d)).tolist()) for d in lists]
    lens = rng.integers(8, 90, size=doc_count)
    deleted = sorted(set(rng.choice(doc_count, size=doc_count // 50, replace=False).tolist()) | {UNIT, doc_count - 1})
    return segment_from_postings(postings, lens, segment_ord=ord_, deleted=deleted), len(lists)


@pytest.fixture(scope="module")
def corpus():
    from oracle import slo
    a, n_terms = _segment(DEN * 141, 0, 11, True)   # 9024 docs: 40 whole units + 64 docs
    b, _ = _segment(UNIT * 31 + 5, 1, 12, False)
    assert a.doc_count % UNIT and b.doc_count % UNIT
    segs = [a, b]
    gis = {}
    for den in (DEN, 0):
        gi = GpuIndex(0, options=dict(OPTIONS, bitmap_den=den))
        for s in segs:
            gi.load_segment(s)
        gis[den] = gi
    yield segs, [slo.OracleIndex(s) for s in segs], gis, n_terms
    for gi in gis.values():
        gi.close()


def _or_batch(n_terms: int, with_columns: bool, seed: int) -> QueryBatch:
    rng = np.random.default_rng(seed)
    sparse = np.arange(0, n_terms - 6)
    cols = np.arange(n_terms - 6, n_terms)
    qs = []
    for i in range(160):
        n = 2 + i % 4
        t = rng.choice(sparse, size=n, replace=False).tolist()
        if i % 5 == 0:
            t[0] = int(rng.integers(0, 4))  # an edge-case term in every fifth query
        if with_columns:
            t = rng.choice(cols, size=2, replace=False).tolist() + t[:2]
        qs.append(t)
    return QueryBatch.from_term_lists(qs)


def _check(segs, oras, gis, qb: QueryBatch, k: int):
    from oracle import slo
    gi = gis[DEN]
    res = {mode: gi.search_batch(qb, k, mode) for mode in ("bm25", "bmw")}
    for mode in ("bm25", "bmw"):
        assert res[mode][0].tobytes() == res["bm25"][0].tobytes() and res[mode][1].tobytes() == res["bm25"][1].tobytes(), mode
        plain = gis[0].search_batch(qb, k, mode)
        assert res[mode][0].tobytes() == plain[0].tobytes() and res[mode][1].tobytes() == plain[1].tobytes(), mode
    per_seg = [o.search_batch(canonical_batch(gi, qb, s.segment_ord), k, "bm25") for s, o in zip(segs, oras)]
    got_h, got_c = res["bm25"]
    n_hits = 0
    for qi in range(qb.n_queries):
        ref = slo.merge_hits([h[qi, : c[qi]] for h, c in per_seg], k)
        got = got_h[qi, : got_c[qi]]
        assert got.tobytes() == ref.tobytes(), qi  # declared order: bit for bit
        n_hits += len(got)
    assert n_hits > 0


def test_segments_get_rank_bitmaps(corpus):
    segs, _, gis, _ = corpus
    for s in segs:
        r = gis[DEN].segment_residency(s.segment_ord)
        assert r["n_presence_bitmaps"] > 20
        assert r["presence_bitmaps"] == r["n_presence_bitmaps"] * ((s.doc_count + UNIT - 1) // UNIT) * 32  # 32 bytes per 224 docs
        assert gis[0].segment_residency(s.segment_ord)["n_presence_bitmaps"] == 0


@pytest.mark.parametrize("k", [11, 101])
@pytest.mark.parametrize("with_columns", [False, True])
def test_or_batches_match_the_search_path(corpus, k, with_columns):
    segs, oras, gis, n_terms = corpus
    qb = _or_batch(n_terms, with_columns, seed=100 + k + with_columns)
    _check(segs, oras, gis, qb, k)
    assert gis[DEN].counters()["last_postings_scattered"] > 0  # the flat posting scan ran


def test_and_batch_matches_the_search_path(corpus):
    segs, oras, gis, n_terms = corpus
    rng = np.random.default_rng(5)
    qs = []
    for i in range(120):
        t = rng.choice(np.arange(0, n_terms), size=2 + i % 2, replace=False).tolist()
        if i % 4 == 0:
            t[0] = int(rng.integers(0, 4))
        qs.append({"must": t})
    _check(segs, oras, gis, QueryBatch.from_bool(qs), 11)
