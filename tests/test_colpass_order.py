"""The pruned column pass in bound order (slg_columns_ordered_kernel): a query's 512-doc blocks are scored in descending
order of their column bound and skipped once the bound cannot reach the k-th score.  Every skip is a safe bound against a
real k-th score, so results must not move by a bit: against the oracle (declared summation order) and against `bm25`,
which runs the exhaustive column pass.

The segment's column terms have "hot" blocks (high tf, short docs), so bounds differ widely between blocks and the top
of the order holds the top k; a tie term gives many docs the same score in one block and in a second block of the same
bin."""
from __future__ import annotations

import numpy as np
import pytest

from searchlite_b200 import GpuIndex, QueryBatch
from searchlite_b200.engine import FILTER_DTYPE, F_I64_RANGE, HIT_DTYPE
from tests.helpers import canonical_batch, segment_from_postings
from tests.parity import assert_parity

pytestmark = pytest.mark.gpu

OPTIONS = {"dense_den": 8, "dense_min_df": 64}
N_COLS, N_MID, N_RARE = 6, 16, 8
TIE = N_COLS + N_MID + N_RARE  # term id of the tie column
TIE_BLOCKS = (37, 201)          # the tied docs sit in these two blocks; their bounds are equal (same bin)


def _segment(doc_count: int, ord_: int, seed: int, deleted: bool):
    rng = np.random.default_rng(seed)
    n_blocks = (doc_count + 511) // 512
    lens = rng.integers(40, 400, size=doc_count)
    lists = []
    for c in range(N_COLS):  # column terms: df N/4..N/2, tf 1..3, and a few hot blocks of tf 8..30
        docs = np.sort(rng.choice(doc_count, size=int(rng.integers(doc_count // 4, doc_count // 2)), replace=False))
        tfs = rng.integers(1, 4, size=len(docs))
        hot = rng.choice(n_blocks, size=4, replace=False)
        in_hot = np.isin(docs >> 9, hot)
        tfs[in_hot] = rng.integers(8, 31, size=int(in_hot.sum()))
        lists.append((docs.tolist(), tfs.tolist()))
    for _ in range(N_MID):
        docs = np.sort(rng.choice(doc_count, size=int(rng.integers(doc_count // 200, doc_count // 20)), replace=False))
        lists.append((docs.tolist(), rng.integers(1, 6, size=len(docs)).tolist()))
    for _ in range(N_RARE):
        docs = np.sort(rng.choice(doc_count, size=int(rng.integers(3, 40)), replace=False))
        lists.append((docs.tolist(), rng.integers(1, 4, size=len(docs)).tolist()))
    # the tie column: tf 1 on a third of the docs, and 9 docs in each tie block with tf 6 and the same length
    docs = set(rng.choice(doc_count, size=doc_count // 3, replace=False).tolist())
    tied = [b * 512 + 17 * j + 3 for b in TIE_BLOCKS for j in range(9)]
    docs.update(tied)
    docs = sorted(docs)
    tied_set = set(tied)
    lists.append((docs, [6 if d in tied_set else 1 for d in docs]))
    lens[tied] = 50
    dead = None
    if deleted:
        dead = sorted(set(rng.choice(doc_count, size=doc_count // 40, replace=False).tolist()) | {tied[0], tied[10]})
    seg = segment_from_postings(lists, lens, segment_ord=ord_, deleted=dead)
    seg.fast_i64 = {"grp": ((np.arange(doc_count) % 7).astype(np.int64), None)}
    return seg


def _grp_filter(cols):
    n = np.zeros(1, dtype=FILTER_DTYPE)
    n[0]["op"], n[0]["column"], n[0]["i_min"], n[0]["i_max"] = F_I64_RANGE, cols["grp"], 1, 5
    return n


class Env:
    def __init__(self, segs, filtered: bool):
        from oracle import slo
        self.segs = segs
        self.oras = [slo.OracleIndex(s) for s in segs]
        self.gi = GpuIndex(0, options=OPTIONS)
        cols = {}
        for s in segs:
            cols.update(self.gi.load_segment(s))
        self.fid = self.gi.compile_filter(_grp_filter(cols)) if filtered else None
        for s in segs:
            for t in range(N_COLS):
                assert self.gi.term_has_column(s.segment_ord, t)
            assert self.gi.term_has_column(s.segment_ord, TIE)

    def batch(self, term_lists, weights=None) -> QueryBatch:
        qb = QueryBatch.from_term_lists(term_lists, weights)
        if self.fid is not None:
            qb.filter_id = np.full(qb.n_queries, self.fid, dtype=np.int32)
        return qb

    def oracle(self, qb: QueryBatch, k: int):
        from oracle import slo
        per = []
        for s, o in zip(self.segs, self.oras):
            kw = {"filter_nodes": _grp_filter(o.columns)} if self.fid is not None else {}
            per.append(o.search_batch(canonical_batch(self.gi, qb, s.segment_ord), k, "bm25", **kw))
        if len(per) == 1:
            return per[0]
        hits = np.zeros((qb.n_queries, k), dtype=HIT_DTYPE)
        counts = np.zeros(qb.n_queries, dtype=np.uint32)
        for qi in range(qb.n_queries):
            m = slo.merge_hits([h[qi, : c[qi]] for h, c in per], k)
            hits[qi, : len(m)] = m
            counts[qi] = len(m)
        return hits, counts

    def check(self, qb: QueryBatch, k: int, two_step: bool = False):
        ref = self.gi.search_batch(qb, k, "bm25")
        if two_step:
            pb = self.gi.prepare(qb, k, "bmw")
            assert pb.run_seeds()
            pb.run_sweep()
            got = pb.fetch()
            pb.free()
        else:
            got = self.gi.search_batch(qb, k, "bmw")
        ctr = self.gi.counters()
        assert got[0].tobytes() == ref[0].tobytes() and got[1].tobytes() == ref[1].tobytes()
        assert_parity(*self.oracle(qb, k), *got, strict=True)
        assert int(got[1].sum()) > 0
        return ctr

    def close(self):
        self.gi.close()


def _queries(seed: int, kind: str, n: int = 48):
    rng = np.random.default_rng(seed)
    cols = np.arange(N_COLS)
    sparse = np.arange(N_COLS, N_COLS + N_MID + N_RARE)
    qs, ws = [], []
    for i in range(n):
        if kind == "all_columns":
            t = rng.choice(cols, size=2 + i % 3, replace=False).tolist()
        elif kind == "one_column":  # one column among sparse terms: the column is usually essential
            t = rng.choice(sparse, size=1 + i % 3, replace=False).tolist() + [int(rng.choice(cols))]
        elif kind == "tie":
            t = [TIE] if i % 2 == 0 else [TIE, int(rng.choice(cols))]
        else:
            raise ValueError(kind)
        qs.append(t)
        w = [1.0] * len(t)
        if kind == "all_columns" and i % 4 == 3:  # a bound dominated by one boosted column
            w[i % len(t)] = float(rng.choice([50.0, 1e4, 2.0 ** 20]))
        ws.append(w)
    return qs, ws


@pytest.fixture(scope="module", params=["plain", "deleted_filtered", "two_segments"])
def env(request):
    if request.param == "plain":
        segs, filtered = [_segment(512 * 230 + 77, 0, 1, False)], False
    elif request.param == "deleted_filtered":
        segs, filtered = [_segment(512 * 230 + 77, 0, 2, True)], True
    else:
        segs, filtered = [_segment(512 * 230 + 77, 0, 3, True), _segment(512 * 211 + 300, 1, 4, False)], False
    for s in segs:
        assert s.doc_count % 512
    e = Env(segs, filtered)
    yield e
    e.close()


@pytest.mark.parametrize("k", [11, 101])
@pytest.mark.parametrize("kind", ["all_columns", "one_column", "tie"])
def test_ordered_column_pass_matches_bm25_and_oracle(env, kind, k):
    qs, ws = _queries(10 + k, kind)
    before = env.gi.counters()
    ctr = env.check(env.batch(qs, ws), k)
    if kind != "one_column":  # (all-column queries always enter the pass; it reads some blocks and skips others)
        scored = ctr["last_column_blocks_streamed"]
        assert 0 < scored <= ctr["last_subtiles_skipped"]
    assert ctr["kernel_launches"] > before["kernel_launches"]


def test_tie_at_the_kth_key_across_two_blocks():
    """18 docs with the same score in two blocks of the same bin: the top 11 are the lowest doc ids of them"""
    e = Env([_segment(512 * 230 + 77, 0, 5, False)], False)
    try:
        qb = e.batch([[TIE]] * 4)
        h, c = e.gi.search_batch(qb, 11, "bmw")
        e.check(qb, 11)
        docs = h[0]["doc_id"][: c[0]].tolist()
        tied = sorted(b * 512 + 17 * j + 3 for b in TIE_BLOCKS for j in range(9))
        assert docs == tied[:11]
        assert len(set(h[0]["score"][: c[0]].tolist())) == 1
    finally:
        e.close()


def test_two_step_run():
    e = Env([_segment(512 * 230 + 77, 0, 6, True)], False)
    try:
        for kind in ("all_columns", "one_column"):
            qs, ws = _queries(40, kind)
            for k in (11, 101):
                e.check(e.batch(qs, ws), k, two_step=True)
    finally:
        e.close()
