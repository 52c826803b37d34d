"""The posting scan's bound arithmetic (slg_scan_kernel.cuh) where it is fragile: heavily boosted terms, exact score ties at
the k-th key, short results and the residency thresholds.

A scanned doc is verified term by term and dropped once  known contributions + bounds of the terms not yet looked up  falls
below the k-th score.  bm25 runs the same test with bounds taken from the batch's own scores, so an unsafe bound moves bm25,
wand and bmw alike: only a scorer that shares none of the engine's float32 arithmetic catches it.  Every case is therefore
checked five ways: bit for bit against the oracle on the declared summation order, within the 1e-5 rule on the query order,
byte-identical across bm25 / wand / bmw, against the float64 BM25 below (no returned score off by more than 1e-5, no doc
above the k-th score missing, the right count), and, where the batch fits it, on the explicit warp kernel (query order)."""
from __future__ import annotations

import itertools
import math

import numpy as np
import pytest

from searchlite_b200 import GpuIndex, QueryBatch, SearchliteGpuError
from searchlite_b200.engine import FILTER_DTYPE, F_I64_RANGE, HIT_DTYPE
from tests.helpers import canonical_batch, segment_from_postings
from tests.parity import RTOL, assert_parity

pytestmark = pytest.mark.gpu

MODES = ("bm25", "wand", "bmw")
K1, B = float(np.float32(0.9)), float(np.float32(0.4))  # load_segment's defaults, as the engine receives them


# ---- float64 reference -------------------------------------------------------------------------------------------------
def f64_scores(seg, terms, weights, must: bool):
    """BM25 of every doc of `seg` in float64 (query/bm25.rs, query/wand.rs:77-84 and :269-286 restated without float32):
    -> (score per doc, matching mask).  A term the segment lacks has no postings; `must`: every term must hold the doc."""
    n = seg.doc_count
    n_del = 0 if seg.deleted_docs is None else len(np.unique(seg.deleted_docs))
    docs_live = float(n - n_del)
    avgdl = seg.total_tokens / n if n else 0.0
    lens = np.asarray(seg.field_lengths, dtype=np.float64)
    lens = np.where(lens > 0, lens, max(avgdl, 1.0))
    score = np.zeros(n)
    held = np.zeros(n, dtype=np.int64)
    for t, w in zip(terms, weights):
        if t >= seg.n_terms:
            continue
        a, b = int(seg.term_offsets[t]), int(seg.term_offsets[t + 1])
        d = np.asarray(seg.post_docs[a:b], dtype=np.int64)
        if len(d) == 0:
            continue
        tf = np.asarray(seg.post_tfs[a:b], dtype=np.float64)
        df = float(len(d))
        ratio = (docs_live - df + 0.5) / (df + 0.5)
        idf = (max(math.log(ratio), 0.0) if ratio > 0 else 0.0) + 1.0  # f32::max(NaN, 0) = 0
        norm = lens[d] / avgdl if avgdl > 0 else 1.0
        denom = np.maximum(tf + K1 * (1.0 - B + B * norm), 1e-6)
        score[d] += idf * tf * (K1 + 1.0) / denom * float(np.float32(w))
        held[d] += 1
    match = held == len(terms) if must else held > 0
    if seg.deleted_docs is not None and len(seg.deleted_docs):
        match[np.asarray(seg.deleted_docs, dtype=np.int64)] = False
    return score, match


def assert_f64(env, qb: QueryBatch, k: int, hits, counts):
    must = qb.group_off is not None  # (the Bool batches of this file are all-MUST)
    for qi in range(qb.n_queries):
        rows = qb.terms[int(qb.term_off[qi]):int(qb.term_off[qi + 1])]
        ref = []
        for s, acc in zip(env.segs, env.accept):
            sc, m = f64_scores(s, rows["term_id"].tolist(), rows["weight"].tolist(), must)
            ref.append((s.segment_ord, sc, m if acc is None else m & acc))
        n_match = sum(int(m.sum()) for _, _, m in ref)
        got = hits[qi, : counts[qi]]
        assert int(counts[qi]) == min(k, n_match), f"query {qi}: {int(counts[qi])} hits, {n_match} docs match (k {k})"
        by_ord = {o: (sc, m) for o, sc, m in ref}
        for h in got:
            sc, m = by_ord[int(h["segment_ord"])]
            d = int(h["doc_id"])
            assert m[d], f"query {qi}: doc {d} returned but does not match"
            assert abs(float(h["score"]) - sc[d]) <= RTOL * sc[d], f"query {qi}: doc {d} scored {float(h['score'])}, f64 {sc[d]}"
        floor = float(got["score"][-1]) * (1.0 + RTOL) if len(got) == k else -np.inf
        have = {(int(h["segment_ord"]), int(h["doc_id"])) for h in got}
        for o, sc, m in ref:
            for d in np.nonzero(m & (sc > floor))[0].tolist():
                assert (o, d) in have, (f"query {qi} ({rows['term_id'].tolist()}, weights {rows['weight'].tolist()}): doc {d} "
                                        f"of segment {o} lost; f64 score {sc[d]!r} exceeds the k-th score {float(got['score'][-1])!r} "
                                        f"by {sc[d] - float(got['score'][-1]):.6g}")


# ---- the engine against all of it --------------------------------------------------------------------------------------
class Env:
    """segments loaded into an automatic-kernel index (and a warp-kernel one), with their oracles and an optional root filter"""

    def __init__(self, segs, options, filt=None, warp=True):
        from oracle import slo
        self.segs = segs
        self.oras = [slo.OracleIndex(s) for s in segs]
        self.filt = filt  # (column name -> handle) -> filter nodes
        self.gis = {}
        for kernel in ("auto", "warp") if warp else ("auto",):
            gi = GpuIndex(0, kernel=kernel, options=options)
            cols = {}
            for s in segs:
                cols.update(gi.load_segment(s))
            fid = gi.compile_filter(filt(cols)) if filt else None
            self.gis[kernel] = (gi, fid)
        self.accept = [None] * len(segs)
        if filt:
            self.accept = [np.unpackbits(o.filter_bitmap(filt(o.columns)).view(np.uint8), bitorder="little")[: s.doc_count].astype(bool)
                           for o, s in zip(self.oras, segs)]

    @property
    def gi(self):
        return self.gis["auto"][0]

    def close(self):
        for gi, _ in self.gis.values():
            gi.close()

    def batch(self, qb: QueryBatch, kernel: str) -> QueryBatch:
        fid = self.gis[kernel][1]
        if fid is not None:
            qb.filter_id = np.full(qb.n_queries, fid, dtype=np.int32)
            qb._structs = None
        return qb

    def oracle(self, qb: QueryBatch, k: int, canonical: bool):
        from oracle import slo
        kw = {}
        per = []
        for s, o in zip(self.segs, self.oras):
            if self.filt:
                kw = {"filter_nodes": self.filt(o.columns)}
            per.append(o.search_batch(canonical_batch(self.gi, qb, s.segment_ord) if canonical else qb, k, "bm25", **kw))
        if len(per) == 1:
            return per[0]
        hits = np.zeros((qb.n_queries, k), dtype=HIT_DTYPE)
        counts = np.zeros(qb.n_queries, dtype=np.uint32)
        for qi in range(qb.n_queries):
            m = slo.merge_hits([h[qi, : c[qi]] for h, c in per], k)
            hits[qi, : len(m)] = m
            counts[qi] = len(m)
        return hits, counts

    def check(self, qb: QueryBatch, k: int):
        """the five checks (the float64 reference first: it names a lost doc); returns the automatic kernel's (hits, counts)"""
        qb = self.batch(qb, "auto")
        got = {m: self.gi.search_batch(qb, k, m) for m in MODES}
        h, c = got["bm25"]
        for m in MODES:
            assert_f64(self, qb, k, *got[m])
        for m in MODES:
            assert got[m][0].tobytes() == h.tobytes() and got[m][1].tobytes() == c.tobytes(), m
        assert_parity(*self.oracle(qb, k, True), h, c, strict=True)
        assert_parity(*self.oracle(qb, k, False), h, c, strict=False)
        n_terms = int(np.max(qb.term_off[1:] - qb.term_off[:-1]))
        if "warp" in self.gis and qb.group_off is None and k <= 32 and n_terms <= 8:
            wq = self.batch(qb, "warp")
            wh, wc = self.gis["warp"][0].search_batch(wq, k, "bm25")
            assert_parity(*self.oracle(wq, k, False), wh, wc, strict=True)
            assert_f64(self, wq, k, wh, wc)
            self.batch(qb, "auto")
        return h, c


def weighted(term_lists, weights) -> QueryBatch:
    return QueryBatch.from_term_lists(term_lists, weights)


def all_must(term_lists, weights) -> QueryBatch:
    qb = QueryBatch.from_bool([{"must": t} for t in term_lists])
    qb.terms["weight"] = [w for ws in weights for w in ws]
    return qb


def i64_range(name, lo, hi):
    def nodes(cols):
        n = np.zeros(1, dtype=FILTER_DTYPE)
        n[0]["op"], n[0]["column"], n[0]["i_min"], n[0]["i_max"] = F_I64_RANGE, cols[name], lo, hi
        return n
    return nodes


# ---- A. boost cancellation ---------------------------------------------------------------------------------------------
# C (term 0) is held by every 8th doc and is a column; S_j (terms 1..4) by the docs 16 m + 2j + 1, L_j (terms 5..8) by the
# same docs and by every 32nd doc from e_j.  A doc of S_j has length 6000 - m // 40: the later the doc, the higher it scores,
# in steps of about 2e-4, and the S_j list is one scan item, met in doc order.  Every other doc is longer, so L_j's bound is
# reached by S_j's last docs.  Without C, a doc's score is S_j + L_j; once C's bound A (boosted) is taken off the sum of the
# bounds, what is left of L_j's is off by up to ulp(A) / 2: at 1e5 or more, far beyond the 1e-4 relative slack.
A_DOCS = 20_000
BOOSTS = (1.0, 1e4, 1e5, float(2 ** 20), 1e30)
A_OPTIONS = {"dense_den": 8, "dense_min_df": 64}


def _boost_segment(deleted_c: str) -> object:
    rng = np.random.default_rng(3)
    d = np.arange(A_DOCS)
    lens = rng.integers(6000, 7000, size=A_DOCS)
    odd = d % 16 % 2 == 1
    lens[odd] = 6000 - (d[odd] // 16) // 40
    lists = [(d[d % 8 == 0].tolist(), rng.integers(1, 4, size=A_DOCS // 8).tolist())]
    s_lists = [d[d % 16 == 2 * j + 1] for j in range(4)]
    for s in s_lists:
        lists.append((s.tolist(), [1] * len(s)))
    for j, e in enumerate((2, 4, 6, 10)):
        l = np.union1d(s_lists[j], d[d % 32 == e])
        lists.append((l.tolist(), [1] * len(l)))
    c_docs = d[d % 8 == 0]
    deleted = {"all": c_docs, "most": c_docs[5:], "none": None}[deleted_c]
    seg = segment_from_postings(lists, lens, deleted=deleted)
    seg.fast_i64 = {"grp": ((d % 8).astype(np.int64), None)}
    return seg


@pytest.fixture(scope="module", params=["deleted", "filtered", "few_live"])
def boost_env(request):
    """T forced small: (i) every holder of C deleted, (ii) a root filter admitting only non-holders, (iii) 5 live holders"""
    if request.param == "deleted":
        env = Env([_boost_segment("all")], A_OPTIONS)
    elif request.param == "filtered":
        env = Env([_boost_segment("none")], A_OPTIONS, filt=i64_range("grp", 1, 7))
    else:
        env = Env([_boost_segment("most")], A_OPTIONS)
    assert env.gi.term_has_column(0, 0)
    assert not any(env.gi.term_has_column(0, t) for t in range(1, 9))
    yield env
    env.close()


def _boost_queries():
    tl, ws = [], []
    for j in range(4):
        for boost in BOOSTS:
            for sw, lw in ((1.0, 1.0), (1.5, 0.75)):
                w = {0: boost, 1 + j: sw, 5 + j: lw}
                for order in itertools.permutations((1 + j, 5 + j, 0)):
                    tl.append(list(order))
                    ws.append([w[t] for t in order])
    return tl, ws


@pytest.mark.parametrize("k", [11, 101])
def test_boosted_column_term_keeps_the_small_bounds(boost_env, k):
    tl, ws = _boost_queries()
    boost_env.check(weighted(tl, ws), k)
    assert boost_env.gi.counters()["last_postings_scattered"] > 0  # the flat posting scan ran


def test_boosted_and_driver(boost_env):
    tl, ws = [], []
    for j in range(4):
        for boost in BOOSTS:
            tl += [[1 + j, 5 + j], [5 + j, 1 + j]]
            ws += [[boost, 1.0], [1.0, boost]]  # the driver (S_j, the shorter list) boosted; then L_j
    boost_env.check(all_must(tl, ws), 11)


# ---- E (and B). residency edges ----------------------------------------------------------------------------------------
# 18981 = 512 * 37 + 37 = 3^3 * 19 * 37 docs: not a multiple of 32, 224 or 512, and dense_den 9 / bitmap_den 57 put the
# column and bitmap thresholds at whole dfs (2109 and 333)
E_DOCS = 18_981
E_OPTIONS = {"dense_den": 9, "dense_min_df": 64, "bitmap_den": 57}
E_OPTIONS_MIN_DF = {"dense_den": 9, "dense_min_df": 2500, "bitmap_den": 57}
E_EDGE_DFS = (2109, 2108, 333, 332, 2500, 2499)  # terms 0..5: column threshold, one below; bitmap threshold, one below; dense_min_df
E_EDGE_TERM, E_TWINS = 6, (7, 8)


def _edge_segment():
    rng = np.random.default_rng(21)
    last = E_DOCS - 1
    lists = []

    def some(df):
        pick = np.sort(rng.choice(np.arange(1, last), size=df - 2, replace=False))
        return [0] + pick.tolist() + [last]  # every list holds the first and the last doc

    for df in E_EDGE_DFS:
        lists.append(some(df))
    lists.append([0, 1, 31, 32, 223, 224, 511, 512, last - 1, last])  # E_EDGE_TERM
    twin = some(900)
    lists += [twin, twin]
    for df in rng.integers(20, 7000, size=24):
        lists.append(some(int(df)))
    postings = [(l, rng.integers(1, 6, size=len(l)).tolist()) for l in lists]
    postings[7] = (twin, postings[8][1])  # the twins: same docs and tfs, so bit-identical bounds
    postings[E_EDGE_TERM] = (lists[E_EDGE_TERM], [9] * len(lists[E_EDGE_TERM]))
    lens = rng.integers(20, 120, size=E_DOCS)
    lens[[0, last]] = 20
    deleted = rng.choice(np.arange(2, last - 1), size=300, replace=False)
    return segment_from_postings(postings, lens, deleted=np.sort(deleted)), len(lists)


@pytest.fixture(scope="module")
def edge_envs():
    seg, n_terms = _edge_segment()
    envs = {"min_df_64": Env([seg], E_OPTIONS), "min_df_2500": Env([seg], E_OPTIONS_MIN_DF)}
    yield envs, seg, n_terms
    for e in envs.values():
        e.close()


def test_residency_classes(edge_envs):
    envs, seg, n_terms = edge_envs
    dfs = np.diff(np.asarray(seg.term_offsets, dtype=np.int64))
    assert seg.doc_count % 32 and seg.doc_count % 224 and seg.doc_count % 512 == 37
    for name, opts in (("min_df_64", E_OPTIONS), ("min_df_2500", E_OPTIONS_MIN_DF)):
        gi = envs[name].gi
        col = [bool(df >= opts["dense_min_df"] and df * opts["dense_den"] >= seg.doc_count) for df in dfs]
        assert [gi.term_has_column(0, t) for t in range(n_terms)] == col
        bits = sum(1 for t in range(n_terms) if not col[t] and dfs[t] >= 64 and dfs[t] * opts["bitmap_den"] >= seg.doc_count)
        assert gi.segment_residency(0)["n_presence_bitmaps"] == bits
    # the thresholds land where intended: column at 2109 and not at 2108; at dense_min_df 2500, 2500 and not 2499
    assert envs["min_df_64"].gi.term_has_column(0, 0) and not envs["min_df_64"].gi.term_has_column(0, 1)
    assert envs["min_df_2500"].gi.term_has_column(0, 4) and not envs["min_df_2500"].gi.term_has_column(0, 5)
    assert not envs["min_df_2500"].gi.term_has_column(0, 0)


def _edge_queries(n_terms, seed):
    rng = np.random.default_rng(seed)
    tl = []
    for i in range(120):
        t = rng.choice(np.arange(n_terms), size=2 + i % 5, replace=False).tolist()
        t[0] = int(rng.integers(0, E_EDGE_TERM + 1))  # one edge-case term in every query
        if t[0] in t[1:]:
            t = t[1:]
        tl.append(t)
    tl += [[E_EDGE_TERM], [E_EDGE_TERM, 2, 3], [0, 1, 2, 3, 4, 5]]
    return tl


@pytest.mark.parametrize("name", ["min_df_64", "min_df_2500"])
@pytest.mark.parametrize("k", [11, 32, 101])
def test_residency_edges(edge_envs, name, k):
    envs, seg, n_terms = edge_envs
    tl = _edge_queries(n_terms, 30 + k)
    h, c = envs[name].check(QueryBatch.from_term_lists(tl), k)
    edge = h[len(tl) - 3, : c[len(tl) - 3]]["doc_id"].tolist()
    assert 0 in edge and E_DOCS - 1 in edge  # hits at the first and the last doc


def test_residency_edges_and(edge_envs):
    envs, seg, n_terms = edge_envs
    rng = np.random.default_rng(41)
    tl = [rng.choice(np.arange(n_terms), size=2 + i % 2, replace=False).tolist() for i in range(80)]
    tl += [[0, 1], [2, 3], [4, 5], [E_EDGE_TERM, 0], [E_EDGE_TERM, 3]]
    envs["min_df_64"].check(all_must(tl, [[1.0] * len(t) for t in tl]), 11)


# B. priority edges: weights from 1e-3 to 1e5 against the df order, bit-identical bounds, a boosted sparse term, 8 terms
@pytest.mark.parametrize("k", [11, 32, 101])
def test_priority_edges(edge_envs, k):
    envs, seg, n_terms = edge_envs
    dfs = np.diff(np.asarray(seg.term_offsets, dtype=np.int64))
    rng = np.random.default_rng(50 + k)
    tl, ws = [], []
    for i in range(60):
        t = rng.choice(np.arange(n_terms), size=6, replace=False)
        t = t[np.argsort(dfs[t], kind="stable")].tolist()  # rarest first: the rarest gets 1e-3, the densest 1e5
        tl.append(t)
        ws.append([1e-3, 1e-2, 1.0, 10.0, 1e3, 1e5])
    for i in range(30):
        others = rng.choice(np.arange(9, n_terms), size=2 + i % 4, replace=False).tolist()
        tl.append([E_TWINS[0]] + others + [E_TWINS[1]])  # twins: ties to the lower slot
        ws.append([1.0] * (len(others) + 2))
        boosted = int(rng.choice([t for t in range(n_terms) if 64 <= dfs[t] and not envs["min_df_64"].gi.term_has_column(0, t)]))
        row = [boosted] + [t for t in rng.choice(np.arange(n_terms), size=3 + i % 5, replace=False).tolist() if t != boosted]
        tl.append(row)
        ws.append([1e4] + [1.0] * (len(row) - 1))  # a boosted sparse term: the highest priority
    for i in range(20):
        tl.append(rng.choice(np.arange(n_terms), size=8, replace=False).tolist())
        ws.append(rng.choice([1e-3, 0.5, 1.0, 2.0, 1e3], size=8).tolist())
    for name in envs:
        envs[name].check(weighted(tl, ws), k)


# ---- C / D. ties at the k-th key, short results ------------------------------------------------------------------------
# term 0: 4500 sparse postings of one (tf, length): one score.  Term 1: a column held by 6000 docs of that length, tf 1: tied
# docs only column terms hold.  Term 2: 40 rare docs.  Term 3: a column with varied scores.  Term 4: no postings here.
T_DOCS = 40_000
T_OPTIONS = {"dense_den": 8, "dense_min_df": 64}


def _tie_segment(ord_=0):
    rng = np.random.default_rng(61)
    d = np.arange(T_DOCS)
    tie = d[d % 8 == 1][:4500]
    tie_col = d[(d % 8 == 2) | (d % 8 == 4)][:6000]
    rare = np.sort(rng.choice(d[d % 8 == 6], size=40, replace=False))
    col = d[d % 8 % 2 == 1]
    lens = rng.integers(50, 150, size=T_DOCS)
    lens[tie] = 100
    lens[tie_col] = 100
    postings = [(tie.tolist(), [2] * len(tie)), (tie_col.tolist(), [1] * len(tie_col)),
                (rare.tolist(), rng.integers(1, 4, size=40).tolist()), (col.tolist(), rng.integers(1, 5, size=len(col)).tolist()),
                ([], [])]
    seg = segment_from_postings(postings, lens, segment_ord=ord_, deleted=d[d % 97 == 5])
    seg.fast_i64 = {"grp": ((d % 10).astype(np.int64), None)}
    return seg


def _small_segment():
    """segment 1 of the two-segment index: terms 0, 1 and 3 held by a few docs, terms 2 and 4 by none"""
    rng = np.random.default_rng(62)
    n = 3000
    postings = [(list(range(0, n, 7)), [2] * len(range(0, n, 7))), (list(range(1, n, 5)), [1] * len(range(1, n, 5))), ([], []),
                (list(range(3, n, 3)), rng.integers(1, 5, size=len(range(3, n, 3))).tolist()), ([], [])]
    return segment_from_postings(postings, rng.integers(50, 150, size=n), segment_ord=1)


@pytest.fixture(scope="module")
def tie_env():
    env = Env([_tie_segment()], T_OPTIONS)
    assert not env.gi.term_has_column(0, 0) and env.gi.term_has_column(0, 1) and env.gi.term_has_column(0, 3)
    yield env
    env.close()


TIE_QUERIES = [[0], [1], [0, 2], [1, 2], [2, 0], [0, 1], [1, 0, 2], [3, 1], [2, 3], [0, 3, 1, 2]]


@pytest.mark.parametrize("k", [1, 11, 32, 33, 64, 65, 1001])
def test_ties_at_the_kth_key(tie_env, k):
    h, c = tie_env.check(QueryBatch.from_term_lists(TIE_QUERIES), k)
    # [0] and [1]: thousands of equal scores; the smallest live doc ids win
    for qi, term in ((0, 0), (1, 1)):
        seg = tie_env.segs[0]
        docs = np.asarray(seg.post_docs[int(seg.term_offsets[term]):int(seg.term_offsets[term + 1])])
        live = docs[~np.isin(docs, seg.deleted_docs)]
        assert h[qi, : c[qi]]["doc_id"].tolist() == live[:k].tolist()
        assert len(set(h[qi, : c[qi]]["score"].view(np.uint32).tolist())) == 1


@pytest.mark.parametrize("k", [11, 101])
def test_short_results(tie_env, k):
    # k above the matching docs (term 2: 40 docs); every term a column; terms without postings
    tie_env.check(QueryBatch.from_term_lists([[2], [2, 4], [4], [1, 3], [3, 1], [4, 1]]), k)
    tie_env.check(all_must([[0, 4], [2, 4], [0, 3], [3, 0], [1, 3]], [[1.0, 1.0]] * 5), k)


@pytest.mark.parametrize("lo,hi", [(6, 6), (20, 30)])
def test_short_results_filtered(lo, hi):
    """a filter that leaves fewer than k docs, and one that admits nothing"""
    env = Env([_tie_segment()], T_OPTIONS, filt=i64_range("grp", lo, hi))
    try:
        for k in (11, 101):
            h, c = env.check(QueryBatch.from_term_lists([[2], [0], [1], [0, 2], [3, 1, 2]]), k)
            if lo == 20:
                assert not c.any()
    finally:
        env.close()


def test_two_segments_one_without_a_match():
    env = Env([_tie_segment(0), _small_segment()], T_OPTIONS)
    try:
        for k in (11, 32, 101):
            h, c = env.check(QueryBatch.from_term_lists([[2], [2, 4], [0], [1, 2], [0, 3], [3], [4]]), k)
            assert set(h[0, : c[0]]["segment_ord"].tolist()) == {0}
        env.check(all_must([[0, 2], [0, 3], [1, 3], [2, 4]], [[1.0, 1.0]] * 4), 11)
    finally:
        env.close()


# ---- F. contributions that would round to +0 ---------------------------------------------------------------------------
@pytest.mark.parametrize("w", [1e-45, 1e-39, 2.0 ** -101])
def test_weights_that_can_round_a_contribution_to_zero_are_refused(tie_env, w):
    """the kernels read a contribution of +0 as "the doc lacks the term" and never return a doc scored 0, where the reference
    keeps one: a weight below 2^-100 is refused (SLG_ERR_UNSUPPORTED)"""
    for qb in (weighted([[0, 2], [3]], [[w, 1.0], [w]]), all_must([[0, 1]], [[1.0, w]])):
        with pytest.raises(SearchliteGpuError) as e:
            tie_env.gi.search_batch(qb, 11, "bm25")
        assert e.value.code == -4


def test_smallest_accepted_weight_is_exact(tie_env):
    w = 2.0 ** -100
    tie_env.check(weighted([[0, 2], [3], [2, 3, 1], [2]], [[w, 1.0], [w], [w, w, w], [w]]), 11)
    tie_env.check(all_must([[0, 3], [2, 3]], [[w, w], [1.0, w]]), 11)
