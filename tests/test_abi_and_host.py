"""CPU tests: the C-ABI library loads and exports every symbol include/searchlite_gpu.h declares, fails
loudly without a device (no CPU fallback), and the host-side mirrors (struct layouts, query
builders, shard ranges, synthetic generators) behave."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from searchlite_b200 import build as slg_build
from searchlite_b200 import engine, shard, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    return engine.load_library()


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "searchlite_gpu.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(slg_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib):
    declared = _declared_symbols()
    assert len(declared) >= 25
    for sym in declared:
        assert hasattr(lib, sym), f"{sym} is declared in include/searchlite_gpu.h but not exported"
    assert sorted(engine.EXPORTED_SYMBOLS) == declared
    assert b"sm_100a" in lib.slg_version()


def test_rust_sys_crate_is_in_sync_with_the_header():
    """rust/searchlite-gpu-sys/src/lib.rs is generated from the header (tools/gen_rust_sys.py): it must be current and
    declare every exported entry point plus a #[repr(C)] mirror of every struct whose size ctypes can cross-check"""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gen_rust_sys
    text = open(gen_rust_sys.OUT).read()
    assert text == gen_rust_sys.generate(), "run python tools/gen_rust_sys.py"
    fns = sorted(re.findall(r"pub fn (slg_[a-z0-9_]+)\(", text))
    assert fns == _declared_symbols()
    for name in ("slg_term_t", "slg_hit_t", "slg_query_t", "slg_plan_node_t", "slg_stats_t", "slg_segment_view_t", "slg_filter_node_t",
                 "slg_counters_t", "slg_vector_clause_t", "slg_segment_files_t", "slg_segment_info_t"):
        assert f"pub struct {name} {{" in text, name
    # field counts agree with the ctypes / numpy mirrors the tests drive the library through
    def n_fields(struct):
        body = text[text.index(f"pub struct {struct} {{"):]
        return len(re.findall(r"^    pub \w+:", body[: body.index("\n}")], flags=re.M))
    assert n_fields("slg_counters_t") == len(engine.Counters._fields_)
    assert n_fields("slg_vector_clause_t") == len(engine.VectorClause._fields_)
    assert n_fields("slg_hit_t") == len(engine.HIT_DTYPE.names)
    assert n_fields("slg_filter_node_t") == len(engine.FILTER_DTYPE.names)


def test_library_is_built_for_sm_100a_only():
    import subprocess
    cuobjdump = os.path.join(os.path.dirname(slg_build._nvcc()), "cuobjdump")  # the toolkit that built the library, on PATH or not
    out = subprocess.run([cuobjdump, "--list-elf", slg_build.LIB_PATH], capture_output=True, text=True, check=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device error path")
def test_open_fails_loudly_without_a_device(lib):
    h = C.c_void_p()
    rc = lib.slg_open(0, C.byref(h))
    assert rc == -3 and not h.value  # SLG_ERR_NO_DEVICE: there is no CPU fallback
    assert b"no CPU fallback" in lib.slg_last_error(None)
    with pytest.raises(engine.SearchliteGpuError):
        engine.GpuIndex(0)


def test_null_arguments_are_errors_not_crashes(lib):
    assert lib.slg_open(0, None) == -1
    assert lib.slg_close(None) == 0
    assert lib.slg_batch_free(None) == 0
    assert lib.slg_batch_run(None, 1) == -1
    assert lib.slg_configure(None, 0, 0, 0, 0) == -1
    assert lib.slg_get_counters(None, None) == -1


def test_struct_layouts_match_the_header():
    # sizes the C compiler gives the header's structs (x86-64 SysV)
    assert engine.TERM_DTYPE.itemsize == 20
    assert engine.QUERY_DTYPE.itemsize == 72
    assert engine.PLAN_DTYPE.itemsize == 12
    assert engine.HIT_DTYPE.itemsize == 12
    assert engine.STATS_DTYPE.itemsize == 40
    assert engine.FILTER_DTYPE.itemsize == 56
    assert C.sizeof(engine.SegmentView) == 80
    assert C.sizeof(engine.Counters) == 144
    assert C.sizeof(engine.VectorClause) == 24
    src = r'''
    #include "include/searchlite_gpu.h"
    #include <stdio.h>
    int main(void){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(slg_term_t), sizeof(slg_query_t), sizeof(slg_hit_t),
      sizeof(slg_stats_t), sizeof(slg_filter_node_t), sizeof(slg_segment_view_t), sizeof(slg_counters_t),
      sizeof(slg_segment_files_t), sizeof(slg_segment_info_t), sizeof(slg_plan_node_t), sizeof(slg_vector_clause_t));return 0;}
    '''
    import subprocess
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(td, "s")
        subprocess.run(["gcc", "-std=c99", "-I", ROOT, "-o", exe, c], check=True, cwd=ROOT)  # the header is plain C
        sizes = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [20, 72, 12, 40, 56, 80, 144, C.sizeof(engine.SegmentFiles), C.sizeof(engine.SegmentInfo), 12, 24]


def test_query_batch_builders():
    qb = engine.QueryBatch.from_term_lists([[3, 5], [], [7]], [[1.0, 2.0], [], [0.5]])
    s = qb.structs()
    assert s["n_terms"].tolist() == [2, 0, 1] and s["min_should"].tolist() == [1, 1, 1] and s["filter_id"].tolist() == [-1] * 3
    assert qb.terms["leaf"].tolist() == [0, 1, 0] and qb.terms["weight"].tolist() == [1.0, 2.0, 0.5]
    bq = engine.QueryBatch.from_bool([{"must": [1], "should": [2, 3], "must_not": [4]}, {"should": [9]}, {"should": [9], "filter_id": 0}])
    assert bq.group_role.tolist() == [1, 0, 0, 2, 0, 0]
    assert bq.terms["flags"].tolist() == [1, 1, 1, 0, 1, 1]           # must_not terms are not scored
    assert bq.min_should.tolist() == [0, 1, 0]                        # api/reader.rs:1553-1561 defaults
    sub = bq.subset(1, 3)
    assert sub.n_queries == 2 and sub.terms["term_id"].tolist() == [9, 9] and sub.filter_id.tolist() == [-1, 0]
    # ScorePlans: postfix rows of the ScoreExpr tree (query/planner.rs:113-122)
    expr = ("sum", [("dismax", [("leaf", 0), ("leaf", 1)], 0.25), ("leaf", 2)])
    assert engine.plan_postfix(expr) == [(0, 0, 0.0), (0, 1, 0.0), (2, 2, 0.25), (0, 2, 0.0), (1, 2, 0.0)]
    pq = engine.QueryBatch.from_term_lists([[3, 5, 6], [7]]).set_plans([expr, None])
    ps = pq.structs()
    assert ps["n_plan_nodes"].tolist() == [5, 0] and ps["leaf_count"].tolist() == [3, 0] and ps["plan"][1] == 0
    assert pq.subset(0, 1).structs()["n_plan_nodes"].tolist() == [5]


def test_shard_ranges_cover_the_corpus():
    for n, w in ((10, 1), (10, 3), (8_841_823, 8), (5, 8)):
        r = shard.shard_ranges(n, w)
        assert r[0][0] == 0 and r[-1][1] == n and all(a[1] == b[0] for a, b in zip(r, r[1:]))
        sizes = [hi - lo for lo, hi in r]
        assert max(sizes) - min(sizes) <= 1


def test_synthetic_corpus_is_a_valid_inverted_index_and_deterministic():
    spec = synth.CorpusSpec(n_docs=3000, vocab=500, seed=5, len_lo=10, len_hi=40)
    a = synth.generate_segment(spec, "cpu", chunk_docs=1024)
    b = synth.generate_segment(spec, "cpu", chunk_docs=4096)
    for x, y in ((a.term_offsets, b.term_offsets), (a.post_docs, b.post_docs), (a.post_tfs, b.post_tfs), (a.field_lengths, b.field_lengths)):
        assert np.array_equal(x, y)
    off = a.term_offsets.astype(np.int64)
    assert off[0] == 0 and off[-1] == len(a.post_docs) and np.all(np.diff(off) >= 0)
    for t in range(0, 500, 7):
        d = a.post_docs[off[t]:off[t + 1]]
        assert np.all(np.diff(d.astype(np.int64)) > 0)
    # sum of tf over a doc's postings == its `_len:` value; total_tokens == sum of lengths
    per_doc = np.bincount(a.post_docs, weights=a.post_tfs, minlength=spec.n_docs)
    assert np.array_equal(per_doc.astype(np.int64), a.field_lengths)
    assert a.total_tokens == int(a.field_lengths.sum())
    # shards of one logical corpus: doc_base shifts the generator, not the content
    lo = synth.generate_segment(synth.CorpusSpec(n_docs=1000, vocab=500, seed=5, len_lo=10, len_hi=40), "cpu")
    hi = synth.generate_segment(synth.CorpusSpec(n_docs=2000, vocab=500, seed=5, len_lo=10, len_hi=40, doc_base=1000, segment_ord=1), "cpu")
    assert np.array_equal(np.concatenate([lo.field_lengths, hi.field_lengths]), a.field_lengths)
    t = 3
    la, lb = lo.post_docs[int(lo.term_offsets[t]):int(lo.term_offsets[t + 1])], hi.post_docs[int(hi.term_offsets[t]):int(hi.term_offsets[t + 1])]
    assert np.array_equal(np.concatenate([la, lb + 1000]), a.post_docs[off[t]:off[t + 1]])


def test_synthetic_queries_shape():
    qb = synth.generate_queries(500, 10_000, seed=9)
    n = (qb.term_off[1:] - qb.term_off[:-1])
    assert n.min() >= 2 and n.max() <= 5
    for q in range(500):
        t = qb.terms["term_id"][qb.term_off[q]:qb.term_off[q + 1]]
        assert len(set(t.tolist())) == len(t) and t.min() >= 9  # distinct, rank >= 10 (term id = rank - 1)
    again = synth.generate_queries(500, 10_000, seed=9)
    assert np.array_equal(again.terms, qb.terms)
