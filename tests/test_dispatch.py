"""Which scoring path a batch takes (searchlite_b200/csrc/slg_dispatch.h).

On the CPU: the header, compiled on its own with g++, against a transcription of the selection logic it replaced,
over every combination of its facts.  On the GPU: each path forced through the options, against the oracle."""
import os
import subprocess
import tempfile

import pytest

from searchlite_b200 import GpuIndex, QueryBatch, SearchliteGpuError, synth
from tests.helpers import assert_engine_parity

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "searchlite_b200", "csrc")

WARP_MAX_K, WARP_MAX_TERMS = 32, 8
ITEMS_MSG = ("the items kernel handles plain OR queries without a ScorePlan, k <= %u, <= %u terms per query, resident scores, "
             "sub_docs <= 4096" % (WARP_MAX_K, WARP_MAX_TERMS))
WARP_MSG = "the warp kernel handles k <= %u and <= %u terms per query" % (WARP_MAX_K, WARP_MAX_TERMS)
AND_MSG = "an AND batch prepared for the posting scan cannot run on the sub-tile kernels (strict_accumulate)"
TWO_STEP_MSG = ("the two-step run (first part, threshold exchange, rest) needs one segment per handle and the posting scan or "
                "the pruned items kernel")

PREPARE_FACTS = ("small_k", "few_terms", "matcher", "all_must", "has_cursor", "has_plan", "all_scores", "sub_docs_ok",
                 "scan_kernels", "stream_kernels", "has_terms")
RUN_FACTS = ("want_stats", "prune", "scan_kernels", "strict_accumulate", "small_plan_docs")
STEPS = ("run", "seeds", "sweep")

# prepare combination p: kernel_choice = p & 3, then one bit per PREPARE_FACTS; run combination r: one bit per RUN_FACTS.
# Per p one line: the selection (or the refusal), then per (r, step, segments 1 / 2) the path (or the refusal).
DRIVER = r'''
#include "slg_dispatch.h"
#include <cstdio>
#include <string>
using namespace slg;

static std::string selection(const char *refusal, const Selection &s) {
  if (refusal) {
    char b[512];
    snprintf(b, sizeof b, refusal, 32u, 8u);
    return b;
  }
  std::string o;
  for (bool v : {s.canonical, s.pools, s.and_scan, s.warp_tables, s.staged, s.colq}) o += v ? '1' : '0';
  return o;
}

int main() {
  static const char *names[] = {"Scan", "Stream", "Items", "Warp", "Tiles"};
  for (unsigned p = 0; p < (4u << 11); p++) {
    BatchFacts f;
    f.kernel_choice = p & 3u;
    bool *fb[] = {&f.small_k, &f.few_terms, &f.matcher, &f.all_must, &f.has_cursor, &f.has_plan, &f.all_scores,
                  &f.sub_docs_ok, &f.scan_kernels, &f.stream_kernels, &f.has_terms};
    for (unsigned i = 0; i < 11; i++) *fb[i] = (p >> (2 + i)) & 1u;
    Selection s;
    const char *refusal = select_kernels(f, s);
    printf("%s", selection(refusal, s).c_str());
    if (!refusal) {
      for (unsigned r = 0; r < 32; r++)
        for (int step = 0; step < 3; step++)
          for (int segs = 1; segs <= 2; segs++) {
            RunFacts rf;
            bool *rb[] = {&rf.want_stats, &rf.prune, &rf.scan_kernels, &rf.strict_accumulate, &rf.small_plan_docs};
            for (unsigned i = 0; i < 5; i++) *rb[i] = (r >> i) & 1u;
            rf.two_step = step != 0;
            rf.one_segment = segs == 1;
            ScorePath path = ScorePath::Tiles;
            const char *why = choose_path(s, rf, path);
            printf("|%s", why ? why : names[(int)path]);
          }
    }
    printf("\n");
  }
  return 0;
}
'''


def expected_line(kc, f):
    """The selection logic of slg_batch_prepare ("kernel selection") and run_batch before slg_dispatch.h, transcribed."""
    small = f["small_k"] and f["few_terms"]
    matcher = f["matcher"]
    and_scan = matcher and f["all_must"] and f["scan_kernels"] and f["stream_kernels"] and not f["has_cursor"]
    items_ok = small and (not matcher or and_scan) and f["all_scores"] and not f["has_plan"] and f["sub_docs_ok"]
    kc_items = kc in (0, 3)
    can_items = items_ok and kc_items
    big_k = (not f["small_k"] and f["few_terms"] and (not matcher or and_scan) and f["all_scores"] and not f["has_plan"]
             and f["scan_kernels"] and f["stream_kernels"] and kc_items)
    can_items = can_items or big_k
    if kc == 3 and not items_ok and not big_k:
        return ITEMS_MSG
    use_warp = can_items or kc == 2 or (kc == 0 and small)
    if use_warp and not small and not big_k:
        return WARP_MSG
    staged = f["all_scores"] and not matcher and f["has_terms"]
    has_colq = can_items and f["stream_kernels"]
    out = ["".join("1" if v else "0" for v in (can_items, big_k, and_scan, use_warp, staged, has_colq))]
    for r in range(32):
        want_stats, prune, scan_kernels, strict, small_plan_docs = ((r >> i) & 1 == 1 for i in range(5))
        run_items = can_items and not want_stats and not (big_k and (not scan_kernels or (strict and not prune)))
        run_scan = run_items and scan_kernels and has_colq and not (strict and not prune)
        warp_path = use_warp and not (big_k and not run_scan)
        if run_scan:
            path = "Scan"
        elif run_items and not prune and has_colq and small_plan_docs:
            path = "Stream"
        elif run_items:
            path = "Items"
        elif warp_path:
            path = "Warp"
        else:
            path = "Tiles"
        for step in STEPS:
            for n_segs in (1, 2):
                if and_scan and run_items and not run_scan:
                    out.append(AND_MSG)
                elif step != "run" and (n_segs != 1 or not run_items or (not prune and not run_scan)):
                    out.append(TWO_STEP_MSG)
                else:
                    out.append(path)
    return "|".join(out)


def run_driver(source: str) -> list:
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "dispatch.cc")
        with open(src, "w") as f:
            f.write(source)
        exe = os.path.join(td, "dispatch")
        subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-Wno-format-security", "-I", CSRC, "-o", exe, src],
                       check=True)
        return subprocess.run([exe], capture_output=True, text=True, check=True).stdout.splitlines()


def test_dispatch_header_reproduces_the_selection_table():
    got = run_driver(DRIVER)
    assert len(got) == 4 << len(PREPARE_FACTS)
    paths = set()
    for p, line in enumerate(got):
        facts = {name: (p >> (2 + i)) & 1 == 1 for i, name in enumerate(PREPARE_FACTS)}
        want = expected_line(p & 3, facts)
        assert line == want, (p & 3, facts)
        paths.update(line.split("|")[1:])
    assert paths == {"Scan", "Stream", "Items", "Warp", "Tiles", AND_MSG, TWO_STEP_MSG}


# ---- every path on the GPU, against the oracle ----

# small corpus: every term with df >= N/8 (and >= 64 postings) gets a column, so the column passes run
DENSE = {"dense_min_df": 64}

# (options, kernel, execution, k, how it runs, declared order, kernel launches of the run).  "canonical": the order of the
# posting-driven paths (terms without a column first), "query": the reference's term order.  The launch count pins the
# path: Scan 10 (reset, slots, 4 scan prologue kernels, scan, column groups, column pass, finalize); Stream 8 (reset, plan
# walk, bounds, slots, sparse pass, column groups, column pass, finalize); pruned Items 8 (reset, plan walk, bounds, slots,
# seeds, item filter, items, finalize); exhaustive Items 6 (no seeds, no filter); Warp and Tiles under bm25 5 (reset,
# plan walk, slots, the kernel, finalize)
PATH_CASES = {
    "scan-bm25-k11": ({}, "bm25", 11, "one", "canonical", 10),
    "scan-bmw-k11": ({}, "bmw", 11, "one", "canonical", 10),
    "scan-bm25-k101": ({}, "bm25", 101, "one", "canonical", 10),
    "scan-bmw-k101": ({}, "bmw", 101, "one", "canonical", 10),
    "stream-bm25": ({"scan_kernels": 0}, "bm25", 11, "one", "canonical", 8),
    "stream-strict-bm25": ({"strict_accumulate": 1}, "bm25", 11, "one", "canonical", 8),
    "items-bmw": ({"scan_kernels": 0}, "bmw", 11, "one", "canonical", 8),
    "items-bm25-no-stream": ({"scan_kernels": 0, "stream_kernels": 0}, "bm25", 11, "one", "canonical", 6),
    "items-two-step": ({"scan_kernels": 0}, "bmw", 11, "two-step", "canonical", 8),
    "warp-stats": ({}, "bm25", 11, "stats", "canonical", 5),
    "tiles-strict-k101": ({"strict_accumulate": 1}, "bm25", 101, "one", "query", 5),
}


@pytest.fixture(scope="module")
def corpus():
    """the segment, the queries, the oracle and, per k, the Scan path's bm25 result: the bytes every path with the
    canonical order must return"""
    spec = synth.CorpusSpec(n_docs=30_000, vocab=5_000, seed=21, len_lo=20, len_hi=80)
    seg = synth.generate_segment(spec, "cpu", chunk_docs=8192)
    qb = synth.generate_queries(120, spec.vocab, seed=22)
    from oracle import slo
    gi = GpuIndex(0, options=DENSE)
    gi.load_segment(seg)
    canonical = {k: gi.search_batch(qb, k, "bm25") for k in (11, 101)}
    gi.close()
    return seg, qb, slo.OracleIndex(seg), canonical


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(PATH_CASES))
def test_every_scoring_path_matches_the_oracle(corpus, case):
    seg, qb, ora, canonical = corpus
    options, execution, k, how, order, launches = PATH_CASES[case]
    gi = GpuIndex(0, options={**DENSE, **options})
    gi.load_segment(seg)
    c0 = gi.counters()
    if how == "one":
        got = gi.search_batch(qb, k, execution)
    elif how == "stats":
        got = gi.search_batch(qb, k, execution, want_stats=True)[:2]
    else:
        pb = gi.prepare(qb, k, execution)
        assert pb.run_seeds()
        pb.run_sweep()
        got = pb.fetch()
        pb.free()
    c1 = gi.counters()
    assert c1["kernel_launches"] - c0["kernel_launches"] == launches
    assert c1["score_launches"] - c0["score_launches"] == 1
    assert_engine_parity(gi, ora, qb, k, got, exact_order=(order == "query"))
    if order == "canonical":
        assert got[0].tobytes() == canonical[k][0].tobytes() and got[1].tobytes() == canonical[k][1].tobytes()
    gi.close()


@pytest.mark.gpu
def test_and_batch_is_refused_on_the_sub_tile_kernels(corpus):
    seg, qb, _, _ = corpus
    gi = GpuIndex(0, options={**DENSE, "strict_accumulate": 1})
    gi.load_segment(seg)
    tl = [qb.terms["term_id"][int(qb.term_off[q]):int(qb.term_off[q + 1])].tolist() for q in range(qb.n_queries)]
    ab = QueryBatch.from_bool([{"must": t[:2]} for t in tl if len(t) >= 2])
    with pytest.raises(SearchliteGpuError, match=r"an AND batch prepared for the posting scan cannot run on the sub-tile kernels"):
        gi.search_batch(ab, 11, "bm25")
    gi.close()
