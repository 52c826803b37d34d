// slg_dispatch.h — which scoring path a batch takes.  Host-only C++17 with no CUDA includes: the whole decision is
// here, and tests/test_dispatch.py compiles this header on its own to check it against every combination of its facts.
//
// Two steps.  slg_batch_prepare calls select_kernels once: it fixes the term layout and which slab sections exist.  Each
// run calls choose_path again, because statistics and the options can change between prepare and run.
#pragma once
#include <cstdint>

namespace slg {

enum class ScorePath {
  Scan,    // flat posting scan, then the column pass (slg_scan_kernel.cuh)
  Stream,  // exhaustive sub-tile path: sparse pass, then the column pass (slg_stream_kernel.cuh)
  Items,   // posting-driven items kernel, with seeds and the item filter when pruned (slg_items_kernel.cuh)
  Warp,    // warp-per-item kernel (slg_warp_kernel.cuh)
  Tiles,   // CTA-per-item kernel (slg_kernels.cuh)
};

// what slg_batch_prepare knows about a batch and the handle's options
struct BatchFacts {
  uint32_t kernel_choice = 0;   // 0 auto, 1 CTA-per-item, 2 warp-per-item, 3 items kernel required
  bool small_k = false;         // k <= kWarpMaxK
  bool few_terms = false;       // every query keeps <= kWarpMaxTerms terms
  bool matcher = false;         // some query needs the group matcher (Bool roles or unscored terms)
  bool all_must = false;        // every query is Bool{must: one scored term per group}
  bool has_cursor = false;
  bool has_plan = false;
  bool all_scores = false;      // staging is on and every segment holds resident per-posting scores
  bool sub_docs_ok = false;     // sub_docs <= 4096
  bool scan_kernels = false;    // the options at prepare time
  bool stream_kernels = false;
  bool has_terms = false;       // the batch has at least one unique term
};

// what prepare decides; a batch keeps it for its runs
struct Selection {
  // the posting-driven paths may run: scan tables (and items when pruned), and the term tables in canonical order, which
  // a statistics run on the warp kernel shares
  bool canonical = false;
  bool pools = false;        // k > kWarpMaxK on the posting scan: candidate pools instead of the warp's sorted top-k
  bool and_scan = false;     // AND batch: the posting scan drives from each query's rarest list
  bool warp_tables = false;  // per-query QTerm / QHead tables
  bool staged = false;       // the warp kernel's (doc, score) stream form applies
  bool colq = false;         // column-pass tables (ColQ, ucol, col_slot)
};

// fills s; non-null: the batch is refused (SLG_ERR_UNSUPPORTED) with this printf format, which takes kWarpMaxK, kWarpMaxTerms
inline const char *select_kernels(const BatchFacts &f, Selection &s) {
  s = Selection{};
  const bool small = f.small_k && f.few_terms;
  // (AND batches ride the posting scan; without it — scan_kernels 0, statistics — they are ordinary matcher batches)
  s.and_scan = f.matcher && f.all_must && f.scan_kernels && f.stream_kernels && !f.has_cursor;
  const bool posting_form = (!f.matcher || s.and_scan) && f.all_scores && !f.has_plan;  // a batch the posting-driven paths take
  const bool items_ok = small && posting_form && f.sub_docs_ok;
  const bool kc_items = f.kernel_choice == 0 || f.kernel_choice == 3;
  s.pools = !f.small_k && f.few_terms && posting_form && f.scan_kernels && f.stream_kernels && kc_items;
  if (f.kernel_choice == 3 && !items_ok && !s.pools)
    return "the items kernel handles plain OR queries without a ScorePlan, k <= %u, <= %u terms per query, resident scores, sub_docs <= 4096";
  s.canonical = (items_ok && kc_items) || s.pools;
  s.warp_tables = s.canonical || f.kernel_choice == 2 || (f.kernel_choice == 0 && small);
  if (s.warp_tables && !small && !s.pools) return "the warp kernel handles k <= %u and <= %u terms per query";
  s.staged = f.all_scores && !f.matcher && f.has_terms;
  s.colq = s.canonical && f.stream_kernels;
  return nullptr;
}

// what a run knows besides the selection
struct RunFacts {
  bool want_stats = false;
  bool prune = false;              // execution is WAND or BMW
  bool scan_kernels = false;       // the options at run time
  bool strict_accumulate = false;
  bool small_plan_docs = false;    // plan_docs <= 2048: posting numbers of a sub-tile fit the sparse pass's 15 bits
  bool two_step = false;           // slg_batch_run_seeds or slg_batch_run_sweep
  bool one_segment = false;
};

// sets path; non-null: the run is refused (SLG_ERR_UNSUPPORTED) with this message
inline const char *choose_path(const Selection &s, const RunFacts &r, ScorePath &path) {
  const bool exhaustive_strict = r.strict_accumulate && !r.prune;
  const bool posting = s.canonical && !r.want_stats && !(s.pools && (!r.scan_kernels || exhaustive_strict));
  const bool scan = posting && r.scan_kernels && s.colq && !exhaustive_strict;
  if (s.and_scan && posting && !scan) return "an AND batch prepared for the posting scan cannot run on the sub-tile kernels (strict_accumulate)";
  if (r.two_step && (!r.one_segment || !posting || (!r.prune && !scan)))
    return "the two-step run (first part, threshold exchange, rest) needs one segment per handle and the posting scan or the pruned items kernel";
  if (scan) path = ScorePath::Scan;
  else if (posting && !r.prune && s.colq && r.small_plan_docs) path = ScorePath::Stream;
  else if (posting) path = ScorePath::Items;
  else if (s.warp_tables && !s.pools) path = ScorePath::Warp;  // (k > kWarpMaxK without the scan: the CTA-per-item kernel)
  else path = ScorePath::Tiles;
  return nullptr;
}

}  // namespace slg
