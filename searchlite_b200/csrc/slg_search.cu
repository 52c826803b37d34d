// slg_search.cu — batched search of libsearchlite_gpu.so: batch preparation, the kernel schedule of one run, result
// fetch and the shard merge.
//
// Mirrors IndexReader::search_segment (searchlite-core/src/api/reader.rs:2908-3128) and
// execute_top_k_with_stats_and_mode_internal (src/query/wand.rs:398-456) for Q queries at once, and
// hits.sort_by(SortKey) (api/reader.rs:2777).  There is no CPU fallback: every search runs the CUDA kernels or fails.
#include "slg_host.h"
#include "slg_residency.cuh"

using namespace slg;

namespace {

// unique terms of a batch: open addressing over a power-of-two table (a batch holds a few 10^4 term instances)
struct TermSet {
  std::vector<uint32_t> key, val;
  uint32_t mask = 0;
  explicit TermSet(size_t expect) {
    size_t n = 64;
    while (n < expect * 2) n <<= 1;
    key.assign(n, 0xFFFFFFFFu);
    val.assign(n, 0);
    mask = (uint32_t)n - 1;
  }
  // index of `term` among the unique terms, appended to `ut` when new
  uint32_t get(uint32_t term, std::vector<uint32_t> &ut) {
    uint32_t h = (term * 0x9E3779B1u) & mask;
    for (;;) {
      if (key[h] == term) return val[h];
      if (key[h] == 0xFFFFFFFFu) {
        key[h] = term;
        val[h] = (uint32_t)ut.size();
        ut.push_back(term);
        return val[h];
      }
      h = (h + 1) & mask;
    }
  }
};

int32_t select_smem(slg_index *ix, uint32_t tile_docs, uint32_t cap, bool matcher, size_t *out, uint32_t planes = 1) {
  size_t smem = (size_t)tile_docs * 4 * planes + (size_t)cap * 8 + (matcher ? tile_docs : 0);
  if (smem + 1024 > ix->smem_optin)
    return fail(ix, SLG_ERR_UNSUPPORTED, "tile of %u docs with k buffer %u needs %zu B shared memory", tile_docs, cap, smem);
  *out = smem;
  return SLG_OK;
}

// per-segment reset of the running state: thr_key = kThrInit, everything else in the state block zero
__global__ void slg_reset_state_kernel(unsigned long long *thr_key, uint32_t n_queries, uint32_t *rest, uint32_t n_rest_words) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_queries) thr_key[i] = kThrInit;
  if (i < n_rest_words) rest[i] = 0u;
}

// thresholds of other shards (score part only: an equal score may still win on segment order, query/sort.rs:80-93)
__global__ void slg_import_thresholds_kernel(unsigned long long *thr_key, const unsigned long long *other, uint32_t n_queries) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_queries) return;
  const unsigned long long o = other[i] & 0xFFFFFFFF00000000ull;
  if (o > thr_key[i]) thr_key[i] = o;
}

}  // namespace

extern "C" {

int32_t slg_batch_prepare(slg_index_t *ix, const slg_query_t *queries, uint32_t n_queries, uint32_t k, slg_exec_t exec,
                          uint32_t bmw_block_size, slg_batch_t **out) {
  if (!ix || !out) return SLG_ERR_INVALID;
  *out = nullptr;
  if (!queries || n_queries == 0) return fail(ix, SLG_ERR_INVALID, "empty query batch");
  if (k == 0) return fail(ix, SLG_ERR_INVALID, "k must be > 0 (the reference bails on limit == 0, api/reader.rs:2540)");
  if (k > SLG_MAX_K) return fail(ix, SLG_ERR_UNSUPPORTED, "k = %u exceeds the built maximum %u", k, SLG_MAX_K);
  if (exec != SLG_EXEC_BM25 && exec != SLG_EXEC_WAND && exec != SLG_EXEC_BMW) return fail(ix, SLG_ERR_INVALID, "unknown execution strategy");
  if (ix->segs.empty()) return fail(ix, SLG_ERR_INVALID, "no segment loaded");
  (void)bmw_block_size;  // bounds are finer than any block size the reference would rebuild (wand.rs:305-330); the result is exact either way
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  PoolScope pool_scope(ix->stream);
  auto bt = std::make_unique<slg_batch>();
  bt->ix = ix;
  bt->Q = n_queries;
  bt->k = k;
  bt->exec = exec;
  bt->cap = std::max(1024u, 1u << (32 - __builtin_clz(4 * k - 1)));
  const Segment *s0 = ix->segs[0].get();
  uint64_t n_terms_space = 0;
  for (auto &s : ix->segs) n_terms_space = std::max(n_terms_space, s->n_terms);

  size_t t_expect = 0;
  for (uint32_t qi = 0; qi < n_queries; qi++) t_expect += queries[qi].n_terms;
  TermSet uset(t_expect);
  std::vector<uint32_t> ut, q_off(n_queries + 1, 0), qt_u;
  std::vector<float> qt_w;
  std::vector<uint8_t> qt_g, qt_f, q_must(n_queries, 0), q_not(n_queries, 0), q_should(n_queries, 0), q_min(n_queries, 0);
  std::vector<int32_t> q_filter(n_queries, -1);
  std::vector<uint64_t> q_cost(n_queries, 0);
  std::vector<uint8_t> qt_leaf, q_leaves(n_queries, 0);
  std::vector<uint32_t> q_plan_off(n_queries + 1, 0);
  std::vector<PlanNodeDev> plan_nodes;
  qt_u.reserve(t_expect);
  qt_w.reserve(t_expect);
  qt_g.reserve(t_expect);
  qt_f.reserve(t_expect);
  qt_leaf.reserve(t_expect);
  bool matcher = false;
  // AND batches: every query is Bool{must:[t1, t2, ..]} — one scored term per group, every group a MUST, nothing else.  The
  // posting scan then walks only the query's RAREST list and asks the other lists whether they hold the doc
  bool all_must = true;
  for (uint32_t qi = 0; qi < n_queries; qi++) {
    const slg_query_t &q = queries[qi];
    if (q.n_terms && !q.terms) return fail(ix, SLG_ERR_INVALID, "query %u has no terms pointer", qi);
    if (q.n_groups > SLG_MAX_GROUPS) return fail(ix, SLG_ERR_UNSUPPORTED, "query %u has %u term groups; this build supports %u", qi, q.n_groups, SLG_MAX_GROUPS);
    if (q.n_groups && !q.group_role) return fail(ix, SLG_ERR_INVALID, "query %u has no group roles", qi);
    if (q.filter_id >= (int32_t)ix->filters.size()) return fail(ix, SLG_ERR_INVALID, "query %u names unknown filter %d", qi, q.filter_id);
    q_filter[qi] = q.filter_id < 0 ? -1 : q.filter_id;
    if (q.n_plan_nodes) {
      // ScorePlan: a well-formed postfix program over leaves 0..leaf_count-1 (query/planner.rs:113-164)
      if (!q.plan) return fail(ix, SLG_ERR_INVALID, "query %u has no plan pointer", qi);
      if (q.leaf_count == 0 || q.leaf_count > SLG_MAX_PLAN_LEAVES)
        return fail(ix, SLG_ERR_UNSUPPORTED, "query %u: a plan needs 1..%u leaves, got %u", qi, SLG_MAX_PLAN_LEAVES, q.leaf_count);
      if (q.n_plan_nodes > SLG_MAX_PLAN_NODES)
        return fail(ix, SLG_ERR_UNSUPPORTED, "query %u: plan of %u nodes; the maximum is %u", qi, q.n_plan_nodes, SLG_MAX_PLAN_NODES);
      uint32_t depth = 0;
      for (uint32_t n = 0; n < q.n_plan_nodes; n++) {
        const slg_plan_node_t &pn = q.plan[n];
        if (pn.op == SLG_PLAN_LEAF) {
          if (pn.arg >= q.leaf_count) return fail(ix, SLG_ERR_INVALID, "query %u plan node %u: leaf %u out of range", qi, n, pn.arg);
          depth++;
        } else if (pn.op == SLG_PLAN_SUM || pn.op == SLG_PLAN_DISMAX) {
          if (pn.arg > depth) return fail(ix, SLG_ERR_INVALID, "query %u plan node %u: %u children but %u values", qi, n, pn.arg, depth);
          if (pn.op == SLG_PLAN_DISMAX && !(pn.tie_breaker >= 0.0f && pn.tie_breaker <= 1.0f))
            return fail(ix, SLG_ERR_INVALID, "query %u plan node %u: tie_breaker must lie in [0, 1]", qi, n);  // planner.rs:850-858
          depth = depth - pn.arg + 1;
        } else {
          return fail(ix, SLG_ERR_INVALID, "query %u plan node %u: unknown op %u", qi, n, pn.op);
        }
        plan_nodes.push_back(PlanNodeDev{pn.op, pn.arg, pn.tie_breaker});
      }
      if (depth != 1) return fail(ix, SLG_ERR_INVALID, "query %u: the plan leaves %u values instead of one", qi, depth);
      q_leaves[qi] = (uint8_t)q.leaf_count;
      bt->has_plan = true;
      bt->max_leaves = std::max(bt->max_leaves, q.leaf_count);
    }
    q_plan_off[qi + 1] = (uint32_t)plan_nodes.size();
    if (q.has_cursor) {
      if (!(q.cursor.score >= 0.0f) || !std::isfinite(q.cursor.score))
        return fail(ix, SLG_ERR_INVALID, "query %u: the cursor score must be finite and >= 0", qi);
      bt->has_cursor = true;
    }
    if (q.filter_id >= 0)
      for (auto &sg : ix->segs)
        if ((size_t)q.filter_id >= sg->filter_bits.size() || !sg->filter_bits[q.filter_id].p)
          return fail(ix, SLG_ERR_INVALID, "query %u names filter %d, which is freed or not compiled for segment %u", qi, q.filter_id, sg->ord);
    uint32_t kept = 0;
    bool need_mask = q.n_groups > 0;
    for (uint32_t t = 0; t < q.n_terms; t++) {
      const slg_term_t &tm = q.terms[t];
      if (tm.term_id == 0xFFFFFFFFu || tm.term_id >= n_terms_space) continue;  // seg.postings(key) == None
      bool scored = tm.flags & SLG_TERM_SCORED;
      if (scored && !(tm.weight >= 0x1p-100f && std::isfinite(tm.weight)))  // (below: a contribution may round to +0, include/searchlite_gpu.h)
        return fail(ix, SLG_ERR_UNSUPPORTED, "query %u term %u: weight must be finite and >= 2^-100", qi, t);
      if (q.n_groups && tm.group >= q.n_groups) return fail(ix, SLG_ERR_INVALID, "query %u term %u: group out of range", qi, t);
      if (scored && q.n_plan_nodes && tm.leaf >= q.leaf_count)
        return fail(ix, SLG_ERR_INVALID, "query %u term %u: leaf %u but the plan has %u leaves", qi, t, tm.leaf, q.leaf_count);  // wand.rs:489-494
      if (!scored) need_mask = true;
      qt_u.push_back(uset.get(tm.term_id, ut));
      qt_w.push_back(tm.weight);
      qt_g.push_back((uint8_t)(q.n_groups ? tm.group : 0));
      qt_f.push_back(scored ? 1 : 0);
      qt_leaf.push_back((uint8_t)(scored && q.n_plan_nodes ? tm.leaf : 0));
      if (scored && tm.term_id < s0->n_terms) q_cost[qi] += s0->h_df[tm.term_id];
      kept++;
    }
    {
      bool pure = q.n_groups > 0 && kept == q.n_groups && q.n_terms == q.n_groups;  // (a MUST group that lost its term can never match: left to the matcher kernels)
      uint32_t seen_groups = 0;
      for (uint32_t g = 0; pure && g < q.n_groups; g++) pure = q.group_role[g] == SLG_ROLE_MUST;
      for (uint32_t t = 0; pure && t < q.n_terms; t++) {
        pure = (q.terms[t].flags & SLG_TERM_SCORED) && !((seen_groups >> q.terms[t].group) & 1u);
        seen_groups |= 1u << q.terms[t].group;
      }
      all_must = all_must && pure;
    }
    if (kept > SLG_MAX_QUERY_TERMS) return fail(ix, SLG_ERR_UNSUPPORTED, "query %u has %u terms; the maximum is %u", qi, kept, SLG_MAX_QUERY_TERMS);
    q_off[qi + 1] = q_off[qi] + kept;
    bt->max_terms = std::max(bt->max_terms, kept);
    if (need_mask) {
      matcher = true;
      if (q.n_groups == 0) {  // non-scored terms without groups: plain OR over group 0
        q_should[qi] = 1;
        q_min[qi] = 1;
      }
      for (uint32_t g = 0; g < q.n_groups; g++) {
        uint8_t bit = (uint8_t)(1u << g);
        if (q.group_role[g] == SLG_ROLE_MUST) q_must[qi] |= bit;
        else if (q.group_role[g] == SLG_ROLE_MUST_NOT) q_not[qi] |= bit;
        else q_should[qi] |= bit;
      }
      if (q.n_groups) q_min[qi] = (uint8_t)std::min<uint32_t>(q.min_should, 255);
    }
    bt->posting_count += q_cost[qi];
  }
  const uint32_t S = (uint32_t)ix->segs.size();
  std::vector<unsigned long long> bounds;
  if (bt->has_cursor) {
    // key.cmp(cursor) (query/sort.rs:80-93: score desc, segment_ord asc, doc_id asc) folded into one exclusive bound on
    // the 64-bit keys of each segment: same segment (score, ~doc); an earlier segment loses ties; a later one wins them
    bounds.assign((size_t)S * n_queries, ~0ull);
    bt->h_has_cursor.assign(n_queries, 0);
    for (uint32_t qi = 0; qi < n_queries; qi++) {
      const slg_query_t &q = queries[qi];
      if (!q.has_cursor) continue;
      bt->h_has_cursor[qi] = 1;
      uint32_t sb;
      std::memcpy(&sb, &q.cursor.score, 4);
      for (uint32_t si = 0; si < S; si++) {
        const uint32_t ord = ix->segs[si]->ord;
        unsigned long long b;
        if (ord == q.cursor.segment_ord) b = ((unsigned long long)sb << 32) | (unsigned long long)(0xFFFFFFFFu - q.cursor.doc_id);
        else if (ord < q.cursor.segment_ord) b = (unsigned long long)sb << 32;
        else b = ((unsigned long long)sb + 1ull) << 32;
        bounds[(size_t)si * n_queries + qi] = b;
      }
    }
    bt->n_cursor_segs = S;
  }
  bt->matcher = matcher;
  bt->U = (uint32_t)ut.size();
  bt->T = (uint32_t)qt_u.size();

  // ---- kernel selection ----
  // items kernel (posting-driven; the automatic choice): plain OR queries, k <= 32, <= 8 terms per query, resident
  // scores, no plan.  Per-query statistics are counted by the warp kernel, on the same (canonical) term layout.
  const bool small = k <= kWarpMaxK && bt->max_terms <= kWarpMaxTerms;
  bool all_scores = ix->staging;
  for (auto &s : ix->segs) all_scores = all_scores && (s->post_score.p != nullptr || s->n_blocks == 0);
  // (AND batches ride the posting scan; without it — scan_kernels 0, statistics — they are ordinary matcher batches)
  const bool and_scan = matcher && all_must && ix->scan_kernels && ix->stream_kernels && !bt->has_cursor;
  bt->and_scan = and_scan;
  const bool items_ok = small && (!matcher || and_scan) && all_scores && !bt->has_plan && ix->sub_docs <= 4096;
  bt->can_items = items_ok && (ix->kernel_choice == 0 || ix->kernel_choice == 3);
  // k up to SLG_MAX_K on the flat posting scan: candidate pools + radix select instead of the warp's sorted top-k
  bt->big_k = k > kWarpMaxK && bt->max_terms <= kWarpMaxTerms && (!matcher || and_scan) && all_scores && !bt->has_plan && ix->scan_kernels && ix->stream_kernels &&
              (ix->kernel_choice == 0 || ix->kernel_choice == 3);
  if (bt->big_k) bt->can_items = true;
  if (ix->kernel_choice == 3 && !items_ok && !bt->big_k)
    return fail(ix, SLG_ERR_UNSUPPORTED,
                "the items kernel handles plain OR queries without a ScorePlan, k <= %u, <= %u terms per query, resident scores, sub_docs <= 4096",
                kWarpMaxK, kWarpMaxTerms);

  bt->canonical = bt->can_items;
  bt->use_warp = bt->can_items || ix->kernel_choice == 2 || (ix->kernel_choice == 0 && small);
  if (bt->use_warp && !small && !bt->big_k)
    return fail(ix, SLG_ERR_UNSUPPORTED, "the warp kernel handles k <= %u and <= %u terms per query", kWarpMaxK, kWarpMaxTerms);
  bt->staged = all_scores && !matcher && bt->U > 0;

  // processing order inside a tile: most expensive queries first
  std::vector<uint32_t> order(n_queries);
  for (uint32_t i = 0; i < n_queries; i++) order[i] = i;
  std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b2) { return q_cost[a] > q_cost[b2]; });

  // ---- geometry ----
  bt->plan_docs = bt->use_warp ? ix->sub_docs : ix->tile_docs;
  if (bt->has_plan) {
    // one accumulator plane per leaf: shrink the doc tile so that the planes together stay near the configured tile
    uint32_t planes = 1;
    while (planes < bt->max_leaves) planes <<= 1;
    bt->plan_docs = bt->use_warp ? std::max(512u, (ix->sub_docs / planes) & ~127u) : std::max(1024u, (ix->tile_docs / planes) & ~1023u);
  }
  uint32_t max_tiles = 1;
  for (auto &s : ix->segs) max_tiles = std::max(max_tiles, (s->doc_count + bt->plan_docs - 1) / bt->plan_docs);
  bt->sub_tiles_max = max_tiles;
  const uint32_t max_groups = (max_tiles + kSubPerGroup - 1) / kSubPerGroup;

  // ---- packed inputs: one host-to-device copy out of pinned memory ----
  size_t pos = 0;
  auto place = [&](size_t bytes) {
    size_t o = pos;
    pos = align_up(pos + std::max<size_t>(bytes, 4), 256);
    return o;
  };
  bt->off_ut_term = place((size_t)bt->U * 4);
  bt->off_q_term_off = place((size_t)(n_queries + 1) * 4);
  bt->off_qt_uterm = place((size_t)bt->T * 4);
  bt->off_qt_weight = place((size_t)bt->T * 4);
  bt->off_qt_group = place(bt->T);
  bt->off_qt_flags = place(bt->T);
  bt->off_q_order = place((size_t)n_queries * 4);
  bt->off_q_must = place(n_queries);
  bt->off_q_not = place(n_queries);
  bt->off_q_should = place(n_queries);
  bt->off_q_min = place(n_queries);
  bt->off_q_filter = place((size_t)n_queries * 4);
  if (bt->has_plan) {
    bt->off_qt_leaf = place(bt->T);
    bt->off_q_leaves = place(n_queries);
    bt->off_q_plan_off = place((size_t)(n_queries + 1) * 4);
    bt->off_plan_nodes = place(plan_nodes.size() * sizeof(PlanNodeDev));
  }
  if (bt->has_cursor) bt->off_cursor_bounds = place(bounds.size() * 8);
  bt->pack_bytes = pos;

  // ---- the slab ----
  size_t dpos = 0;
  auto carve = [&](size_t bytes) {
    size_t o = dpos;
    dpos = align_up(dpos + std::max<size_t>(bytes, 16), 256);
    return o;
  };
  const size_t o_pack = carve(bt->pack_bytes);
  const size_t o_rng = carve((size_t)std::max(bt->U, 1u) * (max_tiles + 1) * 4);
  const size_t o_ub = (exec != SLG_EXEC_BM25 || bt->can_items) ? carve((size_t)std::max(bt->U, 1u) * max_tiles * 4) : 0;
  // state block, reset per segment: thr_key [Q] u64 | topk_count [Q] | lock [Q] | work_counter [64] | n_items [2]
  uint32_t kp = 1;
  while (kp < k) kp <<= 1;
  bt->pool_cap = bt->big_k ? 2 * kp : 0;
  const size_t state_words = (size_t)n_queries * 2 + 64 + 2 + (bt->big_k ? (size_t)n_queries * 4 : 0);
  const size_t o_thr = carve((size_t)n_queries * 8 + state_words * 4);
  const size_t o_topk = carve((size_t)n_queries * k * 8);
  const size_t o_pools = bt->big_k ? carve((size_t)n_queries * 2 * bt->pool_cap * 8) : 0;
  const size_t o_stats = carve((size_t)n_queries * 5 * 8 + 64);  // [Q][4] counters, [Q] accepted docs, then the items counters [4]
  const size_t o_saw = bt->has_cursor ? carve((size_t)n_queries * 4) : 0;
  const size_t o_qterms = bt->use_warp ? carve((size_t)n_queries * kWarpMaxTerms * sizeof(QTerm)) : 0;
  const size_t o_qheads = bt->use_warp ? carve((size_t)n_queries * sizeof(QHead)) : 0;
  const bool want_items = bt->can_items && exec != SLG_EXEC_BM25;
  bt->items_cap = want_items ? max_groups * n_queries : 0;
  bt->done_bytes = want_items ? (size_t)max_groups * n_queries : 0;
  const size_t o_items = want_items ? carve((size_t)bt->items_cap * sizeof(uint2)) : 0;
  const bool want_stream = bt->can_items && ix->stream_kernels;
  for (auto &s : ix->segs) bt->max_cols = std::max(bt->max_cols, s->n_cols);
  // postings per scan item: 4096 on a 10 M-doc segment (fewer, longer items: less per-item work), smaller on small
  // segments — the shards of a multi-GPU run — where 4096 leaves too few items to balance 4736 warps
  // (profiles/r2_scan_experiments.txt: at 1.25 M docs 1024 takes 2.4 ms against 3.0 ms; at 10 M docs it takes 22 against 9.4)
  {
    uint32_t max_docs = 0;
    for (auto &sg : ix->segs) max_docs = std::max(max_docs, sg->doc_count);
    bt->scan_chunk = ix->scan_chunk ? ix->scan_chunk : (max_docs >= 4000000u ? 4096u : max_docs >= 2000000u ? 2048u : 1024u);
  }
  // flat posting scan: item capacity = the largest segment's sum over scanned term instances of ceil(df / scan_chunk)
  if (bt->can_items) {
    for (auto &sg : ix->segs) {
      uint64_t n = 0;
      for (size_t i = 0; i < qt_u.size(); i++) {
        const uint32_t term = ut[qt_u[i]];
        if (term >= sg->n_terms || !qt_f[i]) continue;
        if (!bt->and_scan && !sg->h_term_col.empty() && sg->h_term_col[term] >= 0) continue;  // (an AND batch may scan any of its terms)
        n += (sg->h_df[term] + bt->scan_chunk - 1) / bt->scan_chunk;
      }
      bt->scan_items_cap = (uint32_t)std::max<uint64_t>(bt->scan_items_cap, std::min<uint64_t>(n, 0xFFFFFFF0ull));
    }
  }
  const bool want_scan = bt->can_items;
  const size_t o_utmax = want_scan ? carve((size_t)std::max(bt->U, 1u) * 4) : 0;
  const size_t o_pairs = want_scan ? carve((size_t)n_queries * kWarpMaxTerms * sizeof(ScanPair)) : 0;
  const size_t o_order = want_scan ? carve((size_t)n_queries * kWarpMaxTerms * 4) : 0;
  const size_t o_istart = want_scan ? carve(((size_t)n_queries * kWarpMaxTerms + 1) * 4) : 0;
  const size_t o_sitems = want_scan ? carve((size_t)std::max(bt->scan_items_cap, 1u) * 4) : 0;
  const size_t o_colq = want_stream ? carve((size_t)n_queries * sizeof(ColQ)) : 0;
  const size_t o_ucol = want_stream ? carve((size_t)(bt->max_cols + 1) * 4) : 0;
  const size_t o_colslot = want_stream ? carve((size_t)(bt->max_cols + 1) * 4) : 0;
  const size_t o_done = want_items ? carve(bt->done_bytes) : 0;
  bt->result_stride = align_up((size_t)n_queries * k * sizeof(HitDev) + (size_t)n_queries * 4 + (size_t)n_queries * k * 4, 256);  // hits | counts | vector scores
  const size_t o_results = carve(bt->result_stride * (S + (S > 1 ? 1 : 0)));
  SLG_CUDA(ix, bt->slab.alloc(dpos));
  unsigned char *base = bt->slab.as<unsigned char>();
  bt->d_pack = base + o_pack;
  bt->ut_rng = reinterpret_cast<uint32_t *>(base + o_rng);
  bt->ut_tile_ub = (exec != SLG_EXEC_BM25 || bt->can_items) ? reinterpret_cast<float *>(base + o_ub) : nullptr;
  bt->thr_key = reinterpret_cast<unsigned long long *>(base + o_thr);
  bt->state = base + o_thr + (size_t)n_queries * 8;
  bt->state_bytes = state_words * 4;
  bt->topk_count = reinterpret_cast<uint32_t *>(bt->state);
  bt->lock = bt->topk_count + n_queries;
  bt->work_counter = bt->lock + n_queries;
  bt->n_items = bt->work_counter + 64;
  bt->pool_count = bt->big_k ? bt->n_items + 2 : nullptr;
  bt->pool_lock = bt->big_k ? bt->pool_count + (size_t)n_queries * 2 : nullptr;
  bt->pool_keys = bt->big_k ? reinterpret_cast<unsigned long long *>(base + o_pools) : nullptr;
  bt->topk_keys = reinterpret_cast<unsigned long long *>(base + o_topk);
  bt->stats = reinterpret_cast<unsigned long long *>(base + o_stats);
  bt->item_counters = bt->stats + (size_t)n_queries * 5;
  bt->cursor_saw = bt->has_cursor ? reinterpret_cast<uint32_t *>(base + o_saw) : nullptr;
  bt->qterms = bt->use_warp ? reinterpret_cast<QTerm *>(base + o_qterms) : nullptr;
  bt->qheads = bt->use_warp ? reinterpret_cast<QHead *>(base + o_qheads) : nullptr;
  bt->items = want_items ? reinterpret_cast<uint2 *>(base + o_items) : nullptr;
  bt->done = want_items ? base + o_done : nullptr;
  bt->ut_max = want_scan ? reinterpret_cast<float *>(base + o_utmax) : nullptr;
  bt->scan_pairs = want_scan ? reinterpret_cast<ScanPair *>(base + o_pairs) : nullptr;
  bt->scan_order = want_scan ? reinterpret_cast<uint32_t *>(base + o_order) : nullptr;
  bt->scan_item_start = want_scan ? reinterpret_cast<uint32_t *>(base + o_istart) : nullptr;
  bt->scan_items = want_scan ? reinterpret_cast<uint32_t *>(base + o_sitems) : nullptr;
  bt->colq = want_stream ? reinterpret_cast<ColQ *>(base + o_colq) : nullptr;
  bt->ucol = want_stream ? reinterpret_cast<uint32_t *>(base + o_ucol) : nullptr;
  bt->col_slot = want_stream ? reinterpret_cast<uint32_t *>(base + o_colslot) : nullptr;
  bt->results = base + o_results;

  // ---- pinned staging: [pack | results | per-query stats + items counters] ----
  bt->pinned_result_off = align_up(bt->pack_bytes, 256);
  bt->pinned_bytes = bt->pinned_result_off + bt->result_stride + (size_t)n_queries * 40 + 64;
  if (!ix->pinned_busy && ix->pinned && ix->pinned_bytes >= bt->pinned_bytes) {
    bt->pinned = ix->pinned;
    bt->pinned_from_index = true;
    ix->pinned_busy = true;
  } else {
    SLG_CUDA(ix, cudaMallocHost(&bt->pinned, bt->pinned_bytes));
  }
  unsigned char *hp = static_cast<unsigned char *>(bt->pinned);
  auto put = [&](size_t off, const void *src, size_t bytes) {
    if (bytes) std::memcpy(hp + off, src, bytes);
  };
  put(bt->off_ut_term, ut.data(), (size_t)bt->U * 4);
  put(bt->off_q_term_off, q_off.data(), (size_t)(n_queries + 1) * 4);
  put(bt->off_qt_uterm, qt_u.data(), (size_t)bt->T * 4);
  put(bt->off_qt_weight, qt_w.data(), (size_t)bt->T * 4);
  put(bt->off_qt_group, qt_g.data(), bt->T);
  put(bt->off_qt_flags, qt_f.data(), bt->T);
  put(bt->off_q_order, order.data(), (size_t)n_queries * 4);
  put(bt->off_q_must, q_must.data(), n_queries);
  put(bt->off_q_not, q_not.data(), n_queries);
  put(bt->off_q_should, q_should.data(), n_queries);
  put(bt->off_q_min, q_min.data(), n_queries);
  put(bt->off_q_filter, q_filter.data(), (size_t)n_queries * 4);
  if (bt->has_plan) {
    put(bt->off_qt_leaf, qt_leaf.data(), bt->T);
    put(bt->off_q_leaves, q_leaves.data(), n_queries);
    put(bt->off_q_plan_off, q_plan_off.data(), (size_t)(n_queries + 1) * 4);
    put(bt->off_plan_nodes, plan_nodes.data(), plan_nodes.size() * sizeof(PlanNodeDev));
  }
  if (bt->has_cursor) put(bt->off_cursor_bounds, bounds.data(), bounds.size() * 8);
  SLG_CUDA(ix, cudaMemcpyAsync(bt->d_pack, hp, bt->pack_bytes, cudaMemcpyHostToDevice, ix->stream));
  ix->ctr.last_h2d_bytes = bt->pack_bytes;
  *out = bt.release();
  return SLG_OK;
}

}  // extern "C"

namespace {

// everything of one run up to (seeds_only) or including the sweep; see the schedule in slg_batch_run
int32_t run_batch(slg_batch *bt, bool do_seeds, bool do_sweep) {
  slg_index *ix = bt->ix;
  cudaStream_t st = ix->stream;
  const bool prune = bt->exec != SLG_EXEC_BM25;
  const uint32_t Q = bt->Q, k = bt->k;
  const bool run_items = bt->can_items && !bt->want_stats && !(bt->big_k && (!ix->scan_kernels || (ix->strict_accumulate && bt->exec == SLG_EXEC_BM25)));
  // flat posting scan + column pass: the automatic choice; scan_kernels 0 keeps the sub-tile kernels (stream / items)
  const bool run_scan = run_items && ix->scan_kernels && bt->colq != nullptr && !(ix->strict_accumulate && !prune);
  if (bt->and_scan && !run_scan && run_items)
    return fail(ix, SLG_ERR_UNSUPPORTED, "an AND batch prepared for the posting scan cannot run on the sub-tile kernels (strict_accumulate)");
  const bool two_step = !(do_seeds && do_sweep);
  if (two_step && (ix->segs.size() != 1 || !run_items || (!prune && !run_scan)))
    return fail(ix, SLG_ERR_UNSUPPORTED, "the two-step run (first part, threshold exchange, rest) needs one segment per handle and the posting scan or the pruned items kernel");
  unsigned char *dp = bt->d_pack;
  size_t smem = 0;
  const bool run_scan_pre = bt->can_items && !bt->want_stats && ix->scan_kernels && bt->colq != nullptr && !(ix->strict_accumulate && !prune);
  const bool warp_path = bt->use_warp && !(bt->big_k && !run_scan_pre);  // k > 32 without the scan: the CTA-per-item kernel
  if (!warp_path) {
    int32_t rc = bt->has_plan ? select_smem(ix, bt->plan_docs, bt->cap, bt->matcher, &smem, bt->max_leaves)
                              : select_smem(ix, ix->tile_docs, bt->cap, bt->matcher, &smem);
    if (rc) return rc;
  }
  uint32_t per_sm = (uint32_t)std::max<size_t>(1, (ix->smem_optin + 1024) / (smem + 1024));
  per_sm = std::min(per_sm, 8u);
  if (ix->ctas_per_sm) per_sm = std::min(per_sm, ix->ctas_per_sm);
  if (do_seeds) {
    SLG_CUDA(ix, cudaEventRecord(ix->ev[0], st));
    SLG_CUDA(ix, cudaMemsetAsync(bt->stats, 0, (size_t)Q * 40 + 64, st));
    if (bt->has_cursor) {
      if (bt->n_cursor_segs != ix->segs.size()) return fail(ix, SLG_ERR_INVALID, "a segment was loaded after the batch with cursors was prepared");
      SLG_CUDA(ix, cudaMemsetAsync(bt->cursor_saw, 0, (size_t)Q * 4, st));
    }
  }
  uint32_t si = 0;
  for (auto &sp : ix->segs) {
    Segment *s = sp.get();
    BatchDev bd{};
    bd.ut_term = reinterpret_cast<const uint32_t *>(dp + bt->off_ut_term);
    bd.ut_rng = bt->ut_rng;
    bd.ut_tile_ub = bt->ut_tile_ub;
    bd.q_term_off = reinterpret_cast<const uint32_t *>(dp + bt->off_q_term_off);
    bd.qt_uterm = reinterpret_cast<const uint32_t *>(dp + bt->off_qt_uterm);
    bd.qt_weight = reinterpret_cast<const float *>(dp + bt->off_qt_weight);
    bd.qt_group = dp + bt->off_qt_group;
    bd.qt_flags = dp + bt->off_qt_flags;
    bd.q_order = reinterpret_cast<const uint32_t *>(dp + bt->off_q_order);
    bd.q_must = dp + bt->off_q_must;
    bd.q_not = dp + bt->off_q_not;
    bd.q_should = dp + bt->off_q_should;
    bd.q_min_should = dp + bt->off_q_min;
    bd.q_filter = reinterpret_cast<const int32_t *>(dp + bt->off_q_filter);
    bd.filter_bits = reinterpret_cast<const uint32_t *const *>(s->filter_ptrs.p);
    if (bt->has_plan) {
      bd.qt_leaf = dp + bt->off_qt_leaf;
      bd.q_leaves = dp + bt->off_q_leaves;
      bd.q_plan_off = reinterpret_cast<const uint32_t *>(dp + bt->off_q_plan_off);
      bd.plan_nodes = reinterpret_cast<const PlanNodeDev *>(dp + bt->off_plan_nodes);
    }
    bd.max_leaves = bt->max_leaves;
    if (bt->has_cursor) {
      bd.q_cursor = reinterpret_cast<const unsigned long long *>(dp + bt->off_cursor_bounds) + (size_t)si * Q;
      bd.q_saw = bt->cursor_saw;
    }
    bd.n_queries = Q;
    bd.n_uterms = bt->U;
    bd.k = k;
    bd.cap = bt->cap;
    const uint32_t plan_docs = bt->plan_docs;
    bd.tile_docs = plan_docs;
    bd.n_tiles = std::max(1u, (s->doc_count + plan_docs - 1) / plan_docs);
    bd.thr_key = bt->thr_key;
    bd.topk_count = bt->topk_count;
    bd.lock = bt->lock;
    bd.topk_keys = bt->topk_keys;
    bd.work_counter = bt->work_counter;
    bd.stats = bt->stats;
    bd.match_count = bd.stats + (size_t)Q * 4;
    // queries that name a filter need its bitmap on every segment
    if (!ix->filters.empty() && s->filter_bits.size() < ix->filters.size())
      return fail(ix, SLG_ERR_INVALID, "segment %u was loaded after its filters were compiled", s->ord);

    WarpBatchDev wb{};
    ItemsDev it{};
    const int warps = kThreads / 32;
    size_t wsmem = 0;
    int wgrid = 1;
    const bool score = bt->U && s->doc_count;
    if (bt->use_warp && score) {
      wb.qterms = bt->qterms;
      wb.qheads = bt->qheads;
      wb.rng = bd.ut_rng;
      wb.sub_ub = bd.ut_tile_ub;
      wb.scores = s->dev.post_score;
      wb.filter_bits = bd.filter_bits;
      wb.n_queries = Q;
      wb.k = k;
      wb.sub_docs = plan_docs;
      wb.q_leaves = bd.q_leaves;
      wb.q_plan_off = bd.q_plan_off;
      wb.plan_nodes = bd.plan_nodes;
      wb.max_leaves = bt->max_leaves;
      wb.n_sub = bd.n_tiles;
      wb.n_groups = (bd.n_tiles + kSubPerGroup - 1) / kSubPerGroup;
      wb.ms_frac = (float)ix->maxscore_pct / 100.0f;
      wb.thr_key = bd.thr_key;
      wb.topk_count = bd.topk_count;
      wb.lock = bd.lock;
      wb.topk_keys = bd.topk_keys;
      wb.work_counter = bd.work_counter;
      wb.stats = bd.stats;
      wb.match_count = bd.match_count;
      wb.q_cursor = bd.q_cursor;
      wb.q_saw = bd.q_saw;
      wb.pool_keys = run_scan ? bt->pool_keys : nullptr;
      wb.pool_count = bt->pool_count;
      wb.pool_lock = bt->pool_lock;
      wb.pool_cap = bt->pool_cap;
      wb.board = run_scan ? bt->board : nullptr;  // (the posting scan and its column pass read and push; the other kernels keep to themselves)
      for (uint32_t p = 0; p < kMaxBoardPeers; p++) wb.peer_board[p] = bt->peer_board[p];
      wb.n_peers = bt->n_board_peers;
      wb.epoch = bt->board_epoch;
      // (plan batches: the matcher form of the kernel unless the staged plain-OR form applies — size for the larger)
      wsmem = run_items ? (size_t)warps * warp_kernel_smem_per_warp(wb.sub_docs, false, true, 1)
                        : (size_t)warps * warp_kernel_smem_per_warp(wb.sub_docs, bt->matcher || (bt->has_plan && !bt->staged), prune,
                                                                    bt->has_plan ? bt->max_leaves : 1u);
      if (wsmem + 1024 > ix->smem_optin) return fail(ix, SLG_ERR_UNSUPPORTED, "sub_docs %u needs %zu B shared memory", ix->sub_docs, wsmem);
      uint32_t wper = (uint32_t)std::max<size_t>(1, (ix->smem_optin + 1024) / (wsmem + 1024));
      wper = std::min(wper, 3u);  // the kernels are compiled for at most 3 CTAs per SM (__launch_bounds__)
      if (ix->ctas_per_sm) wper = std::min(wper, ix->ctas_per_sm);
      wgrid = (int)std::min<uint64_t>((uint64_t)ix->n_sm * wper, ((uint64_t)wb.n_groups * wb.n_queries + warps - 1) / warps);
      it.items = nullptr;
      it.n_items = bt->n_items;
      it.done = bt->done;
      it.items_out = bt->items;
      it.n_items_out = bt->n_items;
      it.items_cap = bt->items_cap;
      it.counters = bt->item_counters;
    }

    if (do_seeds) {
      // ---- reset, plans and per-segment query tables ----
      const uint32_t n_reset = std::max(Q, (uint32_t)(bt->state_bytes / 4));
      slg_reset_state_kernel<<<(n_reset + 255) / 256, 256, 0, st>>>(bd.thr_key, Q, reinterpret_cast<uint32_t *>(bt->state),
                                                                    (uint32_t)(bt->state_bytes / 4));
      count_launch(ix);
      if (score && run_scan) {
        // no doc-range plan: the scan walks whole lists and looks terms up by binary search
        slg_build_qterms_kernel<<<(Q + 127) / 128, 128, 0, st>>>(s->dev, bd, bt->qterms, bt->qheads, bt->canonical, true);
        count_launch(ix);
        SLG_CUDA(ix, cudaGetLastError());
      } else if (score) {
        const uint64_t n2 = (uint64_t)bt->U * bd.n_tiles;
        // every unique term: short lists are walked once, long lists take one binary search per boundary.  The items
        // kernel never walks the postings of a column term, so their rows are not planned for it.
        slg_plan_walk_kernel<<<dim3(bt->U, 8), 256, 0, st>>>(s->dev, bd.ut_term, nullptr, bt->U, bd.tile_docs, bd.n_tiles, !run_items,
                                                            bd.ut_rng);
        count_launch(ix);
        if (bd.ut_tile_ub && (prune || run_items)) {
          if (s->dev.mb_max) {
            slg_items_bounds_kernel<<<(unsigned)((n2 + 255) / 256), 256, 0, st>>>(s->dev, bd.ut_term, bt->U, bd.ut_rng, bd.tile_docs, bd.n_tiles,
                                                                                 bd.ut_tile_ub);
          } else {
            slg_plan_bounds_kernel<<<(unsigned)((n2 + 255) / 256), 256, 0, st>>>(s->dev, bd, nullptr, bt->U);
          }
          count_launch(ix);
        }
        if (bt->use_warp) {
          slg_build_qterms_kernel<<<(Q + 127) / 128, 128, 0, st>>>(s->dev, bd, bt->qterms, bt->qheads, bt->canonical, run_items);
          count_launch(ix);
        }
        SLG_CUDA(ix, cudaGetLastError());
      }
      if (!(score && run_scan)) SLG_CUDA(ix, cudaEventRecord(ix->ev[2], st));
      if (score && run_items && prune && !run_scan) {
        // ---- seeds: every query's best items first ----
        SLG_CUDA(ix, cudaMemsetAsync(bt->done, 0, (size_t)wb.n_groups * Q, st));
        const int sgrid = (int)std::min<uint32_t>((uint32_t)ix->n_sm * 3u, (Q + warps - 1) / warps);
        SLG_CUDA(ix, launch_seed_items(s->dev, wb, it, wsmem, sgrid, st));
        count_launch(ix);
      }
    }
    const bool run_stream = run_items && !prune && bt->colq != nullptr && !run_scan && bt->plan_docs <= 2048;  // (posting numbers of a sub-tile fit 15 bits)
    if ((do_sweep || do_seeds) && score && run_scan) {
      ScanDev sc{};
      sc.ut_term = bd.ut_term;
      sc.ut_max = bt->ut_max;
      sc.pairs = bt->scan_pairs;
      sc.order = bt->scan_order;
      sc.n_pairs = bt->work_counter + 5;
      sc.n_items = bt->work_counter + 6;
      sc.item_start = bt->scan_item_start;
      sc.items = bt->scan_items;
      sc.items_cap = bt->scan_items_cap;
      sc.chunk = bt->scan_chunk;
      sc.must_mode = bt->and_scan ? 1u : 0u;
      sc.counter = bt->work_counter + 7;
      sc.counters = bt->item_counters;
      StreamDev sdv{};
      sdv.colq = bt->colq;
      sdv.n_colq = bt->work_counter + 3;
      sdv.ucol = bt->ucol;
      sdv.n_ucol = bt->work_counter + 4;
      sdv.col_slot = bt->col_slot;
      sdv.sparse_counter = bt->work_counter + 1;
      sdv.col_counter = bt->work_counter + 2;
      sdv.stage_cap = ix->stage_cap;
      sdv.strict = 0;
      sdv.counters = bt->item_counters;
      if (do_seeds) {
        if (prune && s->dev.term_ub) {
          slg_term_ub_gather_kernel<<<(bt->U + 255) / 256, 256, 0, st>>>(s->dev, sc, bt->U);
        } else {  // exhaustive: no index-time bound, the maxima are reduced from the batch's posting scores
          SLG_CUDA(ix, cudaMemsetAsync(bt->ut_max, 0, (size_t)bt->U * 4, st));
          slg_term_max_kernel<<<dim3((bt->U + 7) / 8, kMaxSlices), 256, 0, st>>>(s->dev, sc, bt->U);
        }
        slg_scan_pairs_kernel<<<(Q + 127) / 128, 128, 0, st>>>(s->dev, wb, sc, ix->dbg);
        slg_scan_order_kernel<<<1, 1024, 0, st>>>(wb, sc);
        if (bt->scan_items_cap) slg_scan_items_kernel<<<(bt->scan_items_cap + 255) / 256, 256, 0, st>>>(sc);
        for (int i = 0; i < 4; i++) count_launch(ix);
        SLG_CUDA(ix, cudaGetLastError());
        SLG_CUDA(ix, cudaEventRecord(ix->ev[2], st));  // (the scoring time of this path starts here)
      }
      // one launch over all items, or (sharded runs) the rarest items first, the threshold exchange, then the rest
      sc.two_rounds = (ix->dbg & 8u) ? 1u : 0u;
      sc.part_lo = do_seeds ? 0u : ix->scan_first_part;
      sc.part_hi = do_sweep ? 256u : ix->scan_first_part;
      SLG_CUDA(ix, launch_scan(prune, wb.pool_keys != nullptr, s->dev, wb, sc, ix->n_sm * 4, st));
      count_launch(ix);
      if (do_sweep && s->n_cols && !(ix->dbg & 4u) && !bt->and_scan) {  // (AND: every result holds the scanned term — there is nothing left for a column pass)
        slg_colgroups_kernel<<<1, 1024, 0, st>>>(s->dev, wb, sdv, s->n_cols, prune ? bt->ut_max : nullptr);
        count_launch(ix);
        SLG_CUDA(ix, cudaGetLastError());
        sdv.n_smax = std::min(s->n_cols, kColMaxSlots);
        const size_t fixed = column_smem(0, sdv.n_smax);
        const size_t reserve = 2048 + (size_t)kColWarps * 256 * 4;  // (+ the kernel's static shared memory)
        const size_t budget = ix->smem_optin > fixed + reserve ? ix->smem_optin - fixed - reserve : 0;
        sdv.col_resident = (uint32_t)std::min<size_t>(s->n_cols, budget / (2 * kColBlock * 4));
        const size_t csmem = column_smem(sdv.col_resident, sdv.n_smax);
        const uint32_t n_cblocks = (s->doc_count + kColBlock - 1) / kColBlock;
        if (prune) {
          // few queries keep an essential column term: one warp per (query, slice of the doc range), blocks skipped by col_tmax
          (void)csmem;
          (void)n_cblocks;
          SLG_CUDA(ix, launch_columns_pruned(wb.pool_keys != nullptr, s->dev, wb, sdv, (int)((Q * kColSlices + 7) / 8), st));
        } else {
          SLG_CUDA(ix, launch_score_columns(false, wb.pool_keys != nullptr, s->dev, wb, sdv, csmem, (int)std::min<uint32_t>((uint32_t)ix->n_sm, n_cblocks), st));
        }
        count_launch(ix);
      }
      if (do_sweep) ix->ctr.score_launches++;
    }
    if (do_sweep) {
      // ---- scoring ----
      if (score && run_scan) {
        // (launched above)
      } else if (score && run_stream) {
        // exhaustive: sparse pass (staged posting runs), then column pass (queries grouped by their first column)
        StreamDev sdv{};
        sdv.colq = bt->colq;
        sdv.n_colq = bt->work_counter + 3;
        sdv.ucol = bt->ucol;
        sdv.n_ucol = bt->work_counter + 4;
        sdv.col_slot = bt->col_slot;
        sdv.sparse_counter = bt->work_counter + 1;
        sdv.col_counter = bt->work_counter + 2;
        sdv.stage_cap = ix->stage_cap;
        sdv.strict = ix->strict_accumulate;
        sdv.counters = bt->item_counters;
        const size_t ssmem = (size_t)kSparseWarps * sparse_smem_per_warp(wb.sub_docs, sdv.stage_cap);
        if (ssmem + 1024 > ix->smem_optin) return fail(ix, SLG_ERR_UNSUPPORTED, "sub_docs %u with stage_cap %u needs %zu B shared memory", wb.sub_docs, sdv.stage_cap, ssmem);
        uint32_t sper = (uint32_t)std::max<size_t>(1, (ix->smem_optin + 1024) / (ssmem + 1024));
        sper = std::min(sper, 2048u / (kSparseWarps * 32u));
        if (ix->ctas_per_sm) sper = std::min(sper, ix->ctas_per_sm);
        const int sgrid = (int)std::min<uint64_t>((uint64_t)ix->n_sm * sper, ((uint64_t)wb.n_groups * Q + kSparseWarps - 1) / kSparseWarps);
        SLG_CUDA(ix, launch_score_sparse(s->dev, wb, sdv, ssmem, sgrid, st));
        count_launch(ix);
        if (s->n_cols) {
          slg_colgroups_kernel<<<1, 1024, 0, st>>>(s->dev, wb, sdv, s->n_cols, nullptr);
          count_launch(ix);
          SLG_CUDA(ix, cudaGetLastError());
          // one CTA per SM: as many columns of a block resident in shared memory (double buffered) as fit
          sdv.n_smax = std::min(s->n_cols, kColMaxSlots);
          const size_t fixed = column_smem(0, sdv.n_smax);
          const size_t reserve = 2048 + (size_t)kColWarps * 256 * 4;  // (+ the kernel's static shared memory)
        const size_t budget = ix->smem_optin > fixed + reserve ? ix->smem_optin - fixed - reserve : 0;
          sdv.col_resident = (uint32_t)std::min<size_t>(s->n_cols, budget / (2 * kColBlock * 4));
          const size_t csmem = column_smem(sdv.col_resident, sdv.n_smax);
          const uint32_t n_cblocks = (s->doc_count + kColBlock - 1) / kColBlock;
          SLG_CUDA(ix, launch_score_columns(false, wb.pool_keys != nullptr, s->dev, wb, sdv, csmem, (int)std::min<uint32_t>((uint32_t)ix->n_sm, n_cblocks), st));
          count_launch(ix);
        }
        ix->ctr.score_launches++;
      } else if (score && run_items) {
        if (prune) {
          const uint32_t total = wb.n_groups * Q;
          slg_filter_items_kernel<<<(total + 255) / 256, 256, 0, st>>>(wb, it);
          count_launch(ix);
          SLG_CUDA(ix, cudaGetLastError());
          it.items = bt->items;
        }
        SLG_CUDA(ix, launch_score_items(prune, s->dev, wb, it, wsmem, wgrid, st));
        count_launch(ix);
        ix->ctr.score_launches++;
      } else if (score && warp_path) {
        SLG_CUDA(ix, launch_score_warp(bt->matcher, prune, bt->want_stats, bt->staged, bt->has_plan, s->dev, wb, wsmem, wgrid, st));
        count_launch(ix);
        ix->ctr.score_launches++;
      } else if (score) {
        int grid = (int)std::min<uint64_t>((uint64_t)ix->n_sm * per_sm, (uint64_t)bd.n_tiles * Q);
        SLG_CUDA(ix, launch_score_tiles(bt->matcher, prune, bt->want_stats, bt->has_plan, s->dev, bd, smem, grid, st));
        count_launch(ix);
        ix->ctr.score_launches++;
      }
      SLG_CUDA(ix, cudaEventRecord(ix->ev[3], st));
      HitDev *hits = reinterpret_cast<HitDev *>(bt->results + (size_t)si * bt->result_stride);
      uint32_t *cnts = reinterpret_cast<uint32_t *>(bt->results + (size_t)si * bt->result_stride + (size_t)Q * k * sizeof(HitDev));
      size_t fsmem = (size_t)(1u << (32 - __builtin_clz(std::max(k, 2u) - 1))) * 8;
      if (run_scan && bt->pool_keys && score) {
        const size_t psmem = (size_t)bt->pool_cap * 2 * 8;
        SLG_CUDA(ix, cudaFuncSetAttribute(slg_finalize_pools_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem));
        slg_finalize_pools_kernel<<<Q, kThreads, psmem, st>>>(bt->pool_keys, bt->pool_count, bt->pool_cap, k, s->ord, hits, cnts);
      } else {
        slg_finalize_kernel<<<Q, kThreads, fsmem, st>>>(bd, s->ord, hits, cnts);
      }
      count_launch(ix);
      SLG_CUDA(ix, cudaGetLastError());
      if (ix->segs.size() > 1 && score) {
        // per-segment score time must be read before the events are reused
        SLG_CUDA(ix, cudaEventSynchronize(ix->ev[3]));
        float ms = 0;
        SLG_CUDA(ix, cudaEventElapsedTime(&ms, ix->ev[2], ix->ev[3]));
        ix->ctr.score_ms_total += ms;
        ix->ctr.last_score_ms = ms;
      }
    }
    si++;
  }
  if (do_sweep) {
    bt->n_segs_run = si;
    bt->reranked = false;
    if (si > 1) {
      size_t msmem = (size_t)si * k * sizeof(HitDev);
      if (msmem > ix->smem_optin || si > kMaxMergeLists) return fail(ix, SLG_ERR_UNSUPPORTED, "merge of %u segments x k=%u does not fit shared memory", si, k);
      SLG_CUDA(ix, cudaFuncSetAttribute(slg_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem));
      unsigned char *mo = bt->results + (size_t)si * bt->result_stride;
      slg_merge_kernel<<<Q, kThreads, msmem, st>>>(reinterpret_cast<const uint32_t *>(bt->results), si, Q, k,
                                                   (uint32_t)(bt->result_stride / 4), reinterpret_cast<HitDev *>(mo),
                                                   reinterpret_cast<uint32_t *>(mo + (size_t)Q * k * sizeof(HitDev)));
      count_launch(ix);
      SLG_CUDA(ix, cudaGetLastError());
    }
    SLG_CUDA(ix, cudaEventRecord(ix->ev[1], st));
    ix->ctr.last_posting_count = bt->posting_count;
  }
  return SLG_OK;
}

int32_t finish_timing(slg_batch *bt) {
  slg_index *ix = bt->ix;
  SLG_CUDA(ix, cudaStreamSynchronize(ix->stream));
  float ms = 0;
  SLG_CUDA(ix, cudaEventElapsedTime(&ms, ix->ev[0], ix->ev[1]));
  ix->ctr.last_batch_ms = ms;
  if (ix->segs.size() == 1 && bt->U) {
    SLG_CUDA(ix, cudaEventElapsedTime(&ms, ix->ev[2], ix->ev[3]));
    ix->ctr.score_ms_total += ms;
    ix->ctr.last_score_ms = ms;
  }
  return SLG_OK;
}

}  // namespace

extern "C" {

int32_t slg_batch_run(slg_batch_t *bt, int32_t sync) {
  if (!bt) return SLG_ERR_INVALID;
  slg_index *ix = bt->ix;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  int32_t rc = run_batch(bt, true, true);
  if (rc) return rc;
  bt->seeds_done = false;
  return sync ? finish_timing(bt) : SLG_OK;
}

int32_t slg_batch_run_seeds(slg_batch_t *bt) {
  if (!bt) return SLG_ERR_INVALID;
  slg_index *ix = bt->ix;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  int32_t rc = run_batch(bt, true, false);
  if (rc) return rc;
  bt->seeds_done = true;
  return SLG_OK;
}

int32_t slg_batch_threshold_keys(slg_batch_t *bt, void **dev_keys) {
  if (!bt || !dev_keys) return SLG_ERR_INVALID;
  *dev_keys = bt->thr_key;
  return SLG_OK;
}

int32_t slg_batch_import_thresholds(slg_batch_t *bt, const void *dev_keys) {
  if (!bt || !dev_keys) return SLG_ERR_INVALID;
  slg_index *ix = bt->ix;
  if (!bt->seeds_done) return fail(ix, SLG_ERR_INVALID, "thresholds are imported between slg_batch_run_seeds and slg_batch_run_sweep");
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  slg_import_thresholds_kernel<<<(bt->Q + 255) / 256, 256, 0, ix->stream>>>(bt->thr_key, static_cast<const unsigned long long *>(dev_keys), bt->Q);
  count_launch(ix);
  SLG_CUDA(ix, cudaGetLastError());
  return SLG_OK;
}

int32_t slg_batch_run_sweep(slg_batch_t *bt, int32_t sync) {
  if (!bt) return SLG_ERR_INVALID;
  slg_index *ix = bt->ix;
  if (!bt->seeds_done) return fail(ix, SLG_ERR_INVALID, "slg_batch_run_sweep follows slg_batch_run_seeds");
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  int32_t rc = run_batch(bt, false, true);
  if (rc) return rc;
  bt->seeds_done = false;
  return sync ? finish_timing(bt) : SLG_OK;
}

int32_t slg_batch_set_threshold_board(slg_batch_t *bt, void *local_board, void *const *peer_boards, uint32_t n_peers, uint32_t epoch) {
  if (!bt) return SLG_ERR_INVALID;
  slg_index *ix = bt->ix;
  if (!local_board) {  // switch the exchange off
    bt->board = nullptr;
    bt->n_board_peers = 0;
    return SLG_OK;
  }
  if (n_peers > kMaxBoardPeers || (n_peers && !peer_boards)) return fail(ix, SLG_ERR_INVALID, "a threshold board has at most %u peers", kMaxBoardPeers);
  if (epoch == 0) return fail(ix, SLG_ERR_INVALID, "board epochs start at 1 and rise with every batch");
  if (ix->segs.size() != 1) return fail(ix, SLG_ERR_UNSUPPORTED, "the threshold board needs one segment per handle (shard == segment)");
  bt->board = static_cast<unsigned long long *>(local_board);
  for (uint32_t p = 0; p < kMaxBoardPeers; p++) bt->peer_board[p] = p < n_peers ? static_cast<unsigned long long *>(peer_boards[p]) : nullptr;
  bt->n_board_peers = n_peers;
  bt->board_epoch = epoch;
  return SLG_OK;
}

int32_t slg_batch_enable_stats(slg_batch_t *bt, int32_t on) {
  if (!bt) return SLG_ERR_INVALID;
  bt->want_stats = on != 0;
  return SLG_OK;
}

// the (hits, counts) block of the last run: merged over the handle's segments when there are several
static unsigned char *result_block(slg_batch *bt) {
  return bt->results + (bt->n_segs_run > 1 ? (size_t)bt->n_segs_run * bt->result_stride : 0);
}

int32_t slg_batch_device_results(slg_batch_t *bt, void **dev_hits, void **dev_counts) {
  if (!bt || !dev_hits || !dev_counts) return SLG_ERR_INVALID;
  unsigned char *r = result_block(bt);
  *dev_hits = r;
  *dev_counts = r + (size_t)bt->Q * bt->k * sizeof(HitDev);
  return SLG_OK;
}

int32_t slg_batch_packed_results(slg_batch_t *bt, void **dev_block, uint64_t *n_bytes) {
  if (!bt || !dev_block || !n_bytes) return SLG_ERR_INVALID;
  *dev_block = result_block(bt);
  *n_bytes = (uint64_t)bt->Q * bt->k * sizeof(HitDev) + (uint64_t)bt->Q * 4 + (bt->reranked ? (uint64_t)bt->Q * bt->k * 4 : 0);
  return SLG_OK;
}

int32_t slg_batch_fetch(slg_batch_t *bt, slg_hit_t *out_hits, uint32_t *out_counts, slg_stats_t *out_stats) {
  if (!bt || !out_hits || !out_counts) return SLG_ERR_INVALID;
  slg_index *ix = bt->ix;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  cudaStream_t st = ix->stream;
  static_assert(sizeof(slg_hit_t) == sizeof(HitDev), "hit layout");
  const size_t hb = (size_t)bt->Q * bt->k * sizeof(slg_hit_t), cb = (size_t)bt->Q * 4, sb = (size_t)bt->Q * 40 + 64;
  unsigned char *pin = static_cast<unsigned char *>(bt->pinned) + bt->pinned_result_off;
  SLG_CUDA(ix, cudaMemcpyAsync(pin, result_block(bt), hb + cb, cudaMemcpyDeviceToHost, st));
  SLG_CUDA(ix, cudaMemcpyAsync(pin + bt->result_stride, bt->stats, sb, cudaMemcpyDeviceToHost, st));
  SLG_CUDA(ix, cudaStreamSynchronize(st));
  ix->ctr.last_d2h_bytes = hb + cb + sb;
  std::memcpy(out_hits, pin, hb);
  std::memcpy(out_counts, pin + hb, cb);
  const unsigned long long *sv = reinterpret_cast<const unsigned long long *>(pin + bt->result_stride);
  const unsigned long long *ic = sv + (size_t)bt->Q * 5;
  ix->ctr.last_postings_scattered = ic[0];
  ix->ctr.last_subtiles_skipped = ic[1];
  ix->ctr.last_column_blocks_streamed = ic[2];
  ix->ctr.last_items = ic[3];
  ix->ctr.last_postings_verified = ic[4];
  ix->ctr.last_items_dropped = ic[5];
  // SLG_SCAN_TRACE=1: where the flat scan's verification looked up the other sparse terms of a query
  if (getenv("SLG_SCAN_TRACE"))
    fprintf(stderr, "[slg scan] verified %llu, sparse look-ups answered by a presence bitmap %llu, by lower_bound_interp %llu\n", ic[4], ic[6], ic[7]);
  if (out_stats) {
    for (uint32_t q = 0; q < bt->Q; q++) {
      out_stats[q].scored_docs = sv[q * 4 + 0];
      out_stats[q].postings_advanced = sv[q * 4 + 1];
      out_stats[q].blocks_skipped = sv[q * 4 + 2];
      out_stats[q].candidates_examined = sv[q * 4 + 3];
      out_stats[q].total_matches = sv[(size_t)bt->Q * 4 + q];
    }
  }
  return SLG_OK;
}

int32_t slg_batch_copy_results_device(slg_batch_t *bt, void *dst_hits, void *dst_counts) {
  if (!bt || !dst_hits || !dst_counts) return SLG_ERR_INVALID;
  slg_index *ix = bt->ix;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  void *dh, *dc;
  slg_batch_device_results(bt, &dh, &dc);
  SLG_CUDA(ix, cudaMemcpyAsync(dst_hits, dh, (size_t)bt->Q * bt->k * sizeof(HitDev), cudaMemcpyDeviceToDevice, ix->stream));
  SLG_CUDA(ix, cudaMemcpyAsync(dst_counts, dc, (size_t)bt->Q * 4, cudaMemcpyDeviceToDevice, ix->stream));
  return SLG_OK;
}

int32_t slg_batch_cursor_seen(slg_batch_t *bt, uint8_t *out_seen) {
  if (!bt || !out_seen) return SLG_ERR_INVALID;
  slg_index *ix = bt->ix;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  for (uint32_t q = 0; q < bt->Q; q++) out_seen[q] = 1;  // no cursor: saw_cursor starts true (api/reader.rs:2663)
  if (!bt->has_cursor) return SLG_OK;
  std::vector<uint32_t> saw(bt->Q);
  SLG_CUDA(ix, cudaMemcpyAsync(saw.data(), bt->cursor_saw, (size_t)bt->Q * 4, cudaMemcpyDeviceToHost, ix->stream));
  SLG_CUDA(ix, cudaStreamSynchronize(ix->stream));
  for (uint32_t q = 0; q < bt->Q; q++)
    if (bt->h_has_cursor[q]) out_seen[q] = saw[q] ? 1 : 0;
  return SLG_OK;
}

int32_t slg_batch_free(slg_batch_t *bt) {
  if (!bt) return SLG_OK;
  cudaSetDevice(bt->ix->device);
  {
    PoolScope pool_scope(bt->ix->stream);  // (the slab remembers its stream; freeing is stream-ordered, no host wait)
    delete bt;
  }
  return SLG_OK;
}

int32_t slg_search_batch(slg_index_t *ix, const slg_query_t *queries, uint32_t n_queries, uint32_t k, slg_exec_t exec,
                         uint32_t bmw_block_size, slg_hit_t *out_hits, uint32_t *out_counts, slg_stats_t *out_stats) {
  if (!ix) return SLG_ERR_INVALID;
  if (!out_hits || !out_counts) return fail(ix, SLG_ERR_INVALID, "output buffers are NULL");
  slg_batch_t *bt = nullptr;
  int32_t rc = slg_batch_prepare(ix, queries, n_queries, k, exec, bmw_block_size, &bt);
  if (rc) return rc;
  bt->want_stats = out_stats != nullptr;
  rc = slg_batch_run(bt, 0);
  if (rc == SLG_OK) rc = slg_batch_fetch(bt, out_hits, out_counts, out_stats);
  if (rc == SLG_OK && ix->segs.size() == 1 && bt->U) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ix->ev[2], ix->ev[3]) == cudaSuccess) {
      ix->ctr.score_ms_total += ms;
      ix->ctr.last_score_ms = ms;
    }
    if (cudaEventElapsedTime(&ms, ix->ev[0], ix->ev[1]) == cudaSuccess) ix->ctr.last_batch_ms = ms;
  }
  slg_batch_free(bt);
  return rc;
}

// gathered: n_shards blocks of shard_stride bytes, each [n_queries][k] hits then [n_queries] counts (then, hybrid form,
// [n_queries][k] vector scores) — the layout of slg_batch_packed_results; shard_stride 0 = tightly packed
static int32_t merge_packed(slg_index_t *ix, const void *dev_gathered, uint64_t shard_stride, uint32_t n_shards, uint32_t n_queries, uint32_t k,
                            slg_hit_t *out_hits, uint32_t *out_counts, bool hybrid, float *out_vs) {
  if (!ix || !dev_gathered || !out_hits || !out_counts || !n_shards || !n_queries || !k) return SLG_ERR_INVALID;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  cudaStream_t st = ix->stream;
  const size_t hb = (size_t)n_queries * k * sizeof(HitDev), cb = (size_t)n_queries * 4, vb = hybrid ? (size_t)n_queries * k * 4 : 0;
  if (shard_stride == 0) shard_stride = hb + cb + vb;
  if (shard_stride % 4 || shard_stride < hb + cb + vb)
    return fail(ix, SLG_ERR_INVALID, "shard stride %llu does not hold %zu bytes", (unsigned long long)shard_stride, hb + cb + vb);
  size_t msmem = (size_t)n_shards * k * sizeof(HitDev);
  if (msmem > ix->smem_optin || n_shards > kMaxMergeLists) return fail(ix, SLG_ERR_UNSUPPORTED, "merge of %u shards x k=%u does not fit shared memory", n_shards, k);
  PoolScope pool_scope(st);  // per-call buffers from the stream-ordered pool
  DevBuf ob;
  SLG_CUDA(ix, ob.alloc(hb + cb + vb));
  if (ix->merge_pinned_bytes < hb + cb + vb) {  // the merge has its own staging buffer: a prepared batch may hold the handle's other one
    if (ix->merge_pinned) cudaFreeHost(ix->merge_pinned);
    ix->merge_pinned = nullptr;
    ix->merge_pinned_bytes = 0;
    SLG_CUDA(ix, cudaMallocHost(&ix->merge_pinned, hb + cb + vb));
    ix->merge_pinned_bytes = hb + cb + vb;
  }
  SLG_CUDA(ix, cudaFuncSetAttribute(slg_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem));
  slg_merge_kernel<<<n_queries, kThreads, msmem, st>>>(static_cast<const uint32_t *>(dev_gathered), n_shards, n_queries, k,
                                                       (uint32_t)(shard_stride / 4), ob.as<HitDev>(),
                                                       reinterpret_cast<uint32_t *>(ob.as<unsigned char>() + hb), hybrid ? (uint32_t)((hb + cb) / 4) : 0u,
                                                       hybrid ? reinterpret_cast<float *>(ob.as<unsigned char>() + hb + cb) : nullptr);
  count_launch(ix);
  SLG_CUDA(ix, cudaGetLastError());
  const size_t out_bytes = hb + cb + (out_vs ? vb : 0);
  SLG_CUDA(ix, cudaMemcpyAsync(ix->merge_pinned, ob.p, out_bytes, cudaMemcpyDeviceToHost, st));
  SLG_CUDA(ix, cudaStreamSynchronize(st));
  std::memcpy(out_hits, ix->merge_pinned, hb);
  std::memcpy(out_counts, static_cast<unsigned char *>(ix->merge_pinned) + hb, cb);
  if (out_vs && vb) std::memcpy(out_vs, static_cast<unsigned char *>(ix->merge_pinned) + hb + cb, vb);
  ix->ctr.last_d2h_bytes = out_bytes;
  return SLG_OK;
}

int32_t slg_merge_gathered_packed(slg_index_t *ix, const void *dev_gathered, uint64_t shard_stride, uint32_t n_shards, uint32_t n_queries,
                                  uint32_t k, slg_hit_t *out_hits, uint32_t *out_counts) {
  return merge_packed(ix, dev_gathered, shard_stride, n_shards, n_queries, k, out_hits, out_counts, false, nullptr);
}

int32_t slg_merge_gathered_hybrid(slg_index_t *ix, const void *dev_gathered, uint64_t shard_stride, uint32_t n_shards, uint32_t n_queries,
                                  uint32_t k, slg_hit_t *out_hits, uint32_t *out_counts, float *out_vector_scores) {
  return merge_packed(ix, dev_gathered, shard_stride, n_shards, n_queries, k, out_hits, out_counts, true, out_vector_scores);
}

int32_t slg_merge_gathered(slg_index_t *ix, const void *dev_hits, const void *dev_counts, uint32_t n_shards, uint32_t n_queries,
                           uint32_t k, slg_hit_t *out_hits, uint32_t *out_counts) {
  if (!ix || !dev_hits || !dev_counts || !out_hits || !out_counts || !n_shards || !n_queries || !k) return SLG_ERR_INVALID;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  cudaStream_t st = ix->stream;
  // separate hit / count arrays: repack into the block layout, then the packed merge
  const size_t hb = (size_t)n_queries * k * sizeof(HitDev), cb = (size_t)n_queries * 4;
  DevBuf tmp;
  {
    PoolScope pool_scope(st);
    SLG_CUDA(ix, tmp.alloc((hb + cb) * n_shards));
  }
  for (uint32_t r = 0; r < n_shards; r++) {
    unsigned char *blk = tmp.as<unsigned char>() + (size_t)r * (hb + cb);
    SLG_CUDA(ix, cudaMemcpyAsync(blk, static_cast<const unsigned char *>(dev_hits) + (size_t)r * hb, hb, cudaMemcpyDeviceToDevice, st));
    SLG_CUDA(ix, cudaMemcpyAsync(blk + hb, static_cast<const unsigned char *>(dev_counts) + (size_t)r * cb, cb, cudaMemcpyDeviceToDevice, st));
  }
  return slg_merge_gathered_packed(ix, tmp.p, 0, n_shards, n_queries, k, out_hits, out_counts);
}

}  // extern "C"
