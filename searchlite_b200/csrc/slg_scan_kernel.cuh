// slg_scan_kernel.cuh — K2/K3/K5, flat posting scan: the automatic choice for plain OR queries with k <= 32 and <= 8 terms
// per query on segments with resident scores (the shape of BASELINE.json configs[1]), exhaustive and pruned.
//
// brute_force (query/wand.rs:459-566) sums every posting into its doc and offers every touched doc to push_top_k; wand_loop
// (:659-903) walks the lists document-at-a-time and skips what cannot beat the k-th score.  For small k both produce a top k
// that almost no doc enters, so this kernel never builds per-doc accumulators.  A term WITHOUT a dense column is scanned flat:
//
//   work item  = (query, term, chunk of kScanChunk postings), handed out from a global counter, RAREST TERMS FIRST: the
//                docs that end up in a query's top k nearly always hold its rarest term, so every query's k-th score is close
//                to final before its long lists are streamed
//   scan       = the resident unit-weight scores of the chunk, 128-bit loads, 128 postings per warp step.  Terms have a
//                priority (larger bound first) and a doc is the business of its highest-priority holder, so a posting is
//                looked at further only if  contribution + (largest contribution of every LOWER-priority term of the
//                query)  can reach the query's running k-th score.  Doc ids are not even read for the rest
//   verify     = the doc of such a posting gets its EXACT score: every term of the query in slot (= declared) order — the
//                posting's own contribution, the other sparse terms by binary search in their lists, the column terms by one
//                4-byte gather — the sum brute_force computes for that doc, then accept (api/reader.rs:3009-3036) and the
//                warp's candidate buffer.  A doc held by several scanned lists is offered by the posting of its
//                highest-priority list; should two passes still offer the same doc, equal keys collapse in the merge
//
// Exhaustive execution (bm25): every posting of every sparse term is read and compared; the "largest contribution of the other
// terms" comes from slg_term_max_kernel, a reduction over the batch's own posting scores at run time — no index-time bound is
// consulted.  Docs held by no sparse list are the column pass's (slg_score_columns_kernel), which runs afterwards.
// Pruned execution (wand / bmw): MaxScore over whole lists.  With the terms ordered by their bound, the longest prefix of
// smallest bounds whose sum stays below the k-th score is non-essential: a doc holding only such terms cannot enter the top k,
// so their items are dropped when they come up (the k-th score only rises, so the set only grows); every doc that matters
// holds an essential term, is met in that term's scan and verified exactly as above.  Results are byte-identical to bm25.
//
// Float contract (include/searchlite_gpu.h): slot order = the query's terms WITHOUT a column first, then those WITH one,
// each group in query order (slg_build_qterms_kernel); verify() adds in slot order starting from +0.
#pragma once
#include "slg_stream_kernel.cuh"

namespace slg {

constexpr uint32_t kScanChunk = 4096;  // postings per scan item (default of the scan_chunk option; a multiple of 256)
constexpr int kScanWarps = 8;
constexpr uint32_t kScanQueue = 512;  // ring: a step queues at most 256 candidates on top of a remainder below 32

struct __align__(16) ScanPair {  // one scanned (query, sparse term): 48 B
  uint64_t base;      // first padded posting index of the term
  uint32_t df;
  uint32_t qslot_t;   // qslot << 3 | slot
  uint32_t qi;
  float w;
  float others;       // bounds (weight applied) of the query's column terms and of its lower-priority sparse terms: what a doc first met here can gain
  float ne_prefix;    // sum of the bounds of the terms with a bound <= this term's (this term included): the MaxScore test
  int32_t filter;
  uint32_t first_item;
  uint32_t pad[2];
};

struct ScanDev {
  const uint32_t *ut_term;   // [U] unique terms of the batch
  float *ut_max;             // [U] largest unit-weight contribution of each (slg_term_max_kernel)
  ScanPair *pairs;           // [Q * 8] indexed by qslot * 8 + slot; df == 0: not scanned
  uint32_t *order;           // [Q * 8] pair indices, rarest first
  uint32_t *n_pairs;         // device counters: scanned pairs, items
  uint32_t *n_items;
  uint32_t *item_start;      // [n_pairs + 1] first item of every ordered pair
  uint32_t *items;           // [items_cap] ordered-pair index of every item
  uint32_t items_cap;
  uint32_t *counter;         // work counters: [0] first phase, [1] second phase
  uint32_t chunk;            // postings per item
  uint32_t must_mode;        // AND batches: every term of a query must hold the doc; only the rarest list is scanned
  uint32_t two_rounds;       // verification asks the lower-priority lists first, the higher-priority ones only for the survivors
  uint32_t part_lo, part_hi; // this launch scans items [n_items * part_lo / 256, n_items * part_hi / 256): 0..256 = all.  Sharded
                             // runs scan the rarest items first, exchange the per-query k-th keys, then scan the rest
  unsigned long long *counters;  // [8]: 0 postings scanned, 3 items scanned, 4 postings verified, 5 items dropped by MaxScore,
                                 // sparse look-ups of the verification: 6 answered by a presence bitmap, 7 by lower_bound_interp
};

// largest unit-weight contribution of every unique term of the batch: a reduction over the term's resident scores.
// grid (ceil(U / 8), kMaxSlices): warp (u, slice) reduces one slice of the list and folds it in with atomicMax (scores are
// positive floats: their bit patterns order like the values).  ut_max must be zero on entry.
constexpr uint32_t kMaxSlices = 32;
static __global__ void __launch_bounds__(256) slg_term_max_kernel(SegmentDev seg, ScanDev sc, uint32_t n_uterms) {
  const uint32_t u = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (u >= n_uterms) return;
  const uint32_t term = sc.ut_term ? sc.ut_term[u] : u;  // (no list of terms: every term of the segment, at load)
  if (term >= seg.n_terms) return;
  const uint32_t df = seg.term_df[term];
  const uint32_t quads = (df + 3) >> 2;  // (the padding of a list is zero: whole 16-byte pieces up to the 32-posting boundary are safe to read)
  const uint32_t per = (quads + gridDim.y - 1) / gridDim.y;
  const uint32_t q0 = blockIdx.y * per, q1 = min(quads, q0 + per);
  if (q0 >= q1) return;
  const float4 *p = reinterpret_cast<const float4 *>(seg.post_score + seg.term_start[term]);
  uint32_t m = 0u;
  for (uint32_t i = q0 + lane; i < q1; i += 32) {
    const float4 v = __ldg(p + i);
    m = max(m, max(max(__float_as_uint(v.x), __float_as_uint(v.y)), max(__float_as_uint(v.z), __float_as_uint(v.w))));
  }
  m = __reduce_max_sync(0xFFFFFFFFu, m);
  if (lane == 0 && m) atomicMax(reinterpret_cast<uint32_t *>(sc.ut_max) + u, m);
}

// pruned executions: the same maxima were reduced once at load for every term (seg.term_ub)
static __global__ void slg_term_ub_gather_kernel(SegmentDev seg, ScanDev sc, uint32_t n_uterms) {
  const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= n_uterms) return;
  const uint32_t term = sc.ut_term[u];
  sc.ut_max[u] = term < seg.n_terms ? seg.term_ub[term] : 0.0f;
}

// pruned executions: the column terms of the few queries that still have an essential one.  Warp per (query, slice of
// the doc range): 32 blocks of 512 docs at a time, lane = block: the sum of the columns' exact block maxima (seg.col_tmax,
// slot order) + extra below the k-th score means no doc of the block can enter the top k and the block is not read; the
// others are summed per doc (16 docs per lane, slot order) and the docs that can still qualify are verified exactly.
constexpr uint32_t kColSlices = 64;
// POOLS: k > kWarpMaxK (candidate pools + radix select); compiled out otherwise so that the common small-k kernels stay lean
template <int POOLS>
__global__ void __launch_bounds__(256) slg_columns_pruned_kernel(SegmentDev seg, WarpBatchDev wb, StreamDev sd) {
  __shared__ __align__(16) unsigned long long s_cand[8][kWarpCand];
  __shared__ uint32_t s_hist[8][POOLS ? 256 : 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t n_colq = *sd.n_colq;
  const uint32_t wid = blockIdx.x * 8 + warp;
  const uint32_t qidx = wid / kColSlices, slice = wid % kColSlices;
  if (qidx >= n_colq) return;
  const ColQ cq = sd.colq[qidx];
  const QTerm *qts = wb.qterms + (uint64_t)cq.qslot * kWarpMaxTerms;
  const uint32_t nt = (uint32_t)cq.nsp + cq.ncol;
  const uint32_t n_blocks = (seg.doc_count + 511u) >> 9;
  const uint32_t per = (n_blocks + kColSlices - 1) / kColSlices;
  const uint32_t b0 = slice * per, b1 = min(n_blocks, b0 + per);
  WarpCand wc;
  wc.begin(s_cand[warp], load_threshold(wb, cq.qi), wb.k, lane, 1u, POOLS ? s_hist[warp] : nullptr);
  auto cut_of = [&]() {
    if (wc.thr == kThrInit) return 0u;
    const float cf = __uint_as_float((uint32_t)(wc.thr >> 32)) * 0.99998f - cq.extra * 1.00002f;
    return cf > 0.0f ? __float_as_uint(cf) : 0u;
  };
  for (uint32_t bb = b0; bb < b1; bb += 32) {
    const uint32_t blk = bb + lane;
    float bound = 0.0f;
    if (blk < b1)
      for (uint32_t i = 0; i < cq.ncol; i++) {
        const QTerm &q = qts[cq.nsp + i];
        bound = __fadd_rn(bound, __fmul_rn(__ldg(seg.col_tmax + (uint64_t)q.term * seg.tmax_stride + blk), q.weight));
      }
    uint32_t open = __ballot_sync(0xFFFFFFFFu, blk < b1 && bound != 0.0f && __float_as_uint(bound) >= cut_of());
    while (open) {
      const uint32_t d0 = (bb + (__ffs(open) - 1)) << 9;
      open &= open - 1;
      float4 v[4];
#pragma unroll
      for (int x = 0; x < 4; x++) v[x] = make_float4(0, 0, 0, 0);
      for (uint32_t i = 0; i < cq.ncol; i++) {
        const QTerm &q = qts[cq.nsp + i];
        const float4 *p = reinterpret_cast<const float4 *>(seg.cols + q.sc_base + d0) + lane;
        const float w = q.weight;
#pragma unroll
        for (int x = 0; x < 4; x++) {
          const float4 c = __ldg(p + x * 32);
          v[x].x = __fadd_rn(v[x].x, __fmul_rn(c.x, w));
          v[x].y = __fadd_rn(v[x].y, __fmul_rn(c.y, w));
          v[x].z = __fadd_rn(v[x].z, __fmul_rn(c.z, w));
          v[x].w = __fadd_rn(v[x].w, __fmul_rn(c.w, w));
        }
      }
      uint32_t cut = cut_of();
      uint32_t todo = 0u;
#pragma unroll
      for (int x = 0; x < 4; x++) {
        const uint32_t bx[4] = {__float_as_uint(v[x].x), __float_as_uint(v[x].y), __float_as_uint(v[x].z), __float_as_uint(v[x].w)};
#pragma unroll
        for (int e = 0; e < 4; e++)
          if (bx[e] >= cut && bx[e] != 0u && d0 + x * 128 + lane * 4 + e < seg.doc_count) todo |= 1u << (x * 4 + e);
      }
      while (__any_sync(0xFFFFFFFFu, todo != 0u)) {
        const uint32_t el = todo ? __ffs(todo) - 1 : 0u;
        const bool had = todo != 0u;
        todo &= todo - 1u;
        uint32_t bits = 0u;
#pragma unroll
        for (int x = 0; x < 4; x++) {
          if (el == (uint32_t)x * 4 + 0) bits = __float_as_uint(v[x].x);
          if (el == (uint32_t)x * 4 + 1) bits = __float_as_uint(v[x].y);
          if (el == (uint32_t)x * 4 + 2) bits = __float_as_uint(v[x].z);
          if (el == (uint32_t)x * 4 + 3) bits = __float_as_uint(v[x].w);
        }
        const uint32_t doc = d0 + (el >> 2) * 128 + lane * 4 + (el & 3u);
        cut = cut_of();
        const bool pass = had && bits >= cut;
        if (!__any_sync(0xFFFFFFFFu, pass)) continue;
        float s = __uint_as_float(bits);
        if (cq.nsp) {
          uint32_t holders = 0u;
          s = verify_doc(seg, wb, qts, nt, pass, doc, holders);  // (a sparse list the scan dropped may hold the doc)
        }
        wc.offer(seg, wb, cq.qi, cq.filter, pass, doc, s);
      }
    }
  }
  wc.merge(wb, cq.qi);
}

// per query slot: the scanned pairs with their bounds.  Thread per query.
static __global__ void __launch_bounds__(128) slg_scan_pairs_kernel(SegmentDev seg, WarpBatchDev wb, ScanDev sc, uint32_t dbg) {
  const uint32_t qslot = blockIdx.x * blockDim.x + threadIdx.x;
  if (qslot >= wb.n_queries) return;
  const QHead h = wb.qheads[qslot];
  float ub[kWarpMaxTerms];
  bool is_col[kWarpMaxTerms];
  for (uint32_t t = 0; t < kWarpMaxTerms; t++) {
    ub[t] = 0.0f;
    is_col[t] = false;
    if (t < h.nt) {
      const QTerm &q = wb.qterms[(uint64_t)qslot * kWarpMaxTerms + t];
      if (q.flags & 1u) ub[t] = __fmul_rn(sc.ut_max[q.uterm], q.weight);
      is_col[t] = (q.flags & 4u) != 0u;
    }
  }
  // AND batches: the driver is the scored term with the fewest postings; a term the segment lacks means no doc can match
  uint32_t driver = 0xFFFFFFFFu;
  float total_ub = 0.0f;
  if (sc.must_mode) {
    uint32_t best_df = 0xFFFFFFFFu;
    bool possible = h.nt > 0;
    for (uint32_t t = 0; t < h.nt && t < kWarpMaxTerms; t++) {
      const QTerm &q = wb.qterms[(uint64_t)qslot * kWarpMaxTerms + t];
      const uint32_t term = sc.ut_term[q.uterm];  // (q.term of a column term is its column)
      const uint32_t df = (q.flags & 1u) && term < seg.n_terms ? seg.term_df[term] : 0u;
      if (df == 0u) possible = false;
      if (df < best_df) {
        best_df = df;
        driver = t;
      }
      total_ub += ub[t];
    }
    if (!possible) driver = 0xFFFFFFFFu;
  }
  for (uint32_t t = 0; t < kWarpMaxTerms; t++) {
    ScanPair p;
    p.base = 0;
    p.df = 0;
    p.qslot_t = (qslot << 3) | t;
    p.qi = h.qi;
    p.w = 0.0f;
    p.others = 0.0f;
    p.ne_prefix = 0.0f;
    p.filter = h.filter;
    p.first_item = 0;
    p.pad[0] = p.pad[1] = 0;
    if (t < h.nt) {
      const QTerm &q = wb.qterms[(uint64_t)qslot * kWarpMaxTerms + t];
      if (sc.must_mode) {
        if (t == driver) {
          p.base = q.base;
          p.df = seg.term_df[sc.ut_term[q.uterm]];
          p.w = q.weight;
          // every other term must add its share.  A direct sum: total_ub - ub[t] would round the other bounds to a multiple
          // of ulp(total_ub), far off when the driver is heavily boosted
          float o = 0.0f;
          for (uint32_t u = 0; u < kWarpMaxTerms; u++)
            if (u != t) o += ub[u];
          p.others = o;
          p.ne_prefix = total_ub;       // below the k-th score: no doc of this query can enter the top k
        }
      } else if ((q.flags & 5u) == 1u && q.term < seg.n_terms) {
        p.base = q.base;
        p.df = seg.term_df[q.term];
        p.w = q.weight;
        // priority: larger bound first, ties to the lower slot.  A doc with sparse holders is the business of the
        // highest-priority one of them, so a posting met in this term's scan can still gain: every column term, and the
        // sparse terms of LOWER priority
        float lower = 0.0f, gain = 0.0f;
        for (uint32_t u = 0; u < kWarpMaxTerms; u++) {
          const bool lo = u != t && (ub[u] < ub[t] || (ub[u] == ub[t] && u > t));
          if (lo) lower += ub[u];
          if (u != t && (is_col[u] || lo)) gain += ub[u];
        }
        p.others = gain;
        if (dbg & 1u) { float o = 0.0f; for (uint32_t u = 0; u < kWarpMaxTerms; u++) if (u != t) o += ub[u]; p.others = o; }
        p.ne_prefix = lower + ub[t];
      }
    }
    sc.pairs[(uint64_t)qslot * kWarpMaxTerms + t] = p;
  }
}

// order the scanned pairs rarest first (buckets of log2 df; inside a bucket any order) and lay out their items.  One CTA.
static __global__ void __launch_bounds__(1024) slg_scan_order_kernel(WarpBatchDev wb, ScanDev sc) {
  __shared__ uint32_t s_hist[33], s_cur[33], s_carry;
  const uint32_t tid = threadIdx.x, nthr = blockDim.x;
  const uint32_t n = wb.n_queries * kWarpMaxTerms;
  if (tid < 33) s_hist[tid] = 0u;
  __syncthreads();
  for (uint32_t i = tid; i < n; i += nthr) {
    const uint32_t df = sc.pairs[i].df;
    if (df) atomicAdd(&s_hist[32 - __clz(df)], 1u);
  }
  __syncthreads();
  if (tid == 0) {
    uint32_t run = 0;
    for (int b = 0; b < 33; b++) {
      s_cur[b] = run;
      run += s_hist[b];
    }
    *sc.n_pairs = run;
    s_carry = 0;
  }
  __syncthreads();
  for (uint32_t i = tid; i < n; i += nthr) {
    const uint32_t df = sc.pairs[i].df;
    if (df) sc.order[atomicAdd(&s_cur[32 - __clz(df)], 1u)] = i;
  }
  __syncthreads();
  // exclusive scan of the item counts in order: 1024 pairs per round
  const uint32_t np = *sc.n_pairs;
  __shared__ uint32_t s_scan[1024];
  for (uint32_t b0 = 0; b0 < np; b0 += nthr) {
    const uint32_t i = b0 + tid;
    uint32_t c = 0;
    if (i < np) c = (sc.pairs[sc.order[i]].df + sc.chunk - 1) / sc.chunk;
    s_scan[tid] = c;
    __syncthreads();
    for (uint32_t o = 1; o < nthr; o <<= 1) {
      const uint32_t v = tid >= o ? s_scan[tid - o] : 0u;
      __syncthreads();
      s_scan[tid] += v;
      __syncthreads();
    }
    const uint32_t excl = s_scan[tid] - c + s_carry;
    if (i < np) {
      sc.item_start[i] = excl;
      sc.pairs[sc.order[i]].first_item = excl;
    }
    __syncthreads();
    if (tid == nthr - 1) s_carry += s_scan[tid];
    __syncthreads();
  }
  if (tid == 0) {
    sc.item_start[np] = s_carry;
    *sc.n_items = min(s_carry, sc.items_cap);
  }
}

// items[i] = ordered pair of item i (binary search over item_start).  Grid-wide.
static __global__ void __launch_bounds__(256) slg_scan_items_kernel(ScanDev sc) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t n_items = *sc.n_items, np = *sc.n_pairs;
  if (i >= n_items) return;
  uint32_t lo = 0, hi = np;  // last pair with item_start <= i
  while (lo + 1 < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (sc.item_start[mid] <= i) lo = mid;
    else hi = mid;
  }
  sc.items[i] = lo;
}

// MUST: AND batches (sc.must_mode); compiled out of the plain OR instantiations, which then carry one pointer less per lane
template <bool PRUNE, bool POOLS, bool MUST>
__global__ void __launch_bounds__(kScanWarps * 32, 4) slg_scan_kernel(SegmentDev seg, WarpBatchDev wb, ScanDev sc) {
  __shared__ __align__(16) unsigned long long s_cand[kScanWarps][kWarpCand];
  __shared__ uint32_t s_hist[kScanWarps][POOLS ? 256 : 1];
  __shared__ uint32_t s_qidx[kScanWarps][kScanQueue];
  __shared__ float s_qval[kScanWarps][kScanQueue];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long *cand = s_cand[warp];
  uint32_t *q_idx = s_qidx[warp];
  float *q_val = s_qval[warp];
  const uint32_t k = wb.k;
  const uint32_t n_all = *sc.n_items;
  const uint32_t item_lo = (uint32_t)(((uint64_t)n_all * sc.part_lo) >> 8), n_items = (uint32_t)(((uint64_t)n_all * sc.part_hi) >> 8);
  uint32_t *work = sc.counter + (sc.part_lo ? 1 : 0);
  unsigned long long n_scanned = 0;
  uint32_t n_lane_verified = 0, n_lane_bit_lookups = 0, n_lane_searches = 0;  // (per lane: a few 10^4 per launch)
  uint32_t n_dropped = 0, n_done = 0;
  WarpCand wc;

  uint32_t item = 0;
  if (lane == 0) item = item_lo + atomicAdd(work, 1u);
  item = __shfl_sync(0xFFFFFFFFu, item, 0);
  while (item < n_items) {
    uint32_t next_item = 0;
    if (lane == 0) next_item = item_lo + atomicAdd(work, 1u);
    const uint32_t pi = __ldg(sc.order + __ldg(sc.items + item));
    const ScanPair pr = sc.pairs[pi];
    const unsigned long long thr0 = load_threshold(wb, pr.qi);
    const uint32_t chunk = item - pr.first_item;
    const bool have_thr0 = thr0 != kThrInit;
    const float thr0_score = __uint_as_float((uint32_t)(thr0 >> 32));
    if (PRUNE && have_thr0 && pr.ne_prefix * 1.00002f < thr0_score) {
      n_dropped++;  // this term and everything of lower priority cannot lift a doc into the top k
    } else {
      n_done++;
      wc.begin(cand, thr0, k, lane, 0u, POOLS ? s_hist[warp] : nullptr);
      const uint32_t qslot = pr.qslot_t >> 3, t = pr.qslot_t & 7u;
      const QTerm *qts = wb.qterms + (uint64_t)qslot * kWarpMaxTerms;
      const uint32_t nt = __ldg(&wb.qheads[qslot].nt);
      // lane u < nt keeps term u of the query: what verify needs, handed round by shuffles
      uint64_t m_base = 0;      // first posting of the term's list
      uint64_t m_col = 0;       // column terms: element offset of the column
      uint32_t m_df = 0, m_kind = 0;  // kind: 0 absent / unscored, 1 sparse, 2 column, 3 sparse with a presence bitmap (m_df = its row)
      float m_w = 0.0f, m_ub = 0.0f;
      if (lane < (int)nt) {
        const QTerm q = qts[lane];
        if (q.flags & 1u) {
          m_w = q.weight;
          m_ub = __fmul_rn(sc.ut_max[q.uterm], q.weight);
          if (q.flags & 4u) {
            m_kind = 2;
            if (MUST) {
              m_col = q.sc_base;
              m_base = q.base;
            } else {
              m_base = q.sc_base;  // (plain OR: a column term is never scanned, its posting base is not needed)
            }
          } else if (q.term < seg.n_terms) {
            m_kind = 1;
            m_base = q.base;
            m_df = __ldg(seg.term_df + q.term);
            const int32_t row = seg.term_bits ? __ldg(seg.term_bits + q.term) : -1;
            if (row >= 0) {
              m_kind = 3;
              m_df = (uint32_t)row;
            }
          }
        }
      }
      const float my_ub = __shfl_sync(0xFFFFFFFFu, m_ub, t);
      const float4 *sp = reinterpret_cast<const float4 *>(wb.scores + pr.base);
      const uint32_t i0 = chunk * sc.chunk, i1 = min(pr.df, i0 + sc.chunk);
      n_scanned += i1 - i0;
      uint32_t cut = 0u;
      auto recut = [&]() {
        cut = 0u;
        if (wc.thr != kThrInit) {
          const float cf = __uint_as_float((uint32_t)(wc.thr >> 32)) * 0.99998f - pr.others * 1.00002f;
          cut = cf > 0.0f ? __float_as_uint(cf) : 0u;
        }
      };
      recut();
      // candidates wait in the warp's queue (doc id, contribution) until a full round of 32 can be verified at once:
      // a verification is a chain of dependent memory accesses, so what counts is how many docs share each chain
      uint32_t nq = 0, qhead = 0;
      auto verify_round = [&](uint32_t n) {
        bool alive = lane < (int)n;
        uint32_t doc = 0u;
        float v = 0.0f;
        if (alive) {
          doc = q_idx[(qhead + lane) & (kScanQueue - 1u)];  // (the queue carries the doc id: it was read with the scores, coalesced)
          v = q_val[(qhead + lane) & (kScanQueue - 1u)];
        }
        qhead += n;
        nq -= n;
        alive = alive && __float_as_uint(v) >= cut;  // (the k-th score may have risen since the posting was queued)
        n_lane_verified += alive ? 1u : 0u;
        // a filtered query asks the filter first: one bit, and at a selectivity of a few percent most docs are done here
        if (alive && pr.filter >= 0) alive = (__ldg(wb.filter_bits[pr.filter] + (doc >> 5)) >> (doc & 31)) & 1u;
        const bool must = MUST;
        // ---- verify, cheapest evidence first: the column terms (one gather each), then the other sparse terms (a presence
        // bitmap look-up, or a search for a term without a bitmap), dropping the doc as soon as  known contributions + bounds
        // of the unknown ones  falls below the k-th score.  The exact score is the sum of the contributions in slot order.
        const float thr_s = wc.thr == kThrInit ? 0.0f : __uint_as_float((uint32_t)(wc.thr >> 32)) * 0.99998f;
        float c[kWarpMaxTerms];
        // unknown starts at pr.others (the bounds of exactly the terms that can still add: columns + lower-priority sparse)
        // and loses each bound once its term is looked up.  pr.others is a rounded sum and every subtraction rounds again:
        // up to 8 ulp(pr.others) in all, an absolute error that the relative slacks below do not cover when a boosted term's
        // bound dwarfs the others (after a column bound of 3e5 is taken off, a bound of 1.1 would be left as 1.09375).
        // 2^-19 * pr.others (>= 16 ulp) covers it
        float known = v, unknown = __fadd_rn(pr.others, __fmul_rn(pr.others, 0x1p-19f));
#pragma unroll
        for (int u = 0; u < (int)kWarpMaxTerms; u++) {
          c[u] = 0.0f;
          const uint32_t kind = __shfl_sync(0xFFFFFFFFu, m_kind, u);
          if (kind != 2u || u == (int)t) continue;  // (uniform; an AND batch may scan a term that also has a column)
          const uint64_t cb = __shfl_sync(0xFFFFFFFFu, MUST ? m_col : m_base, u);
          const float w = __shfl_sync(0xFFFFFFFFu, m_w, u), ub = __shfl_sync(0xFFFFFFFFu, m_ub, u);
          if (alive) {
            c[u] = __fmul_rn(__ldg(seg.cols + cb + doc), w);
            known += c[u];
            unknown -= ub;
            if (must && c[u] == 0.0f) alive = false;  // (a posting's contribution is positive: +0 means the list lacks the doc)
          }
        }
        alive = alive && (known + fmaxf(unknown, 0.0f)) * 1.0001f >= thr_s;
        bool stand_back = false;
        // two rounds over the other sparse terms.  First those of LOWER priority: each look-up replaces a bound by the exact
        // contribution, so a doc that cannot reach the k-th score dies here.  Only the few survivors then ask the terms of
        // HIGHER priority (the rarer lists, usually without a presence bitmap: a full search each) whether one of them holds
        // the doc — then that term's scan offers it — their bounds were never part of `unknown`.
        const int n_rounds = sc.two_rounds ? 2 : 1;
#pragma unroll 1
        for (int round = 0; round < n_rounds; round++)
#pragma unroll
        for (int u = 0; u < (int)kWarpMaxTerms; u++) {
          const uint32_t kind = __shfl_sync(0xFFFFFFFFu, m_kind, u);
          if (!(kind & 1u) || u == (int)t) continue;  // (uniform)
          const float ub = __shfl_sync(0xFFFFFFFFu, m_ub, u);
          const bool higher = !must && (ub > my_ub || (ub == my_ub && u < (int)t));  // a holder of higher priority offers the doc itself
          if (n_rounds == 2 && higher != (round == 1)) continue;  // (uniform)
          if (!__any_sync(0xFFFFFFFFu, alive)) break;
          const uint64_t pb = __shfl_sync(0xFFFFFFFFu, m_base, u);
          const uint32_t dfu = __shfl_sync(0xFFFFFFFFu, m_df, u);  // (kind 3: the bitmap row)
          const float w = __shfl_sync(0xFFFFFFFFu, m_w, u);
          if (alive) {
            bool held;
            uint32_t at = 0u;
            if (kind == 3u) {
              // the term's presence bitmap: bit and list position from one sector, post_doc is not read
              n_lane_bit_lookups++;
              held = presence_lookup(seg, (uint64_t)dfu * seg.bits_stride, doc, at);
            } else {
              n_lane_searches++;
              const uint32_t *dp = seg.post_doc + pb;
              at = lower_bound_interp(dp, dfu, doc, (float)dfu * (1.0f / (float)max(seg.doc_count, 1u)));
              held = at < dfu && __ldg(dp + at) == doc;
            }
            if (held) {
              if (higher) {
                stand_back = true;  // (the doc dies here: its contribution is not needed)
              } else {
                c[u] = __fmul_rn(__ldg(wb.scores + pb + at), w);
                known += c[u];
              }
            } else if (must) {
              stand_back = true;  // an AND query's doc must sit in every list
            }
            if (!higher) unknown -= ub;
            alive = !stand_back && (known + fmaxf(unknown, 0.0f)) * 1.0001f >= thr_s;
          }
        }
        if (__any_sync(0xFFFFFFFFu, alive)) {
          float sx = 0.0f;
#pragma unroll
          for (int u = 0; u < (int)kWarpMaxTerms; u++) {
            const float cu = u == (int)t ? v : c[u];
            if (cu != 0.0f) sx = __fadd_rn(sx, cu);
          }
          wc.offer(seg, wb, pr.qi, pr.filter, alive, doc, sx);
          recut();
        }
        __syncwarp();
      };
#pragma unroll 1
      for (uint32_t b = i0; b < i1; b += 256) {
        // two 128-posting steps in flight
        const uint32_t ia = b + lane * 4, ib = ia + 128;
        float4 va = make_float4(0, 0, 0, 0), vb = make_float4(0, 0, 0, 0);
        if (ia < i1) va = __ldg(sp + (ia >> 2));
        if (ib < i1) vb = __ldg(sp + (ib >> 2));
        float x[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
        uint32_t todo = 0u;
#pragma unroll
        for (int e = 0; e < 8; e++) {
          x[e] = __fmul_rn(x[e], pr.w);
          const uint32_t idx = (e < 4 ? ia : ib) + (e & 3);
          if (__float_as_uint(x[e]) >= cut && x[e] != 0.0f && idx < i1) todo |= 1u << e;  // (16-byte pieces may reach past the list's end)
        }
        if (!__any_sync(0xFFFFFFFFu, todo != 0u)) continue;
        // the doc ids of the lanes that hold a candidate: 16 bytes next to the 16 bytes of scores just read — coalesced
        // where candidates cluster, and one random 32-byte sector per candidate less than fetching post_doc[idx] later
        const uint4 *dp4 = reinterpret_cast<const uint4 *>(seg.post_doc + pr.base);
        uint4 da = make_uint4(0, 0, 0, 0), db = make_uint4(0, 0, 0, 0);
        if (todo & 0x0Fu) da = __ldg(dp4 + (ia >> 2));
        if (todo & 0xF0u) db = __ldg(dp4 + (ib >> 2));
        const uint32_t dd[8] = {da.x, da.y, da.z, da.w, db.x, db.y, db.z, db.w};
        // queue this step's candidates: every lane appends its own (an exclusive scan of the counts gives the places)
        {
          const uint32_t mine = __popc(todo);
          uint32_t incl = mine;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const uint32_t nb = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += nb;
          }
          uint32_t at = qhead + nq + incl - mine;
#pragma unroll
          for (int e = 0; e < 8; e++)
            if ((todo >> e) & 1u) {
              q_idx[at & (kScanQueue - 1u)] = dd[e];
              q_val[at & (kScanQueue - 1u)] = x[e];
              at++;
            }
          nq += __shfl_sync(0xFFFFFFFFu, incl, 31);
          __syncwarp();
        }
        while (nq >= 32u) verify_round(32u);
      }
      while (nq) verify_round(min(nq, 32u));
      wc.merge(wb, pr.qi);
    }
    item = __shfl_sync(0xFFFFFFFFu, next_item, 0);
  }
  if (sc.counters) {
    unsigned long long n_verified = n_lane_verified, n_bit_lookups = n_lane_bit_lookups, n_searches = n_lane_searches;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      n_verified += __shfl_xor_sync(0xFFFFFFFFu, n_verified, o);
      n_bit_lookups += __shfl_xor_sync(0xFFFFFFFFu, n_bit_lookups, o);
      n_searches += __shfl_xor_sync(0xFFFFFFFFu, n_searches, o);
    }
    if (lane == 0) {
      if (n_scanned) atomicAdd(sc.counters + 0, n_scanned);
      if (n_verified) atomicAdd(sc.counters + 4, n_verified);
      if (n_dropped) atomicAdd(sc.counters + 5, (unsigned long long)n_dropped);
      if (n_bit_lookups) atomicAdd(sc.counters + 6, n_bit_lookups);
      if (n_searches) atomicAdd(sc.counters + 7, n_searches);
      if (n_done) atomicAdd(sc.counters + 3, (unsigned long long)n_done);
    }
  }
}

}  // namespace slg
