// slg_residency.cuh — per-batch range planner and the residency kernels of the derived arrays
// (resident per-posting scores, dense columns of the high-df terms and their per-512-doc maxima).
#pragma once
#include "slg_kernels.cuh"

namespace slg {

// rng[r][j] = index of the first posting of row r's term with doc >= j * tile_docs, j = 0..n_tiles
// (replaces the cursor movement of TermState::advance_to, query/wand.rs:205-232).  Short lists are
// walked once (posting i fills the boundaries between its predecessor's tile and its own); long
// lists take one binary search per boundary.  grid = (rows, chunks).
static __global__ void __launch_bounds__(256) slg_plan_walk_kernel(SegmentDev seg, const uint32_t *ut_term, const uint32_t *row_u,
                                                              uint32_t n_rows, uint32_t tile_docs, uint32_t n_tiles,
                                                              bool column_rows, uint32_t *rng) {
  const uint32_t r = blockIdx.x;
  if (r >= n_rows) return;
  const uint32_t term = ut_term[row_u ? row_u[r] : r];
  uint32_t *out = rng + (uint64_t)r * (n_tiles + 1);
  const uint32_t step = gridDim.y * blockDim.x;
  const uint32_t first = blockIdx.y * blockDim.x + threadIdx.x;
  if (term >= seg.n_terms) {  // a key this segment does not hold: empty list
    for (uint32_t j = first; j <= n_tiles; j += step) out[j] = 0u;
    return;
  }
  if (!column_rows && seg.term_col && seg.term_col[term] >= 0) return;
  const uint32_t df = seg.term_df[term];
  const uint32_t *d = seg.post_doc + seg.term_start[term];
  if ((uint64_t)df <= 8ull * (n_tiles + 1)) {
    for (uint32_t i = first; i <= df; i += step) {
      const uint32_t a = i ? d[i - 1] / tile_docs + 1 : 0u;
      const uint32_t b = i < df ? d[i] / tile_docs : n_tiles;
      for (uint32_t j = a; j <= b; j++) out[j] = i;
    }
  } else {
    for (uint32_t j = first; j <= n_tiles; j += step) {
      const uint64_t target = (uint64_t)j * tile_docs;
      uint32_t lo = 0, hi = df;
      while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (d[mid] < target) lo = mid + 1;
        else hi = mid;
      }
      out[j] = lo;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// residency: unit-weight contribution of every posting (one CTA of 128 threads per 128-posting
// block, like slg_transcode_csr_kernel), the dense columns and their per-512-doc maxima
static __global__ void __launch_bounds__(128) slg_score_postings_kernel(SegmentDev seg, uint32_t n_blocks, float *post_score, float *mb_max) {
  const uint32_t blk = blockIdx.x;
  if (blk >= n_blocks) return;
  __shared__ uint32_t s_term;
  if (threadIdx.x == 0) {
    uint64_t lo = 0, hi = seg.n_terms;  // last term with term_blk[t] <= blk
    while (lo + 1 < hi) {
      const uint64_t mid = (lo + hi) >> 1;
      if (seg.term_blk[mid] <= blk) lo = mid;
      else hi = mid;
    }
    s_term = (uint32_t)lo;
  }
  __syncthreads();
  const uint32_t term = s_term;
  const uint32_t i = (blk - seg.term_blk[term]) * kBlock + threadIdx.x;
  const uint32_t df = seg.term_df[term];
  const uint64_t base = seg.term_start[term];
  float s = 0.0f;
  if (i < df) {
    const uint32_t doc = seg.post_doc[base + i];
    uint32_t tf = seg.post_tf[base + i];
    const uint64_t wide = seg.term_wide[term];
    if (tf == 255u && wide != ~0ull) tf = seg.tf_wide[wide + i];
    s = bm25_contrib_fast(tf, seg.term_idf[term], seg.k1p1, seg_nk(seg, term)[doc], 1.0f);
    post_score[base + i] = s;
  }
  // one warp = one 32-posting mini-block (term starts are multiples of 32): its maximum is the bound the
  // pruned executions use for the postings of a sub-tile (slg_items_bounds_kernel)
  float m = s;
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
  const uint32_t i0 = (blk - seg.term_blk[term]) * kBlock + (threadIdx.x & ~31u);
  if ((threadIdx.x & 31) == 0 && i0 < ((df + 31u) & ~31u)) mb_max[(base + i0) >> 5] = m;
}

// grid (chunks, n_cols): column c holds the scores of term col_terms[c] at their doc slots
static __global__ void slg_fill_columns_kernel(SegmentDev seg, const uint32_t *col_terms, uint32_t n_cols, float *cols) {
  const uint32_t c = blockIdx.y;
  if (c >= n_cols) return;
  const uint32_t term = col_terms[c];
  const uint32_t df = seg.term_df[term];
  const uint64_t base = seg.term_start[term];
  float *col = cols + (uint64_t)c * seg.col_stride;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < df; i += gridDim.x * blockDim.x)
    col[seg.post_doc[base + i]] = seg.post_score[base + i];
}

// ---- presence bitmaps with interleaved rank ----------------------------------------------------------------------
// A row is an array of 32-byte units, one DRAM sector each.  Word 0 of unit u holds the number of docs the list holds
// before doc 224u (the set bits of every earlier unit of the row); words 1..7 hold one bit per doc of [224u, 224u + 224).
// Lists are strictly ascending, so the position of a held doc in its list is its rank: the bit and the posting index
// come out of the same sector, and a look-up never searches post_doc.  (A 64-byte unit would halve the rank words'
// share, 1/16 instead of 1/8, but touch two sectors per look-up.)
constexpr uint32_t kPresUnitDocs = 224;  // docs per unit
constexpr uint32_t kPresUnitWords = 8;

__host__ __device__ inline uint32_t presence_row_words(uint32_t doc_count) {
  return (doc_count + kPresUnitDocs - 1) / kPresUnitDocs * kPresUnitWords;
}

// does the row at word offset row_off of seg.pres_bits hold doc; if so, at = the doc's position in the term's list.  The
// one place that reads seg.pres_bits: every kernel asks here
__device__ __forceinline__ bool presence_lookup(const SegmentDev &seg, uint64_t row_off, uint32_t doc, uint32_t &at) {
  const uint32_t u = doc / kPresUnitDocs, r = doc - u * kPresUnitDocs;
  const uint4 *p = reinterpret_cast<const uint4 *>(seg.pres_bits + row_off + (uint64_t)u * kPresUnitWords);
  const uint4 a = __ldg(p), b = __ldg(p + 1);  // (both halves of the unit's one sector)
  const uint32_t w[kPresUnitWords] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  const uint32_t wi = 1u + (r >> 5), bit = r & 31u;
  uint32_t word = 0u, n = w[0];
#pragma unroll
  for (uint32_t i = 1; i < kPresUnitWords; i++) {
    if (i < wi) n += __popc(w[i]);
    if (i == wi) word = w[i];
  }
  at = n + __popc(word & ((1u << bit) - 1u));
  return (word >> bit) & 1u;
}

// grid (chunks, n_rows): the bits of row r for term bm_terms[r] (rows are zero on entry; slg_presence_rank_kernel then
// writes the rank words)
static __global__ void slg_fill_presence_kernel(SegmentDev seg, const uint32_t *bm_terms, uint32_t n_rows, uint32_t *bits, uint32_t stride) {
  const uint32_t r = blockIdx.y;
  if (r >= n_rows) return;
  const uint32_t term = bm_terms[r];
  const uint32_t df = seg.term_df[term];
  const uint32_t *d = seg.post_doc + seg.term_start[term];
  uint32_t *row = bits + (uint64_t)r * stride;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < df; i += gridDim.x * blockDim.x) {
    const uint32_t doc = d[i];
    const uint32_t u = doc / kPresUnitDocs, rem = doc - u * kPresUnitDocs;
    atomicOr(row + (uint64_t)u * kPresUnitWords + 1u + (rem >> 5), 1u << (rem & 31));
  }
}

// one CTA per row: word 0 of every unit = exclusive scan of the units' popcounts; totals[r] = the row's set bits (the
// loader checks it against the list's df)
constexpr uint32_t kRankThreads = 1024;
static __global__ void __launch_bounds__(kRankThreads) slg_presence_rank_kernel(uint32_t *bits, uint32_t stride, uint32_t n_rows, uint32_t *totals) {
  __shared__ uint32_t s_warp[kRankThreads / 32 + 1];  // exclusive prefix of every warp's units, then the tile's total
  const uint32_t r = blockIdx.x;
  if (r >= n_rows) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t *row = bits + (uint64_t)r * stride;
  const uint32_t n_units = stride / kPresUnitWords;
  uint32_t carry = 0u;
  for (uint32_t u0 = 0; u0 < n_units; u0 += kRankThreads) {
    const uint32_t u = u0 + threadIdx.x;
    uint32_t c = 0u;
    if (u < n_units) {
      const uint4 *p = reinterpret_cast<const uint4 *>(row + (uint64_t)u * kPresUnitWords);
      const uint4 a = p[0], b = p[1];
      c = __popc(a.y) + __popc(a.z) + __popc(a.w) + __popc(b.x) + __popc(b.y) + __popc(b.z) + __popc(b.w);
    }
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      uint32_t t = s_warp[lane], ti = t;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, ti, o);
        if (lane >= o) ti += v;
      }
      s_warp[lane] = ti - t;
      if (lane == 31) s_warp[kRankThreads / 32] = ti;
    }
    __syncthreads();
    if (u < n_units) row[(uint64_t)u * kPresUnitWords] = carry + s_warp[warp] + incl - c;
    carry += s_warp[kRankThreads / 32];
    __syncthreads();
  }
  if (threadIdx.x == 0) totals[r] = carry;
}

// one warp per (512-doc slice, column): the exact maximum contribution inside the slice
static __global__ void slg_column_tmax_kernel(const float *cols, uint64_t col_stride, uint32_t n_cols, uint32_t tmax_stride, float *tmax) {
  const uint64_t w = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= (uint64_t)n_cols * tmax_stride) return;
  const uint32_t c = (uint32_t)(w / tmax_stride), j = (uint32_t)(w % tmax_stride);
  const float4 *p = reinterpret_cast<const float4 *>(cols + (uint64_t)c * col_stride + (uint64_t)j * 512) + lane;
  float m = 0.0f;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const float4 v = p[i * 32];
    m = fmaxf(m, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
  }
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
  if (lane == 0) tmax[w] = m;
}

}  // namespace slg
