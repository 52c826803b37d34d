// slg_stream_kernel.cuh — K2/K5, exhaustive execution (`bm25`) of plain OR queries with k <= 32 and <= 8 terms
// per query on segments with resident scores: the automatic choice for the shape of BASELINE.json configs[1].
//
// brute_force (query/wand.rs:459-566) adds every posting of every query term to its doc's score and offers every
// touched doc to push_top_k.  Here that work is split by what a term looks like in HBM:
//
//   SPARSE PASS   slg_score_sparse_kernel — terms without a dense column.  One warp takes a (query, group of
//                 kSubPerGroup sub-tiles) item.  The (doc, score) runs of ALL the query's sparse terms inside a span of
//                 sub-tiles are brought into shared memory by bulk asynchronous copies (cp.async.bulk, completion on
//                 a warp-private mbarrier) — every byte of the item is in flight at once and no register is
//                 spent on the copy — and then, sub-tile by sub-tile, scattered from shared memory into the warp's
//                 accumulator A (slot order = declared summation order) and walked again: read A[doc], write 0,
//                 and a partial that can still reach the query's k-th score completes its score with one 4-byte
//                 gather per column term and is offered.  A query with a single sparse term needs no accumulator:
//                 its staged scores are compared as they are.
//   COLUMN PASS   slg_score_columns_kernel — terms with a doc-indexed f32 column (df >= N / dense_den).  Doc-block
//                 major: a CTA takes a block of kColBlock docs, brings that block of EVERY column the batch
//                 names into shared memory with one bulk asynchronous copy per column (double buffered: the next
//                 block lands while this one is scored) — each column block leaves HBM/L2 once per batch instead of
//                 once per query — and then scores all the batch's queries that have a column term against it, 32
//                 queries per warp step.  A query whose only column term is c sees v = c[d] * w for every doc of the
//                 block, and max(v) = max(c) * w (f32 multiplication by a positive weight is monotone), so its
//                 comparisons against the k-th score collapse into one against the block maximum the CTA took from
//                 the values it has just read; a query with several columns sums their blocks per doc, slot order,
//                 from shared memory.  Only where a doc can enter the top k is a block looked at per doc.  A doc
//                 that also sits in one of the query's sparse lists belongs to the sparse pass (its partial is in A
//                 there) and is left alone here.
//
// Every posting of every query term is read and takes part in the comparison that decides its doc; what is
// shared is the READ of a column block between the queries that name the column, and what is skipped is only the
// search for candidates that provably do not exist (as in slg_score_warp_kernel's written-maximum shortcut).  The
// sparse pass runs first so that the column pass starts with every query's k-th score already high.
//
// Float contract (include/searchlite_gpu.h): a doc's contributions are summed over the query's terms WITHOUT a
// column first, then over the terms WITH one, each group in query order — slg_build_qterms_kernel lays the slots
// out in that order, both passes add in slot order, so both produce the bits of brute_force on that permutation.
#pragma once
#include "slg_async.cuh"
#include "slg_items_kernel.cuh"
#include "slg_residency.cuh"

namespace slg {

constexpr uint32_t kColBlock = 256;      // docs per column-pass block (1 KB of every column)
constexpr int kSparseWarps = 4;          // warps per CTA of the sparse pass
constexpr int kColWarps = 16;            // warps per CTA of the column pass
constexpr uint32_t kColMaxSlots = 4096;  // used columns whose block maximum is kept (beyond: always looked at per doc)

struct __align__(16) ColQ {  // one query with >= 1 column term (48 B)
  uint32_t qslot, qi;
  int32_t filter;
  uint8_t nsp, ncol, unit_w, off;  // slots [0, nsp) sparse, [nsp, nsp + ncol) columns; unit_w: every column weight is 1.0;
                                   // off: the query sits this pass out (pruned: no column term of it is essential)
  uint16_t slot[8];                // used-column slots of the column terms, slot order
  float extra;                     // pruned: what the sparse terms a doc may still hold unseen can add (their bounds)
  uint32_t pad[3];
};

struct StreamDev {
  ColQ *colq;            // [Q] the batch's queries with >= 1 column term
  uint32_t *n_colq;      // device counters
  uint32_t *ucol;        // [n_cols] slot -> column (the columns the batch names, densest first)
  uint32_t *n_ucol;
  uint32_t *col_slot;    // [n_cols] column -> slot (scratch of slg_colgroups_kernel)
  uint32_t *sparse_counter, *col_counter;  // work counters of the two passes
  uint32_t stage_cap;    // postings a warp of the sparse pass can stage per span (multiple of 4)
  uint32_t col_resident; // columns of a block the column pass keeps in shared memory (per buffer)
  uint32_t n_smax;       // block maxima kept in shared memory (min(columns of the segment, kColMaxSlots))
  uint32_t strict;       // 1: accumulate every posting per doc (option strict_accumulate); 0: bounded accumulation, see sparse_sub_bounded
  unsigned long long *counters;  // [4] sparse postings visited, (query, column block) pairs looked at per doc, (query, column block) pairs scored, sparse items
};

// ---- the batch's column terms: used columns -> slots, queries with a column term -> ColQ (one CTA) -------------
// Pruned executions (ut_max != nullptr): with the k-th score the posting scan left behind, a query's non-essential terms are
// its longest lowest-priority prefix (priority: larger bound first, ties to the lower slot) whose bounds sum below that
// score.  A query whose column terms are ALL non-essential sits the column pass out — a doc without an essential term
// cannot enter the top k — and the others look at v + extra, extra = the bounds of their non-essential SPARSE terms (lists
// the scan may have dropped, so a doc may hold them unseen).
__device__ __forceinline__ bool colq_prune(const WarpBatchDev &wb, const float *ut_max, uint32_t qslot, uint32_t qi, uint32_t nt, float &extra) {
  const unsigned long long thr = load_threshold(wb, qi);
  float ub[kWarpMaxTerms];
  bool col[kWarpMaxTerms];
  for (uint32_t t = 0; t < kWarpMaxTerms; t++) {
    ub[t] = 0.0f;
    col[t] = false;
    if (t < nt) {
      const QTerm &q = wb.qterms[(uint64_t)qslot * kWarpMaxTerms + t];
      if (q.flags & 1u) ub[t] = __fmul_rn(ut_max[q.uterm], q.weight);
      col[t] = (q.flags & 5u) == 5u;
    }
  }
  extra = 0.0f;
  bool any_essential_col = false;
  for (uint32_t t = 0; t < nt; t++) {
    float pre = 0.0f;
    for (uint32_t u = 0; u < nt; u++)
      if (ub[u] < ub[t] || (ub[u] == ub[t] && u >= t)) pre += ub[u];
    const bool ne = thr != kThrInit && pre * 1.00002f < __uint_as_float((uint32_t)(thr >> 32));
    if (col[t]) any_essential_col = any_essential_col || !ne;
    else if (ne) extra += ub[t];
  }
  return any_essential_col;
}

static __global__ void __launch_bounds__(1024) slg_colgroups_kernel(SegmentDev seg, WarpBatchDev wb, StreamDev sd, uint32_t n_cols, const float *ut_max) {
  const uint32_t tid = threadIdx.x, nthr = blockDim.x;
  for (uint32_t c = tid; c < n_cols; c += nthr) sd.col_slot[c] = 0u;
  if (tid == 0) {
    *sd.n_colq = 0u;
    *sd.n_ucol = 0u;
  }
  __syncthreads();
  for (uint32_t slot = tid; slot < wb.n_queries; slot += nthr) {
    const QHead h = wb.qheads[slot];
    float extra;
    if (ut_max && !colq_prune(wb, ut_max, slot, h.qi, h.nt, extra)) continue;
    for (uint32_t t = 0; t < h.nt; t++) {
      const QTerm &q = wb.qterms[(uint64_t)slot * kWarpMaxTerms + t];
      if ((q.flags & 5u) == 5u) sd.col_slot[q.term] = 1u;
    }
  }
  __syncthreads();
  {  // slots in column order (column 0 is the densest term): a block-wide exclusive scan of the "named" flags, 1024 columns a round
    __shared__ uint32_t s_scan[1024];
    __shared__ uint32_t s_carry;
    if (tid == 0) s_carry = 0u;
    __syncthreads();
    for (uint32_t base = 0; base < n_cols; base += nthr) {
      const uint32_t c = base + tid;
      const uint32_t flag = c < n_cols && sd.col_slot[c] ? 1u : 0u;
      s_scan[tid] = flag;
      __syncthreads();
      for (uint32_t o = 1; o < nthr; o <<= 1) {
        const uint32_t v = tid >= o ? s_scan[tid - o] : 0u;
        __syncthreads();
        s_scan[tid] += v;
        __syncthreads();
      }
      const uint32_t excl = s_scan[tid] - flag + s_carry;
      if (c < n_cols) {
        if (flag) {
          sd.ucol[excl] = c;
          sd.col_slot[c] = excl;
        } else {
          sd.col_slot[c] = 0xFFFFFFFFu;
        }
      }
      __syncthreads();
      if (tid == nthr - 1) s_carry += s_scan[tid];
      __syncthreads();
    }
    if (tid == 0) *sd.n_ucol = s_carry;
  }
  __syncthreads();
  for (uint32_t slot = tid; slot < wb.n_queries; slot += nthr) {
    const QHead h = wb.qheads[slot];
    ColQ r;
    r.qslot = slot;
    r.qi = h.qi;
    r.filter = h.filter;
    r.nsp = 0;
    r.ncol = 0;
    r.unit_w = 1;
    r.off = 0;
    r.extra = 0.0f;
    r.pad[0] = r.pad[1] = r.pad[2] = 0;
    for (int i = 0; i < 8; i++) r.slot[i] = 0;
    for (uint32_t t = 0; t < h.nt; t++) {
      const QTerm &q = wb.qterms[(uint64_t)slot * kWarpMaxTerms + t];
      if (!(q.flags & 1u)) continue;
      if (q.flags & 4u) {
        r.slot[r.ncol++] = (uint16_t)sd.col_slot[q.term];
        if (q.weight != 1.0f) r.unit_w = 0;
      } else {
        r.nsp++;
      }
    }
    if (r.ncol && ut_max) {
      // (the k-th score may have risen since the first loop: a query that now tests out names columns that are all in the table)
      if (!colq_prune(wb, ut_max, slot, h.qi, h.nt, r.extra)) continue;
      bool all_in = true;
      for (uint32_t i = 0; i < r.ncol; i++) all_in = all_in && r.slot[i] != 0xFFFFu;
      if (!all_in) r.off = 1;  // cannot happen (the score only rises); stay safe
    }
    if (r.ncol && !r.off) sd.colq[atomicAdd(sd.n_colq, 1u)] = r;
  }
}

// the 64 keys of the warp's buffer are sorted (descending, zeros last): drop repeated keys, return the number of keys left.
// The same doc can be offered twice with the same exact score when two passes (or two of its postings) both find it.
__device__ __forceinline__ uint32_t warp_dedupe64(unsigned long long *a, int lane) {
  const unsigned long long x0 = a[lane], x1 = a[lane + 32];
  const unsigned long long p0 = lane ? a[lane - 1] : ~0ull, p1 = a[lane + 31];
  const bool k0 = x0 != 0ull && x0 != p0, k1 = x1 != 0ull && x1 != p1;
  const uint32_t b0 = __ballot_sync(0xFFFFFFFFu, k0), b1 = __ballot_sync(0xFFFFFFFFu, k1);
  const uint32_t lt = (1u << lane) - 1u, n0 = __popc(b0), n = n0 + __popc(b1);
  __syncwarp();
  if (k0) a[__popc(b0 & lt)] = x0;
  if (k1) a[n0 + __popc(b1 & lt)] = x1;
  __syncwarp();
  for (uint32_t z = n + lane; z < kWarpCand; z += 32) a[z] = 0ull;
  __syncwarp();
  return n;
}

// ---- the warp's candidate buffer: push_top_k (query/wand.rs:905-916) ------------------------------------------
struct WarpCand {
  unsigned long long *cand;  // [kWarpCand] shared
  unsigned long long thr;    // the query's k-th key as this warp knows it
  uint32_t cnt;
  uint32_t k;
  int lane;
  uint32_t pool;             // k > kWarpMaxK: which of the query's pools this pass appends to
  uint32_t *hist;            // k > kWarpMaxK: 256 counters of shared memory private to the warp (radix select)

  __device__ __forceinline__ void begin(unsigned long long *buf, unsigned long long thr0, uint32_t k_, int lane_, uint32_t pool_ = 0,
                                        uint32_t *hist_ = nullptr) {
    cand = buf;
    thr = thr0;
    cnt = 0;
    k = k_;
    lane = lane_;
    pool = pool_;
    hist = hist_;
  }
  // k > kWarpMaxK.  The pool holds up to pool_cap distinct keys in no order.  When an append would overflow it, the warp
  // holding the lock finds the k-th largest key by radix select (8 bits a pass, histogram in shared memory), keeps the keys
  // >= it (exactly k: the keys of a pool are distinct) and publishes it as the query's threshold.
  __device__ __forceinline__ uint32_t compact_pool(const WarpBatchDev &wb, uint32_t qi, unsigned long long *pk, uint32_t n) {
    unsigned long long prefix = 0ull;
    uint32_t want = k;  // rank (from the top) of the key looked for among the keys that share the prefix
    for (int pass = 0; pass < 8; pass++) {
      const int shift = 56 - 8 * pass;
      for (uint32_t z = lane; z < 256; z += 32) hist[z] = 0u;
      __syncwarp();
      for (uint32_t i = lane; i < n; i += 32) {
        const unsigned long long key = ld_cg_u64(pk + i);
        if (pass == 0 || (key >> (shift + 8)) == (prefix >> (shift + 8))) atomicAdd(hist + (uint32_t)((key >> shift) & 255ull), 1u);
      }
      __syncwarp();
      // bins from the top: lane L owns bins 255 - 8L .. 248 - 8L
      uint32_t mine = 0;
#pragma unroll
      for (int j = 0; j < 8; j++) mine += hist[255 - 8 * lane - j];
      uint32_t incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t nb = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += nb;
      }
      const uint32_t owner = __ffs(__ballot_sync(0xFFFFFFFFu, incl >= want)) - 1;  // (some lane qualifies: n >= want)
      uint32_t before = __shfl_sync(0xFFFFFFFFu, incl - mine, owner);
      uint32_t bin = 0;
      if (lane == (int)owner) {
        for (int j = 0; j < 8; j++) {
          const uint32_t c = hist[255 - 8 * lane - j];
          if (before + c >= want) {
            bin = 255 - 8 * lane - j;
            break;
          }
          before += c;
        }
      }
      bin = __shfl_sync(0xFFFFFFFFu, bin, owner);
      before = __shfl_sync(0xFFFFFFFFu, before, owner);
      want -= before;
      prefix |= (unsigned long long)bin << shift;
      __syncwarp();
    }
    const unsigned long long kth = prefix;
    uint32_t out = 0;
    for (uint32_t b0 = 0; b0 < n; b0 += 32) {
      const uint32_t i = b0 + lane;
      unsigned long long key = 0ull;
      if (i < n) key = ld_cg_u64(pk + i);
      const bool keep = i < n && key >= kth;
      const uint32_t bal = __ballot_sync(0xFFFFFFFFu, keep);
      if (keep) st_cg_u64(pk + out + __popc(bal & ((1u << lane) - 1u)), key);  // (out <= b0: never ahead of the reads)
      out += __popc(bal);
      __syncwarp();
    }
    if (lane == 0) {
      if (atomicMax(wb.thr_key + qi, kth) < kth) push_threshold(wb, qi, kth);
    }
    thr = max(thr, kth);
    return out;
  }
  // k > kWarpMaxK: append the pending keys to the query's pool
  __device__ __forceinline__ void flush(const WarpBatchDev &wb, uint32_t qi) {
    if (cnt == 0) return;
    const unsigned long long thr_now = load_threshold(wb, qi);
    thr = max(thr, thr_now);
    // drop what the published threshold already rules out, then append under the pool's lock
    unsigned long long k0 = lane < (int)cnt ? cand[lane] : 0ull, k1 = 32 + lane < (int)cnt ? cand[32 + lane] : 0ull;
    if (k0 <= thr) k0 = 0ull;
    if (k1 <= thr) k1 = 0ull;
    const uint32_t b0 = __ballot_sync(0xFFFFFFFFu, k0 != 0ull), b1 = __ballot_sync(0xFFFFFFFFu, k1 != 0ull);
    const uint32_t n_new = __popc(b0) + __popc(b1);
    cnt = 0;
    __syncwarp();
    if (n_new == 0) return;
    const uint32_t slot = qi * 2u + pool;
    unsigned long long *pk = wb.pool_keys + (uint64_t)slot * wb.pool_cap;
    if (lane == 0) {
      while (atomicCAS(wb.pool_lock + slot, 0u, 1u) != 0u) __nanosleep(64);
      __threadfence();
    }
    __syncwarp();
    uint32_t n = ld_cg_u32(wb.pool_count + slot);
    if (n + n_new > wb.pool_cap) n = compact_pool(wb, qi, pk, n);
    const uint32_t lt = (1u << lane) - 1u;
    // (the compaction may have raised the threshold: keys it rules out are not written)
    const uint32_t w0 = __ballot_sync(0xFFFFFFFFu, k0 > thr), w1 = __ballot_sync(0xFFFFFFFFu, k1 > thr);
    if (k0 > thr) st_cg_u64(pk + n + __popc(w0 & lt), k0);
    if (k1 > thr) st_cg_u64(pk + n + __popc(w0) + __popc(w1 & lt), k1);
    __threadfence();
    __syncwarp();
    if (lane == 0) {
      st_cg_u32(wb.pool_count + slot, n + __popc(w0) + __popc(w1));
      __threadfence();
      atomicExch(wb.pool_lock + slot, 0u);
    }
    __syncwarp();
  }
  // append one ballot round of keys; past 32 pending: sort, keep the best k, raise the local threshold
  __device__ __forceinline__ void push(bool pass, unsigned long long key) {
    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, pass);
    if (!bal) return;
    if (pass) cand[cnt + __popc(bal & ((1u << lane) - 1u))] = key;
    cnt += __popc(bal);
    __syncwarp();
    if (cnt > 32 && hist) {  // k > kWarpMaxK: no local top-k, the pending keys go to the pool (flush needs wb: see offer)
      return;
    }
    if (cnt > 32) {
      for (uint32_t z = cnt + lane; z < kWarpCand; z += 32) cand[z] = 0ull;
      __syncwarp();
      warp_sort64_desc(cand, lane);
      cnt = min(warp_dedupe64(cand, lane), k);
      if (cnt == k) thr = max(thr, cand[k - 1]);
      __syncwarp();
    }
  }
  // accept (api/reader.rs:3009-3036) for a doc whose exact score is known
  __device__ __forceinline__ void offer(const SegmentDev &seg, const WarpBatchDev &wb, uint32_t qi, int32_t filter, bool have, uint32_t doc,
                                        float s) {
    const unsigned long long key = ((unsigned long long)__float_as_uint(s) << 32) | (unsigned long long)(0xFFFFFFFFu - doc);
    bool pass = have && key > thr && s != 0.0f;
    if (pass) pass = (seg.live_bits[doc >> 5] >> (doc & 31)) & 1u;
    if (pass && filter >= 0) pass = (wb.filter_bits[filter][doc >> 5] >> (doc & 31)) & 1u;
    if (pass) pass = cursor_accepts(wb.q_cursor, wb.q_saw, qi, key);
    push(pass, key);
    if (hist && cnt > 32) flush(wb, qi);
  }
  // merge into the query's global top-k under its lock; returns the query's k-th key afterwards
  __device__ __forceinline__ void merge(const WarpBatchDev &wb, uint32_t qi) {
    if (hist) {
      flush(wb, qi);
      return;
    }
    if (cnt == 0) return;
    const unsigned long long thr_now = load_threshold(wb, qi);
    const bool useful = lane < (int)cnt && cand[lane] > thr_now;  // cnt <= 32 after every push
    if (__any_sync(0xFFFFFFFFu, useful)) {
      if (lane == 0) {
        while (atomicCAS(wb.lock + qi, 0u, 1u) != 0u) __nanosleep(64);
        __threadfence();
      }
      __syncwarp();
      const uint32_t ng = ld_cg_u32(wb.topk_count + qi);
      unsigned long long *gk = wb.topk_keys + (uint64_t)qi * k;
      if (lane < (int)ng) cand[cnt + lane] = ld_cg_u64(gk + lane);
      uint32_t total = cnt + ng;
      for (uint32_t z = total + lane; z < kWarpCand; z += 32) cand[z] = 0ull;
      __syncwarp();
      warp_sort64_desc(cand, lane);
      total = min(warp_dedupe64(cand, lane), k);
      if (lane < (int)total) st_cg_u64(gk + lane, cand[lane]);
      __threadfence();
      __syncwarp();
      if (total == k) thr = max(thr, cand[k - 1]);
      thr = max(thr, thr_now);
      if (lane == 0) {
        st_cg_u32(wb.topk_count + qi, total);
        if (total == k && cand[k - 1] > thr_now) {  // (thr_now may be a bound that came from another shard)
          st_cg_u64(wb.thr_key + qi, cand[k - 1]);
          push_threshold(wb, qi, cand[k - 1]);
        }
        __threadfence();
        atomicExch(wb.lock + qi, 0u);
      }
      __syncwarp();
    } else {
      thr = max(thr, thr_now);
    }
    cnt = 0;
  }
};

// shared memory of one warp of the sparse pass
__host__ __device__ inline size_t sparse_smem_per_warp(uint32_t sub_docs, uint32_t stage_cap) {
  // own u16[sub_docs] | sdoc u32[cap] | ssc f32[cap] | cand u64[64] | qt QTerm[8] | rb u32[8][9] | cum u32[65 (+3)] | rest f32[8] | cmx f32[8] | pend u32[64] | bar u64 (+ pad)
  return (((size_t)sub_docs * 2 + 15) & ~(size_t)15) + (size_t)stage_cap * 8 + kWarpCand * 8 + kWarpMaxTerms * sizeof(QTerm) +
         kWarpMaxTerms * kRbStride * 4 + 68 * 4 + kSubPerGroup * 4 + kWarpMaxTerms * 4 + 64 * 4 + 16;
}

constexpr uint32_t kOwnFlag = 0x8000u;  // own[slot]: index of the posting that owns the doc | this flag when other lists hold it too

// One sub-tile of the sparse pass, posting-parallel over ALL the query's sparse terms at once.
//
// The postings of the sub-tile are numbered p = 0 .. P-1, term after term (slot order).  Accumulating per doc needs
// no float read-modify-write — and therefore no term-by-term ordering of the shared-memory traffic — because a doc
// that sits in ONE of the query's sparse lists (the usual case: the lists are sparse) has a one-term sum:
//   L1  every posting writes its number into own[doc - tile_lo]: some posting of the doc ends up owning the slot
//   L2  every posting reads the slot back; one that finds another number there sets the flag: the doc has several postings
//   L3  the owner of an unflagged slot offers its own contribution (the doc's exact sparse sum); the owner of a flagged
//       slot is parked and later sums the doc over all terms, slot order, finding it in the other terms' runs by
//       binary search (runs are sorted by doc)
// own[] needs no clearing: every slot read in L2/L3 was written in L1 of the same sub-tile.
// STAGED: postings [P0, P1) of the staged stream, cells (term runs, rounded out to 16 bytes) back to back, cell t at
// cb[t] - base .. cb[t+1] - base; postings outside the sub-tile's doc range (the rounding) fail the range test.
// Not staged (a sub-tile whose runs do not fit the staging area): the same three loops straight from global memory.
template <bool STAGED>
__device__ __forceinline__ void sparse_sub(const SegmentDev &seg, const WarpBatchDev &wb, const QHead &head, const QTerm *qt, const uint32_t *rbj,
                                           const uint32_t *cb, const uint32_t base, const uint32_t nsp, const uint32_t colmask, const bool unit_w, const float rest,
                                           const uint32_t tile_lo, const uint32_t sub_docs, unsigned short *own, const uint32_t *sdoc,
                                           const float *ssc, uint32_t *pend, WarpCand &wc, const int lane) {
  // run of term t: STAGED staged indices [cb[t], cb[t+1]); else postings [rbj[t*9], rbj[t*9+1]) of the term's list,
  // numbered from the sum of the earlier runs' lengths
  auto cut_now = [&]() {
    if (wc.thr == kThrInit) return 0u;
    const float cf = __uint_as_float((uint32_t)(wc.thr >> 32)) * 0.99998f - rest * 1.00002f;
    return cf > 0.0f ? __float_as_uint(cf) : 0u;
  };
  // a doc whose sparse sum is v: add the column terms of exactly this doc, slot order
  auto complete = [&](bool pass, uint32_t doc, float v) {
    float s = v;
    if (pass)
      for (uint32_t cm = colmask; cm; cm &= cm - 1) {
        const uint32_t ct = __ffs(cm) - 1;
        const float c = __ldg(seg.cols + qt[ct].sc_base + doc);
        s = __fadd_rn(s, __fmul_rn(c, qt[ct].weight));
      }
    wc.offer(seg, wb, head.qi, head.filter, pass, doc, s);
  };
  uint32_t npend = 0;
  // parked owners of docs with several postings: pend[] holds (slot << 16 | p), resolved 32 at a time
  auto resolve = [&](uint32_t n) {
    const bool have = lane < (int)n;
    const uint32_t e = have ? pend[lane] : 0u;
    const uint32_t slot = e >> 16, pp = e & 0xFFFFu, doc = tile_lo + slot;
    float s = 0.0f;
    if (have) {
      uint32_t start = 0;  // not staged: number of the first posting of term t
      for (uint32_t t = 0; t < nsp; t++) {
        uint32_t lo, hi;
        const uint32_t *dp;
        const float *sp;
        bool mine;
        uint32_t at = 0;
        if (STAGED) {
          lo = cb[t] - base;
          hi = cb[t + 1] - base;
          dp = sdoc;
          sp = ssc;
          mine = pp >= lo && pp < hi;
          at = pp;
        } else {
          lo = rbj[t * kRbStride];
          hi = rbj[t * kRbStride + 1];
          dp = seg.post_doc + qt[t].base;
          sp = wb.scores + qt[t].base;
          mine = pp >= start && pp < start + (hi - lo);
          at = lo + (pp - start);
          start += hi - lo;
        }
        float c = 0.0f;
        if (mine) {
          c = sp[at];
        } else {
          const uint32_t end = hi;
          while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (dp[mid] < doc) lo = mid + 1;
            else hi = mid;
          }
          if (lo < end && dp[lo] == doc) c = sp[lo];
        }
        if (c != 0.0f) s = __fadd_rn(s, __fmul_rn(c, qt[t].weight));  // (a sum that starts at +0 and skips absent terms: brute_force on the doc's lists)
      }
    }
    const bool pass = have && __float_as_uint(s) >= cut_now();
    if (__any_sync(0xFFFFFFFFu, pass)) complete(pass, doc, s);
  };
  auto park = [&](bool conf, uint32_t slot, uint32_t pp) {
    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, conf);
    if (!bal) return;
    if (conf) pend[npend + __popc(bal & ((1u << lane) - 1u))] = (slot << 16) | pp;
    npend += __popc(bal);
    __syncwarp();
    if (npend >= 32u) {
      resolve(32u);
      __syncwarp();
      if (lane < (int)(npend - 32u)) {
        const uint32_t x = pend[32 + lane];
        pend[lane] = x;
      }
      npend -= 32u;
      __syncwarp();
    }
  };
  // the weight of posting number pp (only when some weight differs from 1)
  auto weight_of = [&](uint32_t pp) {
    uint32_t t = 0, start = 0;
    for (uint32_t u = 0; u + 1 < nsp; u++) {
      const uint32_t end = STAGED ? cb[u + 1] - base : start + (rbj[u * kRbStride + 1] - rbj[u * kRbStride]);
      if (pp >= end) t = u + 1;
      start = end;
    }
    return qt[t].weight;
  };

  if (STAGED) {
    const uint32_t P0 = cb[0] - base, P1 = cb[nsp] - base;  // staged indices relative to the span (< stage_cap <= 8192)
    if (P1 <= P0) return;
#pragma unroll 1
    for (uint32_t p = P0 + lane; p < P1; p += 32) {
      const uint32_t slot = sdoc[p] - tile_lo;
      if (slot < sub_docs) own[slot] = (unsigned short)p;
    }
    __syncwarp();
#pragma unroll 1
    for (uint32_t p = P0 + lane; p < P1; p += 32) {
      const uint32_t slot = sdoc[p] - tile_lo;
      if (slot < sub_docs) {
        const uint32_t o = own[slot];
        if ((o & (kOwnFlag - 1u)) != p) own[slot] = (unsigned short)(o | kOwnFlag);
      }
    }
    __syncwarp();
    uint32_t cut = cut_now();
#pragma unroll 1
    for (uint32_t b = P0; b < P1; b += 32) {
      const uint32_t p = b + lane;
      uint32_t slot = 0xFFFFFFFFu;
      if (p < P1) slot = sdoc[p] - tile_lo;
      uint32_t o = 0xFFFFFFFFu;
      if (slot < sub_docs) o = own[slot];
      const bool mine = (o & (kOwnFlag - 1u)) == p && o != 0xFFFFFFFFu;
      const bool conf = mine && (o & kOwnFlag);
      float v = 0.0f;
      if (mine && !conf) {
        v = ssc[p];
        if (!unit_w) v = __fmul_rn(v, weight_of(p));
      }
      const bool pass = mine && !conf && __float_as_uint(v) >= cut;
      if (__any_sync(0xFFFFFFFFu, pass)) {
        complete(pass, tile_lo + slot, v);
        cut = cut_now();
      }
      park(conf, slot, p);
    }
  } else {
    uint32_t start = 0;
    for (uint32_t t = 0; t < nsp; t++) {
      const uint32_t lo = rbj[t * kRbStride], hi = rbj[t * kRbStride + 1];
      const uint32_t *dp = seg.post_doc + qt[t].base;
#pragma unroll 1
      for (uint32_t i = lo + lane; i < hi; i += 32) own[dp[i] - tile_lo] = (unsigned short)(start + (i - lo));
      start += hi - lo;
    }
    __syncwarp();
    start = 0;
    for (uint32_t t = 0; t < nsp; t++) {
      const uint32_t lo = rbj[t * kRbStride], hi = rbj[t * kRbStride + 1];
      const uint32_t *dp = seg.post_doc + qt[t].base;
#pragma unroll 1
      for (uint32_t i = lo + lane; i < hi; i += 32) {
        const uint32_t slot = dp[i] - tile_lo, o = own[slot];
        if ((o & (kOwnFlag - 1u)) != start + (i - lo)) own[slot] = (unsigned short)(o | kOwnFlag);
      }
      start += hi - lo;
    }
    __syncwarp();
    uint32_t cut = cut_now();
    start = 0;
    for (uint32_t t = 0; t < nsp; t++) {
      const uint32_t lo = rbj[t * kRbStride], hi = rbj[t * kRbStride + 1];
      const uint32_t *dp = seg.post_doc + qt[t].base;
      const float *sp = wb.scores + qt[t].base;
      const float w = qt[t].weight;
#pragma unroll 1
      for (uint32_t b = lo; b < hi; b += 32) {
        const uint32_t i = b + lane;
        const bool in = i < hi;
        uint32_t slot = 0, o = 0xFFFFFFFFu;
        const uint32_t pp = start + (i - lo);
        if (in) {
          slot = dp[i] - tile_lo;
          o = own[slot];
        }
        const bool mine = in && (o & (kOwnFlag - 1u)) == pp;
        const bool conf = mine && (o & kOwnFlag);
        float v = 0.0f;
        if (mine && !conf) v = __fmul_rn(sp[i], w);
        const bool pass = mine && !conf && __float_as_uint(v) >= cut;
        if (__any_sync(0xFFFFFFFFu, pass)) {
          complete(pass, tile_lo + slot, v);
          cut = cut_now();
        }
        park(conf, slot, pp);
      }
      start += hi - lo;
    }
  }
  if (npend) resolve(npend);
  __syncwarp();
}

// One sub-tile of the sparse pass with BOUNDED ACCUMULATION (the default; option strict_accumulate 0).
//
// Every staged score of the sub-tile is read and compared; what is bounded is the per-doc summation.  A doc's sparse sum is
// at most (its posting's contribution) + (the largest contribution of every OTHER sparse term inside the sub-tile), and its
// score at most that + what the column terms can add (rest).  The maxima are taken from the staged values themselves — no
// index-time bound is consulted, the pruned executions do that — so:
//   A   the largest staged score M (one pass over the scores).  nsp * M * max weight + rest below the k-th score: no doc of
//       the sub-tile can enter the top k and nothing is summed
//   A2  otherwise the largest contribution per term, cmx[t]
//   B   a posting whose contribution + the other terms' maxima + rest reaches the k-th score has its doc summed exactly:
//       every sparse term in slot order (own contribution; the others found by binary search in their staged runs), then
//       the column terms (complete).  A doc with postings in several lists passes the test with each of them when it
//       matters; the posting of its first list offers it, the others stand back.
// The staging rounds runs out to 16 bytes: the few neighbours it drags in only loosen the maxima, and B tests the doc range.
__device__ __forceinline__ void sparse_sub_bounded(const SegmentDev &seg, const WarpBatchDev &wb, const QHead &head, const QTerm *qt, const uint32_t *cb,
                                                   const uint32_t base, const uint32_t nsp, const uint32_t colmask, const bool unit_w,
                                                   const float wmx, const float rest, const uint32_t tile_lo, const uint32_t sub_docs,
                                                   const uint32_t *sdoc, const float *ssc, float *cmx, WarpCand &wc, const int lane) {
  const uint32_t P0 = cb[0] - base, P1 = cb[nsp] - base;
  if (P1 <= P0) return;
  const bool have_thr = wc.thr != kThrInit;
  float thr_score = __uint_as_float((uint32_t)(wc.thr >> 32));
  if (have_thr) {
    uint32_t m = 0u;
#pragma unroll 1
    for (uint32_t p = P0 + lane; p < P1; p += 32) m = max(m, __float_as_uint(ssc[p]));
    m = __reduce_max_sync(0xFFFFFFFFu, m);
    if (((float)nsp * (__uint_as_float(m) * wmx) + rest) * 1.00002f < thr_score) return;
  }
  // ---- A2: per-term maxima ----
  float sum_all = 0.0f;
  for (uint32_t t = 0; t < nsp; t++) {
    const uint32_t c0 = cb[t] - base, c1 = cb[t + 1] - base;
    uint32_t m = 0u;
#pragma unroll 1
    for (uint32_t p = c0 + lane; p < c1; p += 32) m = max(m, __float_as_uint(ssc[p]));
    m = __reduce_max_sync(0xFFFFFFFFu, m);
    const float mt = __fmul_rn(__uint_as_float(m), qt[t].weight);
    if (lane == 0) cmx[t] = mt;
    sum_all += mt;
  }
  __syncwarp();
  if (have_thr && (sum_all + rest) * 1.00002f < thr_score) return;
  // ---- B: the postings whose docs can still qualify ----
  for (uint32_t t = 0; t < nsp; t++) {
    const uint32_t c0 = cb[t] - base, c1 = cb[t + 1] - base;
    if (c1 <= c0) continue;
    float other = rest;
    for (uint32_t u = 0; u < nsp; u++)
      if (u != t) other += cmx[u];
    const float w = qt[t].weight;
#pragma unroll 1
    for (uint32_t b = c0; b < c1; b += 32) {
      const uint32_t p = b + lane;
      float v = 0.0f;
      if (p < c1) v = unit_w ? ssc[p] : __fmul_rn(ssc[p], w);
      uint32_t cut = 0u;
      if (wc.thr != kThrInit) {
        const float cf = __uint_as_float((uint32_t)(wc.thr >> 32)) * 0.99998f - other * 1.00002f;
        cut = cf > 0.0f ? __float_as_uint(cf) : 0u;
      }
      bool pass = p < c1 && __float_as_uint(v) >= cut;
      if (!__any_sync(0xFFFFFFFFu, pass)) continue;
      uint32_t doc = 0u;
      if (pass) {
        doc = sdoc[p];
        pass = doc - tile_lo < sub_docs;
      }
      // the doc's exact sparse sum, slot order; a doc that an earlier list holds is that posting's to offer
      float s = 0.0f;
      if (pass) {
        for (uint32_t u = 0; u < nsp; u++) {
          float c = 0.0f;
          if (u == t) {
            c = v;
          } else {
            uint32_t lo = cb[u] - base, hi = cb[u + 1] - base;
            const uint32_t end = hi;
            while (lo < hi) {
              const uint32_t mid = (lo + hi) >> 1;
              if (sdoc[mid] < doc) lo = mid + 1;
              else hi = mid;
            }
            if (lo < end && sdoc[lo] == doc) {
              if (u < t) {
                pass = false;
                break;
              }
              c = __fmul_rn(ssc[lo], qt[u].weight);
            }
          }
          if (c != 0.0f) s = __fadd_rn(s, c);
        }
      }
      if (!__any_sync(0xFFFFFFFFu, pass)) continue;
      if (pass)
        for (uint32_t cm = colmask; cm; cm &= cm - 1) {
          const uint32_t ct = __ffs(cm) - 1;
          const float c = __ldg(seg.cols + qt[ct].sc_base + doc);
          s = __fadd_rn(s, __fmul_rn(c, qt[ct].weight));
        }
      wc.offer(seg, wb, head.qi, head.filter, pass, doc, s);
    }
  }
}

// ---- sparse pass -----------------------------------------------------------------------------------------------
template <bool UNUSED>
__global__ void __launch_bounds__(kSparseWarps * 32) slg_score_sparse_kernel(SegmentDev seg, WarpBatchDev wb, StreamDev sd) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t sub_docs = wb.sub_docs, cap = sd.stage_cap, k = wb.k;
  unsigned char *mine = smem_raw + (size_t)warp * sparse_smem_per_warp(sub_docs, cap);
  unsigned short *own = reinterpret_cast<unsigned short *>(mine);
  uint32_t *sdoc = reinterpret_cast<uint32_t *>(mine + (((size_t)sub_docs * 2 + 15) & ~(size_t)15));
  float *ssc = reinterpret_cast<float *>(sdoc + cap);
  unsigned long long *cand = reinterpret_cast<unsigned long long *>(ssc + cap);
  QTerm *qt = reinterpret_cast<QTerm *>(cand + kWarpCand);
  uint32_t *rb = reinterpret_cast<uint32_t *>(qt + kWarpMaxTerms);
  uint32_t *cum = rb + kWarpMaxTerms * kRbStride;                 // [65]: staged offset of cell j*8+t, whole item
  float *rest = reinterpret_cast<float *>(cum + 68);              // [jj] what the column terms can add
  float *cmx = rest + kSubPerGroup;                               // [t] largest contribution of term t inside the sub-tile at hand
  uint32_t *pend = reinterpret_cast<uint32_t *>(cmx + kWarpMaxTerms);
  unsigned long long *bar = reinterpret_cast<unsigned long long *>(pend + 64);
  if (lane == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncwarp();
  uint32_t parity = 0;
  const uint32_t total_items = wb.n_groups * wb.n_queries;
  uint32_t n_post = 0;  // per lane
  unsigned long long n_post_total = 0;
  uint32_t n_items = 0;
  WarpCand wc;

  uint32_t item = 0;
  if (lane == 0) item = atomicAdd(sd.sparse_counter, 1u);
  item = __shfl_sync(0xFFFFFFFFu, item, 0);
  while (item < total_items) {
    uint32_t next_item = 0;
    if (lane == 0) next_item = atomicAdd(sd.sparse_counter, 1u);
    const uint32_t tg = item / wb.n_queries, qslot = item - tg * wb.n_queries;
    const QHead head = wb.qheads[qslot];
    const uint32_t nt = head.nt;
    if (lane < 16) reinterpret_cast<uint4 *>(qt)[lane] = __ldg(reinterpret_cast<const uint4 *>(wb.qterms + (uint64_t)qslot * kWarpMaxTerms) + lane);
    const unsigned long long thr0 = load_threshold(wb, head.qi);
    __syncwarp();
    const uint32_t myflags = lane < (int)nt ? qt[lane].flags : 0u;
    const uint32_t spmask = __ballot_sync(0xFFFFFFFFu, (myflags & 5u) == 1u);  // canonical layout: the low nsp slots
    const uint32_t colmask = __ballot_sync(0xFFFFFFFFu, (myflags & 5u) == 5u);
    if (spmask) {
      n_items++;
      const uint32_t nsp = __popc(spmask);
      const bool unit_w = __all_sync(0xFFFFFFFFu, lane >= (int)nsp || qt[lane & 7].weight == 1.0f);
      float wmx = lane < (int)nsp ? qt[lane & 7].weight : 0.0f;  // largest weight of a sparse term
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) wmx = fmaxf(wmx, __shfl_xor_sync(0xFFFFFFFFu, wmx, o));
      wmx = __shfl_sync(0xFFFFFFFFu, wmx, 0);
      const uint32_t sub0 = tg * kSubPerGroup;
      const uint32_t jmax = min(kSubPerGroup, wb.n_sub - sub0);
      {
        // posting boundaries of the sparse terms: lane = t*4 + c
        const uint32_t t = lane >> 2, c = lane & 3;
        if (t < nsp) {
          const uint32_t *row = wb.rng + (uint64_t)qt[t].uterm * (wb.n_sub + 1);
          for (uint32_t j = c; j <= kSubPerGroup; j += 4) rb[t * kRbStride + j] = __ldg(row + min(sub0 + j, wb.n_sub));
        }
        // what the column terms can add to a partial inside each sub-tile: their exact maxima per 512 docs (seg.col_tmax)
        if (lane < (int)kSubPerGroup) {
          float r = 0.0f;
          if (lane < (int)jmax) {
            const uint32_t d0 = (sub0 + lane) * sub_docs, d1 = min(d0 + sub_docs, seg.doc_count) - 1u;
            for (uint32_t cm = colmask; cm; cm &= cm - 1) {
              const uint32_t ct = __ffs(cm) - 1;
              const float *tm = seg.col_tmax + (uint64_t)qt[ct].term * seg.tmax_stride;
              float b = 0.0f;
              for (uint32_t blk = d0 >> 9; blk <= (d1 >> 9); blk++) b = fmaxf(b, __ldg(tm + blk));
              r = __fadd_rn(r, __fmul_rn(b, qt[ct].weight));
            }
          }
          rest[lane] = r;
        }
      }
      __syncwarp();
      // cells e = j*8 + t, two per lane: the run of term t in sub-tile j rounded out to 16-byte pieces; cum = exclusive scan
      uint32_t len[2], alo[2];
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const uint32_t e = lane + 32 * h, t = e & 7, j = e >> 3;
        len[h] = 0;
        alo[h] = 0;
        if (t < nsp && j < jmax) {
          const uint32_t lo = rb[t * kRbStride + j], hi = rb[t * kRbStride + j + 1];
          if (hi > lo) {
            alo[h] = lo & ~3u;
            len[h] = ((hi + 3u) & ~3u) - alo[h];
            n_post += hi - lo;
          }
        }
      }
      {
        uint32_t s0 = len[0], s1 = len[1];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, s0, o), b2 = __shfl_up_sync(0xFFFFFFFFu, s1, o);
          if (lane >= o) {
            s0 += a;
            s1 += b2;
          }
        }
        s1 += __shfl_sync(0xFFFFFFFFu, s0, 31);
        cum[lane + 1] = s0;
        cum[lane + 33] = s1;
        if (lane == 0) cum[0] = 0;
      }
      __syncwarp();
      wc.begin(cand, thr0, k, lane);

      uint32_t j0 = 0;
      while (j0 < jmax) {
        // the longest span of sub-tiles [j0, j1) that fits the staging area
        const uint32_t base = cum[j0 * 8];
        const uint32_t jc = j0 + 1 + lane;  // lanes 0..7 try j1 = j0+1 .. j0+8
        const uint32_t tot = jc <= jmax ? cum[jc * 8] - base : 0xFFFFFFFFu;
        const uint32_t fits = __ballot_sync(0xFFFFFFFFu, jc <= jmax && tot <= cap);
        if (!(fits & 1u)) {  // a single sub-tile does not fit: straight from global memory
          sparse_sub<false>(seg, wb, head, qt, rb + j0, cum, 0u, nsp, colmask, unit_w, rest[j0], (sub0 + j0) * sub_docs, sub_docs, own, sdoc, ssc, pend, wc,
                            lane);
          j0++;
          continue;
        }
        const uint32_t nspan = __ffs(~fits) - 1;  // fits is a run of ones from bit 0 (cum grows)
        const uint32_t j1 = j0 + nspan;
        const uint32_t span_tot = __shfl_sync(0xFFFFFFFFu, tot, nspan - 1);
        if (span_tot == 0) {
          j0 = j1;
          continue;
        }
        // ---- stage: one bulk copy per non-empty cell and array, each lane its own cells ----
        __syncwarp();  // every lane is done reading the staging area of the previous span
        if (lane == 0) mbar_arrive_expect_tx(bar, span_tot * 8u);
        __syncwarp();
#pragma unroll
        for (int h = 0; h < 2; h++) {
          const uint32_t e = lane + 32 * h, t = e & 7, j = e >> 3;
          if (len[h] && j >= j0 && j < j1) {
            const uint32_t off = cum[e] - base;
            bulk_copy_g2s(sdoc + off, seg.post_doc + qt[t].base + alo[h], len[h] * 4u, bar);
            bulk_copy_g2s(ssc + off, wb.scores + qt[t].base + alo[h], len[h] * 4u, bar);
          }
        }
        mbar_wait(bar, parity);
        parity ^= 1u;
        for (uint32_t j = j0; j < j1; j++) {
          if (sd.strict)
            sparse_sub<true>(seg, wb, head, qt, rb + j, cum + j * 8, base, nsp, colmask, unit_w, rest[j], (sub0 + j) * sub_docs, sub_docs, own, sdoc, ssc,
                             pend, wc, lane);
          else
            sparse_sub_bounded(seg, wb, head, qt, cum + j * 8, base, nsp, colmask, unit_w, wmx, rest[j], (sub0 + j) * sub_docs, sub_docs, sdoc, ssc, cmx,
                               wc, lane);
        }
        j0 = j1;
      }
      wc.merge(wb, head.qi);
    }
    if (n_post > 0x40000000u) {
      n_post_total += n_post;
      n_post = 0;
    }
    item = __shfl_sync(0xFFFFFFFFu, next_item, 0);
  }
  if (sd.counters) {
    n_post_total += n_post;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n_post_total += __shfl_xor_sync(0xFFFFFFFFu, n_post_total, o);
    if (lane == 0) {
      if (n_post_total) atomicAdd(sd.counters + 0, n_post_total);
      if (n_items) atomicAdd(sd.counters + 3, (unsigned long long)n_items);
    }
  }
}

// position of the first posting with doc id >= doc in a list of n ascending doc ids.  Lists are near-uniform samples of the
// doc range, so a few guesses by local density (position + (doc - d) * n / doc_count) close in on the place before a binary
// search finishes in the bracket that is left; the bracket invariant keeps the result exact for any list.
__device__ __forceinline__ uint32_t lower_bound_interp(const uint32_t *dp, uint32_t n, uint32_t doc, float dens) {
  uint32_t lo = 0, hi = n;  // dp[i] < doc for i < lo, dp[i] >= doc for i >= hi
  float est = (float)doc * dens;
#pragma unroll 1
  for (int it = 0; it < 4 && lo < hi; it++) {
    const uint32_t pos = min(max(est < 0.0f ? 0u : (uint32_t)est, lo), hi - 1u);
    const uint32_t d = __ldg(dp + pos);
    if (d < doc) lo = pos + 1u;
    else hi = pos;
    if (d == doc) break;
    est = (float)pos + ((float)doc - (float)d) * dens;
  }
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (__ldg(dp + mid) < doc) lo = mid + 1u;
    else hi = mid;
  }
  return lo;
}

// exact score of one doc per lane: every term of the query in slot order (brute_force on the doc's lists).  holders: bit u set
// when sparse term u holds the doc.
__device__ __forceinline__ float verify_doc(const SegmentDev &seg, const WarpBatchDev &wb, const QTerm *qts, uint32_t nt, bool have, uint32_t doc,
                                            uint32_t &holders) {
  float s = 0.0f;
  holders = 0u;
  if (have) {
    for (uint32_t u = 0; u < nt; u++) {
      const uint32_t flags = __ldg(&qts[u].flags);
      if (!(flags & 1u)) continue;
      float c = 0.0f;
      if (flags & 4u) {
        c = __ldg(seg.cols + __ldg(&qts[u].sc_base) + doc);
      } else {
        const uint32_t term = __ldg(&qts[u].term);
        if (term < seg.n_terms) {
          const uint64_t base = __ldg(&qts[u].base);
          const int32_t row = seg.term_bits ? __ldg(seg.term_bits + term) : -1;
          bool held;
          uint32_t at = 0u;
          if (row >= 0) {
            held = presence_lookup(seg, (uint64_t)row * seg.bits_stride, doc, at);  // bit and list position from one sector
          } else {
            const uint32_t *dp = seg.post_doc + base;
            const uint32_t end = __ldg(seg.term_df + term);
            at = lower_bound_interp(dp, end, doc, (float)end / (float)max(seg.doc_count, 1u));
            held = at < end && __ldg(dp + at) == doc;
          }
          if (held) {
            c = __ldg(wb.scores + base + at);
            holders |= 1u << u;
          }
        }
      }
      if (c != 0.0f) s = __fadd_rn(s, __fmul_rn(c, __ldg(&qts[u].weight)));
    }
  }
  return s;
}

// ---- column pass -----------------------------------------------------------------------------------------------
// shared memory: buf f32[2][resident][kColBlock] | smax f32[n_smax] | cand u64[kColWarps][64] | bar u64[2]
__host__ __device__ inline size_t column_smem(uint32_t resident, uint32_t n_smax) {
  return (size_t)2 * resident * kColBlock * 4 + (((size_t)n_smax * 4 + 15) & ~(size_t)15) + (size_t)kColWarps * kWarpCand * 8 + 16;
}

template <bool PRUNE, bool POOLS>
__global__ void __launch_bounds__(kColWarps * 32) slg_score_columns_kernel(SegmentDev seg, WarpBatchDev wb, StreamDev sd) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint32_t s_hist[kColWarps][POOLS ? 256 : 1];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t n_used = *sd.n_ucol, n_colq = *sd.n_colq;
  const uint32_t resident = min(sd.col_resident, n_used), n_smax = min(n_used, sd.n_smax);
  float *buf = reinterpret_cast<float *>(smem_raw);
  float *smax = buf + (size_t)2 * sd.col_resident * kColBlock;
  unsigned long long *cand = reinterpret_cast<unsigned long long *>(reinterpret_cast<unsigned char *>(smax) + (((size_t)sd.n_smax * 4 + 15) & ~(size_t)15)) +
                             (size_t)warp * kWarpCand;
  unsigned long long *bar = reinterpret_cast<unsigned long long *>(smem_raw + column_smem(sd.col_resident, sd.n_smax) - 16);
  const uint32_t k = wb.k;
  const uint32_t n_blocks = (seg.doc_count + kColBlock - 1) / kColBlock;
  if (n_colq == 0 || n_used == 0) return;
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_init(bar + 1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();
  unsigned long long n_tests = 0, n_looked = 0;
  WarpCand wc;
  // one bulk copy per resident column; the column stride keeps a whole block past doc_count in bounds and zero
  auto fetch = [&](uint32_t blk, uint32_t b) {
    if (warp == 0) {
      if (lane == 0) mbar_arrive_expect_tx(bar + b, resident * kColBlock * 4u);
      __syncwarp();
      for (uint32_t s = lane; s < resident; s += 32)
        bulk_copy_g2s(buf + ((size_t)b * sd.col_resident + s) * kColBlock, seg.cols + (uint64_t)sd.ucol[s] * seg.col_stride + (uint64_t)blk * kColBlock,
                      kColBlock * 4u, bar + b);
    }
  };
  uint32_t parity[2] = {0u, 0u};
  uint32_t blk = blockIdx.x;
  if (blk < n_blocks) fetch(blk, 0);
  uint32_t b = 0;
  for (; blk < n_blocks; blk += gridDim.x, b ^= 1u) {
    const uint32_t nxt = blk + gridDim.x;
    if (nxt < n_blocks) fetch(nxt, b ^ 1u);  // the other buffer was released by the barrier that ended the previous block
    mbar_wait(bar + b, parity[b]);
    parity[b] ^= 1u;
    const float *cb = buf + (size_t)b * sd.col_resident * kColBlock;
    const uint32_t d0 = blk * kColBlock;
    // block maximum of every used column (non-resident columns: from global memory)
    for (uint32_t s = warp; s < n_smax; s += kColWarps) {
      const float4 *p = s < resident ? reinterpret_cast<const float4 *>(cb + (size_t)s * kColBlock)
                                     : reinterpret_cast<const float4 *>(seg.cols + (uint64_t)sd.ucol[s] * seg.col_stride + d0);
      uint32_t top = 0u;
#pragma unroll
      for (uint32_t x = 0; x < kColBlock / 128; x++) {
        const float4 v = p[x * 32 + lane];
        top = max(top, max(max(__float_as_uint(v.x), __float_as_uint(v.y)), max(__float_as_uint(v.z), __float_as_uint(v.w))));
      }
      top = __reduce_max_sync(0xFFFFFFFFu, top);
      if (lane == 0) smax[s] = __uint_as_float(top);
    }
    __syncthreads();
    // ---- every query with a column term against this block: lane g = one query ----
    for (uint32_t c0 = warp * 32; c0 < n_colq; c0 += kColWarps * 32) {
      ColQ cq;
      cq.ncol = 0;
      unsigned long long thr = ~0ull;
      const bool live = c0 + lane < n_colq;
      if (live) {
        cq = sd.colq[c0 + lane];
        thr = load_threshold(wb, cq.qi);
      }
      bool look = false;
      if (live && !cq.off) {
        n_tests++;
        // one column: the maximum over the block of c * w is max(c) * w, the comparison of every doc collapses into one.
        // Several columns: the sum of the maxima (same slot order, every operation monotone) dominates every doc's sum; the
        // strict exhaustive execution sums them per doc regardless.  extra (pruned): what unseen sparse terms could add.
        float bound = 0.0f;
        bool known = true;
        if (PRUNE || !sd.strict || cq.ncol == 1)
          for (uint32_t i = 0; i < cq.ncol; i++) {
            const uint32_t s = cq.slot[i];
            if (s >= n_smax) known = false;
            else bound = __fadd_rn(bound, __fmul_rn(smax[s], cq.unit_w ? 1.0f : __ldg(&wb.qterms[(uint64_t)cq.qslot * kWarpMaxTerms + cq.nsp + i].weight)));
          }
        else known = false;
        const uint32_t thr_bits = thr == kThrInit ? 0u : (uint32_t)(thr >> 32);
        if (PRUNE && cq.extra > 0.0f) bound = (bound + cq.extra) * 1.00002f;
        look = !known || (bound != 0.0f && __float_as_uint(bound) >= thr_bits);
      }
      uint32_t hits = __ballot_sync(0xFFFFFFFFu, look);
      if (!PRUNE && sd.strict) {
        // the common several-column shape — two unit-weight columns resident in shared memory: sum the block per doc
        // (slot order) and leave the query out of the per-doc pass below unless some doc can enter its top k
        const bool two = look && cq.ncol == 2 && cq.unit_w && cq.slot[0] < resident && cq.slot[1] < resident;
        uint32_t m2 = __ballot_sync(0xFFFFFFFFu, two);
        const uint32_t my01 = (uint32_t)cq.slot[0] | ((uint32_t)cq.slot[1] << 16);
        const uint32_t my_thr = thr == kThrInit ? 0u : (uint32_t)(thr >> 32);
        while (m2) {
          const int g = __ffs(m2) - 1;
          m2 &= m2 - 1;
          const uint32_t s01 = __shfl_sync(0xFFFFFFFFu, my01, g);
          const uint32_t tb = __shfl_sync(0xFFFFFFFFu, my_thr, g);
          const float4 *pa = reinterpret_cast<const float4 *>(cb + (size_t)(s01 & 0xFFFFu) * kColBlock) + lane;
          const float4 *pb = reinterpret_cast<const float4 *>(cb + (size_t)(s01 >> 16) * kColBlock) + lane;
          uint32_t mx = 0u;
#pragma unroll
          for (uint32_t x = 0; x < kColBlock / 128; x++) {
            const float4 a = pa[x * 32], c = pb[x * 32];
            const uint32_t m01 = max(__float_as_uint(__fadd_rn(a.x, c.x)), __float_as_uint(__fadd_rn(a.y, c.y)));
            const uint32_t m23 = max(__float_as_uint(__fadd_rn(a.z, c.z)), __float_as_uint(__fadd_rn(a.w, c.w)));
            mx = max(mx, max(m01, m23));
          }
          n_looked++;
          if (!__any_sync(0xFFFFFFFFu, mx >= tb && mx != 0u)) hits &= ~(1u << g);
        }
      }
      while (hits) {
        const int g = __ffs(hits) - 1;
        hits &= hits - 1;
        const uint32_t qslot = __shfl_sync(0xFFFFFFFFu, cq.qslot, g), qi = __shfl_sync(0xFFFFFFFFu, cq.qi, g);
        const uint32_t ncol = __shfl_sync(0xFFFFFFFFu, (uint32_t)cq.ncol, g), nsp = __shfl_sync(0xFFFFFFFFu, (uint32_t)cq.nsp, g);
        const uint32_t unit_w = __shfl_sync(0xFFFFFFFFu, (uint32_t)cq.unit_w, g);
        const int32_t filter = __shfl_sync(0xFFFFFFFFu, cq.filter, g);
        const unsigned long long qthr = __shfl_sync(0xFFFFFFFFu, thr, g);
        const float extra = PRUNE ? __shfl_sync(0xFFFFFFFFu, cq.extra, g) : 0.0f;
        const uint32_t nt = nsp + ncol;
        const uint32_t s01 = __shfl_sync(0xFFFFFFFFu, (uint32_t)cq.slot[0] | ((uint32_t)cq.slot[1] << 16), g);
        const uint32_t s23 = __shfl_sync(0xFFFFFFFFu, (uint32_t)cq.slot[2] | ((uint32_t)cq.slot[3] << 16), g);
        const uint32_t s45 = __shfl_sync(0xFFFFFFFFu, (uint32_t)cq.slot[4] | ((uint32_t)cq.slot[5] << 16), g);
        const uint32_t s67 = __shfl_sync(0xFFFFFFFFu, (uint32_t)cq.slot[6] | ((uint32_t)cq.slot[7] << 16), g);
        const QTerm *qts = wb.qterms + (uint64_t)qslot * kWarpMaxTerms;
        n_looked++;
        // v = sum of the query's columns over the block, slot order (the first product is the exact value of 0 + c * w)
        float4 v[kColBlock / 128];
#pragma unroll
        for (uint32_t x = 0; x < kColBlock / 128; x++) v[x] = make_float4(0, 0, 0, 0);
        for (uint32_t i = 0; i < ncol; i++) {
          const uint32_t pair = i < 2 ? s01 : (i < 4 ? s23 : (i < 6 ? s45 : s67));
          const uint32_t s = (i & 1u) ? pair >> 16 : pair & 0xFFFFu;
          const float w = unit_w ? 1.0f : __ldg(&qts[nsp + i].weight);
          const float4 *p = s < resident ? reinterpret_cast<const float4 *>(cb + (size_t)s * kColBlock)
                                         : reinterpret_cast<const float4 *>(seg.cols + (uint64_t)sd.ucol[s] * seg.col_stride + d0);
#pragma unroll
          for (uint32_t x = 0; x < kColBlock / 128; x++) {
            const float4 c = p[x * 32 + lane];
            v[x].x = __fadd_rn(v[x].x, __fmul_rn(c.x, w));
            v[x].y = __fadd_rn(v[x].y, __fmul_rn(c.y, w));
            v[x].z = __fadd_rn(v[x].z, __fmul_rn(c.z, w));
            v[x].w = __fadd_rn(v[x].w, __fmul_rn(c.w, w));
          }
        }
        // v can enter the top k when v (+ extra) reaches the k-th score
        auto cut_of = [&](unsigned long long th) {
          if (th == kThrInit) return 0u;
          if (!(PRUNE && extra > 0.0f)) return (uint32_t)(th >> 32);
          const float cf = __uint_as_float((uint32_t)(th >> 32)) * 0.99998f - extra * 1.00002f;
          return cf > 0.0f ? __float_as_uint(cf) : 0u;
        };
        uint32_t cut = cut_of(qthr);
        uint32_t mx = 0u;
#pragma unroll
        for (uint32_t x = 0; x < kColBlock / 128; x++)
          mx = max(mx, max(max(__float_as_uint(v[x].x), __float_as_uint(v[x].y)), max(__float_as_uint(v[x].z), __float_as_uint(v[x].w))));
        if (!__any_sync(0xFFFFFFFFu, mx >= cut && mx != 0u)) continue;
        // ---- per doc: the docs that can enter the top k, one per lane and round ----
        wc.begin(cand, qthr, k, lane, 1u, POOLS ? s_hist[warp] : nullptr);
        uint32_t todo = 0u;
#pragma unroll
        for (uint32_t x = 0; x < kColBlock / 128; x++) {
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
          for (uint32_t x = 0; x < kColBlock / 128; x++) {
            if (el == x * 4 + 0) bits = __float_as_uint(v[x].x);
            if (el == x * 4 + 1) bits = __float_as_uint(v[x].y);
            if (el == x * 4 + 2) bits = __float_as_uint(v[x].z);
            if (el == x * 4 + 3) bits = __float_as_uint(v[x].w);
          }
          const uint32_t doc = d0 + (el >> 2) * 128 + lane * 4 + (el & 3u);
          cut = cut_of(wc.thr);
          bool pass = had && bits >= cut;
          if (!__any_sync(0xFFFFFFFFu, pass)) continue;
          float sc_exact = __uint_as_float(bits);
          if (nsp) {
            // exhaustive: a doc of one of the query's sparse lists was met by the posting scan.  Pruned: such a list may have
            // been dropped as non-essential, so the doc gets its exact score here (the merge drops a key offered twice).
            uint32_t holders = 0u;
            sc_exact = verify_doc(seg, wb, qts, nt, pass, doc, holders);
            if (!PRUNE && holders) pass = false;
          }
          wc.offer(seg, wb, qi, filter, pass, doc, sc_exact);
        }
        wc.merge(wb, qi);
      }
    }
    __syncthreads();  // everyone is done with buffer b: the fetch two blocks ahead may overwrite it
  }
  if (sd.counters && lane == 0) {
    if (n_looked) atomicAdd(sd.counters + 1, n_looked);
    if (n_tests) atomicAdd(sd.counters + 2, n_tests);
  }
}

}  // namespace slg
