// slg_host.h — host-side state of libsearchlite_gpu.so shared by its translation units: device buffers, resident
// segments, the index handle and a prepared batch.  Not part of the ABI (include/searchlite_gpu.h is).
#pragma once
#include "../../include/searchlite_gpu.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include <cuda_runtime.h>

#include "slg_dispatch.h"
#include "slg_launch.h"

namespace slg {

// thread-local text of the last failed slg_open (no handle exists yet)
std::string &open_error();

// Per-batch buffers come from the device's stream-ordered pool (cudaMallocAsync): a prepare/free pair
// per batch then costs microseconds instead of a cudaMalloc/cudaFree round trip per buffer.  The scope
// guard names the stream; everything else (segment residency) uses plain cudaMalloc.
cudaStream_t &pool_stream();  // thread-local
struct PoolScope {
  cudaStream_t prev;
  explicit PoolScope(cudaStream_t s) : prev(pool_stream()) { pool_stream() = s; }
  ~PoolScope() { pool_stream() = prev; }
};

struct DevBuf {
  void *p = nullptr;
  size_t bytes = 0;
  cudaStream_t pool = nullptr;  // non-null: allocated with cudaMallocAsync on this stream
  bool borrowed = false;        // a view into another DevBuf's allocation: never freed here
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  DevBuf(DevBuf &&o) noexcept : p(o.p), bytes(o.bytes), pool(o.pool), borrowed(o.borrowed) { o.p = nullptr; o.bytes = 0; }
  DevBuf &operator=(DevBuf &&o) noexcept {
    if (this != &o) {
      release();
      p = o.p;
      bytes = o.bytes;
      pool = o.pool;
      borrowed = o.borrowed;
      o.p = nullptr;
      o.bytes = 0;
    }
    return *this;
  }
  ~DevBuf() { release(); }
  void view(void *ptr, size_t n) {  // borrow [ptr, ptr + n) from a slab that outlives this view
    release();
    p = ptr;
    bytes = n;
    borrowed = true;
  }
  void release() {
    if (p && !borrowed) {
      if (pool) cudaFreeAsync(p, pool);
      else cudaFree(p);
    }
    p = nullptr;
    bytes = 0;
    borrowed = false;
  }
  cudaError_t alloc(size_t n) {
    release();
    if (n == 0) n = 16;
    borrowed = false;
    pool = pool_stream();
    cudaError_t e = pool ? cudaMallocAsync(&p, n, pool) : cudaMalloc(&p, n);
    if (e == cudaSuccess) bytes = n;
    else p = nullptr;
    return e;
  }
  template <class T>
  T *as() const { return reinterpret_cast<T *>(p); }
};

struct CastU64 {
  __host__ __device__ uint64_t operator()(uint32_t v) const { return (uint64_t)v; }
};

struct Column {
  int kind = -1;  // 0 i64, 1 f64, 2 str, 3 i64 list, 4 f64 list, 5 str list; -1 = the segment lacks this column (predicates on it are false)
  DevBuf values; // i64 / f64 / u32 ords: one per doc (scalar kinds) or n_values of them (list kinds)
  DevBuf present;
  DevBuf offsets;  // list kinds: u32[doc_count + 1], the values of doc d are values[offsets[d] .. offsets[d + 1])
  uint64_t n_values = 0;
  std::vector<std::string> dict;
};

struct Vectors {
  uint32_t dim = 0;
  uint64_t n_rows = 0;
  bool bf16 = false;
  DevBuf offsets;  // u32[doc_count]
  DevBuf values;   // f32 or bf16 [n_rows][dim]
};

struct Segment {
  uint32_t ord = 0, doc_count = 0;
  uint64_t n_terms = 0, n_postings = 0, n_post_padded = 0;
  uint32_t n_blocks = 0, n_deleted = 0;
  float k1 = 0.9f, b = 0.4f, avgdl = 0, live_docs = 0, min_doc_len = 1;
  std::vector<uint32_t> h_df;  // host copy (query ordering, validation)
  DevBuf post_doc, post_tf, term_start, term_df, term_idf, term_max_tf, term_wide, tf_wide, term_blk, blk_max_doc,
      blk_max_tf, nk, live_bits, post_score, mb_max, cols, term_col, col_tmax, term_bits, pres_bits, term_ub;
  uint32_t n_bitmaps = 0;
  uint32_t n_cols = 0, tmax_stride = 0;
  uint64_t col_stride = 0;
  std::vector<int32_t> h_term_col;  // host copy (tests, introspection); empty = no columns
  SegmentDev dev{};
  std::vector<Column> columns;
  std::vector<DevBuf> filter_bits;  // per filter id (owning, or a view into one of filter_slabs)
  std::vector<std::shared_ptr<DevBuf>> filter_slabs;  // per filter id: the slab a view borrows from (or null)
  std::vector<uint64_t> h_start;    // host copy of term_start
  DevBuf filter_ptrs;               // device array of pointers into filter_bits
  Vectors vec;
  // term positions (index/postings.rs:117-125), kept for phrase matching: positions of padded posting slot i are
  // pos[pos_begin[i] .. pos_begin[i+1])
  DevBuf pos_begin, pos;
  uint64_t n_positions = 0;
  bool has_positions = false;
  bool avgdl_given = false;  // avgdl comes from the segment's .meta file instead of total_tokens / doc_count
  // further text fields of a handle that scores several ("title:..." next to "body:..."): field 0 is the one the
  // load call passes directly; these are set before finish_segment, which consumes the device copies
  struct ExtraField {
    DevBuf d_lens, d_present;
    float avgdl = 0.0f;
  };
  std::vector<ExtraField> extra_fields;
  std::vector<uint8_t> h_term_field;      // per term, empty = single field
  std::vector<float> f_avgdl, f_min_len;  // per field (index 0 = avgdl / min_doc_len)
  DevBuf term_field;
  size_t resident() const {
    return post_doc.bytes + post_tf.bytes + term_start.bytes + term_df.bytes + term_idf.bytes + term_max_tf.bytes +
           term_wide.bytes + tf_wide.bytes + term_blk.bytes + blk_max_doc.bytes + blk_max_tf.bytes + nk.bytes + term_field.bytes +
           live_bits.bytes + post_score.bytes + mb_max.bytes + cols.bytes + term_col.bytes + col_tmax.bytes + term_bits.bytes + pres_bits.bytes + term_ub.bytes +
           pos_begin.bytes + pos.bytes;
  }
};

struct FilterProg {
  std::vector<slg_filter_node_t> nodes;
  std::vector<std::string> strings;
};


}  // namespace slg

struct slg_index {
  int device = 0;
  int n_sm = 148;
  size_t smem_optin = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // 0/1 batch, 2/3 scoring, 4/5 rerank
  std::vector<std::unique_ptr<slg::Segment>> segs;
  std::vector<slg::FilterProg> filters;
  std::string err;
  slg_counters_t ctr{};
  void *pinned = nullptr;        // host staging buffer kept between batches (one batch at a time uses it)
  size_t pinned_bytes = 0;
  bool pinned_busy = false;
  void *merge_pinned = nullptr;  // staging of slg_merge_gathered*
  size_t merge_pinned_bytes = 0;
  uint32_t tile_docs = 16384;
  uint32_t ctas_per_sm = 0;  // 0 = as many as shared memory allows
  uint32_t sub_docs = 2048;  // warp kernel: docs per warp-private accumulator
  uint32_t kernel_choice = 0;  // 0 auto, 1 CTA-per-item kernel, 2 warp-per-item kernel (query order), 3 posting-driven items kernel (required)
  bool staging = true;         // use the resident per-posting scores (seg.post_score) where a kernel can
  // residency options (slg_set_option), applied to segments loaded afterwards
  bool resident_scores = true;   // build seg.post_score at load
  uint32_t dense_den = 24;       // a term gets a dense column when df * dense_den >= doc_count; 0 = no columns (C2: 8 -> 24 took the pruned batch from 9.5 to 7.6 ms for +8.7 GB)
  uint32_t dense_min_df = 256;   // ... and df >= this
  uint32_t bitmap_den = 512;     // a term without a column gets a presence bitmap with rank (slg_residency.cuh) when df * bitmap_den >= doc_count; 0 = none
  uint64_t max_bitmap_bytes = 16ull << 30;
  uint64_t max_column_bytes = 24ull << 30;
  uint32_t stage_cap = 1024;     // sparse pass: postings a warp stages in shared memory per span (slg_stream_kernel.cuh)
  uint32_t strict_accumulate = 0; // exhaustive stream kernels: 1 = sum every posting per doc; 0 = bounded accumulation (slg_stream_kernel.cuh)
  uint32_t dbg = 0;
  uint32_t scan_chunk = 0;       // flat posting scan: postings per work item (multiple of 256); 0 = by segment size (4096 / 2048 / 1024)
  uint32_t scan_first_part = 24; // two-step (sharded) runs: the first step scans this many 256ths of the items (rarest first) before the threshold exchange
  uint32_t scan_kernels = 1;     // plain OR batches: 1 = flat posting scan + column pass (slg_scan_kernel.cuh), 0 = the sub-tile kernels
  uint32_t stream_kernels = 1;   // exhaustive plain OR batches: 1 = sparse pass + column pass, 0 = the items kernel
  uint32_t maxscore_pct = 35;    // pruned warp kernel: non-essential bounds may sum to this % of the k-th score (0 = tile skip only)
  bool keep_positions = true;    // keep term positions resident when a posting image carries them (SegmentReader keep_positions)
  // term space of segments loaded from the reference's files: "field:token" key -> term id, in order of first appearance
  std::unordered_map<std::string, uint32_t> term_ids;
  std::string term_field;        // the text field(s) those keys belong to, as named at load ("body" or "title,body")
  std::vector<uint8_t> term_field_of;  // term id -> index of its field in that list
  // fast-field columns by name (handles are indices into every segment's `columns`)
  std::vector<std::string> column_names;
  slg::Segment *find(uint32_t ord) {
    for (auto &s : segs)
      if (s->ord == ord) return s.get();
    return nullptr;
  }
};

namespace slg {

inline int32_t fail(slg_index *ix, int32_t code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ix) ix->err = buf;
  else open_error() = buf;
  return code;
}

#define SLG_CUDA(ix, call)                                                                         \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return fail((ix), e__ == cudaErrorMemoryAllocation ? SLG_ERR_OOM : SLG_ERR_CUDA, "%s: %s (%s:%d)", #call, \
                  cudaGetErrorString(e__), __FILE__, __LINE__);                                    \
  } while (0)

inline void count_launch(slg_index *ix, uint64_t n = 1) { ix->ctr.kernel_launches += n; }

// idf exactly as query/bm25.rs:2 with docs = live docs (api/reader.rs:2985) and df = list length
// f32::max returns the non-NaN operand (ln of a negative ratio when df > N + 0.5 after deletions): fmaxf
inline float host_idf(float df, float docs) { return fmaxf(logf((docs - df + 0.5f) / (df + 0.5f)), 0.0f) + 1.0f; }
inline float host_nk(float dl, float avgdl, float k1, float b) {
  volatile float norm = avgdl > 0.0f ? dl / avgdl : 1.0f;
  volatile float bn = b * norm;
  volatile float omb = 1.0f - b;
  volatile float s = omb + bn;
  volatile float r = k1 * s;
  return r;
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// SLG_LOAD_TRACE=1: wall-clock time of every residency stage on stderr (the stream is synchronised at each mark)
struct StageTimer {
  bool on;
  cudaStream_t st;
  std::chrono::steady_clock::time_point t0;
  explicit StageTimer(cudaStream_t s) : on(getenv("SLG_LOAD_TRACE") != nullptr), st(s), t0(std::chrono::steady_clock::now()) {}
  void mark(const char *what) {
    if (!on) return;
    cudaStreamSynchronize(st);
    const auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[slg load] %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  }
};

}  // namespace slg

// One prepared batch (slg_batch_prepare): every device buffer is a view into ONE slab from the stream-ordered
// pool, every host input travels in ONE packed host-to-device copy out of pinned memory, and nothing in
// prepare waits for the device.
struct slg_batch {
  slg_index *ix = nullptr;
  uint32_t Q = 0, k = 0, cap = 0, U = 0, T = 0;
  slg_exec_t exec = SLG_EXEC_BM25;
  bool matcher = false;
  bool want_stats = false;
  uint64_t posting_count = 0;
  slg::DevBuf slab;
  unsigned char *d_pack = nullptr;  // packed inputs (offsets below)
  size_t pack_bytes = 0;
  size_t off_ut_term = 0, off_q_term_off = 0, off_qt_uterm = 0, off_qt_weight = 0, off_qt_group = 0, off_qt_flags = 0,
         off_q_order = 0, off_q_must = 0, off_q_not = 0, off_q_should = 0, off_q_min = 0, off_q_filter = 0,
         off_qt_leaf = 0, off_q_leaves = 0, off_q_plan_off = 0, off_plan_nodes = 0, off_cursor_bounds = 0;
  // state + outputs (views into the slab)
  uint32_t *ut_rng = nullptr;
  float *ut_tile_ub = nullptr;
  unsigned char *state = nullptr;  // thr_key | topk_count | lock | work_counter | item_counters | n_items: reset per segment
  size_t state_bytes = 0;
  unsigned long long *thr_key = nullptr, *topk_keys = nullptr, *stats = nullptr, *item_counters = nullptr;
  uint32_t *topk_count = nullptr, *lock = nullptr, *work_counter = nullptr, *n_items = nullptr, *cursor_saw = nullptr;
  slg::QTerm *qterms = nullptr;
  slg::QHead *qheads = nullptr;
  uint2 *items = nullptr;
  slg::ColQ *colq = nullptr;          // exhaustive two-pass path: queries grouped by their first column, chunk list, scratch
  uint32_t *ucol = nullptr, *col_slot = nullptr;
  // flat posting scan (slg_scan_kernel.cuh)
  float *ut_max = nullptr;
  slg::ScanPair *scan_pairs = nullptr;
  uint32_t *scan_order = nullptr, *scan_item_start = nullptr, *scan_items = nullptr;
  uint32_t scan_items_cap = 0, scan_chunk = 4096;
  uint32_t max_cols = 0;
  uint8_t *done = nullptr;
  size_t done_bytes = 0;
  uint32_t items_cap = 0;
  unsigned char *results = nullptr;   // per segment: hits [Q][k], counts [Q], vector scores [Q][k] (after a rerank); then the merged block (S > 1)
  size_t result_stride = 0;           // bytes of one such block
  uint32_t max_terms = 0;
  slg::Selection sel;                 // which kernels the batch may take (slg_dispatch.h)
  unsigned long long *pool_keys = nullptr;
  uint32_t *pool_count = nullptr, *pool_lock = nullptr;
  uint32_t pool_cap = 0;
  bool has_cursor = false;            // some query carries a search-after cursor
  std::vector<uint8_t> h_has_cursor;
  uint32_t n_cursor_segs = 0;
  bool has_plan = false;              // some query carries a ScorePlan
  uint32_t max_leaves = 1;
  uint32_t plan_docs = 0;             // docs per tile / sub-tile of this batch
  uint32_t sub_tiles_max = 0;
  uint32_t n_segs_run = 0;
  // sharded runs: threshold board in peer-accessible memory (slg_batch_set_threshold_board); board == nullptr: none
  unsigned long long *board = nullptr;
  unsigned long long *peer_board[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  uint32_t n_board_peers = 0, board_epoch = 0;
  bool reranked = false;              // slg_rerank_batch ran on the last results: the blocks carry hybrid scores + vector scores
  bool seeds_done = false;            // two-step run (slg_batch_run_seeds / slg_batch_run_sweep)
  void *pinned = nullptr;             // [pack | results | stats]
  size_t pinned_bytes = 0, pinned_result_off = 0;
  bool pinned_from_index = false;
  ~slg_batch() {
    if (pinned_from_index) ix->pinned_busy = false;
    else if (pinned) {
      if (!ix->pinned_busy && pinned_bytes > ix->pinned_bytes) {  // keep the larger buffer for the next batch
        if (ix->pinned) cudaFreeHost(ix->pinned);
        ix->pinned = pinned;
        ix->pinned_bytes = pinned_bytes;
      } else {
        cudaFreeHost(pinned);
      }
    }
  }
};
