// slg_engine.cu — host side of libsearchlite_gpu.so: residency, batch preparation, kernel
// launches and the C ABI declared in include/searchlite_gpu.h.
//
// Mirrors, for the hot path only:
//   SegmentReader::open / live_docs / avg_field_length   searchlite-core/src/index/segment.rs:1239,1344,1365
//   IndexReader::search_segment                           src/api/reader.rs:2908-3128
//   execute_top_k_with_stats_and_mode_internal            src/query/wand.rs:398-456
//   hits.sort_by(SortKey)                                 src/api/reader.rs:2777
// There is no CPU fallback anywhere in this file: every search runs the CUDA kernels or fails.
#include "slg_host.h"

#include <cub/cub.cuh>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "slg_filter.cuh"
#include "slg_phrase.cuh"
#include "slg_postimage.cuh"
#include "slg_residency.cuh"
#include "slg_segfiles.h"

using namespace slg;

namespace slg {
std::string &open_error() {
  thread_local std::string e;
  return e;
}
cudaStream_t &pool_stream() {
  thread_local cudaStream_t s = nullptr;
  return s;
}
}  // namespace slg

namespace {

struct CastU64 {
  __host__ __device__ uint64_t operator()(uint32_t v) const { return (uint64_t)v; }
};

// --------------------------------------------------------------------------------------------
// residency
int32_t finish_segment(slg_index *ix, std::unique_ptr<Segment> seg, const int64_t *d_lens, const uint8_t *d_present,
                       uint64_t total_tokens, const uint32_t *deleted, uint32_t n_deleted) {
  cudaStream_t st = ix->stream;
  Segment *s = seg.get();
  // compute_avg_lengths index/segment.rs:946-957
  if (!s->avgdl_given) s->avgdl = s->doc_count == 0 ? 0.0f : (float)total_tokens / (float)(uint64_t)s->doc_count;
  // deleted docs -> live bitmap; live_docs index/segment.rs:1365-1370
  uint32_t words = (s->doc_count + 31) / 32;
  std::vector<uint32_t> live(words, 0xFFFFFFFFu);
  if (s->doc_count & 31) live[words - 1] = (1u << (s->doc_count & 31)) - 1u;
  uint32_t nd = 0;
  for (uint32_t i = 0; i < n_deleted; i++) {
    uint32_t d = deleted[i];
    if (d < s->doc_count && (live[d >> 5] >> (d & 31) & 1u)) {
      live[d >> 5] &= ~(1u << (d & 31));
      nd++;
    }
  }
  s->n_deleted = nd;
  s->live_docs = (float)(s->doc_count - nd);
  SLG_CUDA(ix, s->live_bits.alloc((size_t)std::max(words, 1u) * 4));
  if (words) SLG_CUDA(ix, cudaMemcpyAsync(s->live_bits.p, live.data(), (size_t)words * 4, cudaMemcpyHostToDevice, st));
  // idf per term on the host (glibc logf, like the reference's f32::ln)
  std::vector<float> idf(s->n_terms);
  for (uint64_t t = 0; t < s->n_terms; t++) idf[t] = host_idf((float)s->h_df[t], s->live_docs);
  SLG_CUDA(ix, s->term_idf.alloc(s->n_terms * 4));
  if (s->n_terms) SLG_CUDA(ix, cudaMemcpyAsync(s->term_idf.p, idf.data(), s->n_terms * 4, cudaMemcpyHostToDevice, st));
  // norms: one [doc_count] vector per scored text field
  const uint32_t n_fields = 1 + (uint32_t)s->extra_fields.size();
  if (n_fields > kMaxFields) return fail(ix, SLG_ERR_UNSUPPORTED, "more than %u text fields in one handle", kMaxFields);
  const size_t nk_stride = s->doc_count;
  SLG_CUDA(ix, s->nk.alloc(std::max<size_t>(nk_stride * n_fields, 1) * 4));
  s->f_avgdl.assign(n_fields, 0.0f);
  s->f_min_len.assign(n_fields, 1.0f);
  DevBuf minbits;
  SLG_CUDA(ix, minbits.alloc(4));
  for (uint32_t f = 0; f < n_fields; f++) {
    const float avgdl_f = f == 0 ? s->avgdl : s->extra_fields[f - 1].avgdl;
    const int64_t *lens_f = f == 0 ? d_lens : s->extra_fields[f - 1].d_lens.as<int64_t>();
    const uint8_t *pres_f = f == 0 ? d_present : s->extra_fields[f - 1].d_present.as<uint8_t>();
    uint32_t inf_bits = 0x7F800000u;
    SLG_CUDA(ix, cudaMemcpyAsync(minbits.p, &inf_bits, 4, cudaMemcpyHostToDevice, st));
    if (s->doc_count) {
      slg_norms_kernel<<<(s->doc_count + 255) / 256, 256, 0, st>>>(lens_f, pres_f, s->doc_count, avgdl_f, s->k1, s->b,
                                                                     s->nk.as<float>() + nk_stride * f, minbits.as<uint32_t>());
      count_launch(ix);
    }
    uint32_t got = 0;
    SLG_CUDA(ix, cudaMemcpyAsync(&got, minbits.p, 4, cudaMemcpyDeviceToHost, st));
    SLG_CUDA(ix, cudaStreamSynchronize(st));
    float mn;
    std::memcpy(&mn, &got, 4);
    s->f_avgdl[f] = avgdl_f;
    s->f_min_len[f] = std::isfinite(mn) ? mn : std::max(avgdl_f, 1.0f);  // query/wand.rs:117-121
  }
  s->min_doc_len = s->f_min_len[0];
  s->extra_fields.clear();  // the device copies of the length columns are no longer needed
  if (n_fields > 1) {
    if (s->h_term_field.size() != s->n_terms) return fail(ix, SLG_ERR_INVALID, "multi-field segment without a term -> field table");
    SLG_CUDA(ix, s->term_field.alloc(std::max<uint64_t>(s->n_terms, 1)));
    if (s->n_terms) SLG_CUDA(ix, cudaMemcpyAsync(s->term_field.p, s->h_term_field.data(), s->n_terms, cudaMemcpyHostToDevice, st));
  }

  SegmentDev &d = s->dev;
  d.post_doc = s->post_doc.as<uint32_t>();
  d.post_tf = s->post_tf.as<uint8_t>();
  d.term_start = s->term_start.as<uint64_t>();
  d.term_df = s->term_df.as<uint32_t>();
  d.term_idf = s->term_idf.as<float>();
  d.term_max_tf = s->term_max_tf.as<float>();
  d.term_wide = s->term_wide.as<uint64_t>();
  d.tf_wide = s->tf_wide.as<uint32_t>();
  d.term_blk = s->term_blk.as<uint32_t>();
  d.blk_max_doc = s->blk_max_doc.as<uint32_t>();
  d.blk_max_tf = s->blk_max_tf.as<float>();
  d.nk = s->nk.as<float>();
  d.live_bits = s->live_bits.as<uint32_t>();
  d.post_score = nullptr;
  d.mb_max = nullptr;
  d.cols = nullptr;
  d.term_col = nullptr;
  d.col_tmax = nullptr;
  d.tmax_stride = 0;
  d.col_stride = 0;
  d.term_ub = nullptr;
  d.term_bits = nullptr;
  d.pres_bits = nullptr;
  d.bits_stride = 0;
  d.n_terms = s->n_terms;
  d.doc_count = s->doc_count;
  d.k1p1 = s->k1 + 1.0f;
  d.min_nk = host_nk(s->min_doc_len, s->avgdl, s->k1, s->b);
  d.term_field = n_fields > 1 ? s->term_field.as<uint8_t>() : nullptr;
  for (uint32_t f = 0; f < kMaxFields; f++)
    d.min_nk_f[f] = f < n_fields ? host_nk(s->f_min_len[f], s->f_avgdl[f], s->k1, s->b) : d.min_nk;

  // resident unit-weight scores: score_tf(tf, df, doc_len, ...) of every posting, once
  if (ix->resident_scores && s->n_blocks) {
    SLG_CUDA(ix, s->post_score.alloc(s->n_post_padded * 4));
    SLG_CUDA(ix, cudaMemsetAsync(s->post_score.p, 0, s->n_post_padded * 4, st));
    SLG_CUDA(ix, s->mb_max.alloc((s->n_post_padded / 32 + 1) * 4));
    SLG_CUDA(ix, cudaMemsetAsync(s->mb_max.p, 0, (s->n_post_padded / 32 + 1) * 4, st));
    slg_score_postings_kernel<<<s->n_blocks, 128, 0, st>>>(d, s->n_blocks, s->post_score.as<float>(), s->mb_max.as<float>());
    count_launch(ix);
    SLG_CUDA(ix, cudaGetLastError());
    d.post_score = s->post_score.as<float>();
    d.mb_max = s->mb_max.as<float>();
    // dense columns for the high-df terms, largest df first until the byte budget is spent
    if (ix->dense_den && s->doc_count) {
      const uint64_t stride = align_up((uint64_t)s->doc_count, 4096) + 4096;  // a whole staged block past the end stays in bounds and zero
      std::vector<uint32_t> cand;
      for (uint64_t t = 0; t < s->n_terms; t++) {
        const uint64_t df = s->h_df[t];
        if (df >= ix->dense_min_df && df * ix->dense_den >= s->doc_count) cand.push_back((uint32_t)t);
      }
      std::sort(cand.begin(), cand.end(), [&](uint32_t a, uint32_t b2) { return s->h_df[a] != s->h_df[b2] ? s->h_df[a] > s->h_df[b2] : a < b2; });
      const uint64_t max_cols = std::min<uint64_t>(65535, ix->max_column_bytes / (stride * 4));
      if (cand.size() > max_cols) cand.resize(max_cols);
      if (!cand.empty()) {
        std::vector<int32_t> tcol(s->n_terms, -1);
        for (size_t c = 0; c < cand.size(); c++) tcol[cand[c]] = (int32_t)c;
        DevBuf d_terms;
        SLG_CUDA(ix, d_terms.alloc(cand.size() * 4));
        SLG_CUDA(ix, cudaMemcpyAsync(d_terms.p, cand.data(), cand.size() * 4, cudaMemcpyHostToDevice, st));
        SLG_CUDA(ix, s->term_col.alloc(s->n_terms * 4));
        SLG_CUDA(ix, cudaMemcpyAsync(s->term_col.p, tcol.data(), s->n_terms * 4, cudaMemcpyHostToDevice, st));
        SLG_CUDA(ix, s->cols.alloc(cand.size() * stride * 4));
        SLG_CUDA(ix, cudaMemsetAsync(s->cols.p, 0, cand.size() * stride * 4, st));
        s->n_cols = (uint32_t)cand.size();
        s->col_stride = stride;
        d.col_stride = stride;
        for (size_t c0 = 0; c0 < cand.size(); c0 += 32768) {  // gridDim.y limit
          const uint32_t nc = (uint32_t)std::min<size_t>(32768, cand.size() - c0);
          slg_fill_columns_kernel<<<dim3(256, nc), 256, 0, st>>>(d, d_terms.as<uint32_t>() + c0, nc,
                                                                  s->cols.as<float>() + c0 * stride);
          count_launch(ix);
        }
        SLG_CUDA(ix, cudaGetLastError());
        // exact per-512-doc maxima of every column: the tile bounds of the pruned modes
        s->tmax_stride = (uint32_t)(stride / 512);
        SLG_CUDA(ix, s->col_tmax.alloc(cand.size() * s->tmax_stride * 4));
        {
          const uint64_t warps = (uint64_t)cand.size() * s->tmax_stride;
          slg_column_tmax_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(s->cols.as<float>(), stride, (uint32_t)cand.size(),
                                                                                     s->tmax_stride, s->col_tmax.as<float>());
          count_launch(ix);
        }
        SLG_CUDA(ix, cudaGetLastError());
        SLG_CUDA(ix, cudaStreamSynchronize(st));  // host vectors go out of scope
        s->h_term_col = std::move(tcol);
        d.cols = s->cols.as<float>();
        d.term_col = s->term_col.as<int32_t>();
        d.col_tmax = s->col_tmax.as<float>();
        d.tmax_stride = s->tmax_stride;
      }
    }
  }
  // the largest contribution of every term: the bounds of the pruned executions (wand.rs:126-135 takes the stored max tf at the
  // segment's minimum doc length; this is the maximum over the postings themselves, tighter and safe for the same reason)
  if (d.post_score && s->n_terms) {
    SLG_CUDA(ix, s->term_ub.alloc(s->n_terms * 4));
    SLG_CUDA(ix, cudaMemsetAsync(s->term_ub.p, 0, s->n_terms * 4, st));
    ScanDev sc{};
    sc.ut_term = nullptr;
    sc.ut_max = s->term_ub.as<float>();
    slg_term_max_kernel<<<dim3((unsigned)((s->n_terms + 7) / 8), kMaxSlices), 256, 0, st>>>(d, sc, (uint32_t)s->n_terms);
    count_launch(ix);
    SLG_CUDA(ix, cudaGetLastError());
    d.term_ub = s->term_ub.as<float>();
  }
  // presence bitmaps with interleaved rank for the mid-dense terms without a column: the posting scan's verification asks
  // "does this list hold the doc, and where", and one 32-byte sector answers both where a search reads several
  if (ix->resident_scores && ix->bitmap_den && s->doc_count && s->n_blocks) {
    const uint32_t stride = presence_row_words(s->doc_count);
    std::vector<uint32_t> cand;
    for (uint64_t t = 0; t < s->n_terms; t++) {
      const uint64_t df = s->h_df[t];
      if (df >= 64 && df * ix->bitmap_den >= s->doc_count && (s->h_term_col.empty() || s->h_term_col[t] < 0)) cand.push_back((uint32_t)t);
    }
    std::sort(cand.begin(), cand.end(), [&](uint32_t a, uint32_t b2) { return s->h_df[a] != s->h_df[b2] ? s->h_df[a] > s->h_df[b2] : a < b2; });
    const uint64_t max_rows = std::min<uint64_t>(32768, ix->max_bitmap_bytes / ((uint64_t)stride * 4));
    if (cand.size() > max_rows) cand.resize(max_rows);
    if (!cand.empty()) {
      std::vector<int32_t> tb(s->n_terms, -1);
      for (size_t r = 0; r < cand.size(); r++) tb[cand[r]] = (int32_t)r;
      DevBuf d_terms;
      SLG_CUDA(ix, d_terms.alloc(cand.size() * 4));
      SLG_CUDA(ix, cudaMemcpyAsync(d_terms.p, cand.data(), cand.size() * 4, cudaMemcpyHostToDevice, st));
      SLG_CUDA(ix, s->term_bits.alloc(s->n_terms * 4));
      SLG_CUDA(ix, cudaMemcpyAsync(s->term_bits.p, tb.data(), s->n_terms * 4, cudaMemcpyHostToDevice, st));
      SLG_CUDA(ix, s->pres_bits.alloc(cand.size() * (uint64_t)stride * 4));
      SLG_CUDA(ix, cudaMemsetAsync(s->pres_bits.p, 0, cand.size() * (uint64_t)stride * 4, st));
      slg_fill_presence_kernel<<<dim3(64, (unsigned)cand.size()), 256, 0, st>>>(d, d_terms.as<uint32_t>(), (uint32_t)cand.size(), s->pres_bits.as<uint32_t>(), stride);
      count_launch(ix);
      SLG_CUDA(ix, cudaGetLastError());
      DevBuf d_totals;
      SLG_CUDA(ix, d_totals.alloc(cand.size() * 4));
      slg_presence_rank_kernel<<<(unsigned)cand.size(), kRankThreads, 0, st>>>(s->pres_bits.as<uint32_t>(), stride, (uint32_t)cand.size(), d_totals.as<uint32_t>());
      count_launch(ix);
      SLG_CUDA(ix, cudaGetLastError());
      std::vector<uint32_t> totals(cand.size());
      SLG_CUDA(ix, cudaMemcpyAsync(totals.data(), d_totals.p, cand.size() * 4, cudaMemcpyDeviceToHost, st));
      SLG_CUDA(ix, cudaStreamSynchronize(st));
      // every row must count exactly its list: a look-up's rank is a posting index, so a wrong count would read another posting
      for (size_t r = 0; r < cand.size(); r++)
        if (totals[r] != s->h_df[cand[r]])
          return fail(ix, SLG_ERR_INVALID, "segment %u: presence bitmap of term %u counts %u docs, its list holds %u", s->ord, cand[r], totals[r],
                      s->h_df[cand[r]]);
      s->n_bitmaps = (uint32_t)cand.size();
      d.term_bits = s->term_bits.as<int32_t>();
      d.pres_bits = s->pres_bits.as<uint32_t>();
      d.bits_stride = stride;
    }
  }
  ix->ctr.resident_bytes += s->resident();
  // replace a segment with the same ordinal
  for (auto &old : ix->segs)
    if (old->ord == s->ord) {
      ix->ctr.resident_bytes -= old->resident();
      old = std::move(seg);
      return SLG_OK;
    }
  ix->segs.push_back(std::move(seg));
  std::sort(ix->segs.begin(), ix->segs.end(), [](const auto &a, const auto &b2) { return a->ord < b2->ord; });
  return SLG_OK;
}

// layout tables shared by both load paths: df -> padded starts, block starts
int32_t build_layout(slg_index *ix, Segment *s) {
  cudaStream_t st = ix->stream;
  std::vector<uint64_t> start(s->n_terms + 1);
  std::vector<uint32_t> blk(s->n_terms + 1);
  uint64_t pos = 0, nb = 0, np = 0;
  for (uint64_t t = 0; t < s->n_terms; t++) {
    start[t] = pos;
    blk[t] = (uint32_t)nb;
    uint32_t df = s->h_df[t];
    np += df;
    pos += align_up(df, kTermAlign);
    nb += (df + kBlock - 1) / kBlock;
    if (nb > 0xFFFFFFF0ull) return fail(ix, SLG_ERR_UNSUPPORTED, "segment has too many posting blocks");
  }
  start[s->n_terms] = pos;
  blk[s->n_terms] = (uint32_t)nb;
  s->n_postings = np;
  s->n_post_padded = pos + 1024;  // tail slack so that vector loads past a list never leave the buffer
  s->n_blocks = (uint32_t)nb;
  SLG_CUDA(ix, s->term_start.alloc((s->n_terms + 1) * 8));
  SLG_CUDA(ix, s->term_blk.alloc((s->n_terms + 1) * 4));
  SLG_CUDA(ix, s->term_df.alloc(std::max<uint64_t>(s->n_terms, 1) * 4));
  SLG_CUDA(ix, cudaMemcpyAsync(s->term_start.p, start.data(), (s->n_terms + 1) * 8, cudaMemcpyHostToDevice, st));
  SLG_CUDA(ix, cudaMemcpyAsync(s->term_blk.p, blk.data(), (s->n_terms + 1) * 4, cudaMemcpyHostToDevice, st));
  if (s->n_terms) SLG_CUDA(ix, cudaMemcpyAsync(s->term_df.p, s->h_df.data(), s->n_terms * 4, cudaMemcpyHostToDevice, st));
  SLG_CUDA(ix, s->post_doc.alloc(s->n_post_padded * 4));
  SLG_CUDA(ix, s->post_tf.alloc(s->n_post_padded));
  SLG_CUDA(ix, cudaMemsetAsync(s->post_doc.p, 0xFF, s->n_post_padded * 4, st));
  SLG_CUDA(ix, cudaMemsetAsync(s->post_tf.p, 0, s->n_post_padded, st));
  SLG_CUDA(ix, s->blk_max_doc.alloc((size_t)std::max(s->n_blocks, 1u) * 4));
  SLG_CUDA(ix, s->blk_max_tf.alloc((size_t)std::max(s->n_blocks, 1u) * 4));
  SLG_CUDA(ix, s->term_max_tf.alloc(std::max<uint64_t>(s->n_terms, 1) * 4));
  SLG_CUDA(ix, s->term_wide.alloc(std::max<uint64_t>(s->n_terms, 1) * 8));
  SLG_CUDA(ix, cudaMemsetAsync(s->term_wide.p, 0xFF, std::max<uint64_t>(s->n_terms, 1) * 8, st));
  SLG_CUDA(ix, cudaStreamSynchronize(st));  // host vectors go out of scope
  s->h_start = std::move(start);
  return SLG_OK;
}

// after post_tf / blk_max_tf are filled: per-term max tf and the wide-tf side table
int32_t build_wide(slg_index *ix, Segment *s, const uint64_t *d_csr_off, const uint32_t *d_csr_tfs, const uint4 *d_ovf = nullptr,
                   uint32_t n_ovf = 0) {
  cudaStream_t st = ix->stream;
  if (!s->n_terms) return SLG_OK;
  if (s->n_blocks) {  // untrusted input: doc ids inside the segment, lists strictly ascending
    DevBuf bad;
    SLG_CUDA(ix, bad.alloc(4));
    SLG_CUDA(ix, cudaMemsetAsync(bad.p, 0, 4, st));
    slg_validate_postings_kernel<<<s->n_blocks, 128, 0, st>>>(s->term_start.as<uint64_t>(), s->term_blk.as<uint32_t>(), s->term_df.as<uint32_t>(),
                                                              s->n_terms, s->n_blocks, s->post_doc.as<uint32_t>(), s->doc_count, bad.as<uint32_t>());
    count_launch(ix);
    uint32_t n_bad = 0;
    SLG_CUDA(ix, cudaMemcpyAsync(&n_bad, bad.p, 4, cudaMemcpyDeviceToHost, st));
    SLG_CUDA(ix, cudaStreamSynchronize(st));
    if (n_bad)
      return fail(ix, SLG_ERR_INVALID, "segment %u: %u postings name a doc outside the segment's %u docs or break the ascending order of their list",
                  s->ord, n_bad, s->doc_count);
  }
  slg_term_max_tf_kernel<<<(unsigned)((s->n_terms + 255) / 256), 256, 0, st>>>(s->term_blk.as<uint32_t>(), s->blk_max_tf.as<float>(),
                                                                              s->n_terms, s->term_max_tf.as<float>());
  count_launch(ix);
  std::vector<float> mtf(s->n_terms);
  SLG_CUDA(ix, cudaMemcpyAsync(mtf.data(), s->term_max_tf.p, s->n_terms * 4, cudaMemcpyDeviceToHost, st));
  SLG_CUDA(ix, cudaStreamSynchronize(st));
  std::vector<uint32_t> wide_terms;
  std::vector<uint64_t> wide_off;
  uint64_t wpos = 0;
  for (uint64_t t = 0; t < s->n_terms; t++)
    if (mtf[t] >= 255.0f) {
      wide_terms.push_back((uint32_t)t);
      wide_off.push_back(wpos);
      wpos += s->h_df[t];
    }
  if (wide_terms.empty()) return SLG_OK;
  SLG_CUDA(ix, s->tf_wide.alloc(wpos * 4));
  DevBuf d_wt, d_wo;
  SLG_CUDA(ix, d_wt.alloc(wide_terms.size() * 4));
  SLG_CUDA(ix, d_wo.alloc(wide_off.size() * 8));
  SLG_CUDA(ix, cudaMemcpyAsync(d_wt.p, wide_terms.data(), wide_terms.size() * 4, cudaMemcpyHostToDevice, st));
  SLG_CUDA(ix, cudaMemcpyAsync(d_wo.p, wide_off.data(), wide_off.size() * 8, cudaMemcpyHostToDevice, st));
  // term_wide[t] = offset such that tf_wide[term_wide[t] + i] is posting i of the term
  std::vector<uint64_t> tw(s->n_terms, ~0ull);
  for (size_t w = 0; w < wide_terms.size(); w++) tw[wide_terms[w]] = wide_off[w];
  SLG_CUDA(ix, cudaMemcpyAsync(s->term_wide.p, tw.data(), s->n_terms * 8, cudaMemcpyHostToDevice, st));
  dim3 grid(64, (unsigned)wide_terms.size());
  if (d_csr_tfs) {
    slg_wide_tf_kernel<<<grid, 256, 0, st>>>(d_csr_off, d_csr_tfs, d_wt.as<uint32_t>(), d_wo.as<uint64_t>(),
                                             (uint32_t)wide_terms.size(), s->tf_wide.as<uint32_t>());
    count_launch(ix);
  } else {
    // posting-image load: the resident bytes give every tf < 255, the decode's side list the saturated ones
    slg_wide_from_bytes_kernel<<<grid, 256, 0, st>>>(s->term_start.as<uint64_t>(), s->term_df.as<uint32_t>(), s->post_tf.as<uint8_t>(),
                                                     d_wt.as<uint32_t>(), d_wo.as<uint64_t>(), (uint32_t)wide_terms.size(),
                                                     s->tf_wide.as<uint32_t>());
    count_launch(ix);
    if (n_ovf) {
      slg_wide_patch_tf_kernel<<<(n_ovf + 255) / 256, 256, 0, st>>>(d_ovf, n_ovf, s->term_wide.as<uint64_t>(), s->tf_wide.as<uint32_t>());
      count_launch(ix);
    }
  }
  SLG_CUDA(ix, cudaGetLastError());
  SLG_CUDA(ix, cudaStreamSynchronize(st));
  return SLG_OK;
}

template <class T>
int32_t to_device(slg_index *ix, const T *src, size_t n, int space, DevBuf &tmp, const T **out) {
  if (!src || n == 0) {
    *out = nullptr;
    return SLG_OK;
  }
  if (space == SLG_MEM_DEVICE) {
    *out = src;
    return SLG_OK;
  }
  SLG_CUDA(ix, tmp.alloc(n * sizeof(T)));
  SLG_CUDA(ix, cudaMemcpyAsync(tmp.p, src, n * sizeof(T), cudaMemcpyHostToDevice, ix->stream));
  *out = tmp.as<T>();
  return SLG_OK;
}

}  // namespace

/* ================================================================================================ C ABI */
extern "C" {

const char *slg_version(void) { return "searchlite-b200 0.1 (sm_100a)"; }

const char *slg_last_error(const slg_index_t *ix) { return ix ? ix->err.c_str() : open_error().c_str(); }

int32_t slg_open(int32_t device, slg_index_t **out) {
  if (!out) return fail(nullptr, SLG_ERR_INVALID, "out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(nullptr, SLG_ERR_NO_DEVICE, "no CUDA device (%s); this engine has no CPU fallback",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  if (device < 0 || device >= n) return fail(nullptr, SLG_ERR_INVALID, "device %d out of range (have %d)", device, n);
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(nullptr, SLG_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return fail(nullptr, SLG_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major < 10)
    return fail(nullptr, SLG_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major,
                prop.minor);
  slg_index *ix = new slg_index();
  ix->device = device;
  ix->n_sm = prop.multiProcessorCount;
  ix->smem_optin = prop.sharedMemPerBlockOptin;
  {
    // keep freed per-batch buffers in the pool instead of returning them to the driver
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      uint64_t keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
  }
  e = cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking);
  for (int i = 0; i < 6 && e == cudaSuccess; i++) e = cudaEventCreate(&ix->ev[i]);
  if (e != cudaSuccess) {
    int32_t rc = fail(nullptr, SLG_ERR_CUDA, "stream/event creation: %s", cudaGetErrorString(e));
    delete ix;
    return rc;
  }
  *out = ix;
  return SLG_OK;
}

int32_t slg_close(slg_index_t *ix) {
  if (!ix) return SLG_OK;
  cudaSetDevice(ix->device);
  cudaStreamSynchronize(ix->stream);
  if (ix->pinned) cudaFreeHost(ix->pinned);
  if (ix->merge_pinned) cudaFreeHost(ix->merge_pinned);
  ix->segs.clear();
  for (auto &ev : ix->ev)
    if (ev) cudaEventDestroy(ev);
  if (ix->stream) cudaStreamDestroy(ix->stream);
  delete ix;
  return SLG_OK;
}

int32_t slg_configure(slg_index_t *ix, uint32_t tile_docs, uint32_t ctas_per_sm, uint32_t sub_docs, uint32_t kernel_choice) {
  if (!ix) return SLG_ERR_INVALID;
  if (sub_docs) {
    if (sub_docs % 128 || sub_docs > 8192) return fail(ix, SLG_ERR_INVALID, "sub_docs must be a multiple of 128 <= 8192");
    ix->sub_docs = sub_docs;
  }
  if ((kernel_choice & 0xFF) > 3) return fail(ix, SLG_ERR_INVALID, "kernel_choice must be 0..3 (+256 = score postings in place)");
  ix->kernel_choice = kernel_choice & 0xFF;
  ix->staging = !(kernel_choice & 256u);
  if (tile_docs) {
    if (tile_docs % 1024 || tile_docs > 49152) return fail(ix, SLG_ERR_INVALID, "tile_docs must be a multiple of 1024 <= 49152");
    ix->tile_docs = tile_docs;
  }
  ix->ctas_per_sm = ctas_per_sm;
  return SLG_OK;
}

int32_t slg_set_option(slg_index_t *ix, const char *name, uint64_t value) {
  if (!ix || !name) return SLG_ERR_INVALID;
  const std::string n(name);
  if (n == "resident_scores") ix->resident_scores = value != 0;
  else if (n == "dense_den") ix->dense_den = (uint32_t)value;
  else if (n == "dense_min_df") ix->dense_min_df = (uint32_t)value;
  else if (n == "max_column_bytes") ix->max_column_bytes = value;
  else if (n == "bitmap_den") ix->bitmap_den = (uint32_t)value;
  else if (n == "scan_chunk") {
    if (value && (value < 256 || value > (1u << 20) || value % 256)) return fail(ix, SLG_ERR_INVALID, "scan_chunk is a multiple of 256 postings (0 = by segment size)");
    ix->scan_chunk = (uint32_t)value;
  } else if (n == "scan_first_part") {
    if (value < 1 || value > 255) return fail(ix, SLG_ERR_INVALID, "scan_first_part is a number of 256ths: 1..255");
    ix->scan_first_part = (uint32_t)value;
  }
  else if (n == "max_bitmap_bytes") ix->max_bitmap_bytes = value;
  else if (n == "stage_cap") {
    if (value < 64 || value > 8192 || value % 4) return fail(ix, SLG_ERR_INVALID, "stage_cap must be a multiple of 4 in [64, 8192]");
    ix->stage_cap = (uint32_t)value;
  }
  else if (n == "stream_kernels") ix->stream_kernels = value != 0;
  else if (n == "strict_accumulate") ix->strict_accumulate = value != 0;
  else if (n == "scan_kernels") ix->scan_kernels = value != 0;
  else if (n == "dbg") ix->dbg = (uint32_t)value;
  else if (n == "maxscore_pct") ix->maxscore_pct = (uint32_t)std::min<uint64_t>(value, 100);
  else if (n == "heavy_kernel") {  // the tile-sweep front end of round 1 is gone (it carried an unlocalised intermittent fault)
    if (value != 0) return fail(ix, SLG_ERR_UNSUPPORTED, "heavy_kernel 1 (tile-sweep kernel) was removed; the column path is the items kernel");
  }
  else if (n == "keep_positions") ix->keep_positions = value != 0;
  else return fail(ix, SLG_ERR_INVALID, "unknown option '%s'", name);
  return SLG_OK;
}

int32_t slg_load_segment(slg_index_t *ix, const slg_segment_view_t *v, float k1, float b) {
  if (!ix || !v) return SLG_ERR_INVALID;
  if (!v->term_offsets || (v->n_terms && (!v->post_docs || !v->post_tfs)))
    return fail(ix, SLG_ERR_INVALID, "segment view lacks postings");
  if (v->doc_count && !v->field_lengths) return fail(ix, SLG_ERR_INVALID, "segment view lacks field lengths");
  if (!ix->term_field.empty())
    return fail(ix, SLG_ERR_INVALID, "this handle's term ids come from the files of field '%s' (slg_term_lookup); caller-assigned ids need their own handle", ix->term_field.c_str());
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  cudaStream_t st = ix->stream;
  auto seg = std::make_unique<Segment>();
  Segment *s = seg.get();
  s->ord = v->segment_ord;
  s->doc_count = v->doc_count;
  s->n_terms = v->n_terms;
  s->k1 = k1;
  s->b = b;
  // CSR offsets on the host (df, idf and the padded layout are host work: 1 M terms)
  std::vector<uint64_t> off(v->n_terms + 1);
  if (v->memory_space == SLG_MEM_DEVICE) {
    SLG_CUDA(ix, cudaMemcpyAsync(off.data(), v->term_offsets, (v->n_terms + 1) * 8, cudaMemcpyDeviceToHost, st));
    SLG_CUDA(ix, cudaStreamSynchronize(st));
  } else {
    std::memcpy(off.data(), v->term_offsets, (v->n_terms + 1) * 8);
  }
  s->h_df.resize(v->n_terms);
  for (uint64_t t = 0; t < v->n_terms; t++) {
    uint64_t df = off[t + 1] - off[t];
    if (off[t + 1] < off[t] || df > 0xFFFFFFFFull) return fail(ix, SLG_ERR_INVALID, "term_offsets not monotone at term %llu", (unsigned long long)t);
    s->h_df[t] = (uint32_t)df;
  }
  int32_t rc = build_layout(ix, s);
  if (rc) return rc;
  const uint64_t n_post = off[v->n_terms] - off[0];
  DevBuf t_off, t_docs, t_tfs, t_lens, t_pres;
  const uint64_t *d_off;
  const uint32_t *d_docs, *d_tfs;
  const int64_t *d_lens;
  const uint8_t *d_pres;
  if ((rc = to_device(ix, v->term_offsets, (size_t)v->n_terms + 1, v->memory_space, t_off, &d_off))) return rc;
  if ((rc = to_device(ix, v->post_docs ? v->post_docs + 0 : nullptr, (size_t)off[v->n_terms], v->memory_space, t_docs, &d_docs))) return rc;
  if ((rc = to_device(ix, v->post_tfs, (size_t)off[v->n_terms], v->memory_space, t_tfs, &d_tfs))) return rc;
  if ((rc = to_device(ix, v->field_lengths, (size_t)v->doc_count, v->memory_space, t_lens, &d_lens))) return rc;
  if ((rc = to_device(ix, v->field_length_present, (size_t)v->doc_count, v->memory_space, t_pres, &d_pres))) return rc;
  (void)n_post;
  if (s->n_blocks) {
    slg_transcode_csr_kernel<<<s->n_blocks, 128, 0, st>>>(d_off, d_docs, d_tfs, s->n_terms, s->term_start.as<uint64_t>(),
                                                          s->term_blk.as<uint32_t>(), s->n_blocks, s->post_doc.as<uint32_t>(),
                                                          s->post_tf.as<uint8_t>(), s->blk_max_doc.as<uint32_t>(),
                                                          s->blk_max_tf.as<float>());
    count_launch(ix);
    SLG_CUDA(ix, cudaGetLastError());
  }
  if ((rc = build_wide(ix, s, d_off, d_tfs))) return rc;
  rc = finish_segment(ix, std::move(seg), d_lens, d_pres, v->total_tokens, v->deleted_docs, v->n_deleted);
  if (rc) return rc;
  SLG_CUDA(ix, cudaStreamSynchronize(st));
  return SLG_OK;
}

namespace {

// exclusive prefix sum of per-slot position counts -> pos_begin[n_post_padded + 1]; allocates pos
int32_t scan_positions(slg_index *ix, Segment *s, DevBuf &npos) {
  cudaStream_t st = ix->stream;
  const uint64_t n = s->n_post_padded + 1;  // npos holds n entries, the last one zero
  if (n > 0x7FFFFFFFull) return fail(ix, SLG_ERR_UNSUPPORTED, "segment has too many posting slots for the position index");
  SLG_CUDA(ix, s->pos_begin.alloc(n * 8));
  size_t tmp_bytes = 0;
  auto in = cub::TransformInputIterator<uint64_t, CastU64, const uint32_t *>(npos.as<uint32_t>(), CastU64());
  SLG_CUDA(ix, cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, in, s->pos_begin.as<uint64_t>(), (int)n, st));
  DevBuf tmp;
  SLG_CUDA(ix, tmp.alloc(tmp_bytes));
  SLG_CUDA(ix, cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, in, s->pos_begin.as<uint64_t>(), (int)n, st));
  count_launch(ix, 2);
  uint64_t total = 0;
  SLG_CUDA(ix, cudaMemcpyAsync(&total, s->pos_begin.as<uint64_t>() + (n - 1), 8, cudaMemcpyDeviceToHost, st));
  SLG_CUDA(ix, cudaStreamSynchronize(st));
  s->n_positions = total;
  SLG_CUDA(ix, s->pos.alloc(std::max<uint64_t>(total, 1) * 4));
  return SLG_OK;
}

// Residency from a `.post` image.  begin[t] = offset of term t's list (UINT64_MAX: the segment lacks the
// term), end[t] = an offset the list does not reach past.  avgdl: the .meta value or nullptr (derive it).
struct FieldInput {  // a further text field: its `_len:` column (host) and its avgdl
  const int64_t *lens;
  const uint8_t *present;
  float avgdl;
};

int32_t load_post_image(slg_index *ix, const slg_segment_view_t *v, const uint8_t *post_image, uint64_t post_image_bytes,
                        const uint64_t *begin, const uint64_t *end, const float *avgdl, float k1, float b,
                        const std::vector<FieldInput> *more_fields = nullptr, const std::vector<uint8_t> *term_field = nullptr) {
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  cudaStream_t st = ix->stream;
  auto seg = std::make_unique<Segment>();
  Segment *s = seg.get();
  s->ord = v->segment_ord;
  s->doc_count = v->doc_count;
  s->n_terms = v->n_terms;
  s->k1 = k1;
  s->b = b;
  if (avgdl) {
    s->avgdl = *avgdl;
    s->avgdl_given = true;
  }
  // parse the fixed part of every list header on the host (index/postings.rs:142-168)
  std::vector<PostTermHeader> hdr(v->n_terms);
  s->h_df.resize(v->n_terms);
  bool any_positions = false;
  for (uint64_t t = 0; t < v->n_terms; t++) {
    const uint64_t o = begin[t];
    if (o == ~0ull) {  // seg.postings(key) == None
      hdr[t] = PostTermHeader{0, 0, 0, 0};
      s->h_df[t] = 0;
      continue;
    }
    if (post_image_bytes < 17 || o > post_image_bytes - 17)  // (written so that an offset near 2^64 cannot wrap)
      return fail(ix, SLG_ERR_INVALID, "posting header of term %llu is out of bounds", (unsigned long long)t);
    const uint8_t *p = post_image + o;
    uint32_t df, raw_block;
    std::memcpy(&df, p, 4);
    std::memcpy(&raw_block, p + 5, 4);
    uint32_t bc = raw_block & 0x7FFFFFFFu;
    bool has_meta = (raw_block >> 31) != 0;
    uint64_t payload = o + 17 + ((has_meta && bc > 0) ? 4 + 8ull * bc : 0);
    if (payload > post_image_bytes || end[t] > post_image_bytes || end[t] < payload)
      return fail(ix, SLG_ERR_INVALID, "block table of term %llu is out of bounds", (unsigned long long)t);
    hdr[t].payload = payload;
    hdr[t].end = end[t];
    hdr[t].df = df;
    hdr[t].has_positions = p[4] == 1;
    any_positions |= hdr[t].has_positions && df > 0;
    s->h_df[t] = df;
  }
  StageTimer tm(st);
  tm.mark("list headers (host)");
  int32_t rc = build_layout(ix, s);
  if (rc) return rc;
  tm.mark("layout tables");
  const bool keep_pos = any_positions && ix->keep_positions;
  DevBuf d_img, d_hdr, t_lens, t_pres, d_npos, d_posbyte;
  SLG_CUDA(ix, d_img.alloc(post_image_bytes + 16));
  SLG_CUDA(ix, cudaMemcpyAsync(d_img.p, post_image, post_image_bytes, cudaMemcpyHostToDevice, st));
  SLG_CUDA(ix, d_hdr.alloc(std::max<uint64_t>(v->n_terms, 1) * sizeof(PostTermHeader)));
  if (v->n_terms) SLG_CUDA(ix, cudaMemcpyAsync(d_hdr.p, hdr.data(), v->n_terms * sizeof(PostTermHeader), cudaMemcpyHostToDevice, st));
  if (keep_pos) {
    SLG_CUDA(ix, d_npos.alloc((s->n_post_padded + 1) * 4));
    SLG_CUDA(ix, d_posbyte.alloc((s->n_post_padded + 1) * 4));
    SLG_CUDA(ix, cudaMemsetAsync(d_npos.p, 0, (s->n_post_padded + 1) * 4, st));
  }
  DevBuf d_err, d_ovf;
  SLG_CUDA(ix, d_err.alloc(8));
  tm.mark("image -> device");
  // postings with tf >= 255 go to a side list (term, posting number, tf); when it overflows the decode is repeated with room
  uint32_t ovf_cap = 1u << 16, n_ovf = 0, derr = 0;
  for (int attempt = 0; attempt < 2; attempt++) {
    SLG_CUDA(ix, d_ovf.alloc((size_t)ovf_cap * sizeof(uint4)));
    SLG_CUDA(ix, cudaMemsetAsync(d_err.p, 0, 8, st));
    if (v->n_terms) {
      slg_decode_post_image_kernel<<<(unsigned)((v->n_terms + 3) / 4), 128, 0, st>>>(
          d_img.as<uint8_t>(), post_image_bytes, d_hdr.as<PostTermHeader>(), v->n_terms, s->term_start.as<uint64_t>(),
          s->term_blk.as<uint32_t>(), s->post_doc.as<uint32_t>(), s->post_tf.as<uint8_t>(), s->blk_max_doc.as<uint32_t>(),
          s->blk_max_tf.as<float>(), keep_pos ? d_npos.as<uint32_t>() : nullptr, keep_pos ? d_posbyte.as<uint32_t>() : nullptr,
          d_err.as<uint32_t>(), d_err.as<uint32_t>() + 1, ovf_cap, d_ovf.as<uint4>());
      count_launch(ix);
      SLG_CUDA(ix, cudaGetLastError());
    }
    uint32_t back[2] = {0, 0};
    SLG_CUDA(ix, cudaMemcpyAsync(back, d_err.p, 8, cudaMemcpyDeviceToHost, st));
    SLG_CUDA(ix, cudaStreamSynchronize(st));
    derr = back[0];
    n_ovf = back[1];
    if (n_ovf <= ovf_cap) break;
    ovf_cap = n_ovf;
  }
  if (derr == 1) return fail(ix, SLG_ERR_INVALID, "malformed varint in the posting image");
  if (n_ovf && derr == 0) {
    slg_wide_patch_blockmax_kernel<<<(n_ovf + 255) / 256, 256, 0, st>>>(d_ovf.as<uint4>(), n_ovf, s->term_blk.as<uint32_t>(), s->blk_max_tf.as<float>());
    count_launch(ix);
    SLG_CUDA(ix, cudaGetLastError());
  }
  if (derr == 3) return fail(ix, SLG_ERR_UNSUPPORTED, "a posting list with positions is longer than 4 GiB");
  tm.mark("decode docs + tfs");
  if (keep_pos) {
    if ((rc = scan_positions(ix, s, d_npos))) return rc;
    if (s->n_blocks) {
      slg_decode_positions_kernel<<<s->n_blocks, 128, 0, st>>>(d_img.as<uint8_t>(), d_hdr.as<PostTermHeader>(), s->n_terms,
                                                               s->term_start.as<uint64_t>(), s->term_blk.as<uint32_t>(),
                                                               s->term_df.as<uint32_t>(), s->n_blocks, d_posbyte.as<uint32_t>(),
                                                               s->pos_begin.as<uint64_t>(), s->pos.as<uint32_t>(), d_err.as<uint32_t>());
      count_launch(ix);
      SLG_CUDA(ix, cudaGetLastError());
      SLG_CUDA(ix, cudaMemcpyAsync(&derr, d_err.p, 4, cudaMemcpyDeviceToHost, st));
      SLG_CUDA(ix, cudaStreamSynchronize(st));
      if (derr) return fail(ix, SLG_ERR_INVALID, "malformed position varint in the posting image");
    }
    s->has_positions = true;
    tm.mark("decode positions");
  }
  if ((rc = build_wide(ix, s, nullptr, nullptr, d_ovf.as<uint4>(), n_ovf))) return rc;
  const int64_t *d_lens;
  const uint8_t *d_pres;
  if ((rc = to_device(ix, v->field_lengths, (size_t)v->doc_count, SLG_MEM_HOST, t_lens, &d_lens))) return rc;
  if ((rc = to_device(ix, v->field_length_present, (size_t)v->doc_count, SLG_MEM_HOST, t_pres, &d_pres))) return rc;
  if (more_fields && !more_fields->empty()) {
    for (const FieldInput &fi : *more_fields) {
      Segment::ExtraField ef;
      ef.avgdl = fi.avgdl;
      SLG_CUDA(ix, ef.d_lens.alloc(std::max<size_t>(v->doc_count, 1) * 8));
      SLG_CUDA(ix, ef.d_present.alloc(std::max<size_t>(v->doc_count, 1)));
      if (v->doc_count) {
        SLG_CUDA(ix, cudaMemcpyAsync(ef.d_lens.p, fi.lens, (size_t)v->doc_count * 8, cudaMemcpyHostToDevice, st));
        SLG_CUDA(ix, cudaMemcpyAsync(ef.d_present.p, fi.present, v->doc_count, cudaMemcpyHostToDevice, st));
      }
      s->extra_fields.push_back(std::move(ef));
    }
    if (term_field) s->h_term_field = *term_field;
  }
  rc = finish_segment(ix, std::move(seg), d_lens, d_pres, v->total_tokens, v->deleted_docs, v->n_deleted);
  if (rc) return rc;
  SLG_CUDA(ix, cudaStreamSynchronize(st));
  tm.mark("norms, scores, columns");
  return SLG_OK;
}

}  // namespace

int32_t slg_load_segment_post_image(slg_index_t *ix, const slg_segment_view_t *v, const uint8_t *post_image,
                                    uint64_t post_image_bytes, const uint64_t *term_post_offsets, float k1, float b) {
  if (!ix || !v || !post_image || !term_post_offsets) return SLG_ERR_INVALID;
  if (v->doc_count && !v->field_lengths) return fail(ix, SLG_ERR_INVALID, "segment view lacks field lengths");
  if (v->memory_space != SLG_MEM_HOST) return fail(ix, SLG_ERR_INVALID, "post image loads take host memory");
  return load_post_image(ix, v, post_image, post_image_bytes, term_post_offsets, term_post_offsets + 1, nullptr, k1, b);
}

/* ---- residency from the reference's segment files (SegmentReader::open, index/segment.rs:1239-1330) ---- */
namespace {

struct ParsedSegmentFiles {
  std::vector<slgf::TermEntry> terms;      // every key of .terms
  std::vector<slgf::FastColumn> fast;      // every column of .fast
  std::vector<std::string> fields;         // the scored text fields, in the caller's order
  std::vector<const slgf::FastColumn *> len_col;  // `_len:<field>` per field (or null)
  std::vector<float> avgdl;                // per field
  std::vector<int32_t> term_field;         // per entry of `terms`: index into fields or -1
  uint64_t n_field_terms = 0;
  uint64_t df_sum = 0;
  bool any_positions = false;
};

// "body" or "title,body": the text fields a handle scores
std::vector<std::string> split_fields(const char *spec) {
  std::vector<std::string> out;
  std::string cur;
  for (const char *p = spec;; p++) {
    if (*p == ',' || *p == '\0') {
      if (!cur.empty()) out.push_back(cur);
      cur.clear();
      if (!*p) break;
    } else {
      cur.push_back(*p);
    }
  }
  return out;
}

// verify_checksums + read_terms + FastFieldsReader::open + the .meta fields the search path reads
bool parse_segment_files(const slg_segment_files_t *f, const char *field_spec, ParsedSegmentFiles &out, std::string &err) {
  if (!f->terms || !f->post || !f->fast || !f->meta) {
    err = "segment files: terms, post, fast and meta images are all required";
    return false;
  }
  out.fields = split_fields(field_spec);
  if (out.fields.empty()) {
    err = "no text field named";
    return false;
  }
  if (out.fields.size() > kMaxFields) {
    err = "more than " + std::to_string(kMaxFields) + " text fields in one handle";
    return false;
  }
  if (f->checksums) {  // SegmentMeta.checksums, index/segment.rs:1140-1200
    const char *label[4] = {"terms", "postings", "fast", "meta"};
    const uint8_t *img[4] = {f->terms, f->post, f->fast, f->meta};
    const uint64_t len[4] = {f->terms_bytes, f->post_bytes, f->fast_bytes, f->meta_bytes};
    for (int i = 0; i < 4; i++) {
      const uint32_t actual = slgf::crc32_parallel(img[i], len[i]);
      if (actual != f->checksums[i]) {
        err = std::string("segment failed checksum for ") + label[i] + " (expected " + std::to_string(f->checksums[i]) +
              ", found " + std::to_string(actual) + ")";
        return false;
      }
    }
  }
  if (!slgf::parse_terms(f->terms, f->terms_bytes, out.terms, err)) return false;
  if (!slgf::parse_fast(f->fast, f->fast_bytes, out.fast, err)) return false;
  slgf::Json root = slgf::json_root(f->meta, f->meta_bytes);
  if (root.kind() != '{') {
    err = "segment meta is not a JSON object";
    return false;
  }
  for (auto &c : out.fast)
    if (c.kind() >= 0 && c.doc_len != f->doc_count) {
      err = "fast-field column '" + c.name + "' has " + std::to_string(c.doc_len) + " rows, the segment " + std::to_string(f->doc_count) + " docs";
      return false;
    }
  const slgf::Json avgs = slgf::json_get(root, "avg_field_lengths");
  for (auto &field : out.fields) {
    const std::string len_key = "_len:" + field;  // doc_length_key, index/fastfields.rs:1162-1164
    const slgf::FastColumn *lc = nullptr;
    for (auto &c : out.fast)
      if (c.name == len_key && c.type == 0) lc = &c;
    out.len_col.push_back(lc);
    // SegmentReader::avg_field_length, index/segment.rs:1344-1351: missing field => 0.0; serde_json reads an f32 as f64 -> f32
    out.avgdl.push_back((float)slgf::json_number(slgf::json_get(avgs, field.c_str()), 0.0));
  }
  out.term_field.assign(out.terms.size(), -1);
  for (size_t i = 0; i < out.terms.size(); i++) {
    const slgf::TermEntry &t = out.terms[i];
    if (f->post_bytes < 17 || t.offset > f->post_bytes - 17) {  // (an offset near 2^64 must not wrap)
      err = "a term's posting offset lies outside the posting file";
      return false;
    }
    // keys are "<field>:<token>" (index/segment.rs:675-679); field names hold no ':' in the reference's schemas,
    // so the field is the text before the first colon
    const char *colon = static_cast<const char *>(std::memchr(t.key, ':', t.key_len));
    if (!colon) continue;
    const size_t fl = (size_t)(colon - t.key);
    for (size_t fi = 0; fi < out.fields.size(); fi++)
      if (out.fields[fi].size() == fl && std::memcmp(t.key, out.fields[fi].data(), fl) == 0) {
        out.term_field[i] = (int32_t)fi;
        out.n_field_terms++;
        uint32_t df;
        std::memcpy(&df, f->post + t.offset, 4);
        out.df_sum += df;
        out.any_positions |= f->post[t.offset + 4] == 1;
        break;
      }
  }
  return true;
}

}  // namespace

int32_t slg_inspect_segment_files(const slg_segment_files_t *files, const char *field, slg_segment_info_t *out, char *err,
                                  uint64_t err_cap) {
  if (!files || !field || !out) return SLG_ERR_INVALID;
  ParsedSegmentFiles ps;
  std::string e;
  if (!parse_segment_files(files, field, ps, e)) {
    if (err && err_cap) snprintf(err, (size_t)err_cap, "%s", e.c_str());
    return SLG_ERR_INVALID;
  }
  std::memset(out, 0, sizeof(*out));
  out->n_terms_total = ps.terms.size();
  out->n_terms_field = ps.n_field_terms;
  out->n_postings = ps.df_sum;
  out->avgdl = ps.avgdl[0];
  out->has_positions = ps.any_positions;
  out->has_length_column = ps.len_col[0] != nullptr;
  out->n_fast_columns = (uint32_t)ps.fast.size();
  for (auto &c : ps.fast) out->n_scalar_columns += c.type <= 2;
  for (auto &c : ps.fast) out->n_list_columns += c.kind() >= 3;
  out->crc_terms = slgf::crc32_parallel(files->terms, files->terms_bytes);
  out->crc_postings = slgf::crc32_parallel(files->post, files->post_bytes);
  out->crc_fast = slgf::crc32_parallel(files->fast, files->fast_bytes);
  out->crc_meta = slgf::crc32_parallel(files->meta, files->meta_bytes);
  return SLG_OK;
}

int32_t slg_load_segment_files(slg_index_t *ix, const slg_segment_files_t *f, const char *field, float k1, float b) {
  if (!ix || !f || !field) return SLG_ERR_INVALID;
  if (!ix->term_field.empty() && ix->term_field != field)
    return fail(ix, SLG_ERR_UNSUPPORTED, "this handle scores field(s) '%s'; every segment of a handle names the same field list", ix->term_field.c_str());
  if (ix->term_field.empty() && !ix->segs.empty())
    return fail(ix, SLG_ERR_INVALID, "this handle holds segments loaded with caller-assigned term ids; file segments need their own handle");
  ParsedSegmentFiles ps;
  std::string e;
  StageTimer tm(ix->stream);
  if (!parse_segment_files(f, field, ps, e)) return fail(ix, SLG_ERR_INVALID, "%s", e.c_str());
  tm.mark("crc32 + parse files (host)");
  // every list's end: the next list's offset in file order (lists of all fields share the file)
  std::vector<uint64_t> all_off;
  all_off.reserve(ps.terms.size() + 1);
  for (auto &t : ps.terms) all_off.push_back(t.offset);
  all_off.push_back(f->post_bytes);
  std::sort(all_off.begin(), all_off.end());
  // the handle's term space grows by the keys this segment adds
  struct Mine {
    uint32_t id;
    uint64_t offset;
    uint8_t field;
  };
  std::vector<Mine> mine;
  mine.reserve((size_t)ps.n_field_terms);
  for (size_t i = 0; i < ps.terms.size(); i++) {
    if (ps.term_field[i] < 0) continue;
    const slgf::TermEntry &t = ps.terms[i];
    auto it = ix->term_ids.emplace(std::string(t.key, t.key_len), (uint32_t)ix->term_ids.size()).first;
    if (it->second >= ix->term_field_of.size()) ix->term_field_of.resize(it->second + 1, 0);
    ix->term_field_of[it->second] = (uint8_t)ps.term_field[i];
    mine.push_back(Mine{it->second, t.offset, (uint8_t)ps.term_field[i]});
  }
  ix->term_field = field;
  const uint64_t n_terms = ix->term_ids.size();
  std::vector<uint64_t> begin(n_terms, ~0ull), end(n_terms, 0);
  for (auto &m : mine) {
    begin[m.id] = m.offset;
    end[m.id] = *std::upper_bound(all_off.begin(), all_off.end(), m.offset);
  }
  // `_len:<field>` per field (field_lengths_for, api/reader.rs:3604-3621: absent column or value => 0)
  const size_t n_fields = ps.fields.size();
  std::vector<std::vector<int64_t>> lens(n_fields, std::vector<int64_t>(f->doc_count, 0));
  std::vector<std::vector<uint8_t>> pres(n_fields, std::vector<uint8_t>(f->doc_count, 0));
  uint64_t total = 0;
  for (size_t fi = 0; fi < n_fields; fi++) {
    if (!ps.len_col[fi]) continue;
    std::memcpy(lens[fi].data(), ps.len_col[fi]->values, (size_t)f->doc_count * 8);
    std::memcpy(pres[fi].data(), ps.len_col[fi]->presence, f->doc_count);
    if (fi == 0)
      for (uint32_t d = 0; d < f->doc_count; d++)
        if (pres[0][d] && lens[0][d] > 0) total += (uint64_t)lens[0][d];
  }
  tm.mark("term space + lengths (host)");
  std::vector<FieldInput> more;
  for (size_t fi = 1; fi < n_fields; fi++) more.push_back(FieldInput{lens[fi].data(), pres[fi].data(), ps.avgdl[fi]});
  std::vector<uint8_t> term_field(ix->term_field_of.begin(), ix->term_field_of.end());
  term_field.resize(n_terms, 0);
  slg_segment_view_t v{};
  v.segment_ord = f->segment_ord;
  v.doc_count = f->doc_count;
  v.n_terms = n_terms;
  v.field_lengths = lens[0].data();
  v.field_length_present = pres[0].data();
  v.total_tokens = total;
  v.deleted_docs = f->deleted_docs;
  v.n_deleted = f->n_deleted;
  v.memory_space = SLG_MEM_HOST;
  int32_t rc = load_post_image(ix, &v, f->post, f->post_bytes, begin.data(), end.data(), &ps.avgdl[0], k1, b, &more, &term_field);
  if (rc) {
    if (ix->segs.empty()) {  // nothing loaded yet: a failed first load leaves no term space behind
      ix->term_ids.clear();
      ix->term_field_of.clear();
      ix->term_field.clear();
    }
    return rc;
  }
  // scalar fast-field columns, by name (the file's field order is HashMap order, index/fastfields.rs:414)
  Segment *s = ix->find(f->segment_ord);
  for (auto &c : ps.fast) {
    if (c.kind() < 0 || c.name.compare(0, 5, "_len:") == 0) continue;  // nested bookkeeping (types 9, 10) is not filterable
    size_t h = 0;
    while (h < ix->column_names.size() && ix->column_names[h] != c.name) h++;
    if (h == ix->column_names.size()) ix->column_names.push_back(c.name);
    if (s->columns.size() <= h) s->columns.resize(h + 1);
    Column col;
    col.kind = c.kind();
    const size_t elem = (col.kind == 2 || col.kind == 5) ? 4 : 8;
    if (col.kind >= 3) {
      // list and (flattened) nested columns: offsets + values, "any value" semantics in the filter kernel
      col.n_values = c.n_values;
      SLG_CUDA(ix, col.offsets.alloc(c.list_offsets.size() * 4));
      SLG_CUDA(ix, cudaMemcpy(col.offsets.p, c.list_offsets.data(), c.list_offsets.size() * 4, cudaMemcpyHostToDevice));
      SLG_CUDA(ix, col.values.alloc(std::max<size_t>((size_t)c.n_values * elem, 16)));
      if (c.n_values) SLG_CUDA(ix, cudaMemcpy(col.values.p, c.values, (size_t)c.n_values * elem, cudaMemcpyHostToDevice));
      col.dict = c.dict;
      s->columns[h] = std::move(col);
      continue;
    }
    SLG_CUDA(ix, col.values.alloc(std::max<size_t>((size_t)s->doc_count * elem, 1)));
    SLG_CUDA(ix, cudaMemcpy(col.values.p, c.values, (size_t)s->doc_count * elem, cudaMemcpyHostToDevice));
    if (c.type != 2) {
      SLG_CUDA(ix, col.present.alloc(std::max<size_t>(s->doc_count, 1)));
      SLG_CUDA(ix, cudaMemcpy(col.present.p, c.presence, s->doc_count, cudaMemcpyHostToDevice));
    }
    col.dict = c.dict;
    s->columns[h] = std::move(col);
  }
  return SLG_OK;
}

int32_t slg_load_vector_file(slg_index_t *ix, uint32_t segment_ord, const uint8_t *bytes, uint64_t n_bytes, int32_t store_bf16,
                             int32_t *metric_out) {
  if (!ix || !bytes) return SLG_ERR_INVALID;
  Segment *s = ix->find(segment_ord);
  if (!s) return fail(ix, SLG_ERR_INVALID, "no segment %u", segment_ord);
  slgf::VectorFile vf;
  std::string e;
  if (!slgf::parse_vector_file(bytes, n_bytes, vf, e)) return fail(ix, SLG_ERR_INVALID, "%s", e.c_str());
  if (vf.doc_count != s->doc_count)
    return fail(ix, SLG_ERR_INVALID, "vector doc count mismatch: expected %u, found %u", s->doc_count, vf.doc_count);
  if (metric_out) *metric_out = vf.metric;
  // slg_load_vectors only copies from these pointers (no host dereference), so the image needs no alignment and no staging
  // copy — the rows of a 100 M-doc shard are 19 GB
  return slg_load_vectors(ix, segment_ord, vf.dim, reinterpret_cast<const uint32_t *>(vf.offsets),
                          reinterpret_cast<const float *>(vf.values), vf.vector_count, store_bf16);
}

namespace {
// read-only mapping of a file: the `.post` of a 10 M-doc index is ~12 GB, so no private copy is made —
// crc32 and the host-to-device copy read the page cache directly
struct MappedFile {
  const uint8_t *p = nullptr;
  size_t n = 0;
  MappedFile() = default;
  MappedFile(const MappedFile &) = delete;
  MappedFile &operator=(const MappedFile &) = delete;
  ~MappedFile() {
    if (p && n) munmap(const_cast<uint8_t *>(p), n);
  }
  bool open(const std::string &path) {
    const int fd = ::open(path.c_str(), O_RDONLY);
    if (fd < 0) return false;
    struct stat st;
    if (fstat(fd, &st) != 0) {
      ::close(fd);
      return false;
    }
    n = (size_t)st.st_size;
    if (n) {
      void *m = mmap(nullptr, n, PROT_READ, MAP_PRIVATE, fd, 0);
      if (m == MAP_FAILED) {
        ::close(fd);
        n = 0;
        return false;
      }
      madvise(m, n, MADV_SEQUENTIAL);
      p = static_cast<const uint8_t *>(m);
    } else {
      static const uint8_t empty = 0;
      p = &empty;
    }
    ::close(fd);
    return true;
  }
  const uint8_t *data() const { return p; }
  size_t size() const { return n; }
};
// the manifest stores `root.join(name)` strings (index/directory.rs:16-46); the index may have moved since
std::string in_dir(const std::string &dir, const std::string &stored) {
  size_t slash = stored.find_last_of('/');
  return dir + "/" + (slash == std::string::npos ? stored : stored.substr(slash + 1));
}
}  // namespace

int32_t slg_load_index_dir(slg_index_t *ix, const char *dir, const char *field, float k1, float b, const char *vector_field,
                           int32_t store_bf16, uint32_t *n_segments_out) {
  return slg_load_index_dir_shard(ix, dir, field, k1, b, vector_field, store_bf16, 0, 1, n_segments_out);
}

int32_t slg_load_index_dir_shard(slg_index_t *ix, const char *dir, const char *field, float k1, float b, const char *vector_field,
                                 int32_t store_bf16, uint32_t shard_rank, uint32_t shard_world, uint32_t *n_segments_out) {
  if (!ix || !dir || !field) return SLG_ERR_INVALID;
  if (shard_world == 0 || shard_rank >= shard_world) return fail(ix, SLG_ERR_INVALID, "shard %u of %u", shard_rank, shard_world);
  MappedFile man;
  const std::string d(dir);
  if (!man.open(d + "/MANIFEST.json")) return fail(ix, SLG_ERR_INVALID, "cannot read %s/MANIFEST.json", dir);
  slgf::Json root = slgf::json_root(man.data(), man.size());
  std::vector<slgf::Json> segs;
  if (!slgf::json_elements(slgf::json_get(root, "segments"), segs)) return fail(ix, SLG_ERR_INVALID, "manifest has no segments array");
  uint32_t ord = 0, loaded = 0;
  for (auto &sm : segs) {  // IndexReader::open keeps manifest order; segment_ord is that index (api/reader.rs:2670)
    if (ord % shard_world != shard_rank) {  // another GPU's segment (segment == shard, DESIGN.md §4)
      ord++;
      continue;
    }
    slgf::Json paths = slgf::json_get(sm, "paths");
    MappedFile terms, post, fast, meta;
    const char *names[4] = {"terms", "postings", "fast", "meta"};
    MappedFile *bufs[4] = {&terms, &post, &fast, &meta};
    uint32_t crcs[4];
    bool have_crc = true;
    slgf::Json sums = slgf::json_get(sm, "checksums");
    for (int i = 0; i < 4; i++) {
      const std::string stored = slgf::json_string(slgf::json_get(paths, names[i]));
      if (stored.empty()) return fail(ix, SLG_ERR_INVALID, "segment %u: manifest lacks paths.%s", ord, names[i]);
      if (!bufs[i]->open(in_dir(d, stored))) return fail(ix, SLG_ERR_INVALID, "cannot read %s", in_dir(d, stored).c_str());
      slgf::Json c = slgf::json_get(sums, names[i]);
      if (c.ok()) crcs[i] = (uint32_t)slgf::json_number(c);
      else have_crc = false;
    }
    std::vector<uint32_t> deleted;
    std::vector<slgf::Json> del;
    slgf::json_elements(slgf::json_get(sm, "deleted_docs"), del);
    for (auto &x : del) deleted.push_back((uint32_t)slgf::json_number(x));
    slg_segment_files_t f{};
    f.segment_ord = ord;
    f.doc_count = (uint32_t)slgf::json_number(slgf::json_get(sm, "doc_count"));
    f.terms = terms.data();
    f.terms_bytes = terms.size();
    f.post = post.data();
    f.post_bytes = post.size();
    f.fast = fast.data();
    f.fast_bytes = fast.size();
    f.meta = meta.data();
    f.meta_bytes = meta.size();
    f.deleted_docs = deleted.data();
    f.n_deleted = (uint32_t)deleted.size();
    f.checksums = have_crc ? crcs : nullptr;
    int32_t rc = slg_load_segment_files(ix, &f, field, k1, b);
    if (rc) return rc;
    if (vector_field && *vector_field) {
      const std::string vdir = slgf::json_string(slgf::json_get(paths, "vector_dir"));
      if (vdir.empty()) return fail(ix, SLG_ERR_INVALID, "segment missing vector directory path");  // segment.rs:969-972
      MappedFile vb;
      const std::string vp = in_dir(d, vdir) + "/" + vector_field + ".bin";
      if (!vb.open(vp)) return fail(ix, SLG_ERR_INVALID, "cannot read %s", vp.c_str());
      if ((rc = slg_load_vector_file(ix, ord, vb.data(), vb.size(), store_bf16, nullptr))) return rc;
    }
    ord++;
    loaded++;
  }
  if (n_segments_out) *n_segments_out = loaded;
  return SLG_OK;
}

int32_t slg_term_lookup(const slg_index_t *ix, const char *key, uint32_t *term_id) {
  if (!ix || !key || !term_id) return SLG_ERR_INVALID;
  auto it = ix->term_ids.find(key);
  *term_id = it == ix->term_ids.end() ? 0xFFFFFFFFu : it->second;
  return SLG_OK;
}

int32_t slg_column_lookup(const slg_index_t *ix, const char *name) {
  if (!ix || !name) return SLG_ERR_INVALID;
  for (size_t h = 0; h < ix->column_names.size(); h++)
    if (ix->column_names[h] == name) return (int32_t)h;
  return -1;
}

/* ---- term positions handed over as CSR (the positions of PostingEntry, index/postings.rs:14-19) ---- */
int32_t slg_load_positions(slg_index_t *ix, uint32_t segment_ord, const uint64_t *term_offsets, const uint64_t *position_offsets,
                           const uint32_t *positions, int32_t memory_space) {
  if (!ix || !term_offsets || !position_offsets) return SLG_ERR_INVALID;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  cudaStream_t st = ix->stream;
  Segment *s = ix->find(segment_ord);
  if (!s) return fail(ix, SLG_ERR_INVALID, "no segment %u", segment_ord);
  const bool dev = memory_space == SLG_MEM_DEVICE;
  std::vector<uint64_t> off(s->n_terms + 1);
  if (dev) SLG_CUDA(ix, cudaMemcpy(off.data(), term_offsets, (s->n_terms + 1) * 8, cudaMemcpyDeviceToHost));
  else std::memcpy(off.data(), term_offsets, (s->n_terms + 1) * 8);
  for (uint64_t t = 0; t < s->n_terms; t++)
    if (off[t + 1] - off[t] != s->h_df[t])
      return fail(ix, SLG_ERR_INVALID, "term offsets do not match the loaded postings at term %llu", (unsigned long long)t);
  const uint64_t n_post = off[s->n_terms];
  uint64_t n_pos = 0;
  if (dev) SLG_CUDA(ix, cudaMemcpy(&n_pos, position_offsets + n_post, 8, cudaMemcpyDeviceToHost));
  else n_pos = position_offsets[n_post];
  if (n_pos && !positions) return SLG_ERR_INVALID;
  ix->ctr.resident_bytes -= s->pos_begin.bytes + s->pos.bytes;
  s->has_positions = false;
  DevBuf t_off, t_poff, t_pos, d_npos;
  const uint64_t *d_off, *d_poff;
  const uint32_t *d_pos;
  int32_t rc;
  if ((rc = to_device(ix, term_offsets, (size_t)s->n_terms + 1, memory_space, t_off, &d_off))) return rc;
  if ((rc = to_device(ix, position_offsets, (size_t)n_post + 1, memory_space, t_poff, &d_poff))) return rc;
  if ((rc = to_device(ix, positions, (size_t)n_pos, memory_space, t_pos, &d_pos))) return rc;
  SLG_CUDA(ix, d_npos.alloc((s->n_post_padded + 1) * 4));
  SLG_CUDA(ix, cudaMemsetAsync(d_npos.p, 0, (s->n_post_padded + 1) * 4, st));
  if (s->n_blocks) {
    slg_csr_position_counts_kernel<<<s->n_blocks, 128, 0, st>>>(d_off, d_poff, s->n_terms, s->term_start.as<uint64_t>(),
                                                                s->term_blk.as<uint32_t>(), s->n_blocks, d_npos.as<uint32_t>());
    count_launch(ix);
  }
  if ((rc = scan_positions(ix, s, d_npos))) return rc;
  if (s->n_positions != n_pos) return fail(ix, SLG_ERR_INVALID, "position offsets are inconsistent");
  if (s->n_blocks) {
    slg_csr_position_copy_kernel<<<s->n_blocks, 128, 0, st>>>(d_off, d_poff, d_pos, s->n_terms, s->term_start.as<uint64_t>(), s->term_blk.as<uint32_t>(),
                                                              s->n_blocks, s->pos_begin.as<uint64_t>(), s->pos.as<uint32_t>());
    count_launch(ix);
  }
  SLG_CUDA(ix, cudaGetLastError());
  SLG_CUDA(ix, cudaStreamSynchronize(st));
  s->has_positions = true;
  ix->ctr.resident_bytes += s->pos_begin.bytes + s->pos.bytes;
  return SLG_OK;
}

int32_t slg_segment_stats(const slg_index_t *ixc, uint32_t segment_ord, float *avgdl, float *live_docs, float *min_doc_len,
                          uint64_t *n_postings) {
  slg_index *ix = const_cast<slg_index *>(ixc);
  if (!ix) return SLG_ERR_INVALID;
  Segment *s = ix->find(segment_ord);
  if (!s) return fail(ix, SLG_ERR_INVALID, "no segment %u", segment_ord);
  if (avgdl) *avgdl = s->avgdl;
  if (live_docs) *live_docs = s->live_docs;
  if (min_doc_len) *min_doc_len = s->min_doc_len;
  if (n_postings) *n_postings = s->n_postings;
  return SLG_OK;
}

int32_t slg_segment_residency(const slg_index_t *ixc, uint32_t segment_ord, char *json_out, uint64_t json_len) {
  slg_index *ix = const_cast<slg_index *>(ixc);
  if (!ix || !json_out || json_len < 2) return SLG_ERR_INVALID;
  Segment *s = ix->find(segment_ord);
  if (!s) return fail(ix, SLG_ERR_INVALID, "no segment %u", segment_ord);
  size_t cols_fast = 0, filters = 0;
  for (auto &c : s->columns) cols_fast += c.values.bytes + c.present.bytes + c.offsets.bytes;
  for (auto &f : s->filter_bits)
    if (!f.borrowed) filters += f.bytes;
  std::vector<const DevBuf *> seen;  // (the phrases of a batch share one slab)
  for (auto &sl : s->filter_slabs)
    if (sl && std::find(seen.begin(), seen.end(), sl.get()) == seen.end()) {
      seen.push_back(sl.get());
      filters += sl->bytes;
    }
  const int n = snprintf(
      json_out, (size_t)json_len,
      "{\"post_doc\": %zu, \"post_tf\": %zu, \"post_score\": %zu, \"mb_max\": %zu, \"term_tables\": %zu, \"block_tables\": %zu, \"norms\": %zu, "
      "\"score_columns\": %zu, \"column_block_maxima\": %zu, \"presence_bitmaps\": %zu, \"wide_tf\": %zu, \"live_bits\": %zu, "
      "\"positions\": %zu, \"fast_field_columns\": %zu, \"filter_bitmaps\": %zu, \"vectors\": %zu, \"n_score_columns\": %u, \"n_presence_bitmaps\": %u}",
      s->post_doc.bytes, s->post_tf.bytes, s->post_score.bytes, s->mb_max.bytes,
      s->term_start.bytes + s->term_df.bytes + s->term_idf.bytes + s->term_max_tf.bytes + s->term_wide.bytes + s->term_blk.bytes + s->term_field.bytes +
          s->term_col.bytes + s->term_bits.bytes + s->term_ub.bytes,
      s->blk_max_doc.bytes + s->blk_max_tf.bytes, s->nk.bytes, s->cols.bytes, s->col_tmax.bytes, s->pres_bits.bytes, s->tf_wide.bytes, s->live_bits.bytes,
      s->pos_begin.bytes + s->pos.bytes, cols_fast, filters, s->vec.offsets.bytes + s->vec.values.bytes, s->n_cols, s->n_bitmaps);
  if (n < 0 || (uint64_t)n >= json_len) return fail(ix, SLG_ERR_INVALID, "residency report needs %d bytes", n + 1);
  return SLG_OK;
}

int32_t slg_field_stats(const slg_index_t *ixc, uint32_t segment_ord, uint32_t field_index, float *avgdl, float *min_doc_len) {
  slg_index *ix = const_cast<slg_index *>(ixc);
  if (!ix) return SLG_ERR_INVALID;
  Segment *s = ix->find(segment_ord);
  if (!s) return fail(ix, SLG_ERR_INVALID, "no segment %u", segment_ord);
  if (field_index >= s->f_avgdl.size()) return fail(ix, SLG_ERR_INVALID, "segment %u scores %zu field(s)", segment_ord, s->f_avgdl.size());
  if (avgdl) *avgdl = s->f_avgdl[field_index];
  if (min_doc_len) *min_doc_len = s->f_min_len[field_index];
  return SLG_OK;
}

int32_t slg_term_has_column(const slg_index_t *ixc, uint32_t segment_ord, uint32_t term_id) {
  slg_index *ix = const_cast<slg_index *>(ixc);
  if (!ix) return SLG_ERR_INVALID;
  Segment *s = ix->find(segment_ord);
  if (!s) return fail(ix, SLG_ERR_INVALID, "no segment %u", segment_ord);
  return term_id < s->h_term_col.size() && s->h_term_col[term_id] >= 0 ? 1 : 0;
}

/* ---- fast-field columns + filters ---- */
static int32_t add_column(slg_index *ix, uint32_t segment_ord, int kind, const void *values, size_t elem,
                          const uint8_t *present, const char *const *dict, uint32_t n_dict) {
  if (!ix || !values) return SLG_ERR_INVALID;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  Segment *s = ix->find(segment_ord);
  if (!s) return fail(ix, SLG_ERR_INVALID, "no segment %u", segment_ord);
  Column c;
  c.kind = kind;
  SLG_CUDA(ix, c.values.alloc((size_t)s->doc_count * elem));
  SLG_CUDA(ix, cudaMemcpy(c.values.p, values, (size_t)s->doc_count * elem, cudaMemcpyHostToDevice));
  if (kind != 2) {
    SLG_CUDA(ix, c.present.alloc(std::max<size_t>(s->doc_count, 1)));
    if (present) SLG_CUDA(ix, cudaMemcpy(c.present.p, present, s->doc_count, cudaMemcpyHostToDevice));
    else SLG_CUDA(ix, cudaMemset(c.present.p, 1, std::max<size_t>(s->doc_count, 1)));
  }
  for (uint32_t i = 0; i < n_dict; i++) c.dict.emplace_back(dict[i]);
  s->columns.push_back(std::move(c));
  return (int32_t)s->columns.size() - 1;
}

int32_t slg_add_i64_column(slg_index_t *ix, uint32_t segment_ord, const int64_t *values, const uint8_t *present) {
  return add_column(ix, segment_ord, 0, values, 8, present, nullptr, 0);
}
int32_t slg_add_f64_column(slg_index_t *ix, uint32_t segment_ord, const double *values, const uint8_t *present) {
  return add_column(ix, segment_ord, 1, values, 8, present, nullptr, 0);
}
int32_t slg_add_str_column(slg_index_t *ix, uint32_t segment_ord, const char *const *dict, uint32_t n_dict,
                           const uint32_t *ords) {
  if (n_dict && !dict) return SLG_ERR_INVALID;
  return add_column(ix, segment_ord, 2, ords, 4, nullptr, dict, n_dict);
}

// list columns (I64List / F64List / StrList, index/fastfields.rs:926-940, 1000-1010, 1045-1068): offsets[doc_count + 1]
// running sums, values[offsets[doc_count]]
static int32_t add_list_column(slg_index *ix, uint32_t segment_ord, int kind, const uint32_t *offsets, const void *values, size_t elem,
                               const char *const *dict, uint32_t n_dict) {
  if (!ix || !offsets) return SLG_ERR_INVALID;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  Segment *s = ix->find(segment_ord);
  if (!s) return fail(ix, SLG_ERR_INVALID, "no segment %u", segment_ord);
  if (offsets[0] != 0) return fail(ix, SLG_ERR_INVALID, "list column offsets must start at 0");
  for (uint32_t d = 0; d < s->doc_count; d++)
    if (offsets[d + 1] < offsets[d]) return fail(ix, SLG_ERR_INVALID, "list column offsets descend at doc %u", d);
  const uint64_t nv = offsets[s->doc_count];
  if (nv && !values) return SLG_ERR_INVALID;
  Column c;
  c.kind = kind;
  c.n_values = nv;
  SLG_CUDA(ix, c.offsets.alloc(((size_t)s->doc_count + 1) * 4));
  SLG_CUDA(ix, cudaMemcpy(c.offsets.p, offsets, ((size_t)s->doc_count + 1) * 4, cudaMemcpyHostToDevice));
  SLG_CUDA(ix, c.values.alloc(std::max<size_t>(nv * elem, 16)));
  if (nv) SLG_CUDA(ix, cudaMemcpy(c.values.p, values, nv * elem, cudaMemcpyHostToDevice));
  for (uint32_t i = 0; i < n_dict; i++) c.dict.emplace_back(dict[i]);
  s->columns.push_back(std::move(c));
  return (int32_t)s->columns.size() - 1;
}

int32_t slg_add_i64_list_column(slg_index_t *ix, uint32_t segment_ord, const uint32_t *offsets, const int64_t *values) {
  return add_list_column(ix, segment_ord, 3, offsets, values, 8, nullptr, 0);
}
int32_t slg_add_f64_list_column(slg_index_t *ix, uint32_t segment_ord, const uint32_t *offsets, const double *values) {
  return add_list_column(ix, segment_ord, 4, offsets, values, 8, nullptr, 0);
}
int32_t slg_add_str_list_column(slg_index_t *ix, uint32_t segment_ord, const char *const *dict, uint32_t n_dict, const uint32_t *offsets,
                                const uint32_t *ords) {
  if (n_dict && !dict) return SLG_ERR_INVALID;
  return add_list_column(ix, segment_ord, 5, offsets, ords, 4, dict, n_dict);
}

// Unicode lowercase of one code point as Rust's char::to_lowercase gives it for the bicameral blocks a keyword field is
// likely to hold: Latin-1, Latin Extended-A / -B (the regular pairs) / Additional, Greek (+ tonos forms), Cyrillic (+ the
// extended pairs), Armenian, fullwidth Latin.  U+0130 (İ) lowers to two code points ("i̇"), the only multi-character mapping.
static void lower_cp(uint32_t c, std::u32string &out, bool final_sigma) {
  if (c < 0x80) {
    out.push_back(c >= 'A' && c <= 'Z' ? c + 32 : c);
    return;
  }
  if (c == 0x130) {
    out.push_back('i');
    out.push_back(0x307);
    return;
  }
  uint32_t r = c;
  if ((c >= 0xC0 && c <= 0xDE && c != 0xD7)) r = c + 0x20;
  else if ((c >= 0x100 && c <= 0x12F) || (c >= 0x132 && c <= 0x137) || (c >= 0x14A && c <= 0x177)) r = (c & 1u) ? c : c + 1;
  else if ((c >= 0x139 && c <= 0x148) || (c >= 0x179 && c <= 0x17E)) r = (c & 1u) ? c + 1 : c;
  else if (c == 0x178) r = 0xFF;
  else if (c == 0x1C4 || c == 0x1C5) r = 0x1C6;  // the DŽ / LJ / NJ / DZ digraphs: upper and title case lower to one letter
  else if (c == 0x1C7 || c == 0x1C8) r = 0x1C9;
  else if (c == 0x1CA || c == 0x1CB) r = 0x1CC;
  else if (c == 0x1F1 || c == 0x1F2) r = 0x1F3;
  else if ((c >= 0x1CD && c <= 0x1DC)) r = (c & 1u) ? c + 1 : c;
  else if ((c >= 0x1DE && c <= 0x1EF) || (c >= 0x1F8 && c <= 0x21F) || (c >= 0x222 && c <= 0x233)) r = (c & 1u) ? c : c + 1;
  else if (c == 0x386) r = 0x3AC;
  else if (c >= 0x388 && c <= 0x38A) r = c + 37;
  else if (c == 0x38C) r = 0x3CC;
  else if (c == 0x38E || c == 0x38F) r = c + 63;
  else if (c >= 0x391 && c <= 0x3AB && c != 0x3A2) r = (c == 0x3A3 && final_sigma) ? 0x3C2 : c + 0x20;
  else if (c >= 0x400 && c <= 0x40F) r = c + 0x50;
  else if (c >= 0x410 && c <= 0x42F) r = c + 0x20;
  else if ((c >= 0x460 && c <= 0x481) || (c >= 0x48A && c <= 0x4BF) || (c >= 0x4D0 && c <= 0x52F)) r = (c & 1u) ? c : c + 1;
  else if (c >= 0x4C1 && c <= 0x4CE) r = (c & 1u) ? c + 1 : c;
  else if (c == 0x4C0) r = 0x4CF;
  else if (c >= 0x531 && c <= 0x556) r = c + 0x30;
  else if (c >= 0x1E00 && c <= 0x1E95) r = (c & 1u) ? c : c + 1;
  else if (c >= 0x1EA0 && c <= 0x1EFF) r = (c & 1u) ? c : c + 1;
  else if (c >= 0xFF21 && c <= 0xFF3A) r = c + 0x20;
  out.push_back(r);
}
static bool is_cased_letter(uint32_t c) {  // enough of Unicode's "cased" for the final-sigma rule
  return (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z') || (c >= 0xC0 && c <= 0x24F && c != 0xD7 && c != 0xF7) ||
         (c >= 0x370 && c <= 0x3FF) || (c >= 0x400 && c <= 0x52F) || (c >= 0x531 && c <= 0x586) || (c >= 0x1E00 && c <= 0x1FFF);
}
static std::u32string utf8_lower(const std::string &s) {
  std::u32string cps;
  for (size_t i = 0; i < s.size();) {
    const unsigned char b = (unsigned char)s[i];
    uint32_t c = b;
    int n = 1;
    if (b >= 0xF0 && i + 3 < s.size()) {
      c = ((b & 7u) << 18) | (((unsigned char)s[i + 1] & 63u) << 12) | (((unsigned char)s[i + 2] & 63u) << 6) | ((unsigned char)s[i + 3] & 63u);
      n = 4;
    } else if (b >= 0xE0 && i + 2 < s.size()) {
      c = ((b & 15u) << 12) | (((unsigned char)s[i + 1] & 63u) << 6) | ((unsigned char)s[i + 2] & 63u);
      n = 3;
    } else if (b >= 0xC0 && i + 1 < s.size()) {
      c = ((b & 31u) << 6) | ((unsigned char)s[i + 1] & 63u);
      n = 2;
    }
    cps.push_back(c);
    i += n;
  }
  std::u32string out;
  for (size_t i = 0; i < cps.size(); i++) {
    // Final_Sigma: preceded by a cased letter and not followed by one (Unicode SpecialCasing, as Rust implements it)
    const bool fin = cps[i] == 0x3A3 && i > 0 && is_cased_letter(cps[i - 1]) && !(i + 1 < cps.size() && is_cased_letter(cps[i + 1]));
    lower_cp(cps[i], out, fin);
  }
  return out;
}

// index/fastfields.rs:475-481: eq_ignore_ascii_case when both sides are ASCII, else a.to_lowercase() == b.to_lowercase()
static bool ci_equals(const std::string &a, const std::string &b) {
  bool ascii = true;
  for (unsigned char ch : a) ascii = ascii && ch < 0x80;
  for (unsigned char ch : b) ascii = ascii && ch < 0x80;
  if (!ascii) return utf8_lower(a) == utf8_lower(b);
  if (a.size() != b.size()) return false;
  for (size_t i = 0; i < a.size(); i++) {
    unsigned char x = a[i], y = b[i];
    if (x >= 'A' && x <= 'Z') x += 32;
    if (y >= 'A' && y <= 'Z') y += 32;
    if (x != y) return false;
  }
  return true;
}

// A filter id names one bitmap per loaded segment (root filters, phrases and their combinations alike).
static int32_t register_filter(slg_index *ix, FilterProg fp, std::vector<DevBuf> &per_seg) {
  const size_t id = ix->filters.size();
  for (size_t si = 0; si < ix->segs.size(); si++) {
    Segment *s = ix->segs[si].get();
    s->filter_bits.resize(id + 1);
    s->filter_slabs.resize(id + 1);
    s->filter_bits[id] = std::move(per_seg[si]);
    std::vector<const uint32_t *> ptrs;
    for (auto &fb : s->filter_bits) ptrs.push_back(fb.as<uint32_t>());
    if (s->filter_ptrs.bytes < ptrs.size() * sizeof(void *)) {
      SLG_CUDA(ix, cudaStreamSynchronize(ix->stream));  // a running batch may still read the old table
      SLG_CUDA(ix, s->filter_ptrs.alloc(std::max<size_t>(64, ptrs.size() * 2) * sizeof(void *)));
    }
    SLG_CUDA(ix, cudaMemcpy(s->filter_ptrs.p, ptrs.data(), ptrs.size() * sizeof(void *), cudaMemcpyHostToDevice));
  }
  ix->filters.push_back(std::move(fp));
  return (int32_t)id;
}

static int32_t compile_filter_for_segment(slg_index *ix, Segment *s, const FilterProg &fp, DevBuf &bits_out) {
  // Resolve keyword predicates to dictionary-ordinal sets on the host (string compares happen once
  // per dictionary entry instead of once per doc, index/fastfields.rs:490-530), then evaluate the
  // program for every doc on the device.
  std::vector<FilterNodeDev> nodes(fp.nodes.size());
  std::vector<uint32_t> ordset;  // concatenated bitsets over dictionaries
  for (size_t i = 0; i < fp.nodes.size(); i++) {
    const slg_filter_node_t &n = fp.nodes[i];
    FilterNodeDev &d = nodes[i];
    d.op = n.op;
    d.n_children = n.n_children;
    d.i_min = n.i_min;
    d.i_max = n.i_max;
    d.f_min = n.f_min;
    d.f_max = n.f_max;
    d.values = nullptr;
    d.present = nullptr;
    d.offsets = nullptr;
    d.set_off = 0;
    d.set_words = 0;
    const Column *c = (n.column >= 0 && (size_t)n.column < s->columns.size()) ? &s->columns[n.column] : nullptr;
    bool leaf = n.op <= SLG_F_F64_RANGE;
    if (!leaf) continue;
    int want = (n.op == SLG_F_I64_RANGE) ? 0 : (n.op == SLG_F_F64_RANGE ? 1 : 2);
    if (!c || (c->kind != want && c->kind != want + 3)) {
      d.op = FOP_FALSE;  // unknown field or wrong column type: predicate is false (fastfields.rs `_ => false`)
      continue;
    }
    d.values = c->values.p;
    d.present = c->present.as<uint8_t>();
    d.offsets = c->offsets.as<uint32_t>();
    if (c->kind == want + 3) d.op = want == 0 ? FOP_I64_LIST : (want == 1 ? FOP_F64_LIST : FOP_KEYWORD_LIST);  // "any value", fastfields.rs:497-509, 548-562, 602-609, 632-639
    if (want == 2) {
      uint32_t words = ((uint32_t)c->dict.size() + 31) / 32;
      d.set_off = (uint32_t)ordset.size();
      d.set_words = words;
      ordset.resize(ordset.size() + words, 0u);
      if (n.value_end < n.value_begin || n.value_end > fp.strings.size()) return fail(ix, SLG_ERR_INVALID, "filter value range out of bounds");
      for (uint32_t o = 0; o < c->dict.size(); o++)
        for (uint32_t vi = n.value_begin; vi < n.value_end; vi++)
          if (ci_equals(c->dict[o], fp.strings[vi])) {
            ordset[d.set_off + (o >> 5)] |= 1u << (o & 31);
            break;
          }
    }
  }
  uint32_t words = (s->doc_count + 31) / 32;
  SLG_CUDA(ix, bits_out.alloc(std::max<size_t>(words, 1) * 4));
  DevBuf d_nodes, d_set;
  SLG_CUDA(ix, d_nodes.alloc(nodes.size() * sizeof(FilterNodeDev)));
  SLG_CUDA(ix, cudaMemcpyAsync(d_nodes.p, nodes.data(), nodes.size() * sizeof(FilterNodeDev), cudaMemcpyHostToDevice, ix->stream));
  SLG_CUDA(ix, d_set.alloc(std::max<size_t>(ordset.size(), 1) * 4));
  if (!ordset.empty()) SLG_CUDA(ix, cudaMemcpyAsync(d_set.p, ordset.data(), ordset.size() * 4, cudaMemcpyHostToDevice, ix->stream));
  if (words) {
    slg_filter_bitmap_kernel<<<(s->doc_count + 255) / 256, 256, 0, ix->stream>>>(d_nodes.as<FilterNodeDev>(), (uint32_t)nodes.size(),
                                                                                 d_set.as<uint32_t>(), s->doc_count,
                                                                                 bits_out.as<uint32_t>());
    count_launch(ix);
    SLG_CUDA(ix, cudaGetLastError());
  }
  SLG_CUDA(ix, cudaStreamSynchronize(ix->stream));
  return SLG_OK;
}

int32_t slg_filter_compile(slg_index_t *ix, const slg_filter_node_t *nodes, uint32_t n_nodes, const char *const *strings) {
  if (!ix || !nodes || !n_nodes) return SLG_ERR_INVALID;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  if (n_nodes > kMaxFilterNodes) return fail(ix, SLG_ERR_UNSUPPORTED, "filter has more than %u nodes", kMaxFilterNodes);
  FilterProg fp;
  fp.nodes.assign(nodes, nodes + n_nodes);
  uint32_t max_val = 0;
  for (auto &n : fp.nodes) {
    if (n.op > SLG_F_NOT) return fail(ix, SLG_ERR_INVALID, "unknown filter op %u", n.op);
    if (n.op <= SLG_F_KEYWORD_IN) max_val = std::max(max_val, n.value_end);
  }
  if (max_val && !strings) return fail(ix, SLG_ERR_INVALID, "keyword filter without strings");
  for (uint32_t i = 0; i < max_val; i++) fp.strings.emplace_back(strings[i]);
  // validate the prefix encoding
  {
    uint32_t pos = 0;
    std::vector<uint32_t> pending{1};
    while (!pending.empty()) {
      if (pending.back() == 0) {
        pending.pop_back();
        continue;
      }
      pending.back()--;
      if (pos >= n_nodes) return fail(ix, SLG_ERR_INVALID, "filter program is truncated");
      const auto &n = fp.nodes[pos++];
      if (n.op == SLG_F_NOT && n.n_children != 1) return fail(ix, SLG_ERR_INVALID, "Not takes one child");
      if (n.op >= SLG_F_AND) pending.push_back(n.n_children);
      if (pending.size() > kMaxFilterDepth) return fail(ix, SLG_ERR_UNSUPPORTED, "filter nesting deeper than %u", kMaxFilterDepth);
    }
    if (pos != n_nodes) return fail(ix, SLG_ERR_INVALID, "filter program has trailing nodes");
  }
  std::vector<DevBuf> per_seg(ix->segs.size());
  for (size_t si = 0; si < ix->segs.size(); si++) {
    int32_t rc = compile_filter_for_segment(ix, ix->segs[si].get(), fp, per_seg[si]);
    if (rc) return rc;
  }
  return register_filter(ix, std::move(fp), per_seg);
}

int32_t slg_filter_bitmap(slg_index_t *ix, int32_t filter_id, uint32_t segment_ord, uint32_t *bitmap_out) {
  if (!ix || !bitmap_out) return SLG_ERR_INVALID;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  Segment *s = ix->find(segment_ord);
  if (!s) return fail(ix, SLG_ERR_INVALID, "no segment %u", segment_ord);
  if (filter_id < 0 || (size_t)filter_id >= s->filter_bits.size() || !s->filter_bits[filter_id].p)
    return fail(ix, SLG_ERR_INVALID, "filter %d is not compiled for segment %u", filter_id, segment_ord);
  uint32_t words = (s->doc_count + 31) / 32;
  SLG_CUDA(ix, cudaMemcpy(bitmap_out, s->filter_bits[filter_id].p, (size_t)words * 4, cudaMemcpyDeviceToHost));
  return SLG_OK;
}

// n consecutive filter ids whose bitmaps are rows of one slab per segment
static int32_t register_slabs(slg_index *ix, std::vector<std::shared_ptr<DevBuf>> &slabs, const std::vector<uint64_t> &stride,
                              uint32_t n, int32_t *out_ids) {
  const size_t id0 = ix->filters.size();
  for (size_t si = 0; si < ix->segs.size(); si++) {
    Segment *s = ix->segs[si].get();
    s->filter_bits.resize(id0 + n);
    s->filter_slabs.resize(id0 + n);
    for (uint32_t i = 0; i < n; i++) {
      s->filter_bits[id0 + i].view(slabs[si]->as<uint32_t>() + (uint64_t)i * stride[si], stride[si] * 4);
      s->filter_slabs[id0 + i] = slabs[si];
    }
    std::vector<const uint32_t *> ptrs;
    for (auto &fb : s->filter_bits) ptrs.push_back(fb.as<uint32_t>());
    if (s->filter_ptrs.bytes < ptrs.size() * sizeof(void *)) {
      SLG_CUDA(ix, cudaStreamSynchronize(ix->stream));  // a running batch may still read the old table
      SLG_CUDA(ix, s->filter_ptrs.alloc(std::max<size_t>(64, ptrs.size() * 2) * sizeof(void *)));
    }
    SLG_CUDA(ix, cudaMemcpy(s->filter_ptrs.p, ptrs.data(), ptrs.size() * sizeof(void *), cudaMemcpyHostToDevice));
  }
  for (uint32_t i = 0; i < n; i++) {
    ix->filters.push_back(FilterProg{});
    out_ids[i] = (int32_t)(id0 + i);
  }
  return SLG_OK;
}

/* ---- phrases (query/phrase.rs:4-48) and bitmap algebra ---- */
int32_t slg_phrase_compile_batch(slg_index_t *ix, const uint32_t *term_ids, const uint32_t *phrase_offsets, const uint32_t *slops,
                                 uint32_t n_phrases, int32_t *out_ids) {
  if (!ix || !term_ids || !phrase_offsets || !n_phrases || !out_ids) return SLG_ERR_INVALID;
  if (ix->segs.empty()) return fail(ix, SLG_ERR_INVALID, "no segment loaded");
  for (uint32_t i = 0; i < n_phrases; i++) {
    const uint32_t n = phrase_offsets[i + 1] - phrase_offsets[i];
    if (phrase_offsets[i + 1] <= phrase_offsets[i]) return fail(ix, SLG_ERR_INVALID, "phrase %u has no terms", i);
    if (n > kMaxPhraseTerms) return fail(ix, SLG_ERR_UNSUPPORTED, "phrase %u has more than %u terms", i, kMaxPhraseTerms);
  }
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  cudaStream_t st = ix->stream;
  // per segment: one slab holding every phrase's bitmap, one table of phrase descriptors, one launch
  std::vector<std::shared_ptr<DevBuf>> slabs(ix->segs.size());
  std::vector<uint64_t> stride(ix->segs.size());
  for (size_t si = 0; si < ix->segs.size(); si++) {
    Segment *s = ix->segs[si].get();
    if (!s->has_positions) return fail(ix, SLG_ERR_INVALID, "segment %u holds no term positions (index without positions, or keep_positions = 0)", s->ord);
    const uint64_t words = align_up(std::max<uint64_t>((s->doc_count + 31) / 32, 1), 32);  // 128-byte rows
    stride[si] = words;
    slabs[si] = std::make_shared<DevBuf>();
    SLG_CUDA(ix, slabs[si]->alloc(words * 4 * n_phrases));
    SLG_CUDA(ix, cudaMemsetAsync(slabs[si]->p, 0, words * 4 * n_phrases, st));
    std::vector<PhraseDev> ph(n_phrases);
    std::vector<uint32_t> blk_off(n_phrases + 1, 0);
    for (uint32_t i = 0; i < n_phrases; i++) {
      PhraseDev &p = ph[i];
      std::memset(&p, 0, sizeof(p));
      const uint32_t *t = term_ids + phrase_offsets[i];
      p.n = phrase_offsets[i + 1] - phrase_offsets[i];
      p.slop = slops ? slops[i] : 0;
      bool absent = false;
      for (uint32_t j = 0; j < p.n; j++) {
        if (t[j] == 0xFFFFFFFFu || t[j] >= s->n_terms || s->h_df[t[j]] == 0) {  // api/reader.rs:1690-1697: no postings => no variant => no match
          absent = true;
          break;
        }
        p.df[j] = s->h_df[t[j]];
        p.start[j] = s->h_start[t[j]];
        if (p.df[j] < p.df[p.driver]) p.driver = j;
      }
      const uint64_t blocks = absent ? 0 : ((uint64_t)p.df[p.driver] + 255) / 256;
      if (absent) p.n = 0;
      if (blk_off[i] + blocks > 0x7FFFFFFFull) return fail(ix, SLG_ERR_UNSUPPORTED, "phrase batch is too large for one launch");
      blk_off[i + 1] = blk_off[i] + (uint32_t)blocks;
    }
    if (blk_off[n_phrases]) {
      DevBuf d_ph, d_off;
      SLG_CUDA(ix, d_ph.alloc(ph.size() * sizeof(PhraseDev)));
      SLG_CUDA(ix, d_off.alloc(blk_off.size() * 4));
      SLG_CUDA(ix, cudaMemcpyAsync(d_ph.p, ph.data(), ph.size() * sizeof(PhraseDev), cudaMemcpyHostToDevice, st));
      SLG_CUDA(ix, cudaMemcpyAsync(d_off.p, blk_off.data(), blk_off.size() * 4, cudaMemcpyHostToDevice, st));
      slg_phrase_bitmap_kernel<<<blk_off[n_phrases], 256, 0, st>>>(d_ph.as<PhraseDev>(), d_off.as<uint32_t>(), n_phrases,
                                                                 s->post_doc.as<uint32_t>(), s->pos_begin.as<uint64_t>(),
                                                                 s->pos.as<uint32_t>(), s->doc_count, slabs[si]->as<uint32_t>(), words);
      count_launch(ix);
      SLG_CUDA(ix, cudaGetLastError());
      SLG_CUDA(ix, cudaStreamSynchronize(st));  // the host tables go out of scope
    }
  }
  SLG_CUDA(ix, cudaStreamSynchronize(st));
  return register_slabs(ix, slabs, stride, n_phrases, out_ids);
}

int32_t slg_phrase_compile(slg_index_t *ix, const uint32_t *term_ids, uint32_t n_terms, uint32_t slop) {
  if (!ix || !term_ids || !n_terms) return SLG_ERR_INVALID;
  const uint32_t off[2] = {0, n_terms};
  int32_t id = -1;
  const int32_t rc = slg_phrase_compile_batch(ix, term_ids, off, &slop, 1, &id);
  return rc ? rc : id;
}

int32_t slg_filter_combine(slg_index_t *ix, uint32_t op, int32_t a, int32_t b) {
  if (!ix) return SLG_ERR_INVALID;
  if (op > SLG_COMBINE_AND_NOT) return fail(ix, SLG_ERR_INVALID, "unknown combine op %u", op);
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  cudaStream_t st = ix->stream;
  std::vector<DevBuf> per_seg(ix->segs.size());
  for (size_t si = 0; si < ix->segs.size(); si++) {
    Segment *s = ix->segs[si].get();
    for (int32_t f : {a, b})
      if (f < 0 || (size_t)f >= s->filter_bits.size() || !s->filter_bits[f].p)
        return fail(ix, SLG_ERR_INVALID, "filter %d is not compiled for segment %u", f, s->ord);
    const uint32_t words = (s->doc_count + 31) / 32;
    SLG_CUDA(ix, per_seg[si].alloc(std::max<size_t>(words, 1) * 4));
    if (words) {
      slg_bitmap_combine_kernel<<<(words + 255) / 256, 256, 0, st>>>(s->filter_bits[a].as<uint32_t>(), s->filter_bits[b].as<uint32_t>(),
                                                                    words, op, per_seg[si].as<uint32_t>());
      count_launch(ix);
    }
  }
  SLG_CUDA(ix, cudaGetLastError());
  SLG_CUDA(ix, cudaStreamSynchronize(st));
  return register_filter(ix, FilterProg{}, per_seg);
}

int32_t slg_filter_combine_batch(slg_index_t *ix, uint32_t op, const int32_t *a, const int32_t *b, uint32_t n, int32_t *out_ids) {
  if (!ix || !a || !b || !n || !out_ids) return SLG_ERR_INVALID;
  if (op > SLG_COMBINE_AND_NOT) return fail(ix, SLG_ERR_INVALID, "unknown combine op %u", op);
  if (n > 65535) return fail(ix, SLG_ERR_UNSUPPORTED, "at most 65535 combinations per call");
  if (ix->segs.empty()) return fail(ix, SLG_ERR_INVALID, "no segment loaded");
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  cudaStream_t st = ix->stream;
  std::vector<std::shared_ptr<DevBuf>> slabs(ix->segs.size());
  std::vector<uint64_t> stride(ix->segs.size());
  for (size_t si = 0; si < ix->segs.size(); si++) {
    Segment *s = ix->segs[si].get();
    std::vector<const uint32_t *> pa(n), pb(n);
    for (uint32_t i = 0; i < n; i++) {
      for (int32_t f : {a[i], b[i]})
        if (f < 0 || (size_t)f >= s->filter_bits.size() || !s->filter_bits[f].p)
          return fail(ix, SLG_ERR_INVALID, "filter %d is freed or not compiled for segment %u", f, s->ord);
      pa[i] = s->filter_bits[a[i]].as<uint32_t>();
      pb[i] = s->filter_bits[b[i]].as<uint32_t>();
    }
    const uint32_t words = (s->doc_count + 31) / 32;
    stride[si] = align_up(std::max<uint64_t>(words, 1), 32);
    slabs[si] = std::make_shared<DevBuf>();
    SLG_CUDA(ix, slabs[si]->alloc(stride[si] * 4 * n));
    SLG_CUDA(ix, cudaMemsetAsync(slabs[si]->p, 0, stride[si] * 4 * n, st));
    if (words) {
      DevBuf d_a, d_b;
      SLG_CUDA(ix, d_a.alloc(n * sizeof(void *)));
      SLG_CUDA(ix, d_b.alloc(n * sizeof(void *)));
      SLG_CUDA(ix, cudaMemcpyAsync(d_a.p, pa.data(), n * sizeof(void *), cudaMemcpyHostToDevice, st));
      SLG_CUDA(ix, cudaMemcpyAsync(d_b.p, pb.data(), n * sizeof(void *), cudaMemcpyHostToDevice, st));
      slg_bitmap_combine_batch_kernel<<<dim3((words + 255) / 256, n), 256, 0, st>>>(
          d_a.as<const uint32_t *>(), d_b.as<const uint32_t *>(), words, op, slabs[si]->as<uint32_t>(), stride[si]);
      count_launch(ix);
      SLG_CUDA(ix, cudaGetLastError());
      SLG_CUDA(ix, cudaStreamSynchronize(st));  // the host tables go out of scope
    }
  }
  return register_slabs(ix, slabs, stride, n, out_ids);
}

int32_t slg_filter_free(slg_index_t *ix, int32_t filter_id) {
  if (!ix) return SLG_ERR_INVALID;
  if (filter_id < 0 || (size_t)filter_id >= ix->filters.size()) return fail(ix, SLG_ERR_INVALID, "no filter %d", filter_id);
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  SLG_CUDA(ix, cudaStreamSynchronize(ix->stream));
  for (auto &s : ix->segs)
    if ((size_t)filter_id < s->filter_bits.size()) {
      s->filter_bits[filter_id].release();
      if ((size_t)filter_id < s->filter_slabs.size()) s->filter_slabs[filter_id].reset();  // the slab goes with its last view
    }
  return SLG_OK;
}

// PaginationCursor::encode / decode, api/reader.rs:630-691, and the generation check of decode_cursor, :821-841
int32_t slg_cursor_encode(uint32_t generation, uint32_t returned, const slg_hit_t *last_hit, char *out43) {
  if (!last_hit || !out43) return SLG_ERR_INVALID;
  uint32_t sb;
  std::memcpy(&sb, &last_hit->score, 4);
  unsigned char buf[21];
  buf[0] = 1;  // CURSOR_VERSION
  const uint32_t words[5] = {generation, sb, last_hit->segment_ord, last_hit->doc_id, returned};
  for (int w = 0; w < 5; w++)
    for (int b = 0; b < 4; b++) buf[1 + w * 4 + b] = (unsigned char)(words[w] >> (24 - 8 * b));
  static const char HEX[] = "0123456789abcdef";
  for (int i = 0; i < 21; i++) {
    out43[2 * i] = HEX[buf[i] >> 4];
    out43[2 * i + 1] = HEX[buf[i] & 15];
  }
  out43[42] = 0;
  return SLG_OK;
}

int32_t slg_cursor_decode(const char *raw, uint32_t manifest_generation, slg_hit_t *key, uint32_t *returned, char *err,
                          uint64_t err_len) {
  auto bail = [&](const char *fmt, auto... a) {
    if (err && err_len) std::snprintf(err, (size_t)err_len, fmt, a...);
    return (int32_t)SLG_ERR_INVALID;
  };
  if (!raw || !key || !returned) return bail("%s", "null argument");
  const size_t len = std::strlen(raw);
  if (len != 42) return bail("invalid cursor length: expected 42 hex chars, got %zu", len);
  unsigned char bytes[21];
  for (int i = 0; i < 21; i++) {
    int v = 0;
    for (int h = 0; h < 2; h++) {
      const char c = raw[2 * i + h];
      int d;
      if (c >= '0' && c <= '9') d = c - '0';
      else if (c >= 'a' && c <= 'f') d = c - 'a' + 10;
      else if (c >= 'A' && c <= 'F') d = c - 'A' + 10;  // u8::from_str_radix accepts both cases
      else return bail("decoding cursor at byte index %d", i);
      v = v * 16 + d;
    }
    bytes[i] = (unsigned char)v;
  }
  if (bytes[0] != 1) return bail("unsupported cursor version %u", (unsigned)bytes[0]);
  uint32_t words[5];
  for (int w = 0; w < 5; w++)
    words[w] = ((uint32_t)bytes[1 + w * 4] << 24) | ((uint32_t)bytes[2 + w * 4] << 16) | ((uint32_t)bytes[3 + w * 4] << 8) | bytes[4 + w * 4];
  if (words[4] > 50000u) return bail("cursor requests %u hits, which exceeds max supported 50000", words[4]);
  if (words[0] != manifest_generation)
    return bail("stale cursor for this index generation: expected %u, got %u", manifest_generation, words[0]);
  std::memcpy(&key->score, &words[1], 4);
  key->segment_ord = words[2];
  key->doc_id = words[3];
  *returned = words[4];
  return SLG_OK;
}

/* ---- vectors + rerank ---- */
int32_t slg_selftest_div(slg_index_t *ix, uint64_t n, uint64_t seed, uint64_t *mismatches) {
  if (!ix || !mismatches) return SLG_ERR_INVALID;
  SLG_CUDA(ix, cudaSetDevice(ix->device));
  DevBuf d;
  SLG_CUDA(ix, d.alloc(8));
  SLG_CUDA(ix, cudaMemsetAsync(d.p, 0, 8, ix->stream));
  slg_selftest_div_kernel<<<ix->n_sm * 8, 256, 0, ix->stream>>>(n, seed, d.as<unsigned long long>());
  count_launch(ix);
  SLG_CUDA(ix, cudaGetLastError());
  unsigned long long v = 0;
  SLG_CUDA(ix, cudaMemcpyAsync(&v, d.p, 8, cudaMemcpyDeviceToHost, ix->stream));
  SLG_CUDA(ix, cudaStreamSynchronize(ix->stream));
  *mismatches = v;
  return SLG_OK;
}

int32_t slg_get_stream(const slg_index_t *ix, void **cuda_stream) {
  if (!ix || !cuda_stream) return SLG_ERR_INVALID;
  *cuda_stream = (void *)ix->stream;
  return SLG_OK;
}

int32_t slg_get_counters(const slg_index_t *ix, slg_counters_t *out) {
  if (!ix || !out) return SLG_ERR_INVALID;
  *out = ix->ctr;
  return SLG_OK;
}

}  // extern "C"
