/*
 * searchlite_gpu.h — C ABI of the B200-native retrieval engine (libsearchlite_gpu.so).
 *
 * This is the drop-in boundary for searchlite-core's per-segment search hot path.  The
 * reference has no inbound plugin interface (SURVEY.md §8b); the seam a Rust
 * `#[cfg(feature = "gpu")]` shim would bind is
 *
 *   IndexReader::search_segment            searchlite-core/src/api/reader.rs:2908-3128
 *     -> execute_top_k_with_stats_and_mode_internal   src/query/wand.rs:398-456
 *   SegmentReader::open (residency)         src/index/segment.rs:1239
 *   hits.sort_by(SortKey) (segment merge)   src/api/reader.rs:2777, src/query/sort.rs:80-93
 *   gpu::rerank (identity stub)             src/gpu/rerank.rs:3-5
 *
 * Conventions: plain pointers and sizes only; the caller owns every host buffer; handles own
 * device memory; no callbacks cross the ABI (the reference's `accept` closure is replaced by
 * data: matcher roles, filter programs, deleted-doc list).  Every function returns 0 on success
 * and a negative slg_status on failure, never aborts or unwinds; slg_last_error() gives the text.
 * A handle is thread-compatible: one in-flight call per handle, several handles may run
 * concurrently.  All calls are synchronous unless stated otherwise.  There is no CPU fallback:
 * without a usable CUDA device slg_open fails.
 */
#ifndef SEARCHLITE_GPU_H
#define SEARCHLITE_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct slg_index slg_index_t;
typedef struct slg_batch slg_batch_t;

typedef enum {
  SLG_OK = 0,
  SLG_ERR_INVALID = -1,     /* bad argument */
  SLG_ERR_CUDA = -2,        /* CUDA runtime error (text in slg_last_error) */
  SLG_ERR_NO_DEVICE = -3,   /* no CUDA device: there is no CPU fallback */
  SLG_ERR_UNSUPPORTED = -4, /* valid request outside the built scope (e.g. k too large) */
  SLG_ERR_OOM = -5
} slg_status;

/* ExecutionStrategy, src/api/types.rs:6-13.  All three return the EXACT top-k (bm25 == wand,
 * query/wand.rs:459-566, :659-903).  BM25 scores every posting; WAND and BMW add safe
 * block-max pruning (the reference's own `bmw` is not exact, SURVEY.md §8c — not reproduced). */
typedef enum { SLG_EXEC_BM25 = 0, SLG_EXEC_WAND = 1, SLG_EXEC_BMW = 2 } slg_exec_t;

/* term-group roles of the flat matcher, src/api/reader.rs:1485-1565 */
enum { SLG_ROLE_SHOULD = 0, SLG_ROLE_MUST = 1, SLG_ROLE_MUST_NOT = 2 };
enum { SLG_TERM_SCORED = 1u };
#define SLG_MAX_QUERY_TERMS 64u
#define SLG_MAX_GROUPS 8u
#define SLG_MAX_K 2048u

/* One "field:term" key of a query after search_segment's weight merge (api/reader.rs:2971-2983). */
typedef struct {
  uint32_t term_id; /* ordinal of the key in the handle's term space; UINT32_MAX = absent */
  float weight;     /* sum of group.boost*field.boost over duplicate keys.  A scored term's weight must be finite and
                       >= 2^-100 (about 7.9e-31), else the batch fails with SLG_ERR_UNSUPPORTED: the kernels read a
                       contribution of +0 as "the doc lacks the term" and never return a doc scored 0, while the reference
                       keeps one.  From 2^-100 up, a posting's contribution stays above 2^-133 for any k1 >= 0, b in [0, 1]
                       and doc less than 2^32 times longer than the average */
  uint32_t leaf;    /* ScorePlan leaf (Sum-of-leaves plan; list terms in leaf order) */
  uint32_t group;   /* matcher term group */
  uint32_t flags;   /* SLG_TERM_SCORED if it contributes to the score */
} slg_term_t;

/* RankedHit as merged by SortKey: score desc, segment_ord asc, doc_id asc */
typedef struct {
  uint32_t segment_ord;
  uint32_t doc_id;
  float score;
} slg_hit_t;

/* ScorePlan (query/planner.rs:113-164): the ScoreExpr tree in POSTFIX order, evaluated per doc on the
 * per-leaf sums `leaves[term.leaf] += score_tf(..)` of query/wand.rs:470-497 (terms added in listed order):
 *   LEAF   arg = leaf index                      -> leaves[arg]                      (planner.rs:134)
 *   SUM    arg = number of children              -> ((0 + c0) + c1) + ..             (planner.rs:135)
 *   DISMAX arg = number of children, tie_breaker -> max + tie_breaker * (sum - max)  (planner.rs:136-151)
 * tie_breaker must lie in [0, 1] (validate_tie_breaker, planner.rs:850-858).  Every leaf of a scored
 * term must be read by the plan (the planner guarantees it, planner.rs:284-460). */
enum { SLG_PLAN_LEAF = 0, SLG_PLAN_SUM = 1, SLG_PLAN_DISMAX = 2 };
#define SLG_MAX_PLAN_LEAVES 8u
#define SLG_MAX_PLAN_NODES 32u
typedef struct {
  uint32_t op;
  uint32_t arg;
  float tie_breaker;
} slg_plan_node_t;

typedef struct {
  uint32_t n_terms;
  const slg_term_t *terms;
  uint32_t n_groups;         /* 0 = plain OR of the scored terms (QueryString, min_should 1) */
  const uint8_t *group_role; /* n_groups entries */
  uint32_t min_should;       /* resolved minimum_should_match */
  uint32_t leaf_count;       /* number of ScorePlan leaves when `plan` is given (1..SLG_MAX_PLAN_LEAVES) */
  int32_t filter_id;         /* root filter from slg_filter_compile, -1 = none */
  uint32_t n_plan_nodes;     /* 0 = no plan: the score is the running sum of the terms in listed order */
  const slg_plan_node_t *plan; /* n_plan_nodes postfix nodes leaving exactly one value */
  /* search-after cursor (SearchRequest.cursor, api/reader.rs:3019-3028): with has_cursor != 0 a doc is accepted only
   * if its SortKey (score desc, segment_ord asc, doc_id asc; query/sort.rs:80-93) is strictly after `cursor`; the doc
   * whose key equals the cursor is rejected and reported by slg_batch_cursor_seen (saw_cursor, api/reader.rs:2747). */
  uint32_t has_cursor;
  slg_hit_t cursor;
} slg_query_t;

/* QueryStats, src/query/wand.rs:45-50 (+ pruning counters the example prints, examples/pruning.rs:198-203) */
typedef struct {
  uint64_t scored_docs;       /* docs that received at least one contribution */
  uint64_t postings_advanced; /* postings decoded and scored */
  uint64_t blocks_skipped;    /* (query, tile) items skipped by the block-max bound */
  uint64_t candidates_examined;
  uint64_t total_matches;     /* docs accepted by the accept closure (match counter, api/reader.rs:3029-3031): exact under
                               * BM25; under WAND/BMW an estimate, as the reference's total_hits_estimate is (skipped
                               * tiles and MaxScore-skipped terms are not visited).  Counted by the warp / CTA kernels (a batch with statistics runs there). */
} slg_stats_t;

/* Where the arrays of a view live. */
enum { SLG_MEM_HOST = 0, SLG_MEM_DEVICE = 1 };

/* One segment as SegmentReader holds it, already parsed into SoA (CSR postings + `_len:` column).
 * Replaces SegmentReader::open + PostingsReader::read_at + field_lengths_for
 * (index/segment.rs:1239, index/postings.rs:142-212, api/reader.rs:3604-3621). */
typedef struct {
  uint32_t segment_ord;
  uint32_t doc_count;
  uint64_t n_terms;
  const uint64_t *term_offsets;        /* n_terms+1, CSR */
  const uint32_t *post_docs;           /* ascending per term */
  const uint32_t *post_tfs;
  const int64_t *field_lengths;        /* `_len:<field>` i64 column, doc_count entries */
  const uint8_t *field_length_present; /* nullable */
  uint64_t total_tokens;               /* sum of field lengths: avgdl = total/doc_count, segment.rs:946-957 */
  const uint32_t *deleted_docs;        /* HOST array, nullable */
  uint32_t n_deleted;
  int32_t memory_space;                /* SLG_MEM_HOST or SLG_MEM_DEVICE for the five arrays above */
} slg_segment_view_t;

/* Filter AST, src/api/types.rs:670-680, evaluated as src/query/filters.rs:84-149 over flat
 * columns.  Prefix encoding: a node is followed by its n_children sub-trees. */
enum {
  SLG_F_KEYWORD_EQ = 0,
  SLG_F_KEYWORD_IN = 1,
  SLG_F_I64_RANGE = 2,
  SLG_F_F64_RANGE = 3,
  SLG_F_AND = 4,
  SLG_F_OR = 5,
  SLG_F_NOT = 6
};
typedef struct {
  uint32_t op;
  int32_t column;       /* handle from slg_add_*_column; -1 = unknown field (predicate false) */
  int64_t i_min, i_max; /* inclusive */
  double f_min, f_max;  /* inclusive */
  uint32_t n_children;
  uint32_t value_begin, value_end; /* keyword values: range in the strings array */
} slg_filter_node_t;

typedef enum { SLG_METRIC_COSINE = 0, SLG_METRIC_L2 = 1 } slg_metric_t;

/* Engine counters (cumulative since open unless noted). */
typedef struct {
  uint64_t kernel_launches;    /* kernels this library launched */
  uint64_t score_launches;     /* launches of the dominant scoring kernel */
  double score_ms_total;       /* CUDA-event time of those launches, on the handle's stream */
  double last_score_ms;
  double last_batch_ms;        /* device time of the last slg_batch_run (all kernels) */
  uint64_t last_posting_count; /* sum over queries of df of their scored terms, last batch */
  uint64_t resident_bytes;     /* device bytes held by loaded segments */
  uint64_t last_h2d_bytes;     /* host->device bytes of the last slg_batch_prepare */
  uint64_t last_d2h_bytes;     /* device->host bytes of the last slg_batch_fetch / slg_merge_gathered */
  /* work of the last fetched run of the posting-driven kernels (whole batch, all segments): */
  uint64_t last_postings_scattered;     /* postings read and accumulated (compare with last_posting_count) */
  uint64_t last_subtiles_skipped;       /* (query, sub-tile) pairs dropped inside the sweep by the bound */
  uint64_t last_column_blocks_streamed; /* 512-doc blocks of dense columns read */
  uint64_t last_items;                  /* (query, doc-range) items scored, seeds included; flat scan: (query, term, chunk) items scanned */
  uint64_t last_postings_verified;      /* flat scan: postings whose doc got its exact score (binary searches + column gathers) */
  uint64_t last_items_dropped;          /* flat scan, pruned: items of non-essential terms dropped (MaxScore) */
  /* hybrid rerank (slg_rerank_batch with sync != 0): */
  uint64_t rerank_launches;    /* calls timed */
  double rerank_ms_total;      /* CUDA-event time of their kernels (scores + sort per segment, merge) */
  double last_rerank_ms;
} slg_counters_t;

/* One vector clause of a hybrid request (VectorClausePlan, api/reader.rs:2162-2171).  query_vecs: n_queries x dim f32,
 * host or device memory, already normalised for cosine fields (normalize_in_place is the planner's step,
 * api/reader.rs:2119-2125).  The clause's similarity is multiplied by boost (api/reader.rs:2421) and blended with the
 * BM25 score by alpha (compute_hybrid_score, api/reader.rs:226-254); several clauses are averaged. */
typedef struct {
  const float *query_vecs;
  float alpha;          /* 0..1; >= 1 keeps the BM25 score, <= 0 the vector score */
  float boost;          /* >= 0, finite; 1.0 = none */
  slg_metric_t metric;  /* the field's metric */
  uint32_t reserved;
} slg_vector_clause_t;

/* ---- lifetime ---- */
int32_t slg_open(int32_t device, slg_index_t **out);
int32_t slg_close(slg_index_t *);
/* text of the last error on this handle (or of the last failed slg_open when NULL) */
const char *slg_last_error(const slg_index_t *);
/* tuning knobs; 0 keeps the default.  tile_docs: docs per shared-memory tile of the CTA-per-item
 * kernel (multiple of 1024); sub_docs: docs per warp-private tile of the warp-per-item kernel
 * (multiple of 128); kernel_choice: 0 = automatic — plain OR queries with <= 8 terms per query and
 * k <= 2048 on the flat posting scan + column pass, queries with a Bool matcher, a ScorePlan, a cursor
 * or statistics on the warp kernel (k <= 32, <= 8 terms) or the CTA kernel (everything else);
 * 1 = CTA kernel, 2 = warp kernel (the reference's query summation order), 3 = the posting-driven
 * path or an error; add 256 to ignore the resident per-posting scores and score postings in place. */
int32_t slg_configure(slg_index_t *, uint32_t tile_docs, uint32_t ctas_per_sm, uint32_t sub_docs,
                      uint32_t kernel_choice);
/* residency / tuning options; the residency ones apply to segments loaded AFTER the call:
 *   "resident_scores"  1/0  keep the unit-weight BM25 contribution of every posting in HBM (default 1)
 *   "dense_den"        n    terms with df * n >= doc_count also get a doc-indexed f32 score column: they
 *                           are never scanned posting by posting; verification reads them with one gather
 *                           (default 24; 0 = no columns)
 *   "dense_min_df"     n    ... and df >= n (default 256)
 *   "max_column_bytes" n    byte budget of the columns of one segment, largest df first (default 24 GiB)
 *   "bitmap_den"       n    terms with df * n >= doc_count (and df >= 64) and no column get a presence bitmap
 *                           with interleaved rank, 32 bytes per 224 docs: the verification learns whether the
 *                           list holds the doc and, if so, its position in the list from one 32-byte sector,
 *                           without searching the list (default 512; 0 = none: every look-up searches)
 *   "max_bitmap_bytes" n    byte budget of those bitmaps, largest df first, at most 32768 rows (default 16 GiB)
 *   "keep_positions"   1/0  keep term positions resident when a posting image carries them (default 1)
 *   "scan_kernels"     1/0  plain OR batches on the flat posting scan (default 1); 0 = the sub-tile kernels
 *   "stream_kernels"   1/0  with scan_kernels 0: exhaustive batches on the sparse pass + column pass (default 1)
 *   "strict_accumulate" 0/1 exhaustive sub-tile kernels: 1 = add every posting into its doc's accumulator even where
 *                           the doc provably cannot enter the top k (default 0)
 *   "scan_chunk"       n    flat posting scan: postings per work item (multiple of 256; default 0 = by segment size:
 *                           4096 from 4 M docs, 2048 from 2 M, else 1024)
 *   "scan_first_part"  n    two-step runs (slg_batch_run_seeds / _sweep): 256ths of the items scanned before the
 *                           threshold exchange (default 24)
 *   "stage_cap"        n    sparse pass: postings a warp stages in shared memory per span (default 1024)
 *   "maxscore_pct"     n    pruned executions of the warp kernel (MaxScore): per (query, tile) the terms whose
 *                           bounds sum to less than n % of the running k-th score are not scattered; docs touched
 *                           by the other terms are rescored exactly if they can still qualify (default 35;
 *                           0 = tile skipping only).  The result is bit-identical to the exhaustive run.
 *   "heavy_kernel"     0    (round 1's tile-sweep kernel was removed; 1 is refused)
 * Float contract: the posting-driven kernels (flat scan, column pass, items / stream kernels) sum a doc's
 * contributions over the query's terms WITHOUT a dense column first, then over the terms WITH one, each
 * group in query order (one left fold from +0) — brute_force (query/wand.rs:527-548) on that
 * permutation of the query, reproduced bit for bit; the warp and CTA kernels sum in query order.  Both
 * agree with the reference within the 1e-5 rule (the reference's own order follows HashMap iteration). */
int32_t slg_set_option(slg_index_t *, const char *name, uint64_t value);
/* 1 if `term_id` of the segment has a dense column (it is summed first by the column front ends) */
int32_t slg_term_has_column(const slg_index_t *, uint32_t segment_ord, uint32_t term_id);

/* ---- residency (SegmentReader::open) ---- */
int32_t slg_load_segment(slg_index_t *, const slg_segment_view_t *view, float k1, float b);
/* Same, from the reference's on-disk `.post` image (index/postings.rs:78-129): term t's list
 * starts at post_image[term_post_offsets[t]]; decoded on the device. */
int32_t slg_load_segment_post_image(slg_index_t *, const slg_segment_view_t *view_without_postings,
                                    const uint8_t *post_image, uint64_t post_image_bytes,
                                    const uint64_t *term_post_offsets, float k1, float b);
/* ---- residency from the reference's own segment files (SURVEY.md §8f row 1) ----
 * One segment as the reference's writer left it on disk; the caller reads or mmaps the files and passes
 * their bytes (SegmentReader::open, index/segment.rs:1239-1330, reads the same four):
 *   terms  seg_<id>.terms  index/terms.rs:10-25        post  seg_<id>.post  index/postings.rs:78-129
 *   fast   seg_<id>.fast   index/fastfields.rs:409-424 meta  seg_<id>.meta  index/segment.rs:43-53 (JSON)
 * doc_count / deleted_docs / checksums come from the segment's MANIFEST.json entry (SegmentMeta,
 * index/manifest.rs:24-37).  checksums (nullable) = crc32 of the whole {terms, postings, fast, meta} files,
 * verified like verify_checksums (index/segment.rs:1140-1200). */
typedef struct {
  uint32_t segment_ord;
  uint32_t doc_count;
  const uint8_t *terms;
  uint64_t terms_bytes;
  const uint8_t *post;
  uint64_t post_bytes;
  const uint8_t *fast;
  uint64_t fast_bytes;
  const uint8_t *meta;
  uint64_t meta_bytes;
  const uint32_t *deleted_docs;
  uint32_t n_deleted;
  const uint32_t *checksums;
} slg_segment_files_t;

typedef struct {
  uint64_t n_terms_total;     /* keys in .terms, all fields */
  uint64_t n_terms_field;     /* keys "<field>:..." */
  uint64_t n_postings;        /* sum of their df */
  float avgdl;                /* .meta avg_field_lengths[field] (0 when absent, index/segment.rs:1344-1351) */
  uint32_t has_positions;     /* some list of the field carries positions */
  uint32_t has_length_column; /* `_len:<field>` is present in .fast */
  uint32_t n_fast_columns, n_scalar_columns;
  uint32_t crc_terms, crc_postings, crc_fast, crc_meta; /* crc32 of the images as given */
  uint32_t n_list_columns;    /* list and nested value columns (types 3..8), loaded with "any value" semantics */
  uint32_t reserved;
} slg_segment_info_t;

/* Host-only: parse + validate the files (checksums, crc of .terms, structure of .fast, .meta JSON) without
 * touching a device.  err (nullable) receives the message on failure. */
int32_t slg_inspect_segment_files(const slg_segment_files_t *files, const char *field, slg_segment_info_t *out, char *err,
                                  uint64_t err_cap);
/* Load one segment for scoring the text field(s) `field`: one name, or several separated by commas
 * ("title,body") — every "f:token" key of a named field enters the term space and is scored with ITS field's
 * `_len:<f>` column, avg_field_lengths[f] and minimum doc length (ScoredTerm carries them per key,
 * api/reader.rs:2990-2994), which is what a QueryString over several default fields needs
 * (query/planner.rs:284-312: one key per field in the term's group, all on one leaf).  Every segment of a
 * handle must name the same list.  Term ids of such a handle
 * are handed out per "field:token" key in order of first appearance across the loaded segments —
 * slg_term_lookup resolves a key; a segment that lacks a key treats it as an empty list
 * (seg.postings(key) == None, api/reader.rs:2986-2988).  avgdl is the .meta value, N/df/min_doc_len are
 * per segment as in the reference; postings are decoded on the device; I64/F64/Str fast fields, their list forms
 * (I64List / F64List / StrList) and their nested forms (flattened: any value of any object) become filter columns
 * addressed by name (slg_column_lookup); a predicate on a list column holds when ANY value of the doc satisfies it
 * (index/fastfields.rs:490-657).
 * Positions stay resident for slg_phrase_compile unless option "keep_positions" is 0. */
int32_t slg_load_segment_files(slg_index_t *, const slg_segment_files_t *files, const char *field, float k1, float b);
/* The same for every segment of an index directory, in MANIFEST.json order (segment_ord = position).
 * vector_field (nullable): also load seg_<id>_vectors/<vector_field>.bin of every segment. */
int32_t slg_load_index_dir(slg_index_t *, const char *dir, const char *field, float k1, float b, const char *vector_field,
                           int32_t store_bf16, uint32_t *n_segments_out);
/* One process per GPU: load only the manifest segments with position % shard_world == shard_rank (segment == shard;
 * N, df, avgdl are per segment in the reference, so no statistics cross GPUs).  segment_ord stays the manifest
 * position; every rank resolves query keys against its own term space (slg_term_lookup) and the local top-k lists
 * meet in slg_merge_gathered.  *n_segments_out = segments this rank loaded. */
int32_t slg_load_index_dir_shard(slg_index_t *, const char *dir, const char *field, float k1, float b, const char *vector_field,
                                 int32_t store_bf16, uint32_t shard_rank, uint32_t shard_world, uint32_t *n_segments_out);
/* <field>.bin image ("VCTR", index/segment.rs:1030-1119) -> slg_load_vectors.  metric_out nullable: 0 cosine, 1 l2 */
int32_t slg_load_vector_file(slg_index_t *, uint32_t segment_ord, const uint8_t *bytes, uint64_t n_bytes, int32_t store_bf16,
                             int32_t *metric_out);
/* *term_id = id of "field:token" in the handle's term space, UINT32_MAX if no loaded segment holds it */
int32_t slg_term_lookup(const slg_index_t *, const char *key, uint32_t *term_id);
/* column handle of a fast field loaded from files, -1 if unknown */
int32_t slg_column_lookup(const slg_index_t *, const char *name);

/* Term positions of a segment loaded through slg_load_segment (PostingEntry.positions, index/postings.rs:14-19):
 * term_offsets is the view's CSR, position_offsets has one entry per posting + 1, positions are absolute and
 * ascending per posting.  memory_space: SLG_MEM_HOST or SLG_MEM_DEVICE for the three arrays. */
int32_t slg_load_positions(slg_index_t *, uint32_t segment_ord, const uint64_t *term_offsets, const uint64_t *position_offsets,
                           const uint32_t *positions, int32_t memory_space);

/* fast-field columns of the last loaded segment (index/fastfields.rs:910-1039); return handle >= 0 */
int32_t slg_add_i64_column(slg_index_t *, uint32_t segment_ord, const int64_t *values, const uint8_t *present);
int32_t slg_add_f64_column(slg_index_t *, uint32_t segment_ord, const double *values, const uint8_t *present);
int32_t slg_add_str_column(slg_index_t *, uint32_t segment_ord, const char *const *dict, uint32_t n_dict,
                           const uint32_t *ords /* UINT32_MAX = missing */);
/* list columns (I64List / F64List / StrList, index/fastfields.rs:926-940, 1045-1068): offsets[doc_count + 1] are running
 * sums starting at 0, the values of doc d are values[offsets[d] .. offsets[d + 1]); a filter leaf on such a column holds
 * when any value of the doc satisfies it (matches_keyword / matches_i64_range / ..., index/fastfields.rs:490-657) */
int32_t slg_add_i64_list_column(slg_index_t *, uint32_t segment_ord, const uint32_t *offsets, const int64_t *values);
int32_t slg_add_f64_list_column(slg_index_t *, uint32_t segment_ord, const uint32_t *offsets, const double *values);
int32_t slg_add_str_list_column(slg_index_t *, uint32_t segment_ord, const char *const *dict, uint32_t n_dict,
                                const uint32_t *offsets, const uint32_t *ords);
/* segment statistics as the reference derives them (for the host shim and for tests) */
int32_t slg_segment_stats(const slg_index_t *, uint32_t segment_ord, float *avgdl, float *live_docs,
                          float *min_doc_len, uint64_t *n_postings);
/* avgdl and minimum positive doc length of the field_index-th scored field (0 = the first / only one) */
int32_t slg_field_stats(const slg_index_t *, uint32_t segment_ord, uint32_t field_index, float *avgdl, float *min_doc_len);
/* device bytes of the segment per resident array, as a JSON object (post_doc, post_score, score_columns,
 * presence_bitmaps, positions, vectors, ...; plus the number of score columns and presence bitmaps) */
int32_t slg_segment_residency(const slg_index_t *, uint32_t segment_ord, char *json_out, uint64_t json_len);

/* ---- filters (query/filters.rs) ---- */
/* compiles a root filter against every loaded segment (one bitmap per segment); returns id >= 0 */
int32_t slg_filter_compile(slg_index_t *, const slg_filter_node_t *nodes, uint32_t n_nodes,
                           const char *const *strings);
/* copy the filter's bitmap for one segment to the host: ceil(doc_count/32) words, LSB first */
int32_t slg_filter_bitmap(slg_index_t *, int32_t filter_id, uint32_t segment_ord, uint32_t *bitmap_out);

/* ---- phrases (SURVEY.md §8f row 2; query/phrase.rs:4-48, api/reader.rs:1584-1597) ----
 * A phrase is compiled, like a root filter, into one doc bitmap per loaded segment and the returned id is used
 * wherever a filter id is (slg_query_t.filter_id, slg_filter_bitmap): a doc is in the bitmap iff it holds every
 * term, each with at least one position, and positions p_0 < p_1 < ... (phrase order) exist whose gaps
 * sum to <= slop.  A term the segment lacks gives an empty bitmap.  Needs resident positions.
 * The matcher requires every phrase of a query (api/reader.rs:1504-1508): AND them, and the root filter,
 * with slg_filter_combine. */
int32_t slg_phrase_compile(slg_index_t *, const uint32_t *term_ids, uint32_t n_terms, uint32_t slop);
/* The phrases of a whole query batch in one launch per segment: phrase i = term_ids[phrase_offsets[i] ..
 * phrase_offsets[i+1]) with slops[i] (slops nullable = all 0); out_ids receives n_phrases consecutive ids. */
int32_t slg_phrase_compile_batch(slg_index_t *, const uint32_t *term_ids, const uint32_t *phrase_offsets, const uint32_t *slops,
                                 uint32_t n_phrases, int32_t *out_ids);
enum { SLG_COMBINE_AND = 0, SLG_COMBINE_OR = 1, SLG_COMBINE_AND_NOT = 2 };
/* new filter id = a op b, per segment */
int32_t slg_filter_combine(slg_index_t *, uint32_t op, int32_t a, int32_t b);
/* n combinations in one launch per segment (a query batch's phrase-and-filter conjunctions): out_ids[i] = a[i] op b[i] */
int32_t slg_filter_combine_batch(slg_index_t *, uint32_t op, const int32_t *a, const int32_t *b, uint32_t n, int32_t *out_ids);
/* release the bitmaps of a filter / phrase id (ids are not reused; a batch naming a freed id is rejected) */
int32_t slg_filter_free(slg_index_t *, int32_t filter_id);

/* ---- batched search (search_segment + execute_top_k for Q queries, all loaded segments) ---- */
/* k is the INTERNAL k (the reference passes limit+1, api/reader.rs:2595-2619).  out_hits has
 * n_queries*k entries, per query sorted by (score desc, segment_ord asc, doc_id asc);
 * out_counts[q] <= k.  out_stats nullable (n_queries entries). */
int32_t slg_search_batch(slg_index_t *, const slg_query_t *queries, uint32_t n_queries, uint32_t k,
                         slg_exec_t exec, uint32_t bmw_block_size, slg_hit_t *out_hits, uint32_t *out_counts,
                         slg_stats_t *out_stats);

/* The same in three steps, so a caller can keep a batch resident and re-run it:
 * prepare = validate + upload; run = all kernels (asynchronous on the handle's stream unless
 * sync != 0); fetch = device->host copy of the results of the last run. */
int32_t slg_batch_prepare(slg_index_t *, const slg_query_t *queries, uint32_t n_queries, uint32_t k,
                          slg_exec_t exec, uint32_t bmw_block_size, slg_batch_t **out);
/* collect slg_stats_t counters in later runs (off by default: the counting costs a few percent) */
int32_t slg_batch_enable_stats(slg_batch_t *, int32_t on);
int32_t slg_batch_run(slg_batch_t *, int32_t sync);
/* The run in two steps for one-segment-per-GPU sharding (SURVEY.md §8e): the first step (the seed pass of the sub-tile
 * kernels, or the first "scan_first_part" of the posting scan's items, rarest terms first) gives every query a local k-th
 * key; the caller max-reduces the keys over the shards (e.g. ncclAllReduce(max) on the uint64 array of
 * slg_batch_threshold_keys, n_queries entries in query order, on the handle's stream) and hands the result to
 * slg_batch_import_thresholds, which keeps the score part (a global k-th score is a safe bound for every shard; an
 * equal score may still win on segment order, query/sort.rs:80-93); the sweep then prunes against the global bound.
 * The merged result over all shards is exact; a shard's own list may lack docs that cannot reach the global top k.
 * Needs one segment in the handle and a batch the posting scan (any execution) or the pruned items kernel handles.
 * slg_batch_set_threshold_board below does the same exchange inside ONE launch over peer-mapped memory. */
int32_t slg_batch_run_seeds(slg_batch_t *);
int32_t slg_batch_threshold_keys(slg_batch_t *, void **dev_keys);
int32_t slg_batch_import_thresholds(slg_batch_t *, const void *dev_keys);
int32_t slg_batch_run_sweep(slg_batch_t *, int32_t sync);
/* Sharded runs over NVLink / NVSwitch, one segment per handle: a THRESHOLD BOARD in peer-accessible device memory (CUDA IPC
 * or symmetric-memory mappings the caller set up; n_queries x 8 bytes per shard, zero-initialised once).  While the posting
 * scan runs, a shard that raises a query's k-th score pushes it into every peer's board (system-scope atomic max on the peer
 * mapping) and folds what its peers pushed into its own pruning bound — the largest k-th score of any shard is a lower
 * bound of the global one — so all shards prune against (nearly) the global threshold with no kernel boundary, collective
 * or host round trip.  local_board: this shard's board; peer_boards: the mappings of the OTHER shards' boards (at most 7);
 * epoch: a number >= 1 that is the same on every shard for one batch and rises with every batch (stale pushes are ignored).
 * The results are exact with or without a board.  local_board NULL switches it off. */
int32_t slg_batch_set_threshold_board(slg_batch_t *, void *local_board, void *const *peer_boards, uint32_t n_peers,
                                      uint32_t epoch);
int32_t slg_batch_fetch(slg_batch_t *, slg_hit_t *out_hits, uint32_t *out_counts, slg_stats_t *out_stats);
/* device pointers of the last run's results (n_queries*k slg_hit_t, n_queries u32) for an
 * allgather by the caller; valid until the batch is re-run or freed */
int32_t slg_batch_device_results(slg_batch_t *, void **dev_hits, void **dev_counts);
/* the same as ONE block — n_queries*k hits followed by n_queries counts, *n_bytes long — the send buffer of a single
 * allgather (slg_merge_gathered_packed takes the gathered blocks) */
int32_t slg_batch_packed_results(slg_batch_t *, void **dev_block, uint64_t *n_bytes);
/* device->device copy of the last run's results into caller buffers (e.g. the send buffer of an
 * allgather), asynchronous on the handle's stream */
int32_t slg_batch_copy_results_device(slg_batch_t *, void *dst_dev_hits, void *dst_dev_counts);
/* saw_cursor per query after slg_batch_run: 1 if the doc named by the query's cursor was met (and rejected) by accept.
 * The reference fails the request with "stale or invalid cursor for this result set" when it was not (api/reader.rs:2747-2749).
 * Queries without a cursor report 1 (api/reader.rs:2663). */
int32_t slg_batch_cursor_seen(slg_batch_t *, uint8_t *out_seen);
int32_t slg_batch_free(slg_batch_t *);

/* PaginationCursor of the score-sorted fast path (api/reader.rs:614-691): 21 bytes — version 1, generation, score bits,
 * segment_ord, doc_id, returned, all big-endian — as 42 lowercase hex characters.  encode writes 43 bytes (NUL included).
 * decode checks length, hex digits, version, returned <= 50000 (MAX_CURSOR_ADVANCE, :55) and the manifest generation
 * (decode_cursor, :821-841) and writes the reference's message into err on failure (returns SLG_ERR_INVALID). */
int32_t slg_cursor_encode(uint32_t generation, uint32_t returned, const slg_hit_t *last_hit, char *out43);
int32_t slg_cursor_decode(const char *raw, uint32_t manifest_generation, slg_hit_t *key, uint32_t *returned, char *err,
                          uint64_t err_len);

/* ---- shard merge (api/reader.rs:2777): gathered is n_shards x n_queries x k hits (DEVICE memory),
 * counts n_shards x n_queries (DEVICE).  Writes n_queries x k merged hits / counts to HOST buffers. */
int32_t slg_merge_gathered(slg_index_t *, const void *dev_gathered_hits, const void *dev_gathered_counts,
                           uint32_t n_shards, uint32_t n_queries, uint32_t k, slg_hit_t *out_hits,
                           uint32_t *out_counts);

/* gathered blocks of slg_batch_packed_results, shard_stride bytes apart (0 = tightly packed), DEVICE memory */
int32_t slg_merge_gathered_packed(slg_index_t *, const void *dev_gathered, uint64_t shard_stride, uint32_t n_shards,
                                  uint32_t n_queries, uint32_t k, slg_hit_t *out_hits, uint32_t *out_counts);

/* ---- vectors + rerank (what gpu::rerank should have been; vectors/mod.rs:63-129, api/reader.rs:218-254) ----
 * offsets: doc -> row in values or UINT32_MAX (VectorStore, index/segment.rs:1030-1053); offsets past n_rows are
 * refused (SLG_ERR_INVALID).  offsets / values may be host or device memory.
 * store_bf16 != 0 keeps the rows as bf16 in HBM (rounded once; the arithmetic stays f32), else f32. */
int32_t slg_load_vectors(slg_index_t *, uint32_t segment_ord, uint32_t dim, const uint32_t *offsets,
                         const float *values, uint64_t n_rows, int32_t store_bf16);
/* the same from rows that already are bf16 (host or device memory) */
int32_t slg_load_vectors_bf16(slg_index_t *, uint32_t segment_ord, uint32_t dim, const uint32_t *offsets,
                              const uint16_t *values_bf16, uint64_t n_rows);
/* For each query: score every candidate hit as compute_hybrid_score (one clause, boost 1):
 * alpha*bm25 + (1-alpha)*similarity, missing vector => -1 (cosine) / f32::MIN (L2); re-sort by
 * (score desc, segment_ord asc, doc_id asc).  cands is n_queries*cand_stride hits (HOST memory).  The dot product /
 * squared distance is folded in dimension order with unfused multiply and add, like the reference's iterator sum:
 * f32 rows give the reference's bits.  Any dim; multiples of 32 (f32 rows) / 64 (bf16 rows) take the coalesced path. */
int32_t slg_rerank(slg_index_t *, const float *query_vecs, uint32_t n_queries, uint32_t dim,
                   const slg_hit_t *cands, const uint32_t *cand_counts, uint32_t cand_stride, float alpha,
                   slg_metric_t metric, slg_hit_t *out_hits, float *out_vector_scores);
/* The same for up to 8 clauses (MAX_VECTOR_CLAUSES, api/reader.rs:134): final = mean of the clause blends.  When every
 * clause has alpha <= 0, candidates without a vector are dropped (api/reader.rs:2474-2476) and out_counts (nullable)
 * receives the new counts.  out_vector_scores (nullable): RankedHit.vector_score = sum of the clause similarities,
 * 0.0 where the candidate has no vector. */
int32_t slg_rerank_clauses(slg_index_t *, const slg_vector_clause_t *clauses, uint32_t n_clauses, uint32_t n_queries,
                           uint32_t dim, const slg_hit_t *cands, const uint32_t *cand_counts, uint32_t cand_stride,
                           slg_hit_t *out_hits, uint32_t *out_counts, float *out_vector_scores);
/* Pipeline form (no host round trip): rescore and re-sort the DEVICE-resident top-k of the batch's last slg_batch_run —
 * every segment's own list, as the reference hands the concatenated per-segment lists to merge_vector_hits
 * (api/reader.rs:2752-2773) — then merge the segments again by hybrid score.  Afterwards slg_batch_fetch,
 * slg_batch_device_results and slg_batch_packed_results (now hits, counts AND vector scores) describe the hybrid
 * ranking.  Asynchronous on the handle's stream unless sync != 0. */
int32_t slg_rerank_batch(slg_batch_t *, const slg_vector_clause_t *clauses, uint32_t n_clauses, uint32_t dim, int32_t sync);
/* n_queries x k vector scores of the hits slg_batch_fetch returns after slg_rerank_batch */
int32_t slg_batch_fetch_vector_scores(slg_batch_t *, float *out_vector_scores);
/* shard merge of reranked blocks (slg_batch_packed_results after slg_rerank_batch: hits, counts, vector scores);
 * out_vector_scores nullable */
int32_t slg_merge_gathered_hybrid(slg_index_t *, const void *dev_gathered, uint64_t shard_stride, uint32_t n_shards,
                                  uint32_t n_queries, uint32_t k, slg_hit_t *out_hits, uint32_t *out_counts,
                                  float *out_vector_scores);

/* ---- introspection ---- */
int32_t slg_get_counters(const slg_index_t *, slg_counters_t *out);
/* the cudaStream_t every call on this handle is ordered on (for callers that enqueue their own
 * work — an NCCL allgather, timing events — between calls) */
int32_t slg_get_stream(const slg_index_t *, void **cuda_stream);
/* device self-test: the scorer's division sequence against IEEE division on n pseudo-random
 * operand pairs from the scorer's range; *mismatches must come back 0 */
int32_t slg_selftest_div(slg_index_t *, uint64_t n, uint64_t seed, uint64_t *mismatches);
const char *slg_version(void);

#ifdef __cplusplus
}
#endif
#endif
