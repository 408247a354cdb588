/*
 * tantivy_b200.h — C ABI of the B200-native query-execution path for tantivy segments.
 *
 * The reference (quickwit-oss/tantivy, Rust) has no FFI; its boundary for this path is the
 * trait surface  Searcher::search -> Collector::collect_segment -> Weight::for_each_pruning
 * (src/core/searcher.rs:180-237, src/collector/mod.rs:173-184, src/query/weight.rs:123-132).
 * The entry points below are what a Rust shim implementing `Collector::collect_segment`
 * (or a `gpu_search(&Searcher, &dyn Query, k)` wrapper) would bind; INTEGRATION.md shows
 * that shim.  Every pointer is a plain host pointer unless its name ends in `_dev`.
 * No exceptions cross this boundary: every call returns TQ_OK or a negative error code and
 * `tq_last_error` gives the message.  All entry points are thread-safe per `tq_ctx`
 * (rayon threads call collect_segment concurrently, src/core/executor.rs:60-100).
 *
 * Doc ids are bit-exact w.r.t. the reference CPU path; scores are f32 computed with the
 * reference's operation order (src/query/bm25.rs:158-175).
 */
#ifndef TANTIVY_B200_H
#define TANTIVY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TQ_OK 0
#define TQ_ERR_INVALID_ARGUMENT (-1)
#define TQ_ERR_CUDA (-2)
#define TQ_ERR_NOT_FOUND (-3)
#define TQ_ERR_UNSUPPORTED (-4)
#define TQ_ERR_OOM (-5)
#define TQ_ERR_CORRUPT (-6)

/* schema::IndexRecordOption (src/schema/index_record_option.rs): decides the skip record
 * size 5 / 8 / 12 bytes (src/postings/skip.rs:205-253). */
#define TQ_RECORD_BASIC 0
#define TQ_RECORD_FREQS 1
#define TQ_RECORD_FREQS_POSITIONS 2

/* Query shapes accelerated: the three specialised scorers of the reference
 * (TermWeight::for_each_pruning, term_weight.rs:118; SpecializedScorer::TermIntersection /
 * TermUnion, boolean_weight.rs:17-21,581-600). */
#define TQ_OP_TERM 0
#define TQ_OP_AND 1
#define TQ_OP_OR 2
/* PhraseQuery (PhraseWeight / PhraseScorer, src/query/phrase_query/phrase_scorer.rs:349-589; slop > 0 for two-term phrases only,
 * intersection_count_with_slop :145-186 -- sloppy phrases of more terms return TQ_ERR_UNSUPPORTED): docs that hold
 * every term, at positions that line up with the terms' offsets in the phrase; score = bm25(fieldnorm, phrase_count)
 * under ONE Bm25Weight for the whole phrase (Bm25Weight::for_terms: the idfs add up, bm25.rs:95-129).  Needs a field
 * indexed WithFreqsAndPositions and its `.pos` bytes (tq_segment_register_positions). */
#define TQ_OP_PHRASE 3
/* BooleanQuery of TermQuery leaves with mixed Occurs, and one level of all-SHOULD sub-queries under MUST
 * (`+a +(b OR c)`, `+(c OR b) +(d OR e)`, `a b -c`, minimum_number_should_match): BooleanWeight::complex_scorer
 * (src/query/boolean_query/boolean_weight.rs:236-431) for these shapes.  Per clause term_occur[t] = TQ_OCCUR_*;
 * MUST clauses that share term_group[t] are alternatives of one required group (a MUST clause of its own: a group of
 * one).  A doc matches when every MUST group has a clause that lists it, at least `min_should_match` SHOULD clauses list
 * it (at least one when there is no MUST group: boolean_weight.rs:354-366), and no MUST_NOT clause lists it (Exclude).
 * Score = (sum over the MUST groups, ascending cost, of the sum of their matching clauses) + (sum of the matching SHOULD
 * clauses) -- Intersection::score / RequiredOptionalScorer::score (intersection.rs:325-329, reqopt_scorer.rs:78-94).
 * Runs on both engines with the same rows: the tile engine when the query fits a tile group, else (and with TQ_TILE=0, and
 * when an overflowing tile-engine run is repeated) the per-query kernel k_bool. */
#define TQ_OP_BOOL 4
#define TQ_OCCUR_SHOULD 0
#define TQ_OCCUR_MUST 1
#define TQ_OCCUR_MUST_NOT 2

/* TERMINATED sentinel of src/docset.rs:12 */
#define TQ_TERMINATED 0x7FFFFFFFu
/* Largest k the device path keeps on chip. */
#define TQ_MAX_K 1024u
/* Largest number of clauses in one query on the device path. */
#define TQ_MAX_TERMS 32u
/* Largest number of terms in a phrase on the device path. */
#define TQ_MAX_PHRASE_TERMS 8u

typedef struct tq_ctx tq_ctx;
typedef struct tq_batch tq_batch;

/* One (clause, segment) posting list: postings::TermInfo (src/postings/term_info.rs:9-16) as
 * returned by InvertedIndexReader::get_term_info (src/index/inverted_index_reader.rs:96).
 * postings_start/end are relative to the field's postings body, i.e. AFTER the 8-byte
 * total_num_tokens header (inverted_index_reader.rs:72-73).  A (clause, segment) pair in
 * which the term does not occur is simply not listed. */
typedef struct {
  uint32_t term_idx;    /* clause ordinal inside the query, 0..n_terms */
  uint32_t segment_ord; /* as given to tq_segment_register */
  uint32_t field;
  uint32_t doc_freq;
  uint64_t postings_start;
  uint64_t postings_end;
} tq_term_seg;

/* TermInfo::positions_range of one (clause, segment) (src/postings/term_info.rs:9-16): byte range of the term's position
 * stream inside the field's `.pos` sub-file (layout: src/positions/mod.rs:22-28).  Only read for TQ_OP_PHRASE. */
typedef struct {
  uint64_t positions_start;
  uint64_t positions_end;
} tq_term_pos;

/* One query = one `Weight` (built once for all segments, searcher.rs:226).
 * weight[i]        = Bm25Weight.weight = idf * (1 + K1) * boost        (bm25.rs:141-151)
 * avg_fieldnorm[i] = Bm25Weight.average_fieldnorm of clause i's field; the 256-entry tf
 *                    cache is recomputed from it exactly as bm25.rs:56-69 does.
 * tf_cache         = optional explicit caches [n_terms][256]; overrides avg_fieldnorm.
 * term_flags       = optional [n_terms] bytes (NULL = all 0).  TQ_TERM_IGNORE_FREQ: the clause is a
 *                    TermQuery::new(term, IndexRecordOption::Basic) on a field indexed WITH term
 *                    frequencies: the reference then skips the tf blocks and scores with tf = 1
 *                    (FreqReadingOption::SkipFreq, block_segment_postings.rs:97-140,343-360).
 * flags/threshold  = TQ_QUERY_HAS_THRESHOLD: only docs with score > threshold are collected -- the initial
 *                    `threshold` argument of Weight::for_each_pruning (src/query/weight.rs:123-132); a caller that
 *                    already holds k hits (another shard, an earlier page) passes its k-th score to prune more. */
#define TQ_TERM_IGNORE_FREQ 1u
#define TQ_QUERY_HAS_THRESHOLD 1u
typedef struct {
  int32_t op;
  uint32_t n_terms;
  uint32_t k; /* TopDocs limit+offset, 1..TQ_MAX_K */
  uint32_t n_term_segs;
  const tq_term_seg* term_segs;
  const float* weight;
  const float* avg_fieldnorm;
  const float* tf_cache;
  const uint8_t* term_flags;
  uint32_t flags;
  float threshold;
  /* TQ_OP_PHRASE only (NULL / 0 otherwise): term_pos[i] belongs to term_segs[i]; term_offset[t] = position of clause t
   * inside the phrase (PhraseQuery::new_with_offset, phrase_query.rs); weight[0] / avg_fieldnorm[0] (or the first
   * tf_cache table) describe the phrase's single Bm25Weight, the other entries are ignored; slop (PhraseQuery::set_slop) may be non-zero
   * for two-term phrases. */
  const tq_term_pos* term_pos;
  const uint32_t* term_offset;
  uint32_t slop;
  uint32_t min_should_match; /* TQ_OP_BOOL: BooleanQuery::minimum_number_should_match */
  /* TQ_OP_BOOL only (NULL otherwise): [n_terms] Occur of every clause; [n_terms] group of every MUST clause (NULL: every
   * MUST clause is a group of its own; ignored for the other Occurs). */
  const uint8_t* term_occur;
  const uint8_t* term_group;
} tq_query;

/* Counters of the last finished batch (per ctx). */
typedef struct {
  uint64_t lists_cached;      /* posting-list block tables resident on the device */
  uint64_t lists_built;       /* block tables built during the last batch */
  uint64_t units;             /* work units launched in the last batch */
  uint64_t kernel_launches;   /* CUDA kernels launched in the last batch */
  uint64_t h2d_bytes;         /* host->device bytes moved by the last batch */
  uint64_t d2h_bytes;         /* device->host bytes moved by the last batch */
  uint64_t algorithmic_bytes; /* SURVEY.md §8(d): sum over (query,segment,term) of postings
                                 range bytes + doc_freq fieldnorm bytes + 12*k output */
  uint64_t postings;          /* sum of doc_freq over all lists touched */
  float kernel_ms;            /* device time of all kernels of the batch (CUDA events on its stream) */
  float total_ms;             /* device time of the whole batch incl. copies */
  float term_ms, and_ms, or_ms, final_ms; /* per-kernel device time (CUDA events on the launching stream) */
  uint64_t units_term, units_and, units_or; /* CTAs launched per kernel */
  uint64_t bytes_term, bytes_and, bytes_or; /* algorithmic bytes per kernel (same formula) */
  /* cumulative since ctx creation, written by k_or_strip only: [1] windows scored exhaustively (no non-essential
   * clause under the threshold), [2] hot windows (non-essential clauses applied after the essential ones), [3] cold
   * windows (essential clauses only), [5] bytes of packed postings + fieldnorms actually read (SURVEY.md §8d: the
   * roofline figure of a pruned kernel).  [0], [4], [6] and [7] are always 0. */
  uint64_t or_windows[8];
  uint64_t units_or_strip; /* of units_or: CTAs of the barrier-free strip kernel (k_or_strip); the rest ran k_or */
  /* shared-decode tile engine (k_score_lists + k_tile, csrc/tq_tile.cuh) */
  float score_ms, tile_ms, theta_ms;  /* device time of k_score_lists / all k_tile launches / the k_theta passes of the batch */
  float phrase_ms;                    /* device time of k_phrase */
  uint64_t units_tile;          /* CTAs of k_tile over all its launches */
  uint64_t units_phrase;        /* CTAs of k_phrase */
  uint64_t tile_groups;         /* query groups evaluated together (one decode-and-score pass each) */
  uint64_t tile_postings;       /* postings decoded and scored by k_score_lists (every distinct list once) */
  uint64_t tile_list_bytes;     /* bytes of those lists' postings ranges (skip data + packed blocks + VInt tails) */
  uint64_t tile_scratch_bytes;  /* HBM scratch of the pair arrays, tile indexes and samples */
  uint64_t tile_fallbacks;      /* 1 if the run overflowed a tile engine buffer and was repeated on the per-query kernels */
  uint64_t tile_counters[8];    /* cumulative, with TQ_TILE_COUNTERS=1: (query, tile) pairs seen / skipped / light / heavy,
                                   essential postings applied, docs completed, docs at or above the threshold;
                                   [7] (always): dynamic shared memory bytes of a k_tile CTA of the last prepared group */
  uint64_t units_bool;          /* CTAs of k_bool (TQ_OP_BOOL queries on the per-query kernels) */
  float bool_ms;                /* device time of k_bool */
} tq_stats;

/* ---- context ------------------------------------------------------------------------- */
/* One context drives ONE device (one process per GPU; segments shard across processes). */
int tq_ctx_create(int device, tq_ctx** out);
void tq_ctx_destroy(tq_ctx*);
const char* tq_last_error(tq_ctx*);
int tq_get_stats(tq_ctx*, tq_stats* out);

/* Uploads one field of one segment to HBM (copied; caller keeps ownership of its mmap).
 * idx_body    = the field's sub-file of the `.idx` composite, INCLUDING the 8-byte
 *               total_num_tokens header (serializer.rs:128).
 * fieldnorm   = the field's sub-file of `.fieldnorm` (max_doc bytes); NULL => constant
 *               fieldnorm 1 (term_weight.rs:218).
 * alive_bitset= `.del` payload without its 4-byte max_value header: little-endian 64-bit
 *               words, bit set = alive (common/src/bitset.rs:362-407); NULL => no deletes. */
int tq_segment_register(tq_ctx*, uint32_t segment_ord, uint32_t field, uint32_t max_doc,
                        int record_option, const uint8_t* idx_body, size_t idx_len,
                        const uint8_t* fieldnorm, size_t fieldnorm_len,
                        const uint8_t* alive_bitset, size_t alive_len);
/* The `.pos` sub-file of a registered (segment, field) with record_option TQ_RECORD_FREQS_POSITIONS (copied to HBM):
 * what SegmentReader::inverted_index hands to PositionReader (src/positions/reader.rs:43-55).  Needed by TQ_OP_PHRASE. */
int tq_segment_register_positions(tq_ctx*, uint32_t segment_ord, uint32_t field, const uint8_t* pos_body, size_t pos_len);
int tq_segment_unregister(tq_ctx*, uint32_t segment_ord, uint32_t field);
/* Restricts what THIS context evaluates of a registered (segment, field) to the docs [doc_lo, doc_hi): the intra-segment split of
 * SURVEY.md §8(e) -- one huge segment registered on several contexts / GPUs, each with its own doc range (the posting lists are
 * block-addressable through the skip list, src/postings/skip.rs:205-302, so a doc range is a unit of work like a segment is in
 * Executor::map, src/core/executor.rs:60-100).  Statistics stay the segment's (the caller counts the segment once); the rows of
 * the ranges merge like the rows of segments (merge_fruits).  Call it before the first search on the segment; a range can only be
 * narrowed.  Docs outside the range behave like deleted docs (Count included); the tile engine skips their tiles altogether. */
int tq_segment_set_doc_range(tq_ctx*, uint32_t segment_ord, uint32_t field, uint32_t doc_lo, uint32_t doc_hi);

/* ---- search -------------------------------------------------------------------------- */
/* The whole hot path for a batch of queries, host buffers in / host buffers out:
 * block decode -> AND/OR/term -> BM25 -> per-segment top-k -> merge_fruits.
 * Replaces Searcher::search_with_executor's segment loop + merge (searcher.rs:220-237).
 * Output row q holds out_count[q] <= k hits sorted by (score desc, segment_ord asc, doc asc)
 * (top_score_collector.rs:591-600); rows are out_stride entries apart. */
int tq_search_batch(tq_ctx*, const tq_query* queries, size_t nq, uint32_t out_stride,
                    float* out_scores, uint32_t* out_segment_ord, uint32_t* out_doc,
                    uint32_t* out_count);

/* The Count collector for term / AND / OR / mixed boolean (TQ_OP_BOOL) queries (src/collector/count_collector.rs;
 * Weight::count, term_weight.rs:179-219): out_counts[q] = number of ALIVE docs matching query q over all its segments.
 * k and thresholds of the queries are ignored (TQ_OP_BOOL reads the weights: they order the clauses).  A term query on a
 * segment without deletes is answered from doc_freq, as the reference does. */
int tq_count_batch(tq_ctx*, const tq_query* queries, size_t nq, uint64_t* out_counts);

/* The same split in three so that callers can keep inputs/outputs device resident:
 * prepare = host planning + H2D of descriptors + block-table builds (cached per term),
 * run     = scoring kernels + final top-k, results stay in HBM,
 * fetch   = D2H of the result rows. */
int tq_batch_prepare(tq_ctx*, const tq_query* queries, size_t nq, tq_batch** out);
int tq_batch_run(tq_batch*);
/* The run in tq_batch_phases() consecutive phases, for callers that shard an index over several GPUs/processes:
 * phase 0 = everything up to the unions' first threshold round (each query then holds the exact k-th best score over
 * the windows scored so far), the middle phases = the further threshold rounds, the last phase = the rest.  Between
 * two phases tq_batch_thresholds_export_dev writes the nq score keys (order-preserving u32 image of the f32 score,
 * zero-extended to int64; 0 = no bound yet) to a DEVICE array; the caller takes the element-wise MAX over all shards
 * (e.g. ncclAllReduce) and hands it back with tq_batch_thresholds_import_dev.  Every shard then prunes against the best
 * bound any shard found: a valid lower bound of the global k-th score (SURVEY.md §8e "broadcast the running global
 * threshold").  tq_batch_run == all phases in order. */
int tq_batch_phases(tq_batch*);
int tq_batch_run_phase(tq_batch*, int phase);
int tq_batch_thresholds_export_dev(tq_batch*, int64_t* keys_dev);
int tq_batch_thresholds_import_dev(tq_batch*, const int64_t* keys_dev);
/* The exact form of that exchange (what one GPU holding all segments computes): between two phases every shard exports,
 * per query, the k best score keys it holds so far (u32 order-preserving images of f32 scores, k_stride entries per
 * query, zero padded) -- enqueued on the batch's stream, no host synchronisation; the caller all-gathers the arrays of
 * all shards ON THAT STREAM (tq_batch_stream; e.g. ncclAllGather, or torch.cuda.ExternalStream) into
 * [n_shards][nq][k_stride] and hands them back: the k-th best key of the union becomes every shard's threshold
 * (merge_top_k's bound, sort_key_top_collector.rs:76-95, available before the scoring is over). */
int tq_batch_stream(tq_batch*, void** cuda_stream_out);
int tq_batch_topkeys_export_dev(tq_batch*, uint32_t* keys_dev, uint32_t k_stride);
int tq_batch_thresholds_from_keys_dev(tq_batch*, const uint32_t* gathered_keys_dev, uint32_t n_shards, uint32_t k_stride);
int tq_batch_fetch(tq_batch*, uint32_t out_stride, float* out_scores, uint32_t* out_segment_ord,
                   uint32_t* out_doc, uint32_t* out_count);
/* Device pointers of the result rows of a finished run: row stride = k_max of the batch. */
int tq_batch_results_dev(tq_batch*, const float** scores_dev, const uint32_t** segment_ord_dev,
                         const uint32_t** doc_dev, const uint32_t** count_dev, uint32_t* stride);
/* Copies the result rows of a finished run into caller-owned DEVICE buffers (row stride = k_max of
 * the batch), e.g. torch tensors about to be all-gathered over NCCL. */
int tq_batch_results_copy_dev(tq_batch*, float* scores_dev, uint32_t* segment_ord_dev, uint32_t* doc_dev,
                              uint32_t* count_dev);
void tq_batch_destroy(tq_batch*);

/* Cross-GPU merge_fruits (sort_key_top_collector.rs:76-95): merges `n_lists` result sets
 * (e.g. the ranks' rows after an NCCL all-gather), all device resident, laid out
 * [list][query][stride], into [query][stride] device rows; same ordering as above. */
int tq_merge_topk_dev(tq_ctx*, uint32_t n_lists, uint32_t nq, uint32_t stride, uint32_t k,
                      const float* scores_dev, const uint32_t* segment_ord_dev,
                      const uint32_t* doc_dev, const uint32_t* count_dev, float* out_scores_dev,
                      uint32_t* out_segment_ord_dev, uint32_t* out_doc_dev,
                      uint32_t* out_count_dev);

/* The same for sharded callers that move ONE buffer per shard: packed = [nq*stride scores | nq*stride segment ords |
 * nq*stride docs | nq counts] as 32-bit words (tq_batch_results_pack_dev writes it with stride = k_max of the batch),
 * n_lists of them pitch_words apart -- what one all-gather of the shards' buffers produces.  The merge is enqueued on
 * cuda_stream (a cudaStream_t, e.g. tq_batch_stream's) and does not synchronise with the host. */
int tq_batch_results_pack_dev(tq_batch*, uint32_t* packed_dev);
/* tq_batch_results_pack_dev without the wait: the copies are enqueued behind the run on the batch's stream, so that pack, all-gather,
 * merge and the NEXT batch's run can all be queued before the host waits for this batch (two batches in flight per GPU).
 * packed_dev holds 3 * nq * k_max + nq + 4 words; the last four are the run's overflow flags -- non-zero on any shard: take
 * tq_batch_results_pack_dev instead (it repeats an overflowed run on the per-query kernels). */
int tq_batch_results_pack_dev_async(tq_batch*, uint32_t* packed_dev);
int tq_merge_topk_packed_dev(tq_ctx*, void* cuda_stream, uint32_t n_lists, uint32_t nq, uint32_t stride, uint32_t k,
                             const uint32_t* packed_dev, size_t pitch_words, uint32_t* out_packed_dev);

/* ---- several GPUs behind one handle --------------------------------------------------- */
/* The reference fans a search out over segments inside ONE process (Executor::map, src/core/executor.rs:60-100;
 * Searcher::search_with_executor, src/core/searcher.rs:220-237).  tq_multi is that shape for GPUs: one tq_ctx per
 * device, every (segment, field) lives on one of them (device_index -1 = the least loaded), tq_multi_search_batch runs
 * the devices' shares concurrently (one host thread per device), exchanges the exact k-th best score keys between the
 * phases -- every device prunes like a single device holding all segments -- and merges the rows on the host
 * (merge_fruits, sort_key_top_collector.rs:54-95).  Same arguments and result layout as tq_search_batch. */
typedef struct tq_multi tq_multi;
int tq_multi_create(const int* devices, int n_devices, tq_multi** out);
void tq_multi_destroy(tq_multi*);
const char* tq_multi_last_error(tq_multi*);
int tq_multi_num_devices(tq_multi*);
int tq_multi_segment_register(tq_multi*, int device_index, uint32_t segment_ord, uint32_t field, uint32_t max_doc,
                              int record_option, const uint8_t* idx_body, size_t idx_len,
                              const uint8_t* fieldnorm, size_t fieldnorm_len,
                              const uint8_t* alive_bitset, size_t alive_len);
/* One (huge) segment over ALL devices of the handle: every device holds the segment's bytes and evaluates its own doc range
 * (tq_segment_set_doc_range; ranges are whole 1024-doc tiles, ceil(max_doc / n_devices) docs each). */
int tq_multi_segment_register_split(tq_multi*, uint32_t segment_ord, uint32_t field, uint32_t max_doc,
                                    int record_option, const uint8_t* idx_body, size_t idx_len,
                                    const uint8_t* fieldnorm, size_t fieldnorm_len,
                                    const uint8_t* alive_bitset, size_t alive_len);
int tq_multi_search_batch(tq_multi*, const tq_query* queries, size_t nq, uint32_t out_stride,
                          float* out_scores, uint32_t* out_segment_ord, uint32_t* out_doc,
                          uint32_t* out_count);

/* ---- codec-level access (parity tests and the decode micro-benchmark) ----------------- */
/* Decodes one whole posting list on the device (BlockSegmentPostings::open + advance loop,
 * block_segment_postings.rs:97-140,343-399) into host arrays of doc_freq entries.
 * out_tfs may be NULL. */
int tq_decode_postings(tq_ctx*, const tq_term_seg* list, uint32_t* out_docs, uint32_t* out_tfs);
/* Block-max scores of every full block (SkipReader::block_max_score, skip.rs:175-184) and
 * last_doc_in_block, as the device block table holds them. n = doc_freq / 128 entries. */
int tq_block_table(tq_ctx*, const tq_term_seg* list, float weight, float avg_fieldnorm,
                   uint32_t* out_last_doc, float* out_block_max);

/* ---- BM25 scalars (host; bit-identical to src/query/bm25.rs) -------------------------- */
float tq_bm25_idf(uint64_t doc_freq, uint64_t doc_count);                  /* bm25.rs:52-56 */
float tq_bm25_weight(uint64_t doc_freq, uint64_t doc_count, float boost);  /* bm25.rs:141-151,80-92 */
void tq_bm25_tf_cache(float avg_fieldnorm, float out[256]);               /* bm25.rs:58-69 */
uint32_t tq_id_to_fieldnorm(uint8_t id);                                   /* fieldnorm/code.rs:2-4 */
uint8_t tq_fieldnorm_to_id(uint32_t fieldnorm);                            /* fieldnorm/code.rs:7-11 */

/* ---- segment writer (host; produces tantivy-format bytes for tests and benchmarks) ----- */
/* Restates PostingsSerializer (src/postings/serializer.rs:353-481): appends one term's
 * posting list (docs ascending, tfs >= 1 or NULL) to `body`, returns TermInfo. */
typedef struct tq_field_writer tq_field_writer;
int tq_field_writer_create(int record_option, uint64_t total_num_tokens,
                           const uint8_t* fieldnorm_ids, uint32_t max_doc, tq_field_writer** out);
int tq_field_writer_add_term(tq_field_writer*, const uint32_t* docs, const uint32_t* tfs,
                             uint32_t doc_freq, uint64_t* postings_start, uint64_t* postings_end);
/* Field body = 8-byte LE total_num_tokens followed by every term's postings. */
int tq_field_writer_body(tq_field_writer*, const uint8_t** body, size_t* len);
void tq_field_writer_destroy(tq_field_writer*);

#ifdef __cplusplus
}
#endif
#endif /* TANTIVY_B200_H */
