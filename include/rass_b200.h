/*
 * rass_b200.h -- C ABI of the B200-native retrieval engine that stands in for the
 * OpenSearch server behind RASSEngine's OpenSearchIndexer.
 *
 * Every entry point replaces work the reference sends over HTTP to OpenSearch 2.11.1
 * (file:line are relative to the reference repo, NeuralRevenant/RASSEngine):
 *
 *   rass_create / rass_destroy      client.indices.create(index, body)          app/main.py:576 (vector field :563-572)
 *   rass_append / rass_overwrite    helpers.bulk(client, actions) "_op_type":"index" (insert-or-overwrite by _id)
 *                                                                               app/main.py:1237,1269,1279 (actions :1258-1264)
 *   rass_tombstone                  overwrite of an _id whose new doc has no embedding (same bulk call)
 *   rass_count                      client.count(index)                         app/main.py:1475-1476
 *   rass_search_knn                 client.search(body={"query":{"knn":{"embedding":{"vector","k"}}}})
 *                                                                               app/main.py:1538-1553
 *   rass_bm25_build                 Lucene inverted index built by the same bulk calls (text field `unstructuredText`,
 *                                   mapping app/main.py:555-556)
 *   rass_search_hybrid              client.search(body={"query":{"bool":{"should":[multi_match, multi_match, knn]}}})
 *                                                                               app/main.py:1574-1609
 *   rass_search_hybrid_weighted,    the same query with "fuzziness": "AUTO" on the text clause (FuzzyQuery rewrite)
 *   rass_text_set_vocab,                                                        app/main.py:1577-1585
 *   rass_fuzzy_expand
 *   rass_set_row_filter             bool.filter [term patientId / doc_type] of the hybrid query               app/main.py:1599-1604
 *   rass_create_sharded             settings.index.number_of_shards of the same create call            app/main.py:357
 *   rass_merge_topk_dev             the OpenSearch coordinator's per-shard top-k merge (number_of_shards, app/main.py:357)
 *   rass_save / rass_load           the on-disk Lucene index of the OpenSearch container (docker-compose.yml:4-17)
 *
 * Conventions: C linkage, plain pointers and sizes, no exceptions cross the boundary.  Every function returns an
 * int status (0 = ok, negative = RASS_E_*); rass_last_error(h) gives the message for the last failure on that
 * handle.  The caller owns every input and output buffer; inputs may be freed on return.  One call at a time per
 * handle.  The engine owns device memory, pinned staging and streams.  Row ids are engine-assigned, dense and
 * append-ordered, so "row ascending" is the tie-break Lucene's doc-id order gives.
 *
 * There is no CPU fallback: every compute entry point fails with RASS_E_CUDA when no sm_100 device is present.
 */
#ifndef RASS_B200_H
#define RASS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RASS_ABI_VERSION 1

typedef struct rass_engine rass_engine;

enum {
  RASS_OK = 0,
  RASS_E_INVALID = -1,
  RASS_E_OOM = -2,
  RASS_E_CUDA = -3,
  RASS_E_NCCL = -4,      /* the inter-GPU exchange of a sharded handle failed (peer mapping / peer copy) */
  RASS_E_NOTFOUND = -5,
  RASS_E_UNSUPPORTED = -6,
  RASS_E_AGAIN = -7      /* rass_search_knn_dev_wait: some query failed its certificate; repeat with the blocking call */
};

enum { RASS_METRIC_COSINE = 0, RASS_METRIC_L2 = 1 };

/* rass_create flags */
enum {
  RASS_KEEP_FP32 = 1u,  /* resident fp32 matrix + bf16 shadow (default when flags == 0)               */
  RASS_BF16_ONLY = 2u,  /* bf16 corpus: the bf16 values ARE the data (BASELINE config 5, 100M rows)  */
  RASS_NO_INT8_SHADOW = 4u  /* fp32 store without the int8 shadow (saves dim_pad + 4 bytes per row); the 2..64-query
                            passes then stream the bf16 shadow.  Alone it still means RASS_KEEP_FP32 */
};

/* rass_search_* path selection (rass_set_option RASS_OPT_PATH) */
enum {
  RASS_PATH_AUTO = 0,    /* B = 1: streaming GEMV+select; B <= 64: tcgen05 tiles, 64 queries per pass, over the
                            int8 shadow when the store has one and its quantisation residual is small (else
                            the bf16 shadow); larger: CTA-pair tcgen05 contraction, 128 (B <= 128) or 256
                            queries per pass  */
  RASS_PATH_STREAM = 1,  /* force the CUDA-core streaming scan (passes of <= 2 queries)                */
  RASS_PATH_UMMA = 2,    /* force the TMA + tcgen05 scan (passes of <= 64 queries)                     */
  RASS_PATH_EXACT = 3,   /* force the fp64 full scan (the certificate-failure fallback), for tests     */
  RASS_PATH_GEMM = 4,    /* force the CTA-pair (cta_group::2) tcgen05 scan (groups of 256 queries)     */
  RASS_PATH_UMMA8 = 5    /* force the TMA + tcgen05 kind::i8 scan over the int8 shadow (passes of <= 64 queries);
                            queries it cannot certify get the bf16 pass, then the fp64 scan.  RASS_E_UNSUPPORTED on
                            a store without the int8 shadow */
};

/* rass_stats.path of a hybrid call: the kNN path in the low byte, plus this bit when the text clauses ran through the
 * order-free tile kernel (every query's clause sums provably exact in double, so the order of the additions is free) */
enum { RASS_PATH_HYBRID_ORDER_FREE = 0x100 };

enum {
  RASS_OPT_PATH = 1,
  RASS_OPT_STREAM = 2,   /* value = cudaStream_t to enqueue on (0 = the legacy default stream, which is what
                            torch's default stream is); -1 = back to the engine-owned stream           */
  RASS_OPT_HYBRID_ORDERED = 4,  /* 1: the text clauses of hybrid calls always walk the query terms in order (one barrier
                            per term); 0 (default): queries whose clause sums are exact in double in ANY order take the
                            order-free kernel.  Both give bit-identical scores; the switch exists for tests and A/B runs */
  RASS_OPT_HYBRID_MAXSCORE = 5, /* 1: the order-free text kernel splits a query's terms the way Lucene's MaxScore scorer
                            does once a pruning bound exists: terms whose summed score bounds stay below the bound are only
                            scored for docs an essential term (or the knn clause) already touched.  Results are identical
                            (tests/test_gpu_hybrid.py); off by default because it measures slower at the current tile size */
  RASS_OPT_ASYNC_OVERLAP = 6,   /* 1: each slot of rass_search_knn_dev_async runs on an engine-owned stream of its own,
                            forked from the engine stream when the search is enqueued, and slot 1 has a second search
                            workspace: the fixed costs of batch i (query preparation, threshold seed, merge + rerank) run
                            under the corpus pass of batch i+1.  Results are ordered by rass_search_knn_dev_wait (host) or
                            rass_async_join (a stream), no longer by the engine stream.  0 (default): both slots are
                            enqueued on the engine stream, back to back */
  RASS_OPT_SCAN_RESERVE_SMS = 7, /* value = SMs the 64-query corpus pass leaves free (default 0).  A row-sharded index
                            sets a few so the exchange of batch i (NCCL all-gather + merge, which cannot share an SM with a
                            scan CTA) runs during the pass of batch i+1 instead of after it */
  RASS_OPT_KNN_PREFILTER = 3  /* 1: rass_search_knn honours rass_set_row_filter as an exact PRE-filter (top-k of
                            the rows that pass); 0 (default): the filter only applies to rass_search_hybrid and
                            the host post-filters the k nearest, which is what OpenSearch's nmslib engine does
                            with bool.must[knn] + filter (app/main.py:1543-1550)                          */
};

typedef struct rass_stats {
  double scan_ms;        /* device time of the scan kernels of the last search (CUDA events)           */
  double finish_ms;      /* device time of merge + exact rerank (+ fallback)                           */
  double total_ms;       /* device time first kernel -> last kernel                                    */
  int64_t rows_scanned;  /* live + tombstoned rows each pass streams                                   */
  int64_t bytes_streamed;/* algorithmic bytes of the scan passes (rows * dim_pad * sizeof(elem) * passes) */
  int32_t n_queries;
  int32_t n_certified;   /* queries whose scan candidate set was proven to contain the exact top-k     */
  int32_t n_fallback;    /* queries re-scanned exactly in fp64                                         */
  int32_t path;          /* RASS_PATH_* actually used                                                  */
  int32_t passes;        /* corpus passes of the scan                                                  */
  int32_t launches;      /* kernels launched by this call                                              */
  int32_t max_candidates;/* largest rerank candidate set                                               */
  int32_t n_retried;     /* queries (k > 32) that failed the first certificate and were re-scanned with wider
                            candidate segments before any fp64 fallback                                */
} rass_stats;

const char* rass_version(void);
const char* rass_last_error(const rass_engine* h);  /* h may be NULL: last create failure */

/* dim: embedding dimension (<= 1024; padded to a multiple of 256 on device).  device: CUDA ordinal.
 * capacity_rows: initial reservation (grows by doubling). */
int rass_create(int dim, int metric, int device, int64_t capacity_rows, uint32_t flags, rass_engine** out);
/* One handle over several GPUs of the box, in the caller's process -- the B200 form of `number_of_shards`
 * (settings.index.number_of_shards, app/main.py:357) with the coordinator's merge (SURVEY.md 8b, 8e).  Global row r lives
 * on device_ids[(r >> 10) % n_devices]; EVERY entry point of this header takes the returned handle (debug entries and
 * rass_fuse_hybrid_dev excepted), row ids stay global, dense and append-ordered, and results are bit-identical to a
 * single-device handle holding the same rows.  device_ids[0] is the coordinator: the *_dev entry points take and leave
 * their buffers there.  Each shard's finish kernel stores its [B, k] list straight into the coordinator's gather buffer
 * through peer-mapped memory (NVLink), then one merge kernel runs -- no all-gather.  RASS_E_NCCL = the inter-GPU exchange
 * failed (peer copy / peer mapping).  n_devices == 1 is rass_create. */
int rass_create_sharded(int dim, int metric, int n_devices, const int* device_ids, int64_t capacity_rows,
                        uint32_t flags, rass_engine** out);
int rass_destroy(rass_engine* h);
int rass_set_option(rass_engine* h, int opt, int64_t value);
/* global row id of local row 0 (row-sharded corpora); search outputs carry base + local row */
int rass_set_row_base(rass_engine* h, int64_t base);

/* rows: [n, dim] row-major fp32, host (pageable or pinned).  *out_first_row = local row of rows[0]. */
int rass_append(rass_engine* h, const float* rows_host, int64_t n, int64_t* out_first_row);
/* same, source already in device memory of this engine's device */
int rass_append_dev(rass_engine* h, const float* rows_dev, int64_t n, int64_t* out_first_row);
int rass_overwrite(rass_engine* h, int64_t row, const float* v_host);
int rass_tombstone(rass_engine* h, int64_t row);
int rass_count(const rass_engine* h, int64_t* out_live_rows);
int rass_rows(const rass_engine* h, int64_t* out_total_rows);
/* How the store is held: *capacity_rows = rows the mapped memory holds; *grows_in_place = 1 when the arrays live in
 * reserved virtual address ranges and grow by mapping more physical chunks (no copy, no second resident array:
 * csrc/vmm.cu), 0 when they are cudaMalloc'ed and grow by copy (a driver without the virtual-memory API). */
int rass_store_info(const rass_engine* h, int64_t* capacity_rows, int* grows_in_place);
/* stored values (fp32, or the bf16 values widened when RASS_BF16_ONLY) back to the host: [n, dim] */
int rass_read_rows(rass_engine* h, int64_t first_row, int64_t n, float* out_host);
/* same for a list of rows (the `_source.embedding` of the hits of one search): one gather, one copy */
int rass_read_rows_list(rass_engine* h, const int64_t* rows_host, int64_t n, float* out_host);

/* Exact top-k.  q: [B, dim] fp32 (need not be normalised).  out_rows: [B, k] (base + local row, -1 = no hit),
 * out_scores: [B, k] fp32 = 1/(2 - cos) (cosine) or 1/(1 + d^2) (L2).  out_keys (nullable): [B, k] fp64 cos / d^2.
 * Ranking is (fp64-accumulated key, row ascending).  stats nullable. */
int rass_search_knn(rass_engine* h, const float* q_host, int B, int k,
                    int64_t* out_rows, float* out_scores, double* out_keys, rass_stats* stats);
/* device-pointer flavour: q_dev and outputs in device memory; enqueued on the engine stream and synchronised */
int rass_search_knn_dev(rass_engine* h, const float* q_dev, int B, int k,
                        int64_t* out_rows_dev, float* out_scores_dev, double* out_keys_dev, rass_stats* stats);

/* Pipelined flavour for callers that keep two batches in flight (row-sharded serving: the all-gather and merge of
 * batch i overlap the scan of batch i+1).  _async enqueues the whole search on the engine stream and returns without
 * touching the host; slot is 0 or 1; flag_out_dev (nullable) receives the number of queries whose certificate failed,
 * on the device, so it can travel with the gathered candidates.  _wait blocks until that slot's search is complete:
 * RASS_OK = outputs final; RASS_E_AGAIN = repeat this batch with rass_search_knn_dev (which re-scans those queries). */
int rass_search_knn_dev_async(rass_engine* h, const float* q_dev, int B, int k, int64_t* out_rows_dev,
                              float* out_scores_dev, double* out_keys_dev, int slot, int64_t* flag_out_dev);
int rass_search_knn_dev_wait(rass_engine* h, int slot, rass_stats* stats);
/* Makes `stream` (a cudaStream_t; 0 = the legacy default stream) wait for the search enqueued in `slot`: what a caller
 * needs before it reads the outputs on a stream of its own (the all-gather of a row-sharded index) when
 * RASS_OPT_ASYNC_OVERLAP is on.  No host synchronisation. */
int rass_async_join(rass_engine* h, int slot, void* stream);

/* Merge G per-shard top-k lists (what each rank all-gathers) into the global top-k, (key desc, row asc).
 * keys_dev / rows_dev point at shard 0's [B, k] fp64 keys / int64 rows (-1 = empty); shard g's lists start
 * shard_stride elements further (0 = B * k, i.e. dense [G, B, k]; 2 * B * k when each rank gathers one packed
 * [2, B, k] buffer).  Outputs [B, k], device memory.  Enqueued on the engine stream, not synchronised. */
int rass_merge_topk_dev(rass_engine* h, const double* keys_dev, const int64_t* rows_dev, int64_t shard_stride,
                        int G, int B, int k, int64_t* out_rows_dev, float* out_scores_dev, double* out_keys_dev);

/* The same merge for the per-shard FUSED lists of a row-sharded hybrid query (rass_fuse_hybrid_dev's out_keys_dev /
 * out_rows_dev): the keys are bool.should scores, larger is better whatever the engine's vector metric is, and the
 * merged score is the key itself (app/main.py:1574-1598 executed per shard, merged by the coordinator). */
int rass_merge_scores_dev(rass_engine* h, const double* scores_dev, const int64_t* rows_dev, int64_t shard_stride,
                          int G, int B, int k, int64_t* out_rows_dev, float* out_scores_dev, double* out_keys_dev);

/* CSR postings of the text field: indptr[V+1], doc[nnz] (local rows, ascending per term), tf[nnz], doclen[N]
 * (token count per row).  Statistics (docCount, sumTotalTermFreq, df) are taken from these arrays unless the
 * global_* overrides are given (row-sharded corpora share global statistics so scores are shard-invariant). */
int rass_bm25_build(rass_engine* h, const int64_t* indptr, const int32_t* doc, const uint16_t* tf,
                    const uint32_t* doclen, int64_t V, int64_t N,
                    int64_t global_doc_count, int64_t global_sum_ttf, const int64_t* global_df);

/* Several analysed fields in one CSR (structured FHIR documents share the index with the chunks, app/main.py:1223-1240):
 * term t belongs to field term_field[t] (0 <= field < F <= 255); doclen is [F][N], the token count of the field in the
 * row (0 = the row lacks the field).  docCount, avgdl and idf are per field, as Lucene keeps them. */
int rass_bm25_build_fields(rass_engine* h, const int64_t* indptr, const int32_t* doc, const uint16_t* tf,
                           const int32_t* term_field, const uint32_t* doclen, int64_t V, int64_t N, int F);

/* ---- text ingest on the device (what a bulk request does to the `text` / `keyword` fields, app/main.py:1258-1269) ----
 * rass_text_add_rows hands over the analysed tokens of n_rows rows of one field: rows[n_rows] ascending, distinct row
 * ids; tok_indptr[n_rows + 1] (starting at 0) into tok_terms, the rows' token sequences as term ids LOCAL to the field
 * (repeats included; only the counts matter to BM25).  The bulk becomes a segment on the device (stable radix sort by
 * term, repeats folded into term frequencies); nothing is searchable until rass_text_commit -- OpenSearch's refresh.
 * A row the field already holds is REWRITTEN (an index request with a known _id): what it held is dropped at the
 * commit, like Lucene's delete-then-add; a row with no tokens loses the field.  The _dev flavour takes device pointers
 * (single-device handles; a handle over several GPUs takes the host flavour and splits the stream by its row map). */
int rass_text_add_rows(rass_engine* h, int field, const int64_t* rows, int64_t n_rows, const int64_t* tok_indptr,
                       const int32_t* tok_terms);
int rass_text_add_rows_dev(rass_engine* h, int field, const int64_t* rows_dev, int64_t n_rows,
                           const int64_t* tok_indptr_dev, const int32_t* tok_terms_dev);
/* Folds the pending segments into the CSR the hybrid kernels walk and recomputes lengths, norm bytes, statistics, idf
 * and the kernels' side tables on the device.  field_vocab[F] = terms of each field NOW (vocabularies only grow); the
 * global id of (field f, local term t) is sum(field_vocab[:f]) + t, the layout rass_bm25_build_fields is given by the
 * client.  N = rows of the index.  When the segments only add rows above the ones indexed, a term's merged list is its
 * old list followed by each segment's: one copy pass over the postings.  When some row was rewritten, the live postings
 * of every source (a per-(field, row) generation word says which source owns the row) are re-sorted by (term, doc). */
int rass_text_commit(rass_engine* h, const int64_t* field_vocab, int F, int64_t N);
/* omit = 1: the field omits norms, like a `keyword` field of the mapping -- every document that has a value counts as
 * length 1 however many values (tokens) it sent; takes effect at the next commit.  The host-array path expresses the
 * same by passing lengths of 0 / 1 to rass_bm25_build_fields. */
int rass_text_omit_norms(rass_engine* h, int field, int omit);
/* Sizes of the committed index, and its arrays read back (tests, host-side evaluation); every pointer nullable:
 * indptr [V + 1], doc / tf [nnz], doclen [F][N], norm [F][N] (Lucene's SmallFloat.intToByte4 of doclen). */
int rass_text_size(rass_engine* h, int64_t* V, int64_t* N, int64_t* nnz, int* F);
int rass_text_export(rass_engine* h, int64_t* indptr, int32_t* doc, uint16_t* tf, uint32_t* doclen, uint8_t* norm);
/* The V- and F-sized statistics a host needs to rewrite a query string into weighted term queries (df = diff of
 * indptr; docCount and sumTotalTermFreq per field); every pointer nullable. */
int rass_text_stats(rass_engine* h, int64_t* indptr, int64_t* doc_count, int64_t* sum_ttf);

/* bool.should boosted sum: S(d) = w_text * BM25(q, d) + w_knn * [d in kNN_k(q)] * knn_score(q, d), top-k by
 * (S desc, row asc) over rows matching at least one clause.  qterm_indptr[B+1] / qterms: term ids per query
 * (duplicates count twice; ids outside [0, V) are ignored).  q_host may be NULL (text-only) and qterm_indptr may
 * be NULL (vector-only). */
int rass_search_hybrid(rass_engine* h, const float* q_host, int B, const int32_t* qterm_indptr,
                       const int32_t* qterms, float w_text, float w_knn, int k,
                       int64_t* out_rows, float* out_scores, rass_stats* stats);

/* Same with caller-supplied per-term weights qweights[nnz of qterms] = float(clause boost * field boost * term boost)
 * * idf instead of w_text * idf(term): the boosted TermQuerys a `fuzziness: AUTO` token rewrites to
 * (app/main.py:1577-1585) carry a similarity boost and blended statistics, which the host computes from
 * rass_fuzzy_expand.
 *
 * qflags (nullable) marks structure for multi-field / multi-clause queries (the reference's two multi_match clauses
 * over 26 text and 24 keyword fields, app/main.py:1403-1456, 1576-1594): bit 0 = last term of its field group,
 * bit 1 = last term of its clause.  A clause scores max over its field groups of the group's term sum (best_fields,
 * tie_breaker 0; every group score is a float), the text part of S(d) is the sum over clauses (in double). */
int rass_search_hybrid_weighted(rass_engine* h, const float* q_host, int B, const int32_t* qterm_indptr,
                                const int32_t* qterms, const float* qweights, const uint8_t* qflags, float w_knn,
                                int k, int64_t* out_rows, float* out_scores, rass_stats* stats);

/* Row-sharded hybrid (SURVEY.md 8e: postings sharded by the same row ranges, statistics global): the text clauses of
 * rass_search_hybrid(_weighted) fused with an EXTERNAL knn list -- the global k nearest the caller all-gathered and
 * merged (global rows; rows of other shards are ignored) -- leaving this shard's top-k on the device: out_rows_dev
 * (global rows), out_scores_dev (fused float scores) and, for rass_merge_topk_dev, out_keys_dev (the scores as
 * double).  qweights / qflags / knn_rows_dev may be NULL.  Synchronises the engine stream. */
int rass_fuse_hybrid_dev(rass_engine* h, int B, const int32_t* qterm_indptr, const int32_t* qterms,
                         const float* qweights, const uint8_t* qflags, float w_text, const int64_t* knn_rows_dev,
                         const float* knn_scores_dev, float w_knn, int k, int64_t* out_rows_dev,
                         float* out_scores_dev, double* out_keys_dev);

/* Host-pointer flavour: the k nearest come from an earlier rass_search_knn -- e.g. one corpus pass shared by several
 * concurrent requests -- while text clauses and bool.filter are this request's own.  knn_rows_host (rows as
 * rass_search_knn returned them, -1 = none) may be NULL for a text-only query. */
int rass_fuse_hybrid(rass_engine* h, int B, const int32_t* qterm_indptr, const int32_t* qterms,
                     const float* qweights, const uint8_t* qflags, float w_text, const int64_t* knn_rows_host,
                     const float* knn_scores_host, float w_knn, int k, int64_t* out_rows, float* out_scores);

/* The term dictionary of the text field, terms back to back in blob, term t = blob[offsets[t] .. offsets[t+1]),
 * UTF-8 (offsets in bytes).  The engine keeps it as code points: Lucene's FuzzyQuery counts edits in code points.
 * Needed only for rass_fuzzy_expand. */
int rass_text_set_vocab(rass_engine* h, const char* blob, const int64_t* offsets, int64_t V);
/* Lucene FuzzyQuery term enumeration on the device: every dictionary term within max_edits (0..2) of the token (UTF-8,
 * token_len bytes, at most 64 code points) under
 * the optimal-string-alignment distance (an adjacent swap is one edit), among the terms [term_lo, term_hi) (one
 * field's slice of the dictionary; term_hi < 0 = to the end).  *out_n = number of matches; the first
 * min(*out_n, max_out) (term id, edits) pairs are written, in no particular order. */
int rass_fuzzy_expand(rass_engine* h, const char* token, int token_len, int max_edits, int64_t term_lo,
                      int64_t term_hi, int64_t max_out, int32_t* out_terms, int32_t* out_edits, int64_t* out_n);

/* bool.filter of the following rass_search_hybrid calls (app/main.py:1599-1604) as a per-row pass mask:
 * mask_host[n] bytes, 1 = the row satisfies the filter; rows >= n fail.  NULL clears the filter. */
int rass_set_row_filter(rass_engine* h, const uint8_t* mask_host, int64_t n);
/* The same filter given as the list of rows that pass (a term filter on patientId selects a few hundred rows of
 * millions): the mask over [0, total_rows) is built on the device, the host moves n * 8 bytes. */
int rass_set_row_filter_rows(rass_engine* h, const int64_t* rows_host, int64_t n, int64_t total_rows);

/* Per-query filters in ONE call (every production query carries its own `term patientId` filter, app/main.py:1543-1550,
 * 1599-1604, :2884; a window of coalesced requests holds as many filters as requests).  Query b brings the rows that pass
 * ITS bool.filter: frows[frow_indptr[b] .. frow_indptr[b+1]) (engine rows, any order, no duplicates).  The listed rows are
 * scored directly -- no corpus pass for them, no pass mask.
 *   rass_search_knn_filtered     exact top-k among each query's listed rows (the pre-filter semantics of
 *                                RASS_OPT_KNN_PREFILTER: same keys, ranking and scores)
 *   rass_search_hybrid_filtered  bool.should of the text clauses + knn over each query's listed rows, as rass_search_hybrid
 *                                (_weighted when qweights != NULL; qflags as there) computes it under that filter.  knn_mode
 *                                0: the knn clause is the k nearest of the WHOLE corpus -- one scan pass shared by the batch,
 *                                OpenSearch/nmslib's post-filter behaviour and this engine's default; 1: the k nearest among
 *                                the listed rows.
 * Single-device handles only. */
int rass_search_knn_filtered(rass_engine* h, const float* q_host, int B, int k, const int64_t* frow_indptr,
                             const int64_t* frows, int64_t* out_rows, float* out_scores, double* out_keys);
int rass_search_hybrid_filtered(rass_engine* h, const float* q_host, int B, const int32_t* qterm_indptr,
                                const int32_t* qterms, const float* qweights, const uint8_t* qflags, float w_text,
                                float w_knn, int k, const int64_t* frow_indptr, const int64_t* frows, int knn_mode,
                                int64_t* out_rows, float* out_scores, rass_stats* stats);

int rass_sync(rass_engine* h);
/* statistics of the last blocking search / hybrid / fuse call on the handle (the entry points without a stats argument,
 * rass_fuse_hybrid(_dev), leave theirs here: scan_ms = the kNN scan, finish_ms = text clauses + fusion + select) */
int rass_last_stats(const rass_engine* h, rass_stats* out);

/* Snapshot / restore of the vector store (the reference relies on the OpenSearch container's own Lucene index
 * directory, docker-compose.yml:4-17).  rass_save writes header + tombstones + the stored values; rass_load fills an
 * EMPTY engine of the same dim/metric/corpus type through the normal append path.  Postings are rebuilt by the
 * caller (rass_bm25_build). */
int rass_save(rass_engine* h, const char* path);
int rass_load(rass_engine* h, const char* path);

/* Debug only (no reference counterpart): raw tensor-core dot products bf16(q_hat) . bf16(x) of B <= 64 queries
 * against every row, out_host [rows, 64] fp32.  Used by the tests to check the TMA/tcgen05 descriptors. */
int rass_debug_umma_scores(rass_engine* h, const float* q_host, int B, float* out_host);
/* same for the CTA-pair kernel: B <= 256 queries, out_host [rows, 256] fp32 */
int rass_debug_gemm_scores(rass_engine* h, const float* q_host, int B, float* out_host);
/* same for the int8 pass: the exact int32 accumulators x8 . q8 of B <= 64 queries, acc_host [rows, 128] (columns
 * 0..63 the first int8 part of each query, 64..127 the second), and the int8 operands the pass read (nullable):
 * x8_host [rows, dim_pad] and q8_host [128, dim_pad].  RASS_E_UNSUPPORTED on a store without the int8 shadow. */
int rass_debug_umma8_scores(rass_engine* h, const float* q_host, int B, int32_t* acc_host, int8_t* x8_host,
                            int8_t* q8_host);

#ifdef __cplusplus
}
#endif
#endif /* RASS_B200_H */
