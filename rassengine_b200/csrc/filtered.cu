// Per-query filters in one call: every query of a batch brings its OWN list of rows that pass its bool.filter.
//
// Every production call of the reference carries its own `term patientId` filter (app/main.py:1543-1550, 1599-1604,
// :2884): a window of coalesced requests holds as many different filters as requests, so one pass-mask per call
// (rass_set_row_filter) cannot serve it.  A patient's documents are a few hundred rows of millions; for such lists
// streaming the corpus (or the postings) is the wrong plan -- the rows are scored directly:
//
//   rass_search_knn_filtered     exact top-k among each query's listed rows: fp64 keys of the stored values, the same
//                                function and ranking as the corpus scans' rerank (OpenSearch's "efficient filter" /
//                                the client's knn_filter="pre" semantics), no corpus pass at all
//   rass_search_hybrid_filtered  the reference's bool.should + bool.filter for each query over its listed rows: the text
//                                clauses are looked up in the postings (binary search per term, summed in query order like
//                                the ordered tile kernel), the knn clause is the query's k nearest -- of the whole corpus
//                                (ONE scan pass shared by the batch; nmslib's post-filter semantics, the default) or of the
//                                listed rows (knn_mode 1) -- intersected with the list
//
// Results are bit-identical to rass_search_knn (pre-filter) / rass_search_hybrid with the same filter set per call.
#include <string.h>

#include <algorithm>

#include "common.cuh"

int launch_select_batch(rass_engine* h, size_t entries, int B, int k, int64_t* out_rows, float* out_scores,
                        double* out_keys, cudaStream_t st, const int* only_if);
int launch_exact_select(rass_engine* h, size_t entries, int B, int k, int64_t* out_rows, float* out_scores,
                        double* out_keys, cudaStream_t st);

// one CTA per query, one warp per listed row: the exact key of (row, query) into the query's list
template <bool BF16_ROWS>
__global__ void __launch_bounds__(256) filtered_keys_kernel(const float* __restrict__ x32,
                                                            const __nv_bfloat16* __restrict__ x16,
                                                            const double* __restrict__ norm64,
                                                            const float* __restrict__ sb, const float* __restrict__ q_raw,
                                                            const double* __restrict__ q_norm,
                                                            const int64_t* __restrict__ findptr,
                                                            const int64_t* __restrict__ frows, int64_t n_rows, int dim_pad,
                                                            int metric, double* __restrict__ xkey,
                                                            uint32_t* __restrict__ xrow, size_t entries) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* qs = reinterpret_cast<float*>(smem_raw);
  const int q = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int j = threadIdx.x; j < dim_pad; j += blockDim.x) qs[j] = q_raw[(size_t)q * dim_pad + j];
  __syncthreads();
  const double qn = q_norm[q];
  const int64_t lo = findptr[q], n = findptr[q + 1] - lo;
  double* kq = xkey + (size_t)q * entries;
  uint32_t* rq = xrow + (size_t)q * entries;
  for (int64_t i = warp; i < (int64_t)entries; i += blockDim.x >> 5) {
    int64_t r = i < n ? frows[lo + i] : -1;
    if (r < 0 || r >= n_rows || sb[r] == neg_inf<float>()) r = -1;          // out of range, tombstoned
    double key = 0.0;
    if (r >= 0) key = exact_key_warp<BF16_ROWS>(x32, x16, norm64, (uint32_t)r, qs, qn, dim_pad, metric);
    if (lane == 0) {
      kq[i] = r >= 0 ? key : neg_inf<double>();
      rq[i] = r >= 0 ? (uint32_t)r : 0xffffffffu;
    }
  }
}

struct FilteredTextArgs {
  const int64_t* indptr;       // postings CSR
  const int32_t* doc;
  const uint16_t* tf;
  const uint8_t* norm;
  const float* inv;
  int64_t norm_rows, n_docs;
  const int32_t* qt_indptr;    // per-term arrays of the batch (hybrid_core's staging layout)
  const int64_t* t_lo;
  const uint32_t* t_len;
  const float* t_w;
  const uint8_t* t_field;
  const uint8_t* t_flag;
  int multi;                   // field groups / clauses present (dis-max + clause sums)
  const int64_t* findptr;
  const int64_t* frows;
  const int64_t* knn_rows;     // [B, k] GLOBAL rows of the knn clause (-1 = none) or null
  const float* knn_scores;
  const float* sb;             // tombstones of the vector store do not affect text: unused here, kept for symmetry
  RowMap rmap;
  int k;
  float w_knn;
  double* xkey;
  uint32_t* xrow;
  size_t entries;
};

// one CTA per query, one thread per listed row: the row's bool.should score, like hybrid_tile_kernel computes it
__global__ void __launch_bounds__(256) filtered_text_kernel(const __grid_constant__ FilteredTextArgs a) {
  __shared__ int64_t s_knn[RASS_MAX_K];
  __shared__ float s_kns[RASS_MAX_K];
  const int q = blockIdx.x;
  const bool have_knn = a.knn_rows != nullptr;
  if (have_knn && threadIdx.x < a.k) {
    const int64_t r = a.knn_rows[(size_t)q * a.k + threadIdx.x];
    s_knn[threadIdx.x] = r >= 0 ? row_global_to_local(a.rmap, r) : -1;
    s_kns[threadIdx.x] = a.knn_scores[(size_t)q * a.k + threadIdx.x];
  }
  __syncthreads();
  const int64_t lo = a.findptr[q], n = a.findptr[q + 1] - lo;
  const int j_begin = a.qt_indptr ? a.qt_indptr[q] : 0, j_end = a.qt_indptr ? a.qt_indptr[q + 1] : 0;
  double* kq = a.xkey + (size_t)q * a.entries;
  uint32_t* rq = a.xrow + (size_t)q * a.entries;
  for (int64_t i = threadIdx.x; i < (int64_t)a.entries; i += blockDim.x) {
    const int64_t r = i < n ? a.frows[lo + i] : -1;
    double fused = 0.0;
    bool matched = false;
    if (r >= 0) {
      // text clauses: every query term in order (duplicates count twice); field groups / clauses as in the tile kernel
      double acc = 0.0, total = 0.0;
      float best = 0.f;
      bool group_touched = false, clause_touched = false;
      if (r < a.n_docs) {
        for (int j = j_begin; j < j_end; ++j) {
          const int64_t p0 = a.t_lo[j];
          int64_t x0 = 0, x1 = (int64_t)a.t_len[j];          // first posting with doc >= r
          while (x0 < x1) {
            const int64_t m = (x0 + x1) >> 1;
            if ((int64_t)__ldg(a.doc + p0 + m) < r) x0 = m + 1; else x1 = m;
          }
          if (x0 < (int64_t)a.t_len[j] && (int64_t)__ldg(a.doc + p0 + x0) == r) {
            const int f = a.t_field[j];
            const float w = a.t_w[j];
            const float x = __fmul_rn((float)__ldg(a.tf + p0 + x0), a.inv[f * 256 + a.norm[(size_t)f * a.norm_rows + r]]);
            const float s = __fsub_rn(w, __fdiv_rn(w, __fadd_rn(1.0f, x)));
            if (s > 0.f) { acc += (double)s; group_touched = true; }
          }
          if (a.multi) {
            const int flag = a.t_flag[j];
            if ((flag & 1) && group_touched) {
              if (acc != 0.0) best = fmaxf(best, (float)acc);
              acc = 0.0;
              group_touched = false;
              clause_touched = true;
            }
            if ((flag & 2) && clause_touched) {
              if (best != 0.f) total += (double)best;
              best = 0.f;
              clause_touched = false;
            }
          }
        }
      }
      fused = a.multi ? total : acc;
      matched = fused != 0.0;
      if (have_knn) {
        for (int c = 0; c < a.k; ++c)
          if (s_knn[c] == r) {
            fused = (a.multi ? fused : (double)(float)fused) + (double)__fmul_rn(a.w_knn, s_kns[c]);
            matched = true;
            break;
          }
      }
    }
    // the fused score is a float (Lucene's BooleanScorer casts the double sum); keys travel as its double image
    kq[i] = matched ? (double)(float)fused : neg_inf<double>();
    rq[i] = matched ? (uint32_t)r : 0xffffffffu;
  }
}

static int upload_lists(rass_engine* h, const int64_t* findptr, const int64_t* frows, int B, int64_t** d_indptr,
                        int64_t** d_rows, size_t* max_len, cudaStream_t st) {
  size_t mx = 0;
  for (int q = 0; q < B; ++q) {
    if (findptr[q + 1] < findptr[q]) return rass_fail(h, RASS_E_INVALID, "filter row lists: offsets must not decrease");
    mx = std::max<size_t>(mx, (size_t)(findptr[q + 1] - findptr[q]));
  }
  const size_t total = (size_t)(findptr[B] - findptr[0]);
  const size_t need = (size_t)B + 1 + total;
  if (need > h->flist_cap) {
    CUDA_TRY(h, cudaStreamSynchronize(st));
    cudaFree(h->flist_dev);
    h->flist_dev = nullptr;
    h->flist_cap = 0;
    CUDA_TRY(h, cudaMalloc(&h->flist_dev, std::max<size_t>(need * 2, 4096) * sizeof(int64_t)));
    h->flist_cap = std::max<size_t>(need * 2, 4096);
  }
  std::vector<int64_t> ip((size_t)B + 1);
  for (int q = 0; q <= B; ++q) ip[(size_t)q] = findptr[q] - findptr[0];
  CUDA_TRY(h, cudaMemcpyAsync(h->flist_dev, ip.data(), ((size_t)B + 1) * 8, cudaMemcpyHostToDevice, st));
  if (total) CUDA_TRY(h, cudaMemcpyAsync(h->flist_dev + B + 1, frows + findptr[0], total * 8, cudaMemcpyHostToDevice, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));          // ip is a local; the caller's lists may be freed on return
  *d_indptr = h->flist_dev;
  *d_rows = h->flist_dev + B + 1;
  *max_len = mx;
  return RASS_OK;
}

// exact top-k of the listed rows of every query into (out_rows, out_scores, out_keys) on the device
static int filtered_knn_dev(rass_engine* h, const float* q_dev, int B, int k, const int64_t* d_indptr,
                            const int64_t* d_rows, size_t max_len, int64_t* out_rows, float* out_scores,
                            double* out_keys, cudaStream_t st) {
  int rc;
  SearchWs& ws = h->ws[0];
  if ((rc = ensure_query_workspace(h, ws, B))) return rc;
  if ((rc = launch_query_prep(h, ws, q_dev, B, st))) return rc;
  const size_t entries = std::max<size_t>(max_len, 1);
  if ((rc = ensure_xlist_workspace(h, (entries * B + RASS_EXACT_NQ - 1) / RASS_EXACT_NQ))) return rc;
  const size_t smem = (size_t)h->dim_pad * 4;
  if (h->flags & RASS_BF16_ONLY)
    filtered_keys_kernel<true><<<B, 256, smem, st>>>(h->x32, h->x16, h->norm64, h->sb, ws.q_raw, ws.q_norm, d_indptr,
                                                     d_rows, h->n_rows, h->dim_pad, h->metric, h->xlist_key,
                                                     h->xlist_row, entries);
  else
    filtered_keys_kernel<false><<<B, 256, smem, st>>>(h->x32, h->x16, h->norm64, h->sb, ws.q_raw, ws.q_norm, d_indptr,
                                                      d_rows, h->n_rows, h->dim_pad, h->metric, h->xlist_key,
                                                      h->xlist_row, entries);
  CUDA_TRY(h, cudaGetLastError());
  return launch_exact_select(h, entries, B, k, out_rows, out_scores, out_keys, st);
}

extern "C" int rass_search_knn_filtered(rass_engine* h, const float* q_host, int B, int k, const int64_t* frow_indptr,
                                        const int64_t* frows, int64_t* out_rows, float* out_scores, double* out_keys) {
  if (!h) return RASS_E_INVALID;
  if (h->shards) return rass_fail(h, RASS_E_UNSUPPORTED, "per-query row lists take a single-device handle");
  cudaSetDevice(h->device);
  if (!q_host || !frow_indptr || !out_rows || !out_scores || B < 1 || (frow_indptr[B] > frow_indptr[0] && !frows))
    return rass_fail(h, RASS_E_INVALID, "bad arguments");
  if (k < 1 || k > RASS_MAX_K) return rass_fail(h, RASS_E_INVALID, "k must be in [1, %d], got %d", RASS_MAX_K, k);
  cudaStream_t st = eng_stream(h);
  int rc;
  float* q_dev = nullptr;
  if ((rc = stage_queries(h, q_host, B, &q_dev))) return rc;
  const size_t n_out = (size_t)B * k;
  if ((rc = ensure_out_workspace(h, n_out))) return rc;
  int64_t *d_ip = nullptr, *d_rows = nullptr;
  size_t mx = 0;
  if ((rc = upload_lists(h, frow_indptr, frows, B, &d_ip, &d_rows, &mx, st))) return rc;
  if ((rc = filtered_knn_dev(h, q_dev, B, k, d_ip, d_rows, mx, h->out_rows, h->out_scores,
                             out_keys ? h->out_keys : nullptr, st)))
    return rc;
  CUDA_TRY(h, cudaMemcpyAsync(h->out_rows_host, h->out_rows, n_out * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaMemcpyAsync(h->out_scores_host, h->out_scores, n_out * 4, cudaMemcpyDeviceToHost, st));
  if (out_keys) CUDA_TRY(h, cudaMemcpyAsync(h->out_keys_host, h->out_keys, n_out * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  memcpy(out_rows, h->out_rows_host, n_out * 8);
  memcpy(out_scores, h->out_scores_host, n_out * 4);
  if (out_keys) memcpy(out_keys, h->out_keys_host, n_out * 8);
  return RASS_OK;
}

extern "C" int rass_search_hybrid_filtered(rass_engine* h, const float* q_host, int B, const int32_t* qterm_indptr,
                                           const int32_t* qterms, const float* qweights, const uint8_t* qflags,
                                           float w_text, float w_knn, int k, const int64_t* frow_indptr,
                                           const int64_t* frows, int knn_mode, int64_t* out_rows, float* out_scores,
                                           rass_stats* stats) {
  if (!h) return RASS_E_INVALID;
  if (h->shards) return rass_fail(h, RASS_E_UNSUPPORTED, "per-query row lists take a single-device handle");
  cudaSetDevice(h->device);
  if (B < 1 || !frow_indptr || !out_rows || !out_scores || (frow_indptr[B] > frow_indptr[0] && !frows))
    return rass_fail(h, RASS_E_INVALID, "bad arguments");
  if (k < 1 || k > RASS_MAX_K) return rass_fail(h, RASS_E_INVALID, "k must be in [1, %d], got %d", RASS_MAX_K, k);
  if (!q_host && !qterm_indptr) return rass_fail(h, RASS_E_INVALID, "neither a vector nor a text clause");
  Bm25State& b = h->bm25;
  if (qterm_indptr && (!b.built || !qterms)) return rass_fail(h, RASS_E_INVALID, "text clause without rass_bm25_build");
  if (knn_mode != 0 && knn_mode != 1) return rass_fail(h, RASS_E_INVALID, "knn_mode must be 0 (post) or 1 (pre)");
  cudaStream_t st = eng_stream(h);
  int rc;
  rass_stats s;
  memset(&s, 0, sizeof(s));
  s.n_queries = B;
  const size_t n_out = (size_t)B * k;
  if ((rc = ensure_out_workspace(h, 2 * n_out))) return rc;
  int64_t *d_ip = nullptr, *d_rows = nullptr;
  size_t mx = 0;
  if ((rc = upload_lists(h, frow_indptr, frows, B, &d_ip, &d_rows, &mx, st))) return rc;
  // 1. the knn clause: the k nearest of the whole corpus (one pass shared by the batch) or of each query's list
  int64_t* knn_rows = h->out_rows + n_out;
  float* knn_scores = h->out_scores + n_out;
  const bool have_vec = q_host != nullptr && h->n_rows > 0;
  if (have_vec) {
    float* q_dev = nullptr;
    if ((rc = stage_queries(h, q_host, B, &q_dev))) return rc;
    if (knn_mode == 0) {
      if ((rc = search_core(h, q_dev, B, k, knn_rows, knn_scores, nullptr, &s))) return rc;
    } else {
      if ((rc = filtered_knn_dev(h, q_dev, B, k, d_ip, d_rows, mx, knn_rows, knn_scores, nullptr, st))) return rc;
    }
  }
  // 2. the text clauses + fusion over the listed rows
  FilteredTermArrays ta;
  memset(&ta, 0, sizeof(ta));
  if (qterm_indptr && (rc = stage_hybrid_terms(h, B, qterm_indptr, qterms, qweights, qflags, w_text, &ta, st))) return rc;
  const size_t entries = std::max<size_t>(mx, 1);
  if ((rc = ensure_xlist_workspace(h, (entries * B + RASS_EXACT_NQ - 1) / RASS_EXACT_NQ))) return rc;
  FilteredTextArgs a;
  memset(&a, 0, sizeof(a));
  a.indptr = b.indptr; a.doc = b.doc; a.tf = b.tf; a.norm = b.norm; a.inv = b.inv_dev;
  a.norm_rows = b.N;
  a.n_docs = b.built ? b.N : 0;
  a.qt_indptr = ta.qt_indptr; a.t_lo = ta.t_lo; a.t_len = ta.t_len; a.t_w = ta.t_w; a.t_field = ta.t_field;
  a.t_flag = ta.t_flag;
  a.multi = ta.multi ? 1 : 0;
  a.findptr = d_ip; a.frows = d_rows;
  a.knn_rows = have_vec ? knn_rows : nullptr;
  a.knn_scores = knn_scores;
  a.rmap = h->rmap;
  a.k = k;
  a.w_knn = w_knn;
  a.xkey = h->xlist_key; a.xrow = h->xlist_row; a.entries = entries;
  filtered_text_kernel<<<B, 256, 0, st>>>(a);
  CUDA_TRY(h, cudaGetLastError());
  if ((rc = launch_select_batch(h, entries, B, k, h->out_rows, h->out_scores, nullptr, st, nullptr))) return rc;
  s.launches += 2;
  CUDA_TRY(h, cudaMemcpyAsync(h->out_rows_host, h->out_rows, n_out * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaMemcpyAsync(h->out_scores_host, h->out_scores, n_out * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  memcpy(out_rows, h->out_rows_host, n_out * 8);
  memcpy(out_scores, h->out_scores_host, n_out * 4);
  h->last_stats = s;
  if (stats) *stats = s;
  return RASS_OK;
}
