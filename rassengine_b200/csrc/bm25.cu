// BM25 term scoring over CSR postings and the bool.should boosted-sum fusion with the kNN clause.
//
// Replaces the Lucene side of OpenSearchIndexer.hybrid_search / multi_intent_search (reference app/main.py:1574-1598,
// 1982-2010):
//   multi_match(best_fields, operator or, fuzziness AUTO) over the 26 text fields   -> per-field BM25Similarity postings
//   multi_match(best_fields) over the 24 keyword fields                                walk, max over a clause's fields
//   knn clause                                                                      -> only the k nearest docs score
//   bool.should (+ bool.filter)                                                     -> sum of the matching clauses
// Arithmetic follows oracle/bm25.py, oracle/fuzzy.py, oracle/multifield.py and oracle/fusion.py operation for operation
// (float ops rounded individually, field sums in double cast to float, clause sums in double, final cast to float) so
// ranked ids and scores are identical.  One fused kernel per batch (hybrid_tile_kernel) + one select; the term
// dictionary scan of fuzziness AUTO (fuzzy_scan_kernel) lives here too.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"

template <typename T>
static int upload(rass_engine* h, T** dst, const T* src, size_t n) {
  cudaFree(*dst);
  *dst = nullptr;
  CUDA_TRY(h, cudaMalloc(dst, std::max<size_t>(n, 1) * sizeof(T)));
  if (n) CUDA_TRY(h, cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
  return RASS_OK;
}

#define BM25_MAX_TERMS 1024      // term queries per query string: 12 tokens x <= 50 fuzzy expansions and then some
#define HYB_THREADS 256
#define HYB_LIST 512             // keys that survive the tile's top-k pre-filter (2 per thread)


// ---- kernels ------------------------------------------------------------------------------------------------
struct HybridArgs {
  const int32_t* doc;
  const uint16_t* tf;
  const float* xq;               // per posting: tf * inv[norm of the doc] (the impact the order-free kernel scores from)
  const uint8_t* norm;
  const float* inv;
  const uint32_t* tile_off;
  const int32_t* qt_indptr;      // [B + 1] into the per-term arrays below (terms without postings are dropped)
  const int64_t* t_lo;           // first posting of the term
  const uint32_t* t_len;         // document frequency
  const float* t_w;              // float(clause boost) * idf
  const int32_t* t_row;          // row of tile_off, -1 for rare terms
  const uint8_t* t_field;        // field of the term (selects norm plane and inv table)
  const uint8_t* t_flag;         // bit 0: last term of its field group (dis-max over fields), bit 1: last of its clause
  const float* t_bound;          // order-free kernel: upper bound of the score of a doc matching only this term and the
                                 // terms of the query with smaller bounds (MaxScore); null = no pruning
  const int64_t* knn_rows;       // [B, k] or null
  const float* knn_scores;
  const uint8_t* row_filter;
  int64_t filter_rows;
  RowMap rmap;                   // local doc <-> global row (knn lists and outputs carry global rows)
  int64_t n_docs, norm_rows;     // norm is [F][norm_rows]
  int n_tiles, table_tiles, k;   // tiles of this launch; tiles the offset table covers (docs known to the postings)
  float w_knn;
  double* xkey;                  // [B][n_tiles * k]
  uint32_t* xrow;
  uint32_t* gthr;                // [B] per query: the largest k-th best fused key any tile has found so far (ordered
                                 // integer image, 0 = none): k rows score at least this much, lower keys are out
};

// The rest of a (tile, query) CTA once the text clauses are summed in `fused` (double per doc, 0 = no match): the knn
// clause, then the tile's top-k by (fused float score desc, row asc) into the query's list.  MULTI: `fused` holds clause
// sums in double (the knn score is one more clause); otherwise the single text clause is rounded to float first.
// pre_g (nullable): the query's pruning bound already sitting in shared memory (the caller read it while the tile was
// being scored), which saves the tail a global round trip and two barriers.
template <bool MULTI>
__device__ __forceinline__ void hybrid_tile_tail(const HybridArgs& a, double* fused, int q, int tile, int64_t d0,
                                                 int64_t d1, bool knn_done = false, const uint32_t* pre_g = nullptr) {
  __shared__ __align__(16) int s_cnt[2][HYB_THREADS / 32];
  __shared__ uint32_t s_list[HYB_LIST];
  __shared__ int s_nout, s_nmatch, s_ns;
  __shared__ uint32_t s_g;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) { s_nout = 0; s_nmatch = 0; s_ns = 0; }
  double* acc = fused;
  // ---- knn clause ----
  if (!knn_done && a.knn_rows && tid < a.k) {
    const int64_t r = a.knn_rows[(size_t)q * a.k + tid];
    if (r >= 0) {
      const int64_t d = row_global_to_local(a.rmap, r);     // -1: a row of another shard
      if (d >= d0 && d < d1 && !(a.row_filter && (d >= a.filter_rows || !a.row_filter[d])))
        // a clause's score is a float; the bool sums the clause scores in double (and the final cast to float below
        // is the identity for rows without a knn contribution)
        fused[d - d0] = (MULTI ? fused[d - d0] : (double)(float)fused[d - d0]) +
                        (double)__fmul_rn(a.w_knn, a.knn_scores[(size_t)q * a.k + tid]);
    }
  }
  __syncthreads();

  // ---- top-k of the tile: keys as order-preserving integers, 0 = no match ----
  constexpr int PER = HYB_TILE / HYB_THREADS;
  uint32_t key[PER];
  int nm = 0;
  // With a positive bound at hand only sums that can round to a float >= the bound need a key.  For positive doubles
  // the high words order like the values, so one 32-bit load and an integer compare per doc decide it: thr_hi = high
  // word of the next float BELOW the bound (every double that rounds to the bound or above is larger than that).
  // Without a bound (or a bound <= 0) every doc passes, as before.
  int thr_hi = (int)0x80000000;
  if (pre_g && *pre_g > 0x80000000u) {
    const float gf = unord32(*pre_g);
    thr_hi = __double2hiint((double)__uint_as_float(__float_as_uint(gf) - 1u));
  }
  const int* acc_hi = reinterpret_cast<const int*>(acc) + 1;
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    key[i] = 0u;
    if (acc_hi[2 * (i * HYB_THREADS + tid)] >= thr_hi) {
      const double v = acc[i * HYB_THREADS + tid];          // doc = d0 + i * HYB_THREADS + tid
      key[i] = v != 0.0 ? ord32((float)v) : 0u;
      nm += v != 0.0;
    }
  }
  if (!pre_g) {
    if (nm) atomicAdd(&s_nmatch, nm);
    __syncthreads();
  }
  const int n_match = pre_g ? HYB_TILE : s_nmatch;      // with a bound at hand the survivors are counted below
  double* xk = a.xkey + ((size_t)q * a.n_tiles + tile) * a.k;
  uint32_t* xr = a.xrow + ((size_t)q * a.n_tiles + tile) * a.k;
  int buf = 0;
  auto block_count = [&](int c) {
    c = __reduce_add_sync(0xffffffffu, c);
    if (lane == 0) s_cnt[buf][warp] = c;
    __syncthreads();
    const int4 c0 = *reinterpret_cast<const int4*>(&s_cnt[buf][0]), c1 = *reinterpret_cast<const int4*>(&s_cnt[buf][4]);
    buf ^= 1;       // the next count writes the other buffer, so one barrier per count is enough
    return c0.x + c0.y + c0.z + c0.w + c1.x + c1.y + c1.z + c1.w;
  };
  // Cross-tile pruning: some other tile of this query already holds k rows with key >= g, so keys below g cannot
  // reach the query's top-k.  Most tiles of a batched launch then keep a handful of keys and skip the selection.
  // (read once per CTA: other tiles raise the bound concurrently, and the branches below must be uniform)
  if (!pre_g) {
    if (tid == 0) s_g = n_match > a.k ? __ldcg(a.gthr + q) : 0u;
    __syncthreads();
  }
  const uint32_t g = pre_g ? *pre_g : s_g;
  int n_live = n_match;
  if (g || pre_g) {
    int c = 0;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      if (key[i] < g) key[i] = 0;
      c += key[i] != 0;
    }
    n_live = block_count(c);
  }
  if (n_live <= a.k) {
#pragma unroll
    for (int i = 0; i < PER; ++i)
      if (key[i]) {
        const int pos = atomicAdd(&s_nout, 1);
        xk[pos] = (double)unord32(key[i]);
        xr[pos] = (uint32_t)(d0 + i * HYB_THREADS + tid);
      }
  } else {
    // Pre-filter: b' = k-th largest per-thread maximum is a lower bound of the tile's k-th largest key, so only
    // keys >= b' (normally between k and 2k of them) enter the selection.
    uint32_t mx = 0;
#pragma unroll
    for (int i = 0; i < PER; ++i) mx = max(mx, key[i]);
    uint32_t bp = 0;
#pragma unroll 1
    for (int bit = 31; bit >= 0; --bit) {
      const uint32_t cand = bp | (1u << bit);
      if (__syncthreads_count(mx >= cand) >= a.k) bp = cand;
    }
    if (mx >= bp && mx) {
#pragma unroll
      for (int i = 0; i < PER; ++i)
        if (key[i] && key[i] >= bp) {
          const int pos = atomicAdd(&s_ns, 1);
          if (pos < HYB_LIST) s_list[pos] = key[i];
        }
    }
    __syncthreads();
    const int ns = s_ns;
    // k-th largest key by most-significant-bit-first descent: prefix grows while >= k entries are >= it
    uint32_t prefix = 0;
    if (ns <= HYB_LIST) {
      const uint32_t e0 = tid < ns ? s_list[tid] : 0u, e1 = tid + HYB_THREADS < ns ? s_list[tid + HYB_THREADS] : 0u;
#pragma unroll 1
      for (int bit = 31; bit >= 0; --bit) {
        const uint32_t cand = prefix | (1u << bit);
        if (block_count((e0 >= cand) + (e1 >= cand)) >= a.k) prefix = cand;
      }
    } else {
#pragma unroll 1
      for (int bit = 31; bit >= 0; --bit) {
        const uint32_t cand = prefix | (1u << bit);
        int c = 0;
#pragma unroll
        for (int i = 0; i < PER; ++i) c += key[i] >= cand;
        if (block_count(c) >= a.k) prefix = cand;
      }
    }
    int n_gt = 0, n_eq = 0;
#pragma unroll
    for (int i = 0; i < PER; ++i) { n_gt += key[i] > prefix; n_eq += key[i] == prefix; }
    const int need_eq = a.k - block_count(n_gt);      // entries equal to the k-th key to take, lowest rows first
    const int tot_eq = block_count(n_eq);
    if (tid == 0) atomicMax(a.gthr + q, prefix);      // k rows of this tile score >= prefix: publish for the others
    const bool all_eq = tot_eq == need_eq;    // the usual case: the k-th key is unique in the tile
#pragma unroll
    for (int i = 0; i < PER; ++i)
      if (key[i] > prefix || (all_eq && key[i] == prefix)) {
        const int pos = atomicAdd(&s_nout, 1);
        xk[pos] = (double)unord32(key[i]);
        xr[pos] = (uint32_t)(d0 + i * HYB_THREADS + tid);
      }
    __syncthreads();
    if (!all_eq && tid == 0) {
      // equal scores at the cut: Lucene's doc-id tie-break keeps the lowest rows
      int pos = s_nout, left = need_eq;
      for (int i = 0; i < HYB_TILE && left > 0; ++i) {
        const double v = acc[i];
        if (v != 0.0 && ord32((float)v) == prefix) {
          xk[pos] = (double)(float)v;
          xr[pos] = (uint32_t)(d0 + i);
          ++pos;
          --left;
        }
      }
      s_nout = pos;
    }
  }
  __syncthreads();
  for (int i = s_nout + tid; i < a.k; i += HYB_THREADS) {
    xk[i] = neg_inf<double>();
    xr[i] = 0xffffffffu;
  }
}

// One CTA per (tile of 4096 docs, query): the whole bool.should of the reference for those docs.
//   text clause : for every query term in order, s = w - w / (1 + tf * inv[norm[d]]) in float (each op rounded),
//                 summed in double per doc -- a term's postings name a doc once, so plain shared-memory adds
//                 between barriers are race free and the summation order is the oracle's; cast to float
//   knn clause  : the k nearest rows get float(w_knn * knn_score) added in double
//   bool.filter : rows failing the pass mask never match
//   top-k       : 32-bit radix select over the tile's fused float scores, ties by row ascending
// The tile's best k (score, row) go to the query's list; exact_select_kernel ranks n_tiles * k entries.
// MULTI = false: one analysed field, one text clause (chunk-only indices): the clause sum stays in acc.
// MULTI = true : several field groups / clauses: acc = running sum of the current field group, best = dis-max over
//                the groups of the current clause (float, like every Lucene scorer's score()), total = sum over the
//                finished clauses in double; dynamic shared memory holds total and best behind acc.
template <bool MULTI>
__global__ void __launch_bounds__(HYB_THREADS) hybrid_tile_kernel(const __grid_constant__ HybridArgs a) {
  extern __shared__ __align__(16) unsigned char hyb_smem[];
  double* acc = reinterpret_cast<double*>(hyb_smem);                       // [HYB_TILE]
  double* total = acc + (MULTI ? HYB_TILE : 0);                            // [HYB_TILE] (MULTI)
  float* best = reinterpret_cast<float*>(total + HYB_TILE);               // [HYB_TILE] (MULTI)
  __shared__ float s_inv[256];
  __shared__ int64_t s_lo[HYB_THREADS];
  __shared__ uint32_t s_n[HYB_THREADS];
  __shared__ float s_w[HYB_THREADS];
  __shared__ uint8_t s_field[HYB_THREADS], s_flag[HYB_THREADS];
  const int tid = threadIdx.x;
  const int tile = blockIdx.y, q = blockIdx.x;            // queries fastest: the CTAs in flight cover a few tiles of EVERY
                                                          // query, so a query's pruning bound exists after its first tiles
  const int64_t d0 = (int64_t)tile * HYB_TILE;
  const int64_t d1 = min(d0 + HYB_TILE, a.n_docs);
  for (int i = tid; i < HYB_TILE; i += HYB_THREADS) {
    acc[i] = 0.0;
    if (MULTI) { total[i] = 0.0; best[i] = 0.f; }
  }
  __syncthreads();

  // ---- text clauses ----
  if (a.qt_indptr) {
    const int j_begin = a.qt_indptr[q], j_end = a.qt_indptr[q + 1];
    int cur_field = -1;
    const uint8_t* norm_f = a.norm;
    bool group_touched = false, clause_touched = false;     // uniform across the CTA
    for (int j0 = j_begin; j0 < j_end; j0 += HYB_THREADS) {
      const int nt = min(HYB_THREADS, j_end - j0);
      // posting range of every term inside this tile, fetched by one thread per term (one latency for all terms)
      if (tid < nt) {
        const int j = j0 + tid;
        const int row = a.t_row[j];
        uint32_t pa = 0, pb = a.t_len[j];
        if (row >= 0) {
          if (tile < a.table_tiles) {
            const uint32_t* off = a.tile_off + (size_t)row * (a.table_tiles + 1) + tile;
            pa = off[0];
            pb = off[1];
          } else {
            pb = 0;      // rows appended after rass_bm25_build carry no postings
          }
        }
        s_lo[tid] = a.t_lo[j] + pa;
        s_n[tid] = pb - pa;
        s_w[tid] = a.t_w[j];
        s_field[tid] = a.t_field[j];
        s_flag[tid] = a.t_flag[j];
      }
      __syncthreads();
      for (int j = 0; j < nt; ++j) {
        const uint32_t n = s_n[j];
        if (n != 0) {                         // uniform: a term without postings in the tile needs no barrier
          const int field = s_field[j];
          if (field != cur_field) {           // per-field length table and norm plane
            s_inv[tid] = a.inv[field * 256 + tid];
            norm_f = a.norm + (size_t)field * a.norm_rows;
            cur_field = field;
            __syncthreads();
          }
          const int64_t lo = s_lo[j];
          const float w = s_w[j];
          for (uint32_t p = tid; p < n; p += HYB_THREADS) {
            const int64_t d = (int64_t)__ldg(a.doc + lo + p);
            if (d < d0 || d >= d1) continue;                                             // rare terms scan their whole list
            if (a.row_filter && (d >= a.filter_rows || !a.row_filter[d])) continue;       // bool.filter
            const float x = __fmul_rn((float)__ldg(a.tf + lo + p), s_inv[norm_f[d]]);
            const float s = __fsub_rn(w, __fdiv_rn(w, __fadd_rn(1.0f, x)));
            if (s > 0.f) acc[d - d0] += (double)s;
          }
          group_touched = true;
          __syncthreads();
        }
        if (MULTI) {
          const int flag = s_flag[j];
          if ((flag & 1) && group_touched) {  // end of a field group: dis-max of the float field scores
            for (int i = tid; i < HYB_TILE; i += HYB_THREADS) {
              const double v = acc[i];
              if (v != 0.0) { best[i] = fmaxf(best[i], (float)v); acc[i] = 0.0; }
            }
            group_touched = false;
            clause_touched = true;
            __syncthreads();
          }
          if ((flag & 2) && clause_touched) { // end of a clause: the bool sums clause scores in double
            for (int i = tid; i < HYB_TILE; i += HYB_THREADS) {
              const float v = best[i];
              if (v != 0.f) { total[i] += (double)v; best[i] = 0.f; }
            }
            clause_touched = false;
            __syncthreads();
          }
        }
      }
      __syncthreads();                        // the next chunk overwrites s_lo / s_n / s_w
    }
  }
  hybrid_tile_tail<MULTI>(a, MULTI ? total : acc, q, tile, d0, d1);
}

// Order-free form of the single-clause kernel above, for queries whose clause sums are EXACT in double whatever the
// order of the additions (hybrid_core checks it per query from the per-term score ranges: every addend is a float that
// is a multiple of 2^L, every partial sum stays below 2^(L + 53)).  Exact sums do not depend on the order, so the
// result is bit-identical to the ordered walk -- and the CTA is free to
//   * take the postings of all the query's terms in the tile at once: warps draw 128-posting chunks of any term, no
//     barrier per term, four independent postings in flight per lane, shared-memory atomics (two terms may name the same
//     doc at the same time);
//   * skip work the way Lucene's MaxScore scorer does.  g = the query's pruning bound (k rows already score >= g,
//     published by earlier tiles).  With the terms sorted by their largest possible score, the longest prefix whose
//     summed bounds stay below g is NON-ESSENTIAL: a doc matching only such terms scores below g and cannot reach the
//     top-k.  So essential terms are accumulated first and mark the docs they touch (the knn rows of the tile are marked
//     too); the postings of non-essential terms -- the frequent terms, i.e. most postings -- are then only looked at
//     (one doc id each) and scored for marked docs alone.  Every doc that can still reach the top-k gets its complete,
//     exact score; the others are never emitted.  Tiles that start before a bound exists simply treat every term as
//     essential.
#define HYB_FAST_TERMS 64      // terms staged per round
#define HYB_CHUNK 256          // postings a warp draws at a time (8 per lane; 128: 1.192 ms, 64: 1.356, 256: 1.173 per cfg4 batch)
#define HYB_QUEUE 64           // per-warp queue of non-essential postings that hit a marked doc
#define HYB_SPARSE_CAP 512     // marked docs at or above the bound a tile can rank without the dense select

// one scored posting: s = w - w / (1 + tf * inv[norm]) with every float op rounded (Lucene's BM25Similarity), added to
// the doc's clause sum
// the same from the posting's precomputed impact x = tf * inv[norm] (Bm25State::xq, written by term_xrange_kernel with
// this very multiplication)
__device__ __forceinline__ bool hyb_score_add_x(double* acc, int rel, float x, float w) {
  const float sc = __fsub_rn(w, __fdiv_rn(w, __fadd_rn(1.0f, x)));
  if (sc > 0.f) atomicAdd(&acc[rel], (double)sc);
  return sc > 0.f;
}
__device__ __forceinline__ bool hyb_score_add(double* acc, const float* s_inv, int rel, uint32_t tfv, uint32_t nb, float w) {
  const float x = __fmul_rn((float)tfv, s_inv[nb]);
  const float sc = __fsub_rn(w, __fdiv_rn(w, __fadd_rn(1.0f, x)));
  if (sc > 0.f) atomicAdd(&acc[rel], (double)sc);
  return sc > 0.f;
}

// PRUNE = false (the default) leaves the MaxScore machinery out: 40 registers and 36.6 KB of shared memory, six CTAs per SM
// instead of five (1.53 -> 1.36 ms per 64-query batch at 5M docs).
template <bool FILTER, bool PRUNE>
__global__ void __launch_bounds__(HYB_THREADS, PRUNE ? 5 : 6) hybrid_tile_fast_kernel(const __grid_constant__ HybridArgs a) {
  __shared__ double acc[HYB_TILE];
  __shared__ uint32_t s_bits[PRUNE ? HYB_TILE / 32 : 1];   // docs touched by an essential term or named by the knn clause
  __shared__ float s_inv[PRUNE ? 256 : 1];        // (the MaxScore phases score from tf and norm bytes)
  __shared__ int64_t s_lo[HYB_FAST_TERMS];
  __shared__ uint32_t s_n[HYB_FAST_TERMS];
  __shared__ uint32_t s_cpre[2][HYB_FAST_TERMS + 1];   // chunk prefix of the essential [0] / non-essential [1] terms
  __shared__ float s_w[HYB_FAST_TERMS];
  __shared__ int s_qrel[HYB_THREADS / 32][PRUNE ? HYB_QUEUE : 1];      // per-warp queue: doc slot, posting, weight
  __shared__ uint32_t s_qtf[HYB_THREADS / 32][PRUNE ? HYB_QUEUE : 1];
  __shared__ float s_qw[HYB_THREADS / 32][PRUNE ? HYB_QUEUE : 1];
  __shared__ int s_cn;
  __shared__ uint32_t s_go;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tile = blockIdx.y, q = blockIdx.x;
  const int64_t d0 = (int64_t)tile * HYB_TILE;
  const int64_t d1 = min(d0 + HYB_TILE, a.n_docs);
  const uint32_t tile_len = (uint32_t)(d1 - d0);
  uint32_t go = 0;                          // the query's pruning bound as this CTA starts (ordered image, 0 = none)
  bool pruned = false;
  if (a.qt_indptr) {
    const int j_begin = a.qt_indptr[q], j_end = a.qt_indptr[q + 1];
    const uint8_t* norm_t = a.norm + d0;    // the tile's slice of the norm plane
    // MaxScore needs all essential terms done before the first non-essential one: one staging round only
    const bool may_prune = PRUNE && a.t_bound != nullptr && j_end - j_begin <= HYB_FAST_TERMS;
    // The bound is read ONCE per CTA (other tiles raise it while this one runs, and every branch on it must be
    // uniform): warp 0 reads it and stages the first round right away, the other warps clear the tile meanwhile.
    float g0 = neg_inf<float>();
    if (warp == 0) {
      uint32_t v = 0;
      if (lane == 0) v = __ldcg(a.gthr + q);             // the tail uses it as well (hybrid_tile_tail pre_g)
      v = __shfl_sync(0xffffffffu, v, 0);
      if (lane == 0) s_go = v;
      if (v && may_prune) g0 = unord32(v);
    }
    if (j_begin < j_end) {                  // every term of the query is of one field (hybrid_core checked)
      const int field = a.t_field[j_begin];
      if (PRUNE) s_inv[tid] = a.inv[field * 256 + tid];
      norm_t = a.norm + (size_t)field * a.norm_rows + d0;
    }
    if (warp != 0 || j_begin == j_end) {
      for (int i = tid - (j_begin == j_end ? 0 : 32); i < HYB_TILE; i += HYB_THREADS - (j_begin == j_end ? 0 : 32))
        acc[i] = 0.0;
    }
    if (PRUNE && warp == 1) {
      for (int i = lane; i < HYB_TILE / 32; i += 32) s_bits[i] = 0u;
      if (lane == 0) s_cn = 0;
    }
    for (int j0 = j_begin; j0 < j_end; j0 += HYB_FAST_TERMS) {
      const int nt = min(HYB_FAST_TERMS, j_end - j0);
      if (j0 != j_begin) __syncthreads();   // the previous round is through with the staging arrays
      if (tid < 32) {
        const bool pruned = g0 > neg_inf<float>();
        const float g = g0;
        // posting range of the round's terms inside this tile (two terms per lane), chunk counts per class
        uint32_t ce[2] = {0, 0}, cn[2] = {0, 0};
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int t = 2 * tid + h;
          if (t < nt) {
            const int j = j0 + t;
            const int row = a.t_row[j];
            uint32_t pa = 0, pb = a.t_len[j];
            if (row >= 0) {
              if (tile < a.table_tiles) {
                const uint32_t* off = a.tile_off + (size_t)row * (a.table_tiles + 1) + tile;
                pa = off[0];
                pb = off[1];
              } else {
                pb = 0;      // rows appended after rass_bm25_build carry no postings
              }
            }
            s_lo[t] = a.t_lo[j] + pa;
            s_n[t] = pb - pa;
            s_w[t] = a.t_w[j];
            const uint32_t chunks = (pb - pa + HYB_CHUNK - 1) / HYB_CHUNK;
            const bool ne = pruned && a.t_bound[j] < g;         // summed bounds up to this term stay below g
            if (ne) cn[h] = chunks; else ce[h] = chunks;
          }
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const uint32_t v0 = c ? cn[0] : ce[0], v1 = c ? cn[1] : ce[1];
          uint32_t incl = v0 + v1;
#pragma unroll
          for (int m = 1; m < 32; m <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, incl, m);
            if (tid >= m) incl += o;
          }
          const uint32_t excl = incl - v0 - v1;
          if (2 * tid <= nt) s_cpre[c][2 * tid] = excl;
          if (2 * tid + 1 <= nt) s_cpre[c][2 * tid + 1] = excl + v0;
          if (tid == 31 && nt == HYB_FAST_TERMS) s_cpre[c][HYB_FAST_TERMS] = incl;
        }
      }
      __syncthreads();                      // (first round: the tile is cleared, s_go / s_inv are set as well)
      if (j0 == j_begin) {
        go = s_go;
        pruned = may_prune && go != 0;
        if (pruned && a.knn_rows) {         // the knn rows of the tile can reach the top-k whatever their text score
          if (tid < a.k) {
            const int64_t r = a.knn_rows[(size_t)q * a.k + tid];
            const int64_t d = r >= 0 ? row_global_to_local(a.rmap, r) : -1;
            if (d >= d0 && d < d1) atomicOr(&s_bits[(d - d0) >> 5], 1u << ((d - d0) & 31));
          }
          // (ordered before the non-essential phase by the barrier that phase starts with)
        }
      }
      // ---- essential terms: every posting is scored ----
      {
        const uint32_t n_chunks = s_cpre[0][nt];
        int j = 0;
        uint32_t c_lo = 0, c_hi = s_cpre[0][1];                // chunk range of term j
        for (uint32_t c = warp; c < n_chunks; c += HYB_THREADS / 32) {
          while (c >= c_hi) { ++j; c_lo = c_hi; c_hi = s_cpre[0][j + 1]; }    // warp-uniform: the chunk's term
          const uint32_t first = (c - c_lo) * HYB_CHUNK, n_rem = s_n[j] - first;
          const int64_t p0 = s_lo[j] + first;
          const int32_t* pd = a.doc + p0;
          const float* px = a.xq + p0;
          const float w = s_w[j];
          int rel[HYB_CHUNK / 32];
          float xv[HYB_CHUNK / 32];
#pragma unroll
          for (int u = 0; u < HYB_CHUNK / 32; ++u) {
            const uint32_t i = u * 32 + lane;
            const int dd = i < n_rem ? __ldg(pd + i) : -1;
            rel[u] = dd - (int)d0;                             // in the tile iff 0 <= rel < tile_len (rare terms scan
            if ((uint32_t)rel[u] >= tile_len) rel[u] = -1;     // their whole list); -1 and out-of-range ids fall out
            if (FILTER && rel[u] >= 0 && (dd >= a.filter_rows || !a.row_filter[dd])) rel[u] = -1;      // bool.filter
            xv[u] = rel[u] >= 0 ? __ldg(px + i) : 0.f;
          }
#pragma unroll
          for (int u = 0; u < HYB_CHUNK / 32; ++u) {
            if (rel[u] < 0) continue;
            if (hyb_score_add_x(acc, rel[u], xv[u], w) && PRUNE && pruned)
              atomicOr(&s_bits[rel[u] >> 5], 1u << (rel[u] & 31));
          }
        }
      }
      // ---- non-essential terms: a doc id per posting, scored for marked docs only ----
      if (PRUNE && s_cpre[1][nt] != 0) {                       // uniform over the CTA
        __syncthreads();                                       // the marks are complete
        const uint32_t n_chunks = s_cpre[1][nt];
        int j = 0;
        int qn = 0;                                            // entries queued by this warp (uniform)
        int* qrel = s_qrel[warp];
        uint32_t* qtf = s_qtf[warp];
        float* qw = s_qw[warp];
        auto drain = [&](int n_take) {                         // score the first n_take queued postings, one per lane
          __syncwarp();
          if (lane < n_take) {
            const int r = qrel[lane];
            hyb_score_add(acc, s_inv, r, qtf[lane], norm_t[r], qw[lane]);
          }
          __syncwarp();
          // move what is left to the front
          const int left = qn - n_take;
          int r2 = 0; uint32_t t2 = 0; float w2 = 0.f;
          if (lane < left) { r2 = qrel[n_take + lane]; t2 = qtf[n_take + lane]; w2 = qw[n_take + lane]; }
          __syncwarp();
          if (lane < left) { qrel[lane] = r2; qtf[lane] = t2; qw[lane] = w2; }
          qn = left;
          __syncwarp();
        };
        for (uint32_t c = warp; c < n_chunks; c += HYB_THREADS / 32) {
          while (c >= s_cpre[1][j + 1]) ++j;
          const uint32_t first = (c - s_cpre[1][j]) * HYB_CHUNK, n_rem = s_n[j] - first;
          const int32_t* pd = a.doc + s_lo[j] + first;
          const uint16_t* pt = a.tf + s_lo[j] + first;
          const float w = s_w[j];
          int dd[HYB_CHUNK / 32];
#pragma unroll
          for (int u = 0; u < HYB_CHUNK / 32; ++u) {
            const uint32_t i = u * 32 + lane;
            dd[u] = i < n_rem ? __ldg(pd + i) : -1;
          }
#pragma unroll
          for (int u = 0; u < HYB_CHUNK / 32; ++u) {
            int rel = dd[u] - (int)d0;
            bool hit = (uint32_t)rel < tile_len && ((s_bits[rel >> 5] >> (rel & 31)) & 1u);
            if (FILTER && hit && (dd[u] >= a.filter_rows || !a.row_filter[dd[u]])) hit = false;
            const unsigned bal = __ballot_sync(0xffffffffu, hit);
            if (bal) {                                          // warp-uniform
              if (hit) {
                const int pos = qn + __popc(bal & ((1u << lane) - 1));
                qrel[pos] = rel;
                qtf[pos] = __ldg(pt + u * 32 + lane);
                qw[pos] = w;
              }
              qn += __popc(bal);
              if (qn >= 32) drain(32);                          // qn <= 31 + 32 before, so one drain suffices
            }
          }
        }
        if (qn > 0) drain(qn);
      }
    }
  } else {
    for (int i = tid; i < HYB_TILE; i += HYB_THREADS) acc[i] = 0.0;      // vector-only: nothing but the knn clause
    if (tid == 0) s_go = __ldcg(a.gthr + q);
  }
  __syncthreads();
  if (!PRUNE || !pruned) {
    hybrid_tile_tail<false>(a, acc, q, tile, d0, d1, false, &s_go);
    return;
  }
  // ---- sparse tail: only marked docs can have a score; rank those at or above the bound ----
  static_assert(!PRUNE || HYB_SPARSE_CAP == (HYB_THREADS / 32) * HYB_QUEUE, "the candidate list reuses the warps' queues");
  uint32_t* c_key = reinterpret_cast<uint32_t*>(&s_qrel[0][0]);      // the queues are drained: reuse their memory
  uint32_t* c_doc = &s_qtf[0][0];
  if (a.knn_rows && tid < a.k) {            // the knn clause (see hybrid_tile_tail)
    const int64_t r = a.knn_rows[(size_t)q * a.k + tid];
    if (r >= 0) {
      const int64_t d = row_global_to_local(a.rmap, r);
      if (d >= d0 && d < d1 && !(FILTER && (d >= a.filter_rows || !a.row_filter[d])))
        acc[d - d0] = (double)(float)acc[d - d0] + (double)__fmul_rn(a.w_knn, a.knn_scores[(size_t)q * a.k + tid]);
    }
  }
  __syncthreads();
  if (tid < HYB_TILE / 32) {
    uint32_t wbits = s_bits[tid];
    while (wbits) {
      const int b = __ffs(wbits) - 1;
      wbits &= wbits - 1;
      const int slot = tid * 32 + b;
      const double v = acc[slot];
      if (v != 0.0) {
        const uint32_t key = ord32((float)v);
        if (key >= go) {
          const int pos = atomicAdd(&s_cn, 1);
          if (pos < HYB_SPARSE_CAP) { c_key[pos] = key; c_doc[pos] = (uint32_t)slot; }
        }
      }
    }
  }
  __syncthreads();
  const int n_c = s_cn;
  if (n_c > HYB_SPARSE_CAP) {               // a wall of docs above the bound: the dense select handles any count
    hybrid_tile_tail<false>(a, acc, q, tile, d0, d1, true);
    return;
  }
  double* xk = a.xkey + ((size_t)q * a.n_tiles + tile) * a.k;
  uint32_t* xr = a.xrow + ((size_t)q * a.n_tiles + tile) * a.k;
  for (int c = tid; c < n_c; c += HYB_THREADS) {
    const uint32_t mk = c_key[c], md = c_doc[c];
    int rank = c;
    if (n_c >= a.k) {
      rank = 0;
      for (int j = 0; j < n_c; ++j) rank += (c_key[j] > mk) || (c_key[j] == mk && c_doc[j] < md);
    }
    if (rank < a.k) {
      xk[rank] = (double)unord32(mk);
      xr[rank] = (uint32_t)(d0 + md);
      if (n_c >= a.k && rank == a.k - 1) atomicMax(a.gthr + q, mk);      // k rows of this tile score >= mk
    }
  }
  for (int i = min(n_c, a.k) + tid; i < a.k; i += HYB_THREADS) {
    xk[i] = neg_inf<double>();
    xr[i] = 0xffffffffu;
  }
}

// Per-query top-k of the tile lists.  The tiles left a lower bound of the query's k-th best key in gthr (the largest
// k-th key any tile found); entries below it cannot be in the top-k, and what is left -- normally k .. a few k entries --
// is ranked by counting.  Without a published bound (no tile had more than k matches) the k-th largest per-thread maximum
// serves.  A query with more than HSEL_CAP survivors (a wall of equal scores) is handed to the radix select.
#define HSEL_CAP 2048
__global__ void __launch_bounds__(1024) hybrid_select_kernel(const double* __restrict__ xkey,
                                                             const uint32_t* __restrict__ xrow, size_t entries, int k,
                                                             const uint32_t* __restrict__ gthr, RowMap rmap,
                                                             int64_t* __restrict__ out_rows,
                                                             float* __restrict__ out_scores,
                                                             double* __restrict__ out_keys, int* __restrict__ fallback) {
  __shared__ uint32_t ck[HSEL_CAP], cr[HSEL_CAP];
  __shared__ int s_n;
  const int tid = threadIdx.x, q = blockIdx.x;
  const double* key = xkey + (size_t)q * entries;
  const uint32_t* row = xrow + (size_t)q * entries;
  if (tid == 0) s_n = 0;
  uint32_t thr = gthr[q];
  if (thr == 0) {
    uint32_t mx = 0;
    for (size_t i = tid; i < entries; i += blockDim.x)
      if (row[i] != 0xffffffffu) mx = max(mx, ord32((float)key[i]));
    uint32_t bp = 0;
#pragma unroll 1
    for (int bit = 31; bit >= 0; --bit) {
      const uint32_t cand = bp | (1u << bit);
      if (__syncthreads_count(mx >= cand) >= k) bp = cand;
    }
    thr = bp;
  }
  __syncthreads();
  for (size_t i = tid; i < entries; i += blockDim.x) {
    const uint32_t r = row[i];
    if (r == 0xffffffffu) continue;
    const uint32_t o = ord32((float)key[i]);
    if (o >= thr) {
      const int pos = atomicAdd(&s_n, 1);
      if (pos < HSEL_CAP) { ck[pos] = o; cr[pos] = r; }
    }
  }
  __syncthreads();
  const int n = s_n;
  if (n > HSEL_CAP) {
    if (tid == 0) fallback[q] = 1;
    return;
  }
  if (tid == 0) fallback[q] = 0;
  for (int c = tid; c < n; c += blockDim.x) {
    const uint32_t mk = ck[c], mr = cr[c];
    int rank = 0;
    for (int j = 0; j < n; ++j) rank += (ck[j] > mk) || (ck[j] == mk && cr[j] < mr);
    if (rank < k) {
      const size_t o = (size_t)q * k + rank;
      const float v = unord32(mk);
      out_rows[o] = row_local_to_global(rmap, (int64_t)mr);
      out_scores[o] = v;
      if (out_keys) out_keys[o] = (double)v;
    }
  }
  for (int r = n + tid; r < k; r += blockDim.x) {
    const size_t o = (size_t)q * k + r;
    out_rows[o] = -1;
    out_scores[o] = 0.f;
    if (out_keys) out_keys[o] = 0.0;
  }
}

int launch_select_batch(rass_engine* h, size_t entries, int B, int k, int64_t* out_rows, float* out_scores,
                        double* out_keys, cudaStream_t st, const int* only_if);

static int ensure_hybrid_workspace(rass_engine* h, size_t n_terms_cap, int B) {
  Bm25State& b = h->bm25;
  if (n_terms_cap > b.qt_cap || (size_t)B + 1 > b.qt_q_cap) {
    CUDA_TRY(h, cudaStreamSynchronize(eng_stream(h)));
    const size_t tc = std::max<size_t>(n_terms_cap * 2, 1024), qc = std::max<size_t>((size_t)B * 2 + 2, 256);
    // one pinned + one device block:
    // [t_lo i64 x tc][t_len u32 x tc][t_w f32 x tc][t_row i32 x tc][t_bound f32 x tc][indptr i32 x qc][t_field u8 x tc]
    // [t_flag u8 x tc]
    const size_t bytes = tc * (8 + 4 + 4 + 4 + 4 + 1 + 1) + qc * 4;
    cudaFree(b.hyb_gthr); b.hyb_gthr = nullptr;
    CUDA_TRY(h, cudaMalloc(&b.hyb_gthr, qc * sizeof(uint32_t)));
    cudaFree(b.sel_fallback); b.sel_fallback = nullptr;
    CUDA_TRY(h, cudaMalloc(&b.sel_fallback, qc * sizeof(int)));
    cudaFreeHost(b.qt_host); b.qt_host = nullptr;
    cudaFree(b.qt_dev); b.qt_dev = nullptr;
    CUDA_TRY(h, cudaMallocHost(&b.qt_host, bytes));
    CUDA_TRY(h, cudaMalloc(&b.qt_dev, bytes));
    b.qt_cap = tc;
    b.qt_q_cap = qc;
    b.qt_bytes = bytes;
  }
  return RASS_OK;
}

// qweights == null: weight of a term = float(w_text) * idf(term); otherwise the caller's per-term weights
// (fuzzy expansions carry their own boost and blended idf)
// Row-sharded corpora fuse against the GLOBAL k nearest (all-gathered and merged by the caller) and leave their local
// top-k on the device for the next exchange (HybridExt, common.cuh).
// The query terms of a batch in the layout the text kernels read (one pinned + one device block, see
// ensure_hybrid_workspace): posting ranges, float(boost) * idf weights (or the caller's), structure flags, MaxScore bounds;
// plus what the host decides from them -- whether the batch needs the multi-clause kernel, and whether every query's
// clause sums are exact in double in any order.
int stage_hybrid_terms(rass_engine* h, int B, const int32_t* qterm_indptr, const int32_t* qterms, const float* qweights,
                       const uint8_t* qflags, float w_text, HybridTerms* out, cudaStream_t st) {
  Bm25State& b = h->bm25;
  int rc;
  size_t n_terms = 0;
  bool multi = false;
  static const bool force_ordered = getenv("RASS_DEBUG_HYBRID_ORDERED") != nullptr;   // A/B and test switch
  bool order_free = !force_ordered && !h->bm25.force_ordered;
  int64_t postings = 0;
  {
    if ((rc = ensure_hybrid_workspace(h, (size_t)(qterm_indptr[B] - qterm_indptr[0]), B))) return rc;
    unsigned char* base = b.qt_host;
    int64_t* t_lo = reinterpret_cast<int64_t*>(base);
    uint32_t* t_len = reinterpret_cast<uint32_t*>(base + b.qt_cap * 8);
    float* t_w = reinterpret_cast<float*>(base + b.qt_cap * 12);
    int32_t* t_row = reinterpret_cast<int32_t*>(base + b.qt_cap * 16);
    float* t_bound = reinterpret_cast<float*>(base + b.qt_cap * 20);
    int32_t* indptr = reinterpret_cast<int32_t*>(base + b.qt_cap * 24);
    uint8_t* t_field = base + b.qt_cap * 24 + b.qt_q_cap * 4;
    uint8_t* t_flag = t_field + b.qt_cap;
    std::vector<std::pair<float, size_t>> by_bound;
    const float bo = w_text;
    for (int q = 0; q < B; ++q) {
      indptr[q] = (int32_t)n_terms;
      int in_query = 0;
      // order-free check (hybrid_tile_fast_kernel): sum of the largest scores, smallest score, one field
      double q_sum_max = 0.0;
      float q_min = INFINITY;
      int q_field = -1;
      bool q_ok = true;
      for (int32_t j = qterm_indptr[q]; j < qterm_indptr[q + 1]; ++j) {
        const int32_t t = qterms[j];
        const uint8_t fl = qflags ? qflags[j] : 0;
        const int64_t lo = (t < 0 || t >= b.V) ? 0 : b.indptr_host[(size_t)t];
        const int64_t len = (t < 0 || t >= b.V) ? 0 : b.indptr_host[(size_t)t + 1] - lo;
        if (len == 0) {
          // a dropped term hands its group / clause end marks to the last kept term of the query
          if (fl && in_query > 0) {
            if ((fl & ~t_flag[n_terms - 1]) && j + 1 < qterm_indptr[q + 1]) multi = true;
            t_flag[n_terms - 1] |= fl;
          }
          continue;
        }
        if (++in_query > BM25_MAX_TERMS) return rass_fail(h, RASS_E_INVALID, "more than %d query terms", BM25_MAX_TERMS);
        t_lo[n_terms] = lo;
        t_len[n_terms] = (uint32_t)len;
        volatile float w = bo * b.idf_host[(size_t)t];
        t_w[n_terms] = qweights ? qweights[j] : w;
        t_row[n_terms] = b.table_row_host[(size_t)t];
        t_field[n_terms] = b.term_field_host[(size_t)t];
        t_flag[n_terms] = fl;
        if (fl && j + 1 < qterm_indptr[q + 1]) multi = true;     // a group or clause ends before the query does
        {
          volatile float wq = t_w[n_terms], one = 1.0f;
          volatile float lo_d = one + b.xmin_host[(size_t)t], hi_d = one + b.xmax_host[(size_t)t];
          volatile float lo_q = wq / lo_d, hi_q = wq / hi_d;
          volatile float s_lo = wq - lo_q, s_hi = wq - hi_q;
          if (s_hi > 0.f) {                       // a term whose scores are all <= 0 never adds anything
            if (!(s_lo > 0.f)) q_ok = false;
            q_sum_max += (double)s_hi;
            q_min = std::min(q_min, (float)s_lo);
          }
          t_bound[n_terms] = s_hi > 0.f ? (float)s_hi : 0.f;     // the term's largest score; summed below
          if (q_field < 0) q_field = t_field[n_terms];
          else if (q_field != t_field[n_terms]) q_ok = false;
        }
        postings += len;
        ++n_terms;
      }
      if (q_ok && q_sum_max > 0.0) {
        // every addend is a multiple of 2^(ilogb(q_min) - 23); every partial sum is < 2^(ilogb(q_sum_max) + 1)
        if ((ilogb(q_sum_max) + 1) - (ilogb((double)q_min) - 23) > 53) q_ok = false;
      }
      if (!q_ok) order_free = false;
      // MaxScore bounds: terms by ascending largest score; t_bound = the sum up to and including the term, rounded UP
      // to float -- no doc matching only those terms scores more (its float score is the rounded sum of smaller addends)
      by_bound.clear();
      for (size_t j = (size_t)indptr[q]; j < n_terms; ++j) by_bound.emplace_back(t_bound[j], j);
      std::sort(by_bound.begin(), by_bound.end());
      double cum = 0.0;
      for (const auto& e : by_bound) {
        cum += (double)e.first;
        float f = (float)cum;
        if ((double)f < cum) f = nextafterf(f, INFINITY);
        t_bound[e.second] = f;
      }
    }
    indptr[B] = (int32_t)n_terms;
    CUDA_TRY(h, cudaMemcpyAsync(b.qt_dev, b.qt_host, b.qt_bytes, cudaMemcpyHostToDevice, st));
  }
  unsigned char* base = b.qt_dev;
  out->t_lo = reinterpret_cast<const int64_t*>(base);
  out->t_len = reinterpret_cast<const uint32_t*>(base + b.qt_cap * 8);
  out->t_w = reinterpret_cast<const float*>(base + b.qt_cap * 12);
  out->t_row = reinterpret_cast<const int32_t*>(base + b.qt_cap * 16);
  out->t_bound = reinterpret_cast<const float*>(base + b.qt_cap * 20);
  out->qt_indptr = reinterpret_cast<const int32_t*>(base + b.qt_cap * 24);
  out->t_field = base + b.qt_cap * 24 + b.qt_q_cap * 4;
  out->t_flag = out->t_field + b.qt_cap;
  out->multi = multi;
  out->order_free = order_free;
  out->n_terms = n_terms;
  out->postings = postings;
  return RASS_OK;
}

// qflags (nullable): per term, bit 0 = last term of its field group, bit 1 = last term of its clause; the clause score is
// the maximum over its field groups (multi_match best_fields), the query's text score the sum over clauses.
int hybrid_core(rass_engine* h, const float* q_host, int B, const int32_t* qterm_indptr, const int32_t* qterms,
                const float* qweights, const uint8_t* qflags, float w_text, float w_knn, int k,
                int64_t* out_rows, float* out_scores, rass_stats* stats, const HybridExt* ext) {
  if (!h) return RASS_E_INVALID;
  cudaSetDevice(h->device);
  if (B < 1 || (!ext && (!out_rows || !out_scores))) return rass_fail(h, RASS_E_INVALID, "bad arguments");
  if (k < 1 || k > RASS_MAX_K) return rass_fail(h, RASS_E_INVALID, "k must be in [1, %d], got %d", RASS_MAX_K, k);
  if (!q_host && !qterm_indptr && !(ext && ext->knn_rows_dev))
    return rass_fail(h, RASS_E_INVALID, "neither a vector nor a text clause");
  Bm25State& b = h->bm25;
  if (qterm_indptr && (!b.built || !qterms)) return rass_fail(h, RASS_E_INVALID, "text clause without rass_bm25_build");
  cudaStream_t st = eng_stream(h);
  int rc;
  const size_t n_out = (size_t)B * k;
  if ((rc = ensure_out_workspace(h, 2 * n_out))) return rc;
  rass_stats s;
  memset(&s, 0, sizeof(s));
  s.n_queries = B;
  // 1. the knn clause: exact top-k per query (results stay on the device in the second half of the staging)
  const int64_t* knn_rows = h->out_rows + n_out;
  const float* knn_scores = h->out_scores + n_out;
  bool have_vec = q_host != nullptr && h->n_rows > 0;
  if (ext && ext->knn_rows_dev) {
    knn_rows = ext->knn_rows_dev;
    knn_scores = ext->knn_scores_dev;
    have_vec = true;
  } else if (have_vec) {
    float* q_dev = nullptr;
    if ((rc = stage_queries(h, q_host, B, &q_dev))) return rc;
    if ((rc = search_core(h, q_dev, B, k, h->out_rows + n_out, h->out_scores + n_out, nullptr, &s))) return rc;
  }
  // 2. the query terms: posting ranges and float(boost) * idf weights, in query order
  const bool have_text = qterm_indptr != nullptr;
  HybridTerms ta;
  memset(&ta, 0, sizeof(ta));
  ta.order_free = true;
  if (have_text && (rc = stage_hybrid_terms(h, B, qterm_indptr, qterms, qweights, qflags, w_text, &ta, st))) return rc;
  const bool multi = ta.multi;
  const bool order_free = ta.order_free;
  s.bytes_streamed += ta.postings * 6;
  // 3. one fused kernel over (tile, query), then the per-query top-k of the tile lists
  const int64_t n_docs = std::max<int64_t>(std::max<int64_t>(b.built ? b.N : 0, h->n_rows), 1);
  const int n_tiles = (int)((n_docs + HYB_TILE - 1) / HYB_TILE);
  const size_t entries = (size_t)n_tiles * k;
  if ((rc = ensure_xlist_workspace(h, (entries * B + RASS_EXACT_NQ - 1) / RASS_EXACT_NQ))) return rc;
  cudaEvent_t e0 = h->ev[0], e1 = h->ev[3];
  CUDA_TRY(h, cudaEventRecord(e0, st));
  HybridArgs a;
  memset(&a, 0, sizeof(a));
  a.doc = b.doc; a.tf = b.tf; a.xq = b.xq; a.norm = b.norm; a.inv = b.inv_dev; a.tile_off = b.tile_off;
  if (have_text) {
    a.t_lo = ta.t_lo; a.t_len = ta.t_len; a.t_w = ta.t_w; a.t_row = ta.t_row;
    // MaxScore marks are opt-in (RASS_OPT_HYBRID_MAXSCORE / RASS_HYBRID_MAXSCORE=1): on the cfg4 corpus they remove 88 % of
    // the scoring work but add a barrier-separated phase to a CTA that is latency-bound, not work-bound, and measure
    // 10 % slower (1.69 ms against 1.53 ms per 64-query batch at 5M docs, profiles/r2_hybrid_kernel_ncu.md)
    static const bool env_prune = getenv("RASS_HYBRID_MAXSCORE") != nullptr;
    a.t_bound = (env_prune || h->bm25.maxscore) ? ta.t_bound : nullptr;
    a.qt_indptr = ta.qt_indptr; a.t_field = ta.t_field; a.t_flag = ta.t_flag;
  }
  a.norm_rows = b.N;
  a.knn_rows = have_vec ? knn_rows : nullptr;
  a.knn_scores = knn_scores;
  a.row_filter = h->row_filter;
  a.filter_rows = h->row_filter_rows;
  a.rmap = h->rmap;
  a.n_docs = n_docs;
  a.n_tiles = n_tiles;
  a.table_tiles = b.built ? b.n_tiles : 0;
  a.k = k;
  a.w_knn = w_knn;
  a.xkey = h->xlist_key;
  a.xrow = h->xlist_row;
  if ((rc = ensure_hybrid_workspace(h, 0, B))) return rc;          // vector-only calls have not sized it yet
  a.gthr = b.hyb_gthr;
  CUDA_TRY(h, cudaMemsetAsync(b.hyb_gthr, 0, (size_t)B * sizeof(uint32_t), st));
  const size_t smem_single = (size_t)HYB_TILE * 8, smem_multi = (size_t)HYB_TILE * (8 + 8 + 4);
  CUDA_TRY(h, cudaFuncSetAttribute(hybrid_tile_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_multi));
  if (a.n_tiles > 65535) return rass_fail(h, RASS_E_UNSUPPORTED, "more than 65535 tiles of %d documents", HYB_TILE);
  const bool fast = order_free && !multi;
  if (fast) s.path |= RASS_PATH_HYBRID_ORDER_FREE;
  {
    // grid = (queries, tiles): queries are the fast index, so the CTAs in flight cover a few tiles of every query and
    // a query's cross-tile pruning bound exists after its first tiles
    const dim3 grid((unsigned)B, (unsigned)a.n_tiles);
    if (multi) hybrid_tile_kernel<true><<<grid, HYB_THREADS, smem_multi, st>>>(a);
    else if (fast && a.t_bound) {
      if (a.row_filter) hybrid_tile_fast_kernel<true, true><<<grid, HYB_THREADS, 0, st>>>(a);
      else hybrid_tile_fast_kernel<false, true><<<grid, HYB_THREADS, 0, st>>>(a);
    } else if (fast) {
      if (a.row_filter) hybrid_tile_fast_kernel<true, false><<<grid, HYB_THREADS, 0, st>>>(a);
      else hybrid_tile_fast_kernel<false, false><<<grid, HYB_THREADS, 0, st>>>(a);
    }
    else hybrid_tile_kernel<false><<<grid, HYB_THREADS, smem_single, st>>>(a);
    CUDA_TRY(h, cudaGetLastError());
    s.launches++;
  }
  {
    int64_t* o_rows = ext ? ext->out_rows_dev : h->out_rows;
    float* o_scores = ext ? ext->out_scores_dev : h->out_scores;
    double* o_keys = ext ? ext->out_keys_dev : nullptr;
    hybrid_select_kernel<<<B, 1024, 0, st>>>(h->xlist_key, h->xlist_row, (size_t)a.n_tiles * k, k, b.hyb_gthr,
                                             h->rmap, o_rows, o_scores, o_keys, b.sel_fallback);
    CUDA_TRY(h, cudaGetLastError());
    if ((rc = launch_select_batch(h, (size_t)a.n_tiles * k, B, k, o_rows, o_scores, o_keys, st, b.sel_fallback)))
      return rc;
    s.launches += 2;
  }
  CUDA_TRY(h, cudaEventRecord(e1, st));
  if (!ext) {
    CUDA_TRY(h, cudaMemcpyAsync(h->out_rows_host, h->out_rows, n_out * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaMemcpyAsync(h->out_scores_host, h->out_scores, n_out * 4, cudaMemcpyDeviceToHost, st));
  }
  CUDA_TRY(h, cudaStreamSynchronize(st));
  if (!ext) {
    memcpy(out_rows, h->out_rows_host, n_out * 8);
    memcpy(out_scores, h->out_scores_host, n_out * 4);
  }
  float ms = 0.f;
  CUDA_TRY(h, cudaEventElapsedTime(&ms, e0, e1));
  s.finish_ms += ms;
  s.total_ms += ms;
  h->last_stats = s;
  if (stats) *stats = s;
  return RASS_OK;
}

extern "C" int rass_search_hybrid(rass_engine* h, const float* q_host, int B, const int32_t* qterm_indptr,
                                  const int32_t* qterms, float w_text, float w_knn, int k, int64_t* out_rows,
                                  float* out_scores, rass_stats* stats) {
  SHARDED(h, sharded_search_hybrid(h, q_host, B, qterm_indptr, qterms, nullptr, nullptr, w_text, w_knn, k, out_rows, out_scores, stats));
  return hybrid_core(h, q_host, B, qterm_indptr, qterms, nullptr, nullptr, w_text, w_knn, k, out_rows, out_scores,
                     stats);
}

extern "C" int rass_search_hybrid_weighted(rass_engine* h, const float* q_host, int B, const int32_t* qterm_indptr,
                                           const int32_t* qterms, const float* qweights, const uint8_t* qflags,
                                           float w_knn, int k, int64_t* out_rows, float* out_scores,
                                           rass_stats* stats) {
  SHARDED(h, (qterm_indptr && !qweights) ? rass_fail(h, RASS_E_INVALID, "null weights") : sharded_search_hybrid(h, q_host, B, qterm_indptr, qterms, qweights, qflags, 0.f, w_knn, k, out_rows, out_scores, stats));
  if (h && qterm_indptr && !qweights) return rass_fail(h, RASS_E_INVALID, "null weights");
  return hybrid_core(h, q_host, B, qterm_indptr, qterms, qweights, qflags, 0.f, w_knn, k, out_rows, out_scores,
                     stats);
}

extern "C" int rass_fuse_hybrid_dev(rass_engine* h, int B, const int32_t* qterm_indptr, const int32_t* qterms,
                                    const float* qweights, const uint8_t* qflags, float w_text,
                                    const int64_t* knn_rows_dev, const float* knn_scores_dev, float w_knn, int k,
                                    int64_t* out_rows_dev, float* out_scores_dev, double* out_keys_dev) {
  SHARDED(h, rass_fail(h, RASS_E_UNSUPPORTED, "rass_fuse_hybrid_dev is the per-shard step; a sharded handle fuses through rass_search_hybrid / rass_fuse_hybrid"));
  if (!h) return RASS_E_INVALID;
  if (!out_rows_dev || !out_scores_dev || (knn_rows_dev && !knn_scores_dev))
    return rass_fail(h, RASS_E_INVALID, "null buffer");
  HybridExt ext = {knn_rows_dev, knn_scores_dev, out_rows_dev, out_scores_dev, out_keys_dev};
  return hybrid_core(h, nullptr, B, qterm_indptr, qterms, qweights, qflags, w_text, w_knn, k, nullptr, nullptr, nullptr,
                     &ext);
}

// host-pointer flavour: the k nearest come from an earlier rass_search_knn (possibly shared with other requests by a
// request coalescer), the text clauses and the bool.filter are this request's own
extern "C" int rass_fuse_hybrid(rass_engine* h, int B, const int32_t* qterm_indptr, const int32_t* qterms,
                                const float* qweights, const uint8_t* qflags, float w_text,
                                const int64_t* knn_rows_host, const float* knn_scores_host, float w_knn, int k,
                                int64_t* out_rows, float* out_scores) {
  SHARDED(h, sharded_fuse_hybrid(h, B, qterm_indptr, qterms, qweights, qflags, w_text, knn_rows_host, knn_scores_host, w_knn, k, out_rows, out_scores));
  if (!h) return RASS_E_INVALID;
  cudaSetDevice(h->device);
  if (B < 1 || k < 1 || k > RASS_MAX_K || !out_rows || !out_scores || (knn_rows_host && !knn_scores_host))
    return rass_fail(h, RASS_E_INVALID, "bad arguments");
  cudaStream_t st = eng_stream(h);
  int rc;
  const size_t n_out = (size_t)B * k;
  if ((rc = ensure_out_workspace(h, 2 * n_out))) return rc;
  // second half of the result staging = the external knn list, first half = this call's results
  int64_t* knn_rows_dev = h->out_rows + n_out;
  float* knn_scores_dev = h->out_scores + n_out;
  if (knn_rows_host) {
    memcpy(h->out_rows_host + n_out, knn_rows_host, n_out * 8);
    memcpy(h->out_scores_host + n_out, knn_scores_host, n_out * 4);
    CUDA_TRY(h, cudaMemcpyAsync(knn_rows_dev, h->out_rows_host + n_out, n_out * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(h, cudaMemcpyAsync(knn_scores_dev, h->out_scores_host + n_out, n_out * 4, cudaMemcpyHostToDevice, st));
  }
  HybridExt ext = {knn_rows_host ? knn_rows_dev : nullptr, knn_scores_dev, h->out_rows, h->out_scores, nullptr};
  if ((rc = hybrid_core(h, nullptr, B, qterm_indptr, qterms, qweights, qflags, w_text, w_knn, k, nullptr, nullptr, nullptr,
                        &ext)))
    return rc;
  CUDA_TRY(h, cudaMemcpyAsync(h->out_rows_host, h->out_rows, n_out * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaMemcpyAsync(h->out_scores_host, h->out_scores, n_out * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  memcpy(out_rows, h->out_rows_host, n_out * 8);
  memcpy(out_scores, h->out_scores_host, n_out * 4);
  return RASS_OK;
}

// ---- fuzziness: AUTO -- edit-distance scan of the term dictionary -------------------------------------------
// Lucene's FuzzyQuery measures edits in Unicode code points, so the dictionary is kept on the device as code points
// (decoded once from the UTF-8 the host hands over) and so is the query token.
#define FUZZY_MAX_TOKEN 64

struct FuzzyToken {
  int len;
  uint32_t c[FUZZY_MAX_TOKEN];
};

// UTF-8 -> code points; false on a malformed sequence
static bool utf8_decode(const unsigned char* p, size_t n, std::vector<uint32_t>& out) {
  size_t i = 0;
  while (i < n) {
    const unsigned char b = p[i];
    uint32_t cp;
    int extra;
    if (b < 0x80) { cp = b; extra = 0; }
    else if ((b & 0xe0) == 0xc0) { cp = b & 0x1f; extra = 1; }
    else if ((b & 0xf0) == 0xe0) { cp = b & 0x0f; extra = 2; }
    else if ((b & 0xf8) == 0xf0) { cp = b & 0x07; extra = 3; }
    else return false;
    for (int e = 1; e <= extra; ++e) {
      if (i + e >= n || (p[i + e] & 0xc0) != 0x80) return false;
      cp = (cp << 6) | (p[i + e] & 0x3f);
    }
    out.push_back(cp);
    i += (size_t)extra + 1;
  }
  return true;
}

// One thread per dictionary term: optimal-string-alignment distance (insert / delete / substitute / adjacent swap)
// to the query token, cut off at max_edits; matches are appended to (out_terms, out_edits) in no particular order.
__global__ void __launch_bounds__(256) fuzzy_scan_kernel(const uint32_t* __restrict__ blob,
                                                         const int64_t* __restrict__ off, int64_t t_lo, int64_t V,
                                                         const __grid_constant__ FuzzyToken tok, int max_edits,
                                                         int32_t* __restrict__ out_terms,
                                                         int32_t* __restrict__ out_edits, int* __restrict__ out_n) {
  const int64_t t = t_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= V) return;
  const int64_t o = off[t];
  const int lt = (int)(off[t + 1] - o), m = tok.len;
  if (lt == 0 || abs(lt - m) > max_edits) return;
  const uint32_t* term = blob + o;
  // rows of the DP over the token (columns 0..m); row i = prefix of the term of length i
  unsigned char prev2[FUZZY_MAX_TOKEN + 1], prev[FUZZY_MAX_TOKEN + 1], cur[FUZZY_MAX_TOKEN + 1];
  for (int j = 0; j <= m; ++j) prev[j] = (unsigned char)j;
  for (int i = 1; i <= lt; ++i) {
    const uint32_t ci = term[i - 1];
    cur[0] = (unsigned char)min(i, 255);
    int row_min = cur[0];
    for (int j = 1; j <= m; ++j) {
      const uint32_t cj = tok.c[j - 1];
      int v = min(min(prev[j] + 1, cur[j - 1] + 1), prev[j - 1] + (ci != cj));
      if (i > 1 && j > 1 && ci == tok.c[j - 2] && term[i - 2] == cj) v = min(v, prev2[j - 2] + 1);
      cur[j] = (unsigned char)min(v, 255);
      row_min = min(row_min, v);
    }
    if (row_min > max_edits) return;      // the distance can only grow from here
    for (int j = 0; j <= m; ++j) { prev2[j] = prev[j]; prev[j] = cur[j]; }
  }
  const int ed = prev[m];
  if (ed > max_edits) return;
  const int pos = atomicAdd(out_n, 1);
  out_terms[pos] = (int32_t)t;
  out_edits[pos] = ed;
}

extern "C" int rass_text_set_vocab(rass_engine* h, const char* blob, const int64_t* offsets, int64_t V) {
  SHARDED(h, rass_text_set_vocab(sharded_first(h), blob, offsets, V));
  if (!h) return RASS_E_INVALID;
  cudaSetDevice(h->device);
  if (V < 0 || !offsets || (offsets[V] > 0 && !blob)) return rass_fail(h, RASS_E_INVALID, "bad vocabulary");
  Bm25State& b = h->bm25;
  CUDA_TRY(h, cudaStreamSynchronize(eng_stream(h)));
  std::vector<uint32_t> cps;
  std::vector<int64_t> cp_off((size_t)V + 1, 0);
  cps.reserve((size_t)offsets[V]);
  for (int64_t t = 0; t < V; ++t) {
    if (offsets[t + 1] < offsets[t]) return rass_fail(h, RASS_E_INVALID, "vocabulary offsets must not decrease");
    if (!utf8_decode(reinterpret_cast<const unsigned char*>(blob) + offsets[t], (size_t)(offsets[t + 1] - offsets[t]), cps))
      return rass_fail(h, RASS_E_INVALID, "term %lld is not valid UTF-8", (long long)t);
    cp_off[(size_t)t + 1] = (int64_t)cps.size();
  }
  int rc;
  if ((rc = upload(h, &b.vocab_blob, cps.data(), cps.size()))) return rc;
  if ((rc = upload(h, &b.vocab_off, cp_off.data(), (size_t)V + 1))) return rc;
  cudaFree(b.fz_terms); b.fz_terms = nullptr;
  cudaFree(b.fz_edits); b.fz_edits = nullptr;
  CUDA_TRY(h, cudaMalloc(&b.fz_terms, std::max<size_t>((size_t)V, 1) * sizeof(int32_t)));
  CUDA_TRY(h, cudaMalloc(&b.fz_edits, std::max<size_t>((size_t)V, 1) * sizeof(int32_t)));
  if (!b.fz_n) CUDA_TRY(h, cudaMalloc(&b.fz_n, sizeof(int)));
  b.vocab_V = V;
  return RASS_OK;
}

extern "C" int rass_fuzzy_expand(rass_engine* h, const char* token, int token_len, int max_edits, int64_t term_lo,
                                 int64_t term_hi, int64_t max_out, int32_t* out_terms, int32_t* out_edits,
                                 int64_t* out_n) {
  SHARDED(h, rass_fuzzy_expand(sharded_first(h), token, token_len, max_edits, term_lo, term_hi, max_out, out_terms, out_edits, out_n));
  if (!h) return RASS_E_INVALID;
  cudaSetDevice(h->device);
  Bm25State& b = h->bm25;
  if (!token || token_len < 1 || max_edits < 0 || max_edits > 2 || !out_n || (max_out > 0 && (!out_terms || !out_edits)))
    return rass_fail(h, RASS_E_INVALID, "bad arguments");
  if (!b.vocab_off) return rass_fail(h, RASS_E_INVALID, "rass_fuzzy_expand before rass_text_set_vocab");
  std::vector<uint32_t> cps;
  if (!utf8_decode(reinterpret_cast<const unsigned char*>(token), (size_t)token_len, cps))
    return rass_fail(h, RASS_E_INVALID, "the token is not valid UTF-8");
  if (cps.size() > FUZZY_MAX_TOKEN) return rass_fail(h, RASS_E_INVALID, "token longer than %d code points", FUZZY_MAX_TOKEN);
  *out_n = 0;
  if (term_hi < 0 || term_hi > b.vocab_V) term_hi = b.vocab_V;
  if (term_lo < 0) term_lo = 0;
  if (term_lo >= term_hi) return RASS_OK;
  FuzzyToken tok;
  memset(&tok, 0, sizeof(tok));
  tok.len = (int)cps.size();
  memcpy(tok.c, cps.data(), cps.size() * sizeof(uint32_t));
  cudaStream_t st = eng_stream(h);
  CUDA_TRY(h, cudaMemsetAsync(b.fz_n, 0, sizeof(int), st));
  fuzzy_scan_kernel<<<(unsigned)((term_hi - term_lo + 255) / 256), 256, 0, st>>>(
      b.vocab_blob, b.vocab_off, term_lo, term_hi, tok, max_edits, b.fz_terms, b.fz_edits, b.fz_n);
  CUDA_TRY(h, cudaGetLastError());
  int n = 0;
  CUDA_TRY(h, cudaMemcpyAsync(&n, b.fz_n, sizeof(int), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  *out_n = n;
  const int64_t m = std::min<int64_t>(n, max_out);
  if (m > 0) {
    CUDA_TRY(h, cudaMemcpyAsync(out_terms, b.fz_terms, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaMemcpyAsync(out_edits, b.fz_edits, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
  }
  return RASS_OK;
}
