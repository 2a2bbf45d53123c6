// Candidate merge + exact fp64 rerank + certificate, the fp64 full scan it falls back to, and the shard merge.
//
// These make the final top-k identical to the oracle's definition (oracle/knn.py: fp64-accumulated key of the
// stored values, ranking (key desc, row asc)), which is the exact form of the search the reference delegates to
// OpenSearch's approximate HNSW (app/main.py:1538-1553), and emit OpenSearch's score translation 1/(2 - cos).
//
// Certificate (per query).  The scan kernels leave a pool of (approximate key, row) entries in segments, and a
// bound thr_s per segment such that every row the segment's owner saw and did not keep has approximate key
// <= thr_s.  With t = max_s thr_s and eps >= |approximate key - exact key| for every row:
//   * b' = a lower bound of the k-th best approximate key in the pool, so the exact k-th best s_k >= b' - eps,
//   * every pool entry with approximate key < b' - 2 eps has exact key < s_k and cannot be in the top-k,
//   * if t + eps < s_k no row outside the pool can be in the top-k either.
// So re-ranking the entries >= b' - 2 eps in fp64 gives the exact top-k whenever t + eps < s_k holds; queries
// for which it does not are flagged and re-scanned exactly.
#include "common.cuh"

// ---------------------------------------------------------------------------------------------
// finish: one CTA per query of the group
// ---------------------------------------------------------------------------------------------
struct FinishArgs {
  const float* pool_key;
  const uint32_t* pool_row;
  const float* pool_thr;
  const int* pool_cnt;      // null: every slot of a segment is an entry unless its row is 0xffffffff
  size_t pool_entries;      // per query
  int n_segs, seg_size;
  const float* x32;
  const __nv_bfloat16* x16;
  const double* norm64;
  const float* q_raw;
  const double* q_norm;
  const float* q_rho;       // null when the scan used the fp32 query
  const StoreScalars* store;   // rho_x, rho_x8, max_xnorm
  int int8;                 // the scan read the int8 shadow: rho_x8 bounds its rows (q_rho is then the int8 query's)
  SearchScalars* scal;
  int* flagged;
  int dim_pad, metric, k, g0;
  float acc_eps;
  RowMap rmap;
  int64_t* out_rows;
  float* out_scores;
  double* out_keys;
  int64_t* flag_out;        // null, or where the launch leaves scal->flagged_n once all its CTAs are through
};

template <bool BF16_ROWS>
__global__ void __launch_bounds__(RASS_FINISH_THREADS, 1) finish_kernel(FinishArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* qs = reinterpret_cast<float*>(smem_raw);                          // [dim_pad]
  double* ckey = reinterpret_cast<double*>(qs + a.dim_pad);                // [RASS_CAND_MAX]
  uint32_t* crow = reinterpret_cast<uint32_t*>(ckey + RASS_CAND_MAX);      // [RASS_CAND_MAX]
  __shared__ float s_red[32];
  __shared__ int s_redi[32];
  __shared__ float s_t;
  __shared__ int s_valid, s_ncand, s_have;
  __shared__ double s_sk;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slot = blockIdx.x;          // pool slot within the group
  const int q = a.g0 + slot;            // query id within the search
  const float* pk = a.pool_key + (size_t)slot * a.pool_entries;
  const uint32_t* pr = a.pool_row + (size_t)slot * a.pool_entries;

  for (int j = tid; j < a.dim_pad; j += blockDim.x) qs[j] = a.q_raw[(size_t)q * a.dim_pad + j];
  if (tid == 0) { s_ncand = 0; s_have = 0; }

  // phase 1: per-thread maximum of the valid entries (warp per segment, lanes over its entries),
  // t = max segment bound, number of valid entries
  float mx = neg_inf<float>();
  int nvalid = 0;
  for (int sgm = warp; sgm < a.n_segs; sgm += RASS_FINISH_THREADS / 32) {
    const int cnt = a.pool_cnt ? min(a.pool_cnt[(size_t)slot * a.n_segs + sgm], a.seg_size) : a.seg_size;
    for (int i = lane; i < cnt; i += 32) {
      const size_t o = (size_t)sgm * a.seg_size + i;
      if (a.pool_cnt || pr[o] != 0xffffffffu) {
        ++nvalid;
        mx = fmaxf(mx, pk[o]);
      }
    }
  }
  float t = neg_inf<float>();
  for (int s = tid; s < a.n_segs; s += blockDim.x) t = fmaxf(t, a.pool_thr[(size_t)slot * a.n_segs + s]);
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) {
    t = fmaxf(t, __shfl_xor_sync(0xffffffffu, t, m));
    nvalid += __shfl_xor_sync(0xffffffffu, nvalid, m);
  }
  if (lane == 0) { s_red[warp] = t; s_redi[warp] = nvalid; }
  __syncthreads();
  if (warp == 0) {
    float tt = s_red[lane];
    int nv = s_redi[lane];
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
      tt = fmaxf(tt, __shfl_xor_sync(0xffffffffu, tt, m));
      nv += __shfl_xor_sync(0xffffffffu, nv, m);
    }
    if (lane == 0) { s_t = tt; s_valid = nv; }
  }

  // phase 2: b' = k-th largest per-thread maximum (k distinct entries are >= it): MSB-first radix descent on the
  // order-preserving integer image, one __syncthreads_count per bit.  Threads without an entry hold 0.
  float bprime;
  {
    const uint32_t mine = mx > neg_inf<float>() ? ord32(mx) : 0u;
    uint32_t prefix = 0;
#pragma unroll 1
    for (int bit = 31; bit >= 0; --bit) {
      const uint32_t cand = prefix | (1u << bit);
      if (__syncthreads_count(mine >= cand) >= a.k) prefix = cand;
    }
    bprime = prefix > 0x007fffffu ? unord32(prefix) : neg_inf<float>();   // fewer than k holders -> take everything
  }

  float eps;
  {
    const float rho_x = a.int8 ? a.store->rho_x8 : (BF16_ROWS ? 0.f : a.store->rho_x);
    const float rho_q = a.q_rho ? a.q_rho[q] : 0.f;
    float e = rho_x * (1.f + rho_q) + rho_q + a.acc_eps;
    if (a.metric == RASS_METRIC_L2) {
      const float xm = a.store->max_xnorm;
      e = e * xm * (float)a.q_norm[q] * 1.0001f + 6.0e-8f * xm * xm;
    }
    eps = e * 1.0001f;
  }
  const float cutoff = bprime - 2.f * eps;   // -inf when fewer than k threads hold an entry

  // phase 3: collect the candidates
  for (int sgm = warp; sgm < a.n_segs; sgm += RASS_FINISH_THREADS / 32) {
    const int cnt = a.pool_cnt ? min(a.pool_cnt[(size_t)slot * a.n_segs + sgm], a.seg_size) : a.seg_size;
    for (int i = lane; i < cnt; i += 32) {
      const size_t o = (size_t)sgm * a.seg_size + i;
      if ((a.pool_cnt || pr[o] != 0xffffffffu) && pk[o] >= cutoff) {
        int pos = atomicAdd(&s_ncand, 1);
        if (pos < RASS_CAND_MAX) crow[pos] = pr[o];
      }
    }
  }
  __syncthreads();
  const int ncand_raw = s_ncand;
  const int ncand = min(ncand_raw, RASS_CAND_MAX);

  // phase 4: exact keys
  const double qn = a.q_norm[q];
  for (int c = warp; c < ncand; c += RASS_FINISH_THREADS / 32) {
    double key = exact_key_warp<BF16_ROWS>(a.x32, a.x16, a.norm64, crow[c], qs, qn, a.dim_pad, a.metric);
    if (lane == 0) ckey[c] = key;
  }
  __syncthreads();

  // phase 5: rank by counting, emit the top-k
  const int kk = a.k;
  for (int c = tid; c < ncand; c += blockDim.x) {
    const double key = ckey[c];
    const uint32_t row = crow[c];
    int rank = 0;
    for (int j = 0; j < ncand; ++j) rank += entry_better<double>(ckey[j], crow[j], key, row);
    if (rank < kk) {
      const size_t o = (size_t)q * kk + rank;
      a.out_rows[o] = row_local_to_global(a.rmap, (int64_t)row);
      a.out_scores[o] = score_from_key(key, a.metric);
      if (a.out_keys) a.out_keys[o] = a.metric == RASS_METRIC_COSINE ? key : -key;
      if (rank == kk - 1) { s_sk = key; s_have = 1; }
    }
  }
  for (int r = ncand + tid; r < kk; r += blockDim.x) {
    const size_t o = (size_t)q * kk + r;
    a.out_rows[o] = -1;
    a.out_scores[o] = 0.f;
    if (a.out_keys) a.out_keys[o] = 0.0;
  }
  __syncthreads();

  // phase 6: certificate
  if (tid == 0) {
    bool ok;
    const float tt = s_t;
    if (ncand_raw > RASS_CAND_MAX) {
      ok = false;
    } else if (!s_have) {
      // fewer than k candidates: exact only if nothing at all was excluded
      ok = (tt == neg_inf<float>()) && ncand == s_valid;
    } else if (tt == neg_inf<float>()) {
      ok = true;
    } else {
      // exact key of the k-th hit in the units of the scan key
      double sk = s_sk;
      if (a.metric == RASS_METRIC_L2) sk = 0.5 * (qn * qn + sk);   // sk = -(d^2); surrogate = (|q|^2 - d^2) / 2
      ok = (double)tt + (double)eps < sk;
    }
    if (ok) {
      atomicAdd(&a.scal->n_certified, 1);
    } else {
      int pos = atomicAdd(&a.scal->flagged_n, 1);
      a.flagged[pos] = q;
    }
    atomicMax(&a.scal->max_cand, ncand_raw);
    if (a.flag_out) {
      // the last CTA of the launch publishes the running count of uncertified queries (what a row-sharded caller
      // gathers with the candidates); a later launch of the same search overwrites it with the later count
      __threadfence();
      if (atomicAdd(&a.scal->finish_done, 1) == (int)gridDim.x - 1) {
        a.scal->finish_done = 0;
        *a.flag_out = (int64_t)atomicAdd(&a.scal->flagged_n, 0);
      }
    }
  }
}

static size_t finish_smem(int dim_pad) {
  return (size_t)dim_pad * 4 + RASS_CAND_MAX * 12;
}

int launch_finish(rass_engine* h, const SearchWs& ws, int g0, int ng, int k, int n_segs, int seg_size, bool has_cnt,
                  ScanOperands ops, int64_t* out_rows, float* out_scores, double* out_keys, cudaStream_t st,
                  int64_t* flag_out) {
  FinishArgs a;
  a.flag_out = flag_out;
  a.pool_key = ws.pool_key;
  a.pool_row = ws.pool_row;
  a.pool_thr = ws.pool_thr;
  a.pool_cnt = has_cnt ? ws.pool_cnt : nullptr;
  a.pool_entries = ws.pool_entries;
  a.n_segs = n_segs;
  a.seg_size = seg_size;
  a.x32 = h->x32;
  a.x16 = h->x16;
  a.norm64 = h->norm64;
  a.q_raw = ws.q_raw;
  a.q_norm = ws.q_norm;
  // acc_eps (below) also covers the int8 pass's fp32 combination s1 * acc1 + s2 * acc2 of exact integer dots: a few
  // roundings of 2^-24 relative, against dim_pad * 2^-23
  a.q_rho = ops == SCAN_INT8 ? ws.q_rho8 : (ops == SCAN_BF16 ? ws.q_rho : nullptr);
  a.int8 = ops == SCAN_INT8;
  a.store = h->store_scal;
  a.scal = ws.scal;
  a.flagged = ws.flagged;
  a.dim_pad = h->dim_pad;
  a.metric = h->metric;
  a.k = k;
  a.g0 = g0;
  a.acc_eps = acc_allowance(h->dim_pad);
  a.rmap = h->rmap;
  a.out_rows = out_rows;
  a.out_scores = out_scores;
  a.out_keys = out_keys;
  const size_t smem = finish_smem(h->dim_pad);
  if (h->flags & RASS_BF16_ONLY) {
    CUDA_TRY(h, cudaFuncSetAttribute(finish_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    finish_kernel<true><<<ng, RASS_FINISH_THREADS, smem, st>>>(a);
  } else {
    CUDA_TRY(h, cudaFuncSetAttribute(finish_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    finish_kernel<false><<<ng, RASS_FINISH_THREADS, smem, st>>>(a);
  }
  CUDA_TRY(h, cudaGetLastError());
  return RASS_OK;
}

// ---------------------------------------------------------------------------------------------
// exact fp64 scan: the definition, used for flagged queries, RASS_PATH_EXACT and the tests
// ---------------------------------------------------------------------------------------------
template <bool BF16_ROWS, int M>
__global__ void __launch_bounds__(RASS_WARPS_PER_CTA * 32) exact_scan_kernel(
    const float* __restrict__ x32, const __nv_bfloat16* __restrict__ x16, const double* __restrict__ norm64,
    const float* __restrict__ sb, const float* __restrict__ q_raw, const double* __restrict__ q_norm,
    const int* __restrict__ qids, int nq, int64_t n_rows, int dim_pad, int metric, double* __restrict__ xkey,
    uint32_t* __restrict__ xrow, size_t xlist_entries) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* qs = reinterpret_cast<float*>(smem_raw);   // [RASS_EXACT_NQ][dim_pad]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gw = blockIdx.x * RASS_WARPS_PER_CTA + warp;
  const int W = gridDim.x * RASS_WARPS_PER_CTA;
  for (int i = threadIdx.x; i < nq * dim_pad; i += blockDim.x)
    qs[i] = q_raw[(size_t)qids[i / dim_pad] * dim_pad + (i % dim_pad)];
  __syncthreads();
  double qn[RASS_EXACT_NQ];
  WarpTop<double, M> top[RASS_EXACT_NQ];
#pragma unroll
  for (int i = 0; i < RASS_EXACT_NQ; ++i) {
    top[i].init();
    qn[i] = i < nq ? q_norm[qids[i]] : 0.0;
  }
  for (int64_t row = gw; row < n_rows; row += W) {
    if (sb[row] == neg_inf<float>()) continue;   // tombstone
#pragma unroll
    for (int i = 0; i < RASS_EXACT_NQ; ++i) {
      if (i < nq) {
        double key = exact_key_warp<BF16_ROWS>(x32, x16, norm64, (uint32_t)row, qs + (size_t)i * dim_pad, qn[i],
                                               dim_pad, metric);
        if (top[i].admits_ascending(key)) top[i].insert(key, (uint32_t)row);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < RASS_EXACT_NQ; ++i) {
    if (i < nq) {
      const size_t base = (size_t)i * xlist_entries + (size_t)gw * (32 * M);
#pragma unroll
      for (int s = 0; s < M; ++s) {
        xkey[base + s * 32 + lane] = top[i].key[s];
        xrow[base + s * 32 + lane] = top[i].row[s];
      }
    }
  }
}

__device__ __forceinline__ uint64_t ord64(double d) {
  if (d == 0.0) d = 0.0;  // -0 -> +0
  uint64_t u = (uint64_t)__double_as_longlong(d);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ULL);
}

// One CTA per query: exact top-k of n (key, row) entries in the total order (key desc, row asc).  Rows are
// distinct, so the k-th entry T of that order is unique; a 12-byte radix select finds it, then the k entries
// >= T are ranked by counting.
__global__ void __launch_bounds__(1024, 1) exact_select_kernel(const double* __restrict__ xkey,
                                                               const uint32_t* __restrict__ xrow, size_t xlist_entries,
                                                               int n, int k, const int* __restrict__ qids, int q_fixed,
                                                               int raw_score, int metric,
                                                               RowMap rmap, int64_t* __restrict__ out_rows,
                                                               float* __restrict__ out_scores,
                                                               double* __restrict__ out_keys,
                                                               const int* __restrict__ only_if) {
  if (only_if && !only_if[blockIdx.x]) return;     // hybrid_select_kernel already ranked this query
  __shared__ int hist[256];
  __shared__ int s_bucket, s_remaining, s_nsel, s_nvalid;
  __shared__ double selk[RASS_MAX_K];
  __shared__ uint32_t selr[RASS_MAX_K];
  const int tid = threadIdx.x;
  const int q = qids ? qids[blockIdx.x] : q_fixed + (int)blockIdx.x;
  const double* key = xkey + (size_t)blockIdx.x * xlist_entries;
  const uint32_t* row = xrow + (size_t)blockIdx.x * xlist_entries;

  if (tid == 0) { s_nvalid = 0; s_nsel = 0; }
  __syncthreads();
  int nv = 0;
  for (int i = tid; i < n; i += blockDim.x) nv += row[i] != 0xffffffffu;
  if (nv) atomicAdd(&s_nvalid, nv);
  __syncthreads();
  const int kk = min(k, s_nvalid);

  // composite 96-bit key: (ord64(key), ~row); larger is better
  uint64_t pre_hi = 0, mask_hi = 0;
  uint32_t pre_lo = 0, mask_lo = 0;
  if (kk > 0) {
    if (tid == 0) s_remaining = kk;
    for (int byte = 11; byte >= 0; --byte) {
      for (int b = tid; b < 256; b += blockDim.x) hist[b] = 0;
      __syncthreads();
      for (int i = tid; i < n; i += blockDim.x) {
        const uint32_t r = row[i];
        if (r == 0xffffffffu) continue;
        const uint64_t hi = ord64(key[i]);
        const uint32_t lo = ~r;
        if ((hi & mask_hi) != pre_hi || (lo & mask_lo) != pre_lo) continue;
        const int b = byte >= 4 ? (int)((hi >> ((byte - 4) * 8)) & 255) : (int)((lo >> (byte * 8)) & 255);
        atomicAdd(&hist[b], 1);
      }
      __syncthreads();
      if (tid < 32) {
        // highest bucket whose suffix count reaches the remaining rank: lane L owns buckets [8L, 8L + 8)
        int loc[8], sum = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) { loc[i] = hist[8 * tid + i]; sum += loc[i]; }
        int suf = sum;
#pragma unroll
        for (int m = 1; m < 32; m <<= 1) {
          const int o = __shfl_down_sync(0xffffffffu, suf, m);
          if (tid + m < 32) suf += o;
        }
        const int rem = s_remaining, above = suf - sum;
        if (above < rem && rem <= above + sum) {
          int cum = above;
#pragma unroll
          for (int i = 7; i >= 0; --i) {
            if (cum + loc[i] >= rem) { s_bucket = 8 * tid + i; s_remaining = rem - cum; break; }
            cum += loc[i];
          }
        }
      }
      __syncthreads();
      const int b = s_bucket;
      if (byte >= 4) {
        pre_hi |= (uint64_t)b << ((byte - 4) * 8);
        mask_hi |= (uint64_t)255 << ((byte - 4) * 8);
      } else {
        pre_lo |= (uint32_t)b << (byte * 8);
        mask_lo |= (uint32_t)255 << (byte * 8);
      }
      __syncthreads();
    }
    // (pre_hi, pre_lo) is the k-th entry; gather everything >= it
    for (int i = tid; i < n; i += blockDim.x) {
      const uint32_t r = row[i];
      if (r == 0xffffffffu) continue;
      const uint64_t hi = ord64(key[i]);
      const uint32_t lo = ~r;
      if (hi > pre_hi || (hi == pre_hi && lo >= pre_lo)) {
        int pos = atomicAdd(&s_nsel, 1);
        if (pos < RASS_MAX_K) { selk[pos] = key[i]; selr[pos] = r; }
      }
    }
  }
  __syncthreads();
  const int nsel = min(s_nsel, RASS_MAX_K);
  for (int c = tid; c < nsel; c += blockDim.x) {
    int rank = 0;
    for (int j = 0; j < nsel; ++j) rank += entry_better<double>(selk[j], selr[j], selk[c], selr[c]);
    if (rank < k) {
      const size_t o = (size_t)q * k + rank;
      out_rows[o] = row_local_to_global(rmap, (int64_t)selr[c]);
      out_scores[o] = raw_score ? (float)selk[c] : score_from_key(selk[c], metric);
      if (out_keys) out_keys[o] = metric == RASS_METRIC_COSINE ? selk[c] : -selk[c];
    }
  }
  for (int r = nsel + tid; r < k; r += blockDim.x) {
    const size_t o = (size_t)q * k + r;
    out_rows[o] = -1;
    out_scores[o] = 0.f;
    if (out_keys) out_keys[o] = 0.0;
  }
}

int launch_exact(rass_engine* h, const SearchWs& ws, int k, const int* qids_host, int n_q, int64_t* out_rows,
                 float* out_scores, double* out_keys, cudaStream_t st, int* launches) {
  if (n_q <= 0) return RASS_OK;
  const int M = k <= 32 ? 1 : 4;
  const int grid = h->num_sms * 2;
  const int W = grid * RASS_WARPS_PER_CTA;
  const size_t entries = (size_t)W * 32 * M;
  int rc = ensure_xlist_workspace(h, entries);
  if (rc) return rc;
  const bool bf = (h->flags & RASS_BF16_ONLY) != 0;
  const size_t smem = (size_t)RASS_EXACT_NQ * h->dim_pad * 4;
  // qids live in the (pinned) flagged_host mirror; ship them to the device list
  int* qids_dev = ws.flagged;  // reuse: the flagged list has been consumed by the caller
  CUDA_TRY(h, cudaMemcpyAsync(qids_dev, qids_host, (size_t)n_q * sizeof(int), cudaMemcpyHostToDevice, st));
  for (int p = 0; p < n_q; p += RASS_EXACT_NQ) {
    const int nq = n_q - p < RASS_EXACT_NQ ? n_q - p : RASS_EXACT_NQ;
#define RASS_EX(BF, MM)                                                                                           \
  exact_scan_kernel<BF, MM><<<grid, RASS_WARPS_PER_CTA * 32, smem, st>>>(                                         \
      h->x32, h->x16, h->norm64, h->sb_scan, ws.q_raw, ws.q_norm, qids_dev + p, nq, h->n_rows, h->dim_pad, h->metric, \
      h->xlist_key, h->xlist_row, entries)
    if (bf) { if (M == 1) RASS_EX(true, 1); else RASS_EX(true, 4); }
    else    { if (M == 1) RASS_EX(false, 1); else RASS_EX(false, 4); }
#undef RASS_EX
    CUDA_TRY(h, cudaGetLastError());
    exact_select_kernel<<<nq, 1024, 0, st>>>(h->xlist_key, h->xlist_row, entries, (int)entries, k, qids_dev + p, 0, 0,
                                             h->metric, h->rmap, out_rows, out_scores, out_keys, nullptr);
    CUDA_TRY(h, cudaGetLastError());
    if (launches) *launches += 2;
  }
  return RASS_OK;
}

// exact top-k of B queries' (fp64 key, row) lists of `entries` entries each, scores translated by the engine's metric
int launch_exact_select(rass_engine* h, size_t entries, int B, int k, int64_t* out_rows, float* out_scores,
                        double* out_keys, cudaStream_t st) {
  exact_select_kernel<<<B, 1024, 0, st>>>(h->xlist_key, h->xlist_row, entries, (int)entries, k, nullptr, 0, 0, h->metric,
                                          h->rmap, out_rows, out_scores, out_keys, nullptr);
  CUDA_TRY(h, cudaGetLastError());
  return RASS_OK;
}

// top-k of B queries' fused (score, row) lists of `entries` entries each; the score is emitted as is (bm25.cu)
int launch_select_batch(rass_engine* h, size_t entries, int B, int k, int64_t* out_rows, float* out_scores,
                        double* out_keys, cudaStream_t st, const int* only_if) {
  // raw scores: "larger is better" whatever the vector metric of the engine is
  exact_select_kernel<<<B, 1024, 0, st>>>(h->xlist_key, h->xlist_row, entries, (int)entries, k, nullptr, 0, 1,
                                          RASS_METRIC_COSINE, h->rmap, out_rows, out_scores, out_keys, only_if);
  CUDA_TRY(h, cudaGetLastError());
  return RASS_OK;
}

// ---------------------------------------------------------------------------------------------
// shard merge: G per-shard top-k lists -> global top-k  (the OpenSearch coordinator's merge)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) merge_topk_kernel(const double* __restrict__ keys,
                                                         const int64_t* __restrict__ rows, int64_t shard_stride,
                                                         int G, int B, int k,
                                                         int metric, int raw_score, int64_t* __restrict__ out_rows,
                                                         float* __restrict__ out_scores,
                                                         double* __restrict__ out_keys) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sk = reinterpret_cast<double*>(smem_raw);        // [G*k] "larger is better" key
  int64_t* sr = reinterpret_cast<int64_t*>(sk + G * k);    // [G*k]
  const int q = blockIdx.x, n = G * k;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int g = i / k, j = i % k;
    const size_t src = (size_t)g * shard_stride + (size_t)q * k + j;
    const double v = keys[src];
    sk[i] = (raw_score || metric == RASS_METRIC_COSINE) ? v : -v;     // raw fused scores: larger is better
    sr[i] = rows[src];
  }
  __syncthreads();
  int n_valid = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int64_t r = sr[i];
    if (r < 0) continue;
    const double key = sk[i];
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      const int64_t rj = sr[j];
      if (rj < 0) continue;
      rank += (sk[j] > key) || (sk[j] == key && rj < r);
    }
    if (rank < k) {
      const size_t o = (size_t)q * k + rank;
      out_rows[o] = r;
      out_scores[o] = raw_score ? (float)key : score_from_key(key, metric);
      if (out_keys) out_keys[o] = (raw_score || metric == RASS_METRIC_COSINE) ? key : -key;
    }
  }
  // pad: count the valid entries (every thread, cheap) and blank the tail
  for (int j = 0; j < n; ++j) n_valid += sr[j] >= 0;
  for (int r = n_valid + threadIdx.x; r < k; r += blockDim.x) {
    const size_t o = (size_t)q * k + r;
    out_rows[o] = -1;
    out_scores[o] = 0.f;
    if (out_keys) out_keys[o] = 0.0;
  }
}

int launch_merge_topk(rass_engine* h, const double* keys, const int64_t* rows, int64_t shard_stride, int G, int B,
                      int k, int64_t* out_rows, float* out_scores, double* out_keys, cudaStream_t st, bool raw_score) {
  if (shard_stride <= 0) shard_stride = (int64_t)B * k;
  const size_t smem = (size_t)G * k * 16;
  if (smem > 200 * 1024) return rass_fail(h, RASS_E_INVALID, "merge of %d lists of %d exceeds shared memory", G, k);
  CUDA_TRY(h, cudaFuncSetAttribute(merge_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  merge_topk_kernel<<<B, 256, smem, st>>>(keys, rows, shard_stride, G, B, k, h->metric, raw_score ? 1 : 0, out_rows,
                                          out_scores, out_keys);
  CUDA_TRY(h, cudaGetLastError());
  return RASS_OK;
}
