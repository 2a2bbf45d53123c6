// Engine handle, vector store management and the search orchestration behind the C ABI (include/rass_b200.h).
//
// The store is what OpenSearch keeps for the `embedding` knn_vector field (reference app/main.py:563-572):
// here a device-resident fp32 matrix + bf16 shadow + per-row norms, filled by `bulk index` through pinned,
// double-buffered async copies (reference app/main.py:1247-1269).
#include <stdarg.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"

thread_local std::string g_create_error;

int rass_fail(rass_engine* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  else g_create_error = buf;
  return code;
}

extern "C" const char* rass_version(void) { return "rass-b200 0.1 (abi 1, sm_100a)"; }

extern "C" const char* rass_last_error(const rass_engine* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

#define CHECK_HANDLE(h)                    \
  do {                                     \
    if (!(h)) return RASS_E_INVALID;       \
    cudaSetDevice((h)->device);            \
  } while (0)

template <typename T>
static int dev_realloc(rass_engine* h, T** p, size_t old_n, size_t new_n, cudaStream_t st) {
  T* np = nullptr;
  CUDA_TRY(h, cudaMalloc(&np, new_n * sizeof(T)));
  if (*p && old_n) CUDA_TRY(h, cudaMemcpyAsync(np, *p, old_n * sizeof(T), cudaMemcpyDeviceToDevice, st));
  if (*p) {
    CUDA_TRY(h, cudaStreamSynchronize(st));
    cudaFree(*p);
  }
  *p = np;
  return RASS_OK;
}

static int ensure_capacity(rass_engine* h, int64_t rows) {
  if (rows <= h->cap) return RASS_OK;
  if (rows > 0xfffffff0LL) return rass_fail(h, RASS_E_INVALID, "a shard holds at most 2^32-16 rows");
  cudaStream_t st = eng_stream(h);
  const size_t d = (size_t)h->dim_pad;
  const bool bf16_only = (h->flags & RASS_BF16_ONLY) != 0;
  const bool int8 = has_int8_shadow(h->flags);
  // bytes per row of x32, x16, norm64, sa, sb, x8, sa8
  const size_t per_row[7] = {bf16_only ? 0 : d * 4, d * 2, 8, 4, 4, int8 ? d : 0, int8 ? 4u : 0u};
  if (h->cap == 0 && !h->use_vm && vm_available()) {
    // first allocation: reserve address space for as many rows as the device could ever hold of each array
    size_t free_b = 0, total_b = 0;
    bool ok = cudaMemGetInfo(&free_b, &total_b) == cudaSuccess;
    for (int i = 0; ok && i < 7; ++i)
      if (per_row[i]) {
        const size_t max_rows = std::min<size_t>(0xfffffff0ULL, total_b / per_row[i] + 1);
        ok = vm_reserve(&h->vm[i], h->device, std::max<size_t>(max_rows, (size_t)rows) * per_row[i], 32768 * per_row[i]);
      }
    if (!ok) for (int i = 0; i < 7; ++i) vm_free(&h->vm[i]);
    h->use_vm = ok;
  }
  if (h->use_vm) {
    // grow in place: map enough chunks for `rows` (plus head room: an eighth, at least 64k rows) behind the same
    // pointers -- no copy, no second resident array
    // (none on the first allocation: a caller that passes capacity_rows has sized the store)
    int64_t ncap = std::max<int64_t>(h->cap == 0 ? rows : rows + std::max<int64_t>(rows / 8, 65536), 1024);
    ncap = std::min<int64_t>(ncap, 0xfffffff0LL);
    for (int pass = 0; pass < 2; ++pass) {
      int bad = 0;
      for (int i = 0; i < 7 && !bad; ++i)
        if (per_row[i]) {
          if ((size_t)ncap * per_row[i] > h->vm[i].reserved) ncap = (int64_t)(h->vm[i].reserved / per_row[i]);
          bad = vm_grow(&h->vm[i], (size_t)ncap * per_row[i]);
        }
      if (!bad) break;
      if (pass == 1 || ncap == rows)
        return rass_fail(h, bad == 1 ? RASS_E_OOM : RASS_E_CUDA, "cannot map device memory for %lld rows", (long long)rows);
      ncap = rows;                 // out of memory with the head room: retry with exactly what is needed
    }
    if (ncap < rows) return rass_fail(h, RASS_E_OOM, "%lld rows exceed the address range reserved for the store", (long long)rows);
    // the capacity in rows is what the smallest mapping holds: chunks are not row-aligned, and the last one mapped is
    // usually only partly asked for
    ncap = 0xfffffff0LL;
    for (int i = 0; i < 7; ++i)
      if (per_row[i]) ncap = std::min<int64_t>(ncap, (int64_t)(h->vm[i].mapped / per_row[i]));
    h->x32 = bf16_only ? nullptr : (float*)h->vm[0].base;
    h->x16 = (__nv_bfloat16*)h->vm[1].base;
    h->norm64 = (double*)h->vm[2].base;
    h->sa = (float*)h->vm[3].base;
    h->sb = (float*)h->vm[4].base;
    h->x8 = int8 ? (int8_t*)h->vm[5].base : nullptr;
    h->sa8 = int8 ? (float*)h->vm[6].base : nullptr;
    h->cap = ncap;
    return RASS_OK;
  }
  int64_t ncap = std::max<int64_t>(rows, std::max<int64_t>(h->cap * 2, 1024));
  if (ncap > 0xfffffff0LL) ncap = 0xfffffff0LL;
  const size_t o = (size_t)h->n_rows, n = (size_t)ncap;
  int rc;
  if (!bf16_only)
    if ((rc = dev_realloc(h, &h->x32, o * d, n * d, st))) return rc;
  if ((rc = dev_realloc(h, &h->x16, o * d, n * d, st))) return rc;
  if ((rc = dev_realloc(h, &h->norm64, o, n, st))) return rc;
  if ((rc = dev_realloc(h, &h->sa, o, n, st))) return rc;
  if ((rc = dev_realloc(h, &h->sb, o, n, st))) return rc;
  if (int8) {
    if ((rc = dev_realloc(h, &h->x8, o * d, n * d, st))) return rc;
    if ((rc = dev_realloc(h, &h->sa8, o, n, st))) return rc;
  }
  h->cap = ncap;
  return RASS_OK;
}

extern "C" int rass_create(int dim, int metric, int device, int64_t capacity_rows, uint32_t flags,
                           rass_engine** out) {
  if (!out) return rass_fail(nullptr, RASS_E_INVALID, "out is null");
  *out = nullptr;
  if (dim < 1 || dim > 1024) return rass_fail(nullptr, RASS_E_INVALID, "dim must be in [1, 1024], got %d", dim);
  if (metric != RASS_METRIC_COSINE && metric != RASS_METRIC_L2)
    return rass_fail(nullptr, RASS_E_INVALID, "unknown metric %d", metric);
  if ((flags & RASS_KEEP_FP32) && (flags & RASS_BF16_ONLY))
    return rass_fail(nullptr, RASS_E_INVALID, "RASS_KEEP_FP32 and RASS_BF16_ONLY are exclusive");
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return rass_fail(nullptr, RASS_E_CUDA, "no CUDA device (%s); this engine has no CPU fallback",
                     e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (device < 0 || device >= n_dev) return rass_fail(nullptr, RASS_E_INVALID, "device %d out of range", device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess)
    return rass_fail(nullptr, RASS_E_CUDA, "cudaGetDeviceProperties failed");
  if (prop.major != 10)
    return rass_fail(nullptr, RASS_E_CUDA, "device %d is sm_%d%d; this engine is built for sm_100a only", device,
                     prop.major, prop.minor);
  rass_engine* h = new rass_engine();
  h->dim = dim;
  h->dim_pad = (dim + 255) / 256 * 256;
  h->metric = metric;
  h->device = device;
  h->flags = (flags & (RASS_KEEP_FP32 | RASS_BF16_ONLY)) ? flags : flags | RASS_KEEP_FP32;
  h->num_sms = prop.multiProcessorCount;
  auto bail = [&](int code) {
    g_create_error = h->err;
    rass_destroy(h);
    return code;
  };
  if (cudaSetDevice(device) != cudaSuccess) { h->err = "cudaSetDevice failed"; return bail(RASS_E_CUDA); }
#define CREATE_TRY(call)                                                                            \
  do {                                                                                              \
    cudaError_t e_ = (call);                                                                        \
    if (e_ != cudaSuccess) {                                                                        \
      h->err = std::string(#call) + " failed: " + cudaGetErrorString(e_);                           \
      return bail(e_ == cudaErrorMemoryAllocation ? RASS_E_OOM : RASS_E_CUDA);                      \
    }                                                                                               \
  } while (0)
  CREATE_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CREATE_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 4; ++i) CREATE_TRY(cudaEventCreate(&h->ev[i]));
  for (int i = 0; i < 2; ++i) CREATE_TRY(cudaEventCreateWithFlags(&h->stage_ev[i], cudaEventDisableTiming));
  h->stage_bytes = (size_t)32 << 20;
  for (int i = 0; i < 2; ++i) CREATE_TRY(cudaMallocHost(&h->stage[i], h->stage_bytes));
  CREATE_TRY(cudaMalloc(&h->store_scal, sizeof(StoreScalars)));
  CREATE_TRY(cudaMemset(h->store_scal, 0, sizeof(StoreScalars)));
  CREATE_TRY(cudaMalloc(&h->ws[0].scal, sizeof(SearchScalars)));
  CREATE_TRY(cudaMemset(h->ws[0].scal, 0, sizeof(SearchScalars)));
  CREATE_TRY(cudaMallocHost(&h->scal_host, sizeof(SearchScalars)));
  memset(h->scal_host, 0, sizeof(SearchScalars));
#undef CREATE_TRY
  if (capacity_rows > 0) {
    int rc = ensure_capacity(h, capacity_rows);
    if (rc) return bail(rc);
  }
  *out = h;
  return RASS_OK;
}

static void free_search_ws(SearchWs& w) {
  cudaFree(w.scal);
  cudaFree(w.q_raw); cudaFree(w.q_hat); cudaFree(w.q16); cudaFree(w.q_norm); cudaFree(w.q_rho); cudaFree(w.q_gthr);
  cudaFree(w.q8); cudaFree(w.q8_scale); cudaFree(w.q_rho8);
  cudaFree(w.pool_key); cudaFree(w.pool_row); cudaFree(w.pool_thr); cudaFree(w.pool_cnt);
  cudaFree(w.flagged); cudaFreeHost(w.flagged_host);
  free(w.tmap_q); free(w.tmap_q2); free(w.tmap_q8);
}

extern "C" int rass_destroy(rass_engine* h) {
  SHARDED(h, sharded_destroy(h));
  if (!h) return RASS_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  if (h->use_vm) {
    for (int i = 0; i < 7; ++i) vm_free(&h->vm[i]);
  } else {
    cudaFree(h->x32); cudaFree(h->x16); cudaFree(h->norm64); cudaFree(h->sa); cudaFree(h->sb);
    cudaFree(h->x8); cudaFree(h->sa8);
  }
  cudaFree(h->store_scal); cudaFreeHost(h->scal_host);
  for (SearchWs& w : h->ws) free_search_ws(w);
  cudaFree(h->dev_stage);
  cudaFree(h->xlist_key); cudaFree(h->xlist_row);
  cudaFree(h->out_rows); cudaFree(h->out_scores); cudaFree(h->out_keys);
  cudaFreeHost(h->out_rows_host); cudaFreeHost(h->out_scores_host); cudaFreeHost(h->out_keys_host);
  cudaFreeHost(h->q_stage_host);
  cudaFree(h->q_stage_dev);
  cudaFree(h->row_filter);
  cudaFree(h->filter_rows_dev);
  cudaFree(h->flist_dev);
  cudaFree(h->sb_filtered);
  cudaFree(h->retry_ids); cudaFree(h->retry_q); cudaFree(h->retry_rows); cudaFree(h->retry_scores); cudaFree(h->retry_keys);
  for (int i = 0; i < 2; ++i) {
    if (h->slot_stream[i]) cudaStreamDestroy(h->slot_stream[i]);
    if (h->slot_fork[i]) cudaEventDestroy(h->slot_fork[i]);
  }
  for (cudaEvent_t e : h->ev_pool) if (e) cudaEventDestroy(e);
  for (auto& a : h->aslot) { cudaFreeHost(a.scal_host); if (a.done) cudaEventDestroy(a.done); }
  for (int i = 0; i < 2; ++i) { cudaFreeHost(h->stage[i]); if (h->stage_ev[i]) cudaEventDestroy(h->stage_ev[i]); }
  for (int i = 0; i < 4; ++i) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  Bm25State& b = h->bm25;
  cudaFree(b.indptr); cudaFree(b.doc); cudaFree(b.tf); cudaFree(b.xq); cudaFree(b.norm); cudaFree(b.inv_dev);
  cudaFree(b.tile_off); cudaFree(b.qt_dev); cudaFreeHost(b.qt_host); cudaFree(b.hyb_gthr); cudaFree(b.sel_fallback);
  for (TextSegment& sg : b.pending) { cudaFree(sg.uterm); cudaFree(sg.uptr); cudaFree(sg.doc); cudaFree(sg.tf); }
  cudaFree(b.doclen_dev);
  cudaFree(b.gen_dev);
  cudaFree(b.scratch);
  cudaFree(b.vocab_blob); cudaFree(b.vocab_off); cudaFree(b.fz_terms); cudaFree(b.fz_edits); cudaFree(b.fz_n);
  free(h->tmap_x);
  free(h->tmap_x8);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  delete h;
  return RASS_OK;
}

extern "C" int rass_set_option(rass_engine* h, int opt, int64_t value) {
  SHARDED(h, sharded_set_option(h, opt, value));
  CHECK_HANDLE(h);
  switch (opt) {
    case RASS_OPT_KNN_PREFILTER:
      h->knn_prefilter = value != 0;
      return RASS_OK;
    case RASS_OPT_HYBRID_ORDERED:
      h->bm25.force_ordered = value != 0;
      return RASS_OK;
    case RASS_OPT_HYBRID_MAXSCORE:
      h->bm25.maxscore = value != 0;
      return RASS_OK;
    case RASS_OPT_PATH:
      if (value < RASS_PATH_AUTO || value > RASS_PATH_UMMA8) return rass_fail(h, RASS_E_INVALID, "bad path %lld", (long long)value);
      if (value == RASS_PATH_UMMA8 && !has_int8_shadow(h->flags))
        return rass_fail(h, RASS_E_UNSUPPORTED, "RASS_PATH_UMMA8 needs the int8 shadow (a store without RASS_BF16_ONLY "
                         "and RASS_NO_INT8_SHADOW)");
      h->path = (int)value;
      return RASS_OK;
    case RASS_OPT_ASYNC_OVERLAP:
      for (auto& a : h->aslot)
        if (a.pending) return rass_fail(h, RASS_E_INVALID, "RASS_OPT_ASYNC_OVERLAP cannot change while a search is in flight");
      h->async_overlap = value != 0;
      return RASS_OK;
    case RASS_OPT_SCAN_RESERVE_SMS:
      if (value < 0 || value >= h->num_sms) return rass_fail(h, RASS_E_INVALID, "bad SM reserve %lld", (long long)value);
      h->scan_reserve_sms = (int)value;
      return RASS_OK;
    case RASS_OPT_STREAM:
      if (value == -1) {
        h->has_user_stream = false;
        h->user_stream = nullptr;
      } else {
        h->has_user_stream = true;
        h->user_stream = reinterpret_cast<cudaStream_t>(value);
      }
      return RASS_OK;
    default:
      return rass_fail(h, RASS_E_INVALID, "unknown option %d", opt);
  }
}

extern "C" int rass_set_row_base(rass_engine* h, int64_t base) {
  SHARDED(h, sharded_set_row_base(h, base));
  CHECK_HANDLE(h);
  h->rmap.base = base;
  return RASS_OK;
}

extern "C" int rass_count(const rass_engine* h, int64_t* out) {
  if (!h || !out) return RASS_E_INVALID;
  *out = h->n_live;
  return RASS_OK;
}

extern "C" int rass_rows(const rass_engine* h, int64_t* out) {
  if (!h || !out) return RASS_E_INVALID;
  *out = h->n_rows;
  return RASS_OK;
}

extern "C" int rass_store_info(const rass_engine* h, int64_t* capacity_rows, int* grows_in_place) {
  if (!h) return RASS_E_INVALID;
  const rass_engine* e = h->shards ? sharded_first(const_cast<rass_engine*>(h)) : h;
  if (capacity_rows) *capacity_rows = e->cap;
  if (grows_in_place) *grows_in_place = e->use_vm ? 1 : 0;
  return RASS_OK;
}

extern "C" int rass_last_stats(const rass_engine* h, rass_stats* out) {
  if (!h || !out) return RASS_E_INVALID;
  *out = h->last_stats;
  return RASS_OK;
}

extern "C" int rass_sync(rass_engine* h) {
  SHARDED(h, sharded_sync(h));
  CHECK_HANDLE(h);
  CUDA_TRY(h, cudaStreamSynchronize(eng_stream(h)));
  return RASS_OK;
}

static int ensure_dev_stage(rass_engine* h, size_t bytes) {
  if (bytes <= h->dev_stage_bytes) return RASS_OK;
  CUDA_TRY(h, cudaStreamSynchronize(eng_stream(h)));
  cudaFree(h->dev_stage);
  h->dev_stage = nullptr;
  h->dev_stage_bytes = 0;
  CUDA_TRY(h, cudaMalloc(&h->dev_stage, bytes));
  h->dev_stage_bytes = bytes;
  return RASS_OK;
}

static bool direct_fp32(const rass_engine* h) { return !(h->flags & RASS_BF16_ONLY) && h->dim == h->dim_pad; }

// rows already on the device: [n, dim] fp32
static int append_from_device(rass_engine* h, const float* rows_dev, int64_t first, int64_t n, cudaStream_t st) {
  if (direct_fp32(h)) {
    float* dst = h->x32 + (size_t)first * h->dim_pad;
    if (rows_dev != dst)
      CUDA_TRY(h, cudaMemcpyAsync(dst, rows_dev, (size_t)n * h->dim * 4, cudaMemcpyDeviceToDevice, st));
    return launch_store_convert(h, dst, h->dim_pad, first, n, st);
  }
  return launch_store_convert(h, rows_dev, h->dim, first, n, st);
}

extern "C" int rass_append_dev(rass_engine* h, const float* rows_dev, int64_t n, int64_t* out_first_row) {
  SHARDED(h, sharded_append_dev(h, rows_dev, n, out_first_row));
  CHECK_HANDLE(h);
  if (n < 0 || (n > 0 && !rows_dev)) return rass_fail(h, RASS_E_INVALID, "bad rows");
  int rc = ensure_capacity(h, h->n_rows + n);
  if (rc) return rc;
  cudaStream_t st = eng_stream(h);
  const int64_t first = h->n_rows;
  if ((rc = append_from_device(h, rows_dev, first, n, st))) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  h->n_rows += n;
  h->n_live += n;
  h->dead.resize((size_t)h->n_rows, 0);
  if (out_first_row) *out_first_row = first;
  return RASS_OK;
}

// host rows -> device rows [first, first+n) through the pinned double buffer
static int upload_rows(rass_engine* h, const float* rows_host, int64_t first, int64_t n, cudaStream_t st) {
  const size_t row_bytes = (size_t)h->dim * 4;
  cudaPointerAttributes attr;
  bool pinned = cudaPointerGetAttributes(&attr, rows_host) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  const int64_t chunk = std::max<int64_t>(1, (int64_t)(h->stage_bytes / row_bytes));
  int rc;
  if (!direct_fp32(h) && (rc = ensure_dev_stage(h, (size_t)std::min<int64_t>(chunk, n) * row_bytes))) return rc;
  int buf = 0;
  for (int64_t off = 0; off < n; off += chunk, buf ^= 1) {
    const int64_t m = std::min<int64_t>(chunk, n - off);
    const float* src = rows_host + (size_t)off * h->dim;
    if (!pinned) {
      CUDA_TRY(h, cudaEventSynchronize(h->stage_ev[buf]));
      memcpy(h->stage[buf], src, (size_t)m * row_bytes);
      src = h->stage[buf];
    }
    float* dst = direct_fp32(h) ? h->x32 + (size_t)(first + off) * h->dim_pad : h->dev_stage;
    CUDA_TRY(h, cudaMemcpyAsync(dst, src, (size_t)m * row_bytes, cudaMemcpyHostToDevice, st));
    if (!pinned) CUDA_TRY(h, cudaEventRecord(h->stage_ev[buf], st));
    if ((rc = launch_store_convert(h, dst, direct_fp32(h) ? h->dim_pad : h->dim, first + off, m, st))) return rc;
  }
  return RASS_OK;
}

extern "C" int rass_append(rass_engine* h, const float* rows_host, int64_t n, int64_t* out_first_row) {
  SHARDED(h, sharded_append(h, rows_host, n, out_first_row));
  CHECK_HANDLE(h);
  if (n < 0 || (n > 0 && !rows_host)) return rass_fail(h, RASS_E_INVALID, "bad rows");
  int rc = ensure_capacity(h, h->n_rows + n);
  if (rc) return rc;
  cudaStream_t st = eng_stream(h);
  const int64_t first = h->n_rows;
  if ((rc = upload_rows(h, rows_host, first, n, st))) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  h->n_rows += n;
  h->n_live += n;
  h->dead.resize((size_t)h->n_rows, 0);
  if (out_first_row) *out_first_row = first;
  return RASS_OK;
}

extern "C" int rass_overwrite(rass_engine* h, int64_t row, const float* v_host) {
  SHARDED(h, sharded_overwrite(h, row, v_host));
  CHECK_HANDLE(h);
  if (row < 0 || row >= h->n_rows || !v_host) return rass_fail(h, RASS_E_NOTFOUND, "row %lld out of range", (long long)row);
  cudaStream_t st = eng_stream(h);
  int rc = upload_rows(h, v_host, row, 1, st);
  if (rc) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  if (h->dead[(size_t)row]) { h->dead[(size_t)row] = 0; h->n_live++; }
  return RASS_OK;
}

// sb = -inf for one row (row >= 0) or for the listed rows: stream-ordered, nothing for the host to wait for
__global__ void tombstone_kernel(float* __restrict__ sb, int64_t row, const int64_t* __restrict__ rows, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) sb[rows ? rows[i] : row] = __int_as_float(0xff800000);
}

extern "C" int rass_tombstone(rass_engine* h, int64_t row) {
  SHARDED(h, sharded_tombstone(h, row));
  CHECK_HANDLE(h);
  if (row < 0 || row >= h->n_rows) return rass_fail(h, RASS_E_NOTFOUND, "row %lld out of range", (long long)row);
  if (h->dead[(size_t)row]) return RASS_OK;
  tombstone_kernel<<<1, 32, 0, eng_stream(h)>>>(h->sb, row, nullptr, 1);     // ordered before the next search, no sync
  CUDA_TRY(h, cudaGetLastError());
  h->sb_filtered_dirty = true;
  h->dead[(size_t)row] = 1;
  h->n_live--;
  return RASS_OK;
}

// the tombstones of a snapshot in one launch
static int tombstone_many(rass_engine* h, const std::vector<int64_t>& rows) {
  if (rows.empty()) return RASS_OK;
  cudaStream_t st = eng_stream(h);
  int64_t* dev = nullptr;
  CUDA_TRY(h, cudaMalloc(&dev, rows.size() * 8));
  cudaError_t e = cudaMemcpyAsync(dev, rows.data(), rows.size() * 8, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    tombstone_kernel<<<(unsigned)((rows.size() + 255) / 256), 256, 0, st>>>(h->sb, -1, dev, (int64_t)rows.size());
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(dev);
  if (e != cudaSuccess) return rass_fail(h, RASS_E_CUDA, "tombstones: %s", cudaGetErrorString(e));
  for (int64_t r : rows)
    if (!h->dead[(size_t)r]) { h->dead[(size_t)r] = 1; h->n_live--; }
  h->sb_filtered_dirty = true;
  return RASS_OK;
}

__global__ void widen_rows_kernel(const __nv_bfloat16* __restrict__ x16, int dim, int dim_pad, int64_t first,
                                  int64_t n, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * dim) return;
  const int64_t r = i / dim;
  const int c = (int)(i % dim);
  out[i] = __bfloat162float(x16[(size_t)(first + r) * dim_pad + c]);
}

extern "C" int rass_read_rows(rass_engine* h, int64_t first_row, int64_t n, float* out_host) {
  SHARDED(h, sharded_read_rows(h, first_row, n, out_host));
  CHECK_HANDLE(h);
  if (first_row < 0 || n < 0 || first_row + n > h->n_rows || (n && !out_host))
    return rass_fail(h, RASS_E_NOTFOUND, "rows [%lld, +%lld) out of range", (long long)first_row, (long long)n);
  if (n == 0) return RASS_OK;
  cudaStream_t st = eng_stream(h);
  if (!(h->flags & RASS_BF16_ONLY)) {
    CUDA_TRY(h, cudaMemcpy2DAsync(out_host, (size_t)h->dim * 4, h->x32 + (size_t)first_row * h->dim_pad,
                                  (size_t)h->dim_pad * 4, (size_t)h->dim * 4, (size_t)n, cudaMemcpyDeviceToHost, st));
  } else {
    const int64_t chunk = std::max<int64_t>(1, (int64_t)((size_t)64 << 20) / (h->dim * 4));
    int rc = ensure_dev_stage(h, (size_t)std::min(chunk, n) * h->dim * 4);
    if (rc) return rc;
    for (int64_t off = 0; off < n; off += chunk) {
      const int64_t m = std::min(chunk, n - off);
      const int64_t tot = m * h->dim;
      widen_rows_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(h->x16, h->dim, h->dim_pad, first_row + off, m,
                                                                       h->dev_stage);
      CUDA_TRY(h, cudaGetLastError());
      CUDA_TRY(h, cudaMemcpyAsync(out_host + (size_t)off * h->dim, h->dev_stage, (size_t)tot * 4,
                                  cudaMemcpyDeviceToHost, st));
    }
  }
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return RASS_OK;
}

// ---------------------------------------------------------------------------------------------
// snapshot / restore of the vector store (SURVEY.md 5: checkpoint/resume; 8f N3)
// ---------------------------------------------------------------------------------------------
struct SnapHeader {
  char magic[8];          // "RASSB200"
  uint32_t version, dim, metric, flags;
  int64_t n_rows, n_live;
};

// File = header, tombstone bytes [n_rows], stored values [n_rows, dim] fp32 (the bf16 values widened for a bf16
// corpus).  Restore re-ingests through the normal append path, so shadow, norms and bounds are rebuilt, not trusted.
extern "C" int rass_save(rass_engine* h, const char* path) {
  SHARDED(h, sharded_save(h, path));
  CHECK_HANDLE(h);
  if (!path) return rass_fail(h, RASS_E_INVALID, "null path");
  FILE* f = fopen(path, "wb");
  if (!f) return rass_fail(h, RASS_E_INVALID, "cannot open %s for writing", path);
  SnapHeader hd;
  memset(&hd, 0, sizeof(hd));
  memcpy(hd.magic, "RASSB200", 8);
  hd.version = 1; hd.dim = (uint32_t)h->dim; hd.metric = (uint32_t)h->metric; hd.flags = h->flags;
  hd.n_rows = h->n_rows; hd.n_live = h->n_live;
  bool ok = fwrite(&hd, sizeof(hd), 1, f) == 1;
  if (ok && h->n_rows) ok = fwrite(h->dead.data(), 1, (size_t)h->n_rows, f) == (size_t)h->n_rows;
  const int64_t chunk = std::max<int64_t>(1, (int64_t)(h->stage_bytes / ((size_t)h->dim * 4)));
  int rc = RASS_OK;
  for (int64_t off = 0; ok && off < h->n_rows; off += chunk) {
    const int64_t m = std::min<int64_t>(chunk, h->n_rows - off);
    if ((rc = rass_read_rows(h, off, m, h->stage[0]))) break;
    ok = fwrite(h->stage[0], (size_t)h->dim * 4, (size_t)m, f) == (size_t)m;
  }
  ok = (fclose(f) == 0) && ok;
  if (rc) return rc;
  if (!ok) return rass_fail(h, RASS_E_INVALID, "short write to %s", path);
  return RASS_OK;
}

extern "C" int rass_load(rass_engine* h, const char* path) {
  CHECK_HANDLE(h);
  if (!path) return rass_fail(h, RASS_E_INVALID, "null path");
  if (h->n_rows != 0) return rass_fail(h, RASS_E_INVALID, "rass_load needs an empty engine");
  FILE* f = fopen(path, "rb");
  if (!f) return rass_fail(h, RASS_E_NOTFOUND, "cannot open %s", path);
  SnapHeader hd;
  int rc = RASS_OK;
  std::vector<uint8_t> dead;
  if (fread(&hd, sizeof(hd), 1, f) != 1 || memcmp(hd.magic, "RASSB200", 8) != 0 || hd.version != 1) {
    rc = rass_fail(h, RASS_E_INVALID, "%s is not a rass_b200 snapshot", path);
  } else if ((int)hd.dim != h->dim || (int)hd.metric != h->metric ||
             ((hd.flags ^ h->flags) & RASS_BF16_ONLY)) {
    rc = rass_fail(h, RASS_E_INVALID, "snapshot is dim %u metric %u flags %u, engine is dim %d metric %d flags %u",
                   hd.dim, hd.metric, hd.flags, h->dim, h->metric, h->flags);
  } else {
    dead.resize((size_t)hd.n_rows);
    if (hd.n_rows && fread(dead.data(), 1, dead.size(), f) != dead.size())
      rc = rass_fail(h, RASS_E_INVALID, "%s is truncated", path);
  }
  const size_t stage = h->stage_bytes ? h->stage_bytes : ((size_t)64 << 20);     // a sharded coordinator has no staging
  const int64_t chunk = std::max<int64_t>(1, (int64_t)(stage / ((size_t)h->dim * 4)));
  std::vector<float> buf;
  if (!rc) buf.resize((size_t)std::min<int64_t>(chunk, std::max<int64_t>(hd.n_rows, 1)) * h->dim);
  for (int64_t off = 0; !rc && off < hd.n_rows; off += chunk) {
    const int64_t m = std::min<int64_t>(chunk, hd.n_rows - off);
    if (fread(buf.data(), (size_t)h->dim * 4, (size_t)m, f) != (size_t)m) {
      rc = rass_fail(h, RASS_E_INVALID, "%s is truncated", path);
      break;
    }
    rc = rass_append(h, buf.data(), m, nullptr);
  }
  fclose(f);
  if (!rc) {
    std::vector<int64_t> gone;
    for (int64_t r = 0; r < hd.n_rows; ++r)
      if (dead[(size_t)r]) gone.push_back(r);
    if (h->shards)                                    // a sharded handle routes every row to its shard
      for (size_t i = 0; !rc && i < gone.size(); ++i) rc = rass_tombstone(h, gone[i]);
    else
      rc = tombstone_many(h, gone);
  }
  return rc;
}

// ---------------------------------------------------------------------------------------------
// workspaces
// ---------------------------------------------------------------------------------------------
#define REALLOC_DEV(h, p, n)                                    \
  do {                                                          \
    cudaFree(p);                                                \
    (p) = nullptr;                                              \
    CUDA_TRY(h, cudaMalloc(&(p), (n) * sizeof(*(p))));          \
  } while (0)
#define REALLOC_HOST(h, p, n)                                   \
  do {                                                          \
    cudaFreeHost(p);                                            \
    (p) = nullptr;                                              \
    CUDA_TRY(h, cudaMallocHost(&(p), (n) * sizeof(*(p))));      \
  } while (0)

// a workspace is about to be freed: nothing enqueued may still use it
static int sync_for_realloc(rass_engine* h) {
  CUDA_TRY(h, cudaStreamSynchronize(eng_stream(h)));
  for (int i = 0; i < 2; ++i)
    if (h->slot_stream[i]) CUDA_TRY(h, cudaStreamSynchronize(h->slot_stream[i]));
  return RASS_OK;
}

int ensure_query_workspace(rass_engine* h, SearchWs& ws, int B) {
  if (B <= ws.q_cap) return RASS_OK;
  { const int rc_ = sync_for_realloc(h); if (rc_) return rc_; }
  const size_t cap = (size_t)(B + RASS_QPAD - 1) / RASS_QPAD * RASS_QPAD, d = (size_t)h->dim_pad;
  REALLOC_DEV(h, ws.q_raw, cap * d);
  REALLOC_DEV(h, ws.q_hat, cap * d);
  REALLOC_DEV(h, ws.q16, cap * d);
  REALLOC_DEV(h, ws.q_norm, cap);
  REALLOC_DEV(h, ws.q_rho, cap);
  REALLOC_DEV(h, ws.q_gthr, cap);
  if (has_int8_shadow(h->flags)) {
    REALLOC_DEV(h, ws.q8, cap * 2 * d);
    REALLOC_DEV(h, ws.q8_scale, cap * 2);
    REALLOC_DEV(h, ws.q_rho8, cap);
  }
  REALLOC_DEV(h, ws.flagged, cap);
  REALLOC_HOST(h, ws.flagged_host, cap);
  ws.q_cap = (int)cap;
  ws.tmap_qbase = nullptr;
  ws.tmap_q2base = nullptr;
  ws.tmap_q8base = nullptr;
  return RASS_OK;
}

int ensure_pool(rass_engine* h, SearchWs& ws, size_t entries_per_query, size_t segs_per_query, size_t n_queries) {
  const size_t need_e = entries_per_query * n_queries, need_s = segs_per_query * n_queries;
  if (need_e > ws.pool_alloc_entries) {
    { const int rc_ = sync_for_realloc(h); if (rc_) return rc_; }
    ws.pool_alloc_entries = 0;
    REALLOC_DEV(h, ws.pool_key, need_e);
    REALLOC_DEV(h, ws.pool_row, need_e);
    ws.pool_alloc_entries = need_e;
  }
  if (need_s > ws.pool_alloc_segs) {
    { const int rc_ = sync_for_realloc(h); if (rc_) return rc_; }
    ws.pool_alloc_segs = 0;
    REALLOC_DEV(h, ws.pool_thr, need_s);
    REALLOC_DEV(h, ws.pool_cnt, need_s);
    ws.pool_alloc_segs = need_s;
  }
  ws.pool_entries = entries_per_query;
  ws.pool_segs = segs_per_query;
  return RASS_OK;
}

int ensure_xlist_workspace(rass_engine* h, size_t entries) {
  if (entries <= h->xlist_entries) return RASS_OK;
  CUDA_TRY(h, cudaStreamSynchronize(eng_stream(h)));
  REALLOC_DEV(h, h->xlist_key, entries * RASS_EXACT_NQ);
  REALLOC_DEV(h, h->xlist_row, entries * RASS_EXACT_NQ);
  h->xlist_entries = entries;
  return RASS_OK;
}

int ensure_out_workspace(rass_engine* h, size_t n) {
  if (n <= h->out_cap) return RASS_OK;
  CUDA_TRY(h, cudaStreamSynchronize(eng_stream(h)));
  REALLOC_DEV(h, h->out_rows, n);
  REALLOC_DEV(h, h->out_scores, n);
  REALLOC_DEV(h, h->out_keys, n);
  REALLOC_HOST(h, h->out_rows_host, n);
  REALLOC_HOST(h, h->out_scores_host, n);
  REALLOC_HOST(h, h->out_keys_host, n);
  h->out_cap = n;
  return RASS_OK;
}

// ---------------------------------------------------------------------------------------------
// search
// ---------------------------------------------------------------------------------------------
__global__ void fill_empty_kernel(int64_t* rows, float* scores, double* keys, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  rows[i] = -1;
  scores[i] = 0.f;
  if (keys) keys[i] = 0.0;
}

// sb with the bool.filter folded in: rows failing the pass mask read -inf, exactly like tombstones
__global__ void fold_filter_kernel(const float* __restrict__ sb, const uint8_t* __restrict__ mask, int64_t mask_rows,
                                   int64_t n, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = (i < mask_rows && mask[i]) ? sb[i] : __int_as_float(0xff800000);
}

static int select_scan_offsets(rass_engine* h, cudaStream_t st) {
  h->sb_scan = h->sb;
  if (!h->knn_prefilter || !h->row_filter) return RASS_OK;
  if (h->sb_filtered_cap < h->cap) {
    CUDA_TRY(h, cudaStreamSynchronize(st));
    cudaFree(h->sb_filtered);
    h->sb_filtered = nullptr;
    CUDA_TRY(h, cudaMalloc(&h->sb_filtered, (size_t)h->cap * sizeof(float)));
    h->sb_filtered_cap = h->cap;
    h->sb_filtered_dirty = true;
  }
  if (h->sb_filtered_dirty && h->n_rows > 0) {
    fold_filter_kernel<<<(unsigned)((h->n_rows + 255) / 256), 256, 0, st>>>(h->sb, h->row_filter, h->row_filter_rows,
                                                                           h->n_rows, h->sb_filtered);
    CUDA_TRY(h, cudaGetLastError());
    h->sb_filtered_dirty = false;
  }
  h->sb_scan = h->sb_filtered;
  return RASS_OK;
}

// Largest rho_x8 for which AUTO scans the int8 shadow.  The int8 certificate allowance is eps ~ rho_x8 + rho_q8
// (rho_q8 ~ 4e-5 with the two-part query); a query's rerank set holds the pool entries within 2 eps of the k-th best
// scan key.  Unit rows without outlier channels give rho_x8 ~ 0.014 and ~600 candidates per query at 10M rows x 1024;
// the count grows faster than linearly in eps (the tail of the score distribution), so 0.03 keeps it below
// RASS_CAND_MAX = 2048 with room, and the candidate segments keep t + eps below s_k.  Rows with an outlier channel
// (max|x| far above the rest: s_x = max|x| / 127 quantises everything else coarsely) push rho_x8 past it; the store
// then keeps the bf16 pass.
#define RASS_INT8_RHO_MAX 0.03f

// the store facts raised by store_convert_kernel, on the host (appends and overwrites synchronise before they return)
static int refresh_store_scalars(rass_engine* h) {
  if (!h->store_scal_stale) return RASS_OK;
  cudaStream_t st = eng_stream(h);
  CUDA_TRY(h, cudaMemcpyAsync(&h->store_scal_host, h->store_scal, sizeof(StoreScalars), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  h->store_scal_stale = false;
  return RASS_OK;
}

static int resolve_path(const rass_engine* h, int B, int k) {
  if (h->path != RASS_PATH_AUTO) return h->path;
  // measured at 10M rows: streaming scan 2.79 ms for one query, 3.10 ms for two; one tcgen05 pass 2.98-3.05 ms for
  // 1..64 queries; one 256-query CTA-pair pass ~5.1 ms (two 64-query passes = 6.1 ms).  The int8 pass streams half
  // the bytes of the bf16 one.  RASS_DEBUG_NO_INT8: the bf16 pass (the A/B switch of the measurement)
  static const bool no_int8 = getenv("RASS_DEBUG_NO_INT8") != nullptr;
  if (B <= 1) return RASS_PATH_STREAM;
  if (B > RASS_GROUP_Q) return RASS_PATH_GEMM;
  const bool int8 = !no_int8 && h->x8 && h->store_scal_host.rho_x8 <= RASS_INT8_RHO_MAX && k <= h->int8_k_max;
  return int8 ? RASS_PATH_UMMA8 : RASS_PATH_UMMA;
}

// after an int8 pass AUTO chose: too many uncertified queries at this k -> the bf16 pass for k and above from now on
static void note_int8_outcome(rass_engine* h, int path, int B, int k, int n_flagged, bool robust) {
  if (path == RASS_PATH_UMMA8 && h->path == RASS_PATH_AUTO && !robust && 4 * n_flagged > B)
    h->int8_k_max = std::min(h->int8_k_max, k - 1);
}

static cudaEvent_t get_event(rass_engine* h, size_t i) {
  while (h->ev_pool.size() <= i) {
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    h->ev_pool.push_back(e);
  }
  return h->ev_pool[i];
}

// second-chance pass for queries whose certificate failed: gather them, search with 512-entry segments, scatter back
__global__ void gather_queries_kernel(const float* __restrict__ q, const int* __restrict__ ids, int dim,
                                      float* __restrict__ out) {
  const float* src = q + (size_t)ids[blockIdx.x] * dim;
  float* dst = out + (size_t)blockIdx.x * dim;
  for (int j = threadIdx.x; j < dim; j += blockDim.x) dst[j] = src[j];
}
__global__ void scatter_results_kernel(const int* __restrict__ ids, int k, const int64_t* __restrict__ rows,
                                       const float* __restrict__ scores, const double* __restrict__ keys,
                                       int64_t* __restrict__ out_rows, float* __restrict__ out_scores,
                                       double* __restrict__ out_keys) {
  const size_t src = (size_t)blockIdx.x * k, dst = (size_t)ids[blockIdx.x] * k;
  for (int j = threadIdx.x; j < k; j += blockDim.x) {
    out_rows[dst + j] = rows[src + j];
    out_scores[dst + j] = scores[src + j];
    if (out_keys) out_keys[dst + j] = keys[src + j];
  }
}

// the scan time of a search: the sum over its pairs of timing events (ev_pool[base + i], ev_pool[base + i + 1])
static int scan_ms_of(rass_engine* h, size_t base, size_t n_ev, double* out) {
  double ms = 0.0;
  for (size_t i = 0; i + 1 < n_ev; i += 2) {
    float t = 0.f;
    CUDA_TRY(h, cudaEventElapsedTime(&t, h->ev_pool[base + i], h->ev_pool[base + i + 1]));
    ms += t;
  }
  *out = ms;
  return RASS_OK;
}

// robust = false: 256-entry segments (a compaction keeps 32..64 entries): fastest, and every pivot has >= 32 >= k
// entries above it when k <= 32.  For k > 32 a cluster of near neighbours inside one segment can lift a pivot above
// the k-th best; those queries fail their certificate and get a second pass with robust = true (512-entry segments,
// >= 128 entries above every pivot) at tensor-core speed instead of the fp64 scan.
//
// async_slot >= 0: enqueue only -- no host synchronisation, no fallback; the certificate outcome lands in the slot's
// pinned scalars (and, for row-sharded callers, in *async_flag_dev, which travels with the all-gathered candidates).
static int search_core_body(rass_engine* h, SearchWs& ws, const float* q_dev, int B, int k, int64_t* out_rows,
                            float* out_scores, double* out_keys, rass_stats* stats, bool robust, int async_slot,
                            int64_t* async_flag_dev, cudaStream_t st) {
  int rc;
  if ((rc = ensure_query_workspace(h, ws, B))) return rc;
  rass_stats s;
  memset(&s, 0, sizeof(s));
  s.n_queries = B;
  s.rows_scanned = h->n_rows;
  double retry_scan_ms = 0.0, retry_total_ms = 0.0, first_scan_ms = 0.0, first_total_ms = -1.0;
  const size_t n_out = (size_t)B * k;
  const size_t ev_base = async_slot >= 0 ? (size_t)1024 * (async_slot + 1) : 0;   // per-slot timing events
  rass_engine::AsyncSlot* as = async_slot >= 0 ? &h->aslot[async_slot] : nullptr;
  if (as) {
    if (as->pending) return rass_fail(h, RASS_E_INVALID, "async slot %d still has a search in flight", async_slot);
    if (!as->scal_host) CUDA_TRY(h, cudaMallocHost(&as->scal_host, sizeof(SearchScalars)));
    if (!as->done) CUDA_TRY(h, cudaEventCreateWithFlags(&as->done, cudaEventDisableTiming));
  }
  if (h->n_rows == 0) {
    fill_empty_kernel<<<(unsigned)((n_out + 255) / 256), 256, 0, st>>>(out_rows, out_scores, out_keys, n_out);
    CUDA_TRY(h, cudaGetLastError());
    if (as) {
      if (async_flag_dev) CUDA_TRY(h, cudaMemsetAsync(async_flag_dev, 0, sizeof(int64_t), st));
      CUDA_TRY(h, cudaEventRecord(as->done, st));
      s.n_certified = B;
      s.launches = 1;
      as->stats = s;
      as->n_ev = 0;
      as->trivial = true;
      as->pending = true;
      return RASS_OK;
    }
    CUDA_TRY(h, cudaStreamSynchronize(st));
    s.n_certified = B;
    s.launches = 1;
    if (stats) *stats = s;
    return RASS_OK;
  }
  if ((rc = refresh_store_scalars(h))) return rc;
  int path = resolve_path(h, B, k);
  int64_t* flag_out = as ? async_flag_dev : nullptr;   // published by the last CTA of the last finish launch
  // the second chance is the bf16 tcgen05 pass: the streaming scan keeps 32 per warp only, and the queries an int8
  // pass could not certify need the smaller allowance of the bf16 shadow
  if (robust && (path == RASS_PATH_STREAM || path == RASS_PATH_UMMA8)) path = RASS_PATH_UMMA;
  s.path = path;
  if (!(as && h->async_overlap) && (rc = select_scan_offsets(h, st))) return rc;
  // (query_prep_kernel resets the per-search device counters ws.scal)
  if (!as) CUDA_TRY(h, cudaEventRecord(h->ev[0], st));
  if ((rc = launch_query_prep(h, ws, q_dev, B, st))) return rc;
  s.launches = 1;
  size_t n_ev = 0;
  if (path == RASS_PATH_EXACT) {
    for (int i = 0; i < B; ++i) ws.flagged_host[i] = i;
    CUDA_TRY(h, cudaEventRecord(h->ev[1], st));
    if ((rc = launch_exact(h, ws, k, ws.flagged_host, B, out_rows, out_scores, out_keys, st, &s.launches))) return rc;
    s.n_fallback = B;
    s.passes = (B + RASS_EXACT_NQ - 1) / RASS_EXACT_NQ;
    s.bytes_streamed = (int64_t)s.passes * h->n_rows * h->dim_pad * ((h->flags & RASS_BF16_ONLY) ? 2 : 4);
  } else if (path == RASS_PATH_GEMM) {
    const int n_segs = scan_gemm_segs(h, B);
    const int seg = robust ? rass_tc_seg(k) : 256;
    if ((rc = ensure_pool(h, ws, (size_t)n_segs * seg, (size_t)n_segs, (size_t)B))) return rc;
    bool cleared = false;
    if ((rc = launch_seed_thresholds(h, ws, B, seg, (size_t)n_segs * B, &cleared, st))) return rc;
    CUDA_TRY(h, cudaEventRecord(get_event(h, ev_base + n_ev++), st));
    if ((rc = launch_scan_gemm(h, ws, B, seg, st, cleared))) return rc;
    CUDA_TRY(h, cudaEventRecord(get_event(h, ev_base + n_ev++), st));
    if ((rc = launch_finish(h, ws, 0, B, k, n_segs, seg, true, SCAN_BF16, out_rows, out_scores, out_keys, st, flag_out)))
      return rc;
    s.launches += cleared ? 3 : 4;
    s.passes = (B + 255) / 256;
    s.bytes_streamed = (int64_t)s.passes * h->n_rows * h->dim_pad * 2;
  } else {
    const bool int8 = path == RASS_PATH_UMMA8;
    const bool umma = path == RASS_PATH_UMMA || int8;
    const ScanOperands ops = int8 ? SCAN_INT8 : (umma ? SCAN_BF16 : SCAN_FP32_Q);
    const int n_segs = umma ? scan_umma_segs(h) : scan_stream_segs(h);
    const int seg = umma ? (robust ? rass_tc_seg(k) : 256) : RASS_STREAM_SEG;
    if ((rc = ensure_pool(h, ws, (size_t)n_segs * seg, (size_t)n_segs))) return rc;
    bool cleared = false;
    if (umma) {
      if ((rc = launch_seed_thresholds(h, ws, B, seg, (size_t)n_segs * RASS_GROUP_Q, &cleared, st, int8))) return rc;
      s.launches += 1;
    }
    for (int g0 = 0; g0 < B; g0 += RASS_GROUP_Q) {
      const int ng = std::min(RASS_GROUP_Q, B - g0);
      CUDA_TRY(h, cudaEventRecord(get_event(h, ev_base + n_ev++), st));
      if (umma) {
        const bool skip_clear = cleared && g0 == 0;      // the seed kernel emptied the pool for the first group
        if ((rc = launch_scan_umma(h, ws, g0, ng, seg, st, skip_clear, int8))) return rc;
        s.launches += skip_clear ? 1 : 2;
        s.passes += 1;
      } else {
        for (int q0 = g0; q0 < g0 + ng; q0 += 2) {
          if ((rc = launch_scan_stream(h, ws, q0, std::min(2, g0 + ng - q0), g0, st))) return rc;
          s.launches += 1;
          s.passes += 1;
        }
      }
      CUDA_TRY(h, cudaEventRecord(get_event(h, ev_base + n_ev++), st));
      if ((rc = launch_finish(h, ws, g0, ng, k, n_segs, seg, true, ops, out_rows, out_scores, out_keys, st, flag_out)))
        return rc;
      s.launches += 1;
    }
    s.bytes_streamed = (int64_t)s.passes * h->n_rows * h->dim_pad * (int8 ? 1 : 2);
  }
  if (as) {
    if (path == RASS_PATH_EXACT) return rass_fail(h, RASS_E_INVALID, "the fp64 scan has no async form");
    CUDA_TRY(h, cudaMemcpyAsync(as->scal_host, ws.scal, sizeof(SearchScalars), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaEventRecord(as->done, st));
    as->stats = s;
    as->k = k;
    as->n_ev = n_ev;
    as->trivial = false;
    as->pending = true;
    return RASS_OK;
  }
  if (path != RASS_PATH_EXACT) {
    CUDA_TRY(h, cudaEventRecord(h->ev[1], st));
    CUDA_TRY(h, cudaMemcpyAsync(h->scal_host, ws.scal, sizeof(SearchScalars), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    const int nf = h->scal_host->flagged_n;
    note_int8_outcome(h, s.path, B, k, nf, robust);
    s.n_certified = h->scal_host->n_certified;
    s.max_candidates = h->scal_host->max_cand;
    if (nf > 0) {
      CUDA_TRY(h, cudaMemcpyAsync(ws.flagged_host, ws.flagged, (size_t)nf * sizeof(int), cudaMemcpyDeviceToHost, st));
      CUDA_TRY(h, cudaStreamSynchronize(st));
      std::sort(ws.flagged_host, ws.flagged_host + nf);
      // k > 32: wider segments; an int8 pass: the bf16 pass (with rass_tc_seg(k) segments)
      const bool second_chance = !robust && (path == RASS_PATH_UMMA8 || (k > 32 && rass_tc_seg(k) != 256));
      if (second_chance) {
        // the recursive search also reuses the timing events: keep this pass's times
        float pre = 0.f;
        CUDA_TRY(h, cudaEventElapsedTime(&pre, h->ev[0], h->ev[1]));
        if ((rc = scan_ms_of(h, ev_base, n_ev, &first_scan_ms))) return rc;
        n_ev = 0;
        first_total_ms = pre;
        // the recursive search reuses every workspace of this one, so stage ids, queries and results on the side
        if ((size_t)nf > h->retry_cap || k > h->retry_k) {
          const size_t cap = std::max<size_t>((size_t)nf * 2, 256);
          const int kk = std::max(k, h->retry_k);
          cudaFree(h->retry_ids); cudaFree(h->retry_q); cudaFree(h->retry_rows); cudaFree(h->retry_scores);
          cudaFree(h->retry_keys);
          h->retry_ids = nullptr; h->retry_q = nullptr; h->retry_rows = nullptr; h->retry_scores = nullptr;
          h->retry_keys = nullptr;
          h->retry_cap = 0;
          CUDA_TRY(h, cudaMalloc(&h->retry_ids, cap * sizeof(int)));
          CUDA_TRY(h, cudaMalloc(&h->retry_q, cap * h->dim * sizeof(float)));
          CUDA_TRY(h, cudaMalloc(&h->retry_rows, cap * kk * sizeof(int64_t)));
          CUDA_TRY(h, cudaMalloc(&h->retry_scores, cap * kk * sizeof(float)));
          CUDA_TRY(h, cudaMalloc(&h->retry_keys, cap * kk * sizeof(double)));
          h->retry_cap = cap;
          h->retry_k = kk;
        }
        CUDA_TRY(h, cudaMemcpyAsync(h->retry_ids, ws.flagged_host, (size_t)nf * sizeof(int), cudaMemcpyHostToDevice, st));
        gather_queries_kernel<<<nf, 256, 0, st>>>(q_dev, h->retry_ids, h->dim, h->retry_q);
        CUDA_TRY(h, cudaGetLastError());
        rass_stats s2;
        if ((rc = search_core_body(h, ws, h->retry_q, nf, k, h->retry_rows, h->retry_scores, h->retry_keys, &s2, true,
                                   -1, nullptr, st)))
          return rc;
        scatter_results_kernel<<<nf, 128, 0, st>>>(h->retry_ids, k, h->retry_rows, h->retry_scores, h->retry_keys,
                                                   out_rows, out_scores, out_keys);
        CUDA_TRY(h, cudaGetLastError());
        s.n_certified += s2.n_certified;
        s.n_fallback = s2.n_fallback;
        s.n_retried = nf;
        s.launches += s2.launches + 2;
        s.passes += s2.passes;
        s.bytes_streamed += s2.bytes_streamed;
        retry_scan_ms = s2.scan_ms;
        retry_total_ms = s2.total_ms;
      } else {
        if ((rc = launch_exact(h, ws, k, ws.flagged_host, nf, out_rows, out_scores, out_keys, st, &s.launches))) return rc;
        s.n_fallback = nf;
      }
    }
  }
  CUDA_TRY(h, cudaEventRecord(h->ev[2], st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  if (first_total_ms >= 0.0) {
    s.total_ms = first_total_ms + retry_total_ms;
  } else {
    float ms = 0.f;
    CUDA_TRY(h, cudaEventElapsedTime(&ms, h->ev[0], h->ev[2]));
    s.total_ms = ms;
  }
  double scan = 0.0;
  if ((rc = scan_ms_of(h, ev_base, n_ev, &scan))) return rc;
  s.scan_ms = first_scan_ms + scan + retry_scan_ms;
  s.finish_ms = s.total_ms - s.scan_ms;
  h->last_stats = s;
  if (stats) *stats = s;
  return RASS_OK;
}

int search_core(rass_engine* h, const float* q_dev, int B, int k, int64_t* out_rows, float* out_scores,
                double* out_keys, rass_stats* stats, int async_slot, int64_t* async_flag_dev) {
  if (B < 1) return rass_fail(h, RASS_E_INVALID, "B must be >= 1");
  if (k < 1 || k > RASS_MAX_K) return rass_fail(h, RASS_E_INVALID, "k must be in [1, %d], got %d", RASS_MAX_K, k);
  // the stream and the workspace of the search: the engine stream and ws[0], except for an async slot under
  // RASS_OPT_ASYNC_OVERLAP, which runs on its own stream in its own workspace
  cudaStream_t st = eng_stream(h);
  SearchWs* ws = &h->ws[0];
  if (h->async_overlap && async_slot < 0) {
    // a blocking search shares slot 0's workspace (and must see everything enqueued so far): order it behind the
    // searches in flight
    for (auto& a : h->aslot)
      if (a.pending && a.done) CUDA_TRY(h, cudaStreamWaitEvent(st, a.done, 0));
  } else if (h->async_overlap) {
    if (h->aslot[async_slot].pending)
      return rass_fail(h, RASS_E_INVALID, "async slot %d still has a search in flight", async_slot);
    if (!h->slot_stream[async_slot]) {
      CUDA_TRY(h, cudaStreamCreateWithFlags(&h->slot_stream[async_slot], cudaStreamNonBlocking));
      CUDA_TRY(h, cudaEventCreateWithFlags(&h->slot_fork[async_slot], cudaEventDisableTiming));
    }
    // the folded filter offsets are shared by both slots: (re)build them ahead of the fork, on the engine stream
    const int rc = select_scan_offsets(h, st);
    if (rc) return rc;
    CUDA_TRY(h, cudaEventRecord(h->slot_fork[async_slot], st));
    st = h->slot_stream[async_slot];
    CUDA_TRY(h, cudaStreamWaitEvent(st, h->slot_fork[async_slot], 0));
    ws = &h->ws[async_slot];
    if (!ws->scal) {          // slot 1's workspace, on its first use
      CUDA_TRY(h, cudaMalloc(&ws->scal, sizeof(SearchScalars)));
      CUDA_TRY(h, cudaMemsetAsync(ws->scal, 0, sizeof(SearchScalars), st));
    }
  }
  return search_core_body(h, *ws, q_dev, B, k, out_rows, out_scores, out_keys, stats, false, async_slot,
                          async_flag_dev, st);
}

extern "C" int rass_search_knn_dev_async(rass_engine* h, const float* q_dev, int B, int k, int64_t* out_rows_dev,
                                         float* out_scores_dev, double* out_keys_dev, int slot,
                                         int64_t* flag_out_dev) {
  SHARDED(h, sharded_search_knn_dev_async(h, q_dev, B, k, out_rows_dev, out_scores_dev, out_keys_dev, slot, flag_out_dev));
  CHECK_HANDLE(h);
  if (!q_dev || !out_rows_dev || !out_scores_dev) return rass_fail(h, RASS_E_INVALID, "null buffer");
  if (slot < 0 || slot > 1) return rass_fail(h, RASS_E_INVALID, "slot must be 0 or 1");
  return search_core(h, q_dev, B, k, out_rows_dev, out_scores_dev, out_keys_dev, nullptr, slot, flag_out_dev);
}

extern "C" int rass_search_knn_dev_wait(rass_engine* h, int slot, rass_stats* stats) {
  SHARDED(h, sharded_search_knn_dev_wait(h, slot, stats));
  CHECK_HANDLE(h);
  if (slot < 0 || slot > 1) return rass_fail(h, RASS_E_INVALID, "slot must be 0 or 1");
  rass_engine::AsyncSlot& a = h->aslot[slot];
  if (!a.pending) return rass_fail(h, RASS_E_INVALID, "no search in flight in slot %d", slot);
  CUDA_TRY(h, cudaEventSynchronize(a.done));
  a.pending = false;
  rass_stats s = a.stats;
  int nf = 0;
  if (!a.trivial) {
    nf = a.scal_host->flagged_n;
    note_int8_outcome(h, s.path, s.n_queries, a.k, nf, false);
    s.n_certified = a.scal_host->n_certified;
    s.max_candidates = a.scal_host->max_cand;
    const int rc = scan_ms_of(h, (size_t)1024 * (slot + 1), a.n_ev, &s.scan_ms);
    if (rc) return rc;
  }
  s.n_fallback = nf;          // queries whose outputs are NOT final: the caller repeats the search with the blocking call
  if (stats) *stats = s;
  return nf > 0 ? RASS_E_AGAIN : RASS_OK;
}

extern "C" int rass_async_join(rass_engine* h, int slot, void* stream) {
  SHARDED(h, sharded_async_join(h, slot, stream));
  CHECK_HANDLE(h);
  if (slot < 0 || slot > 1) return rass_fail(h, RASS_E_INVALID, "slot must be 0 or 1");
  rass_engine::AsyncSlot& a = h->aslot[slot];
  if (!a.pending || !a.done) return rass_fail(h, RASS_E_INVALID, "no search in flight in slot %d", slot);
  CUDA_TRY(h, cudaStreamWaitEvent(reinterpret_cast<cudaStream_t>(stream), a.done, 0));
  return RASS_OK;
}

extern "C" int rass_search_knn_dev(rass_engine* h, const float* q_dev, int B, int k, int64_t* out_rows_dev,
                                   float* out_scores_dev, double* out_keys_dev, rass_stats* stats) {
  SHARDED(h, sharded_search_knn_dev(h, q_dev, B, k, out_rows_dev, out_scores_dev, out_keys_dev, stats));
  CHECK_HANDLE(h);
  if (!q_dev || !out_rows_dev || !out_scores_dev) return rass_fail(h, RASS_E_INVALID, "null buffer");
  return search_core(h, q_dev, B, k, out_rows_dev, out_scores_dev, out_keys_dev, stats);
}

int stage_queries(rass_engine* h, const float* q_host, int B, float** q_dev_out) {
  const size_t n = (size_t)B * h->dim;
  if (n > h->q_stage_cap) {
    CUDA_TRY(h, cudaStreamSynchronize(eng_stream(h)));
    REALLOC_HOST(h, h->q_stage_host, n);
    cudaFree(h->q_stage_dev);
    h->q_stage_dev = nullptr;
    CUDA_TRY(h, cudaMalloc(&h->q_stage_dev, n * 4));
    h->q_stage_cap = n;
  }
  memcpy(h->q_stage_host, q_host, n * 4);
  CUDA_TRY(h, cudaMemcpyAsync(h->q_stage_dev, h->q_stage_host, n * 4, cudaMemcpyHostToDevice, eng_stream(h)));
  *q_dev_out = h->q_stage_dev;
  return RASS_OK;
}

extern "C" int rass_search_knn(rass_engine* h, const float* q_host, int B, int k, int64_t* out_rows,
                               float* out_scores, double* out_keys, rass_stats* stats) {
  SHARDED(h, sharded_search_knn(h, q_host, B, k, out_rows, out_scores, out_keys, stats));
  CHECK_HANDLE(h);
  if (!q_host || !out_rows || !out_scores) return rass_fail(h, RASS_E_INVALID, "null buffer");
  if (B < 1) return rass_fail(h, RASS_E_INVALID, "B must be >= 1");
  if (k < 1 || k > RASS_MAX_K) return rass_fail(h, RASS_E_INVALID, "k must be in [1, %d], got %d", RASS_MAX_K, k);
  int rc;
  float* q_dev = nullptr;
  if ((rc = stage_queries(h, q_host, B, &q_dev))) return rc;
  const size_t n_out = (size_t)B * k;
  if ((rc = ensure_out_workspace(h, n_out))) return rc;
  if ((rc = search_core(h, q_dev, B, k, h->out_rows, h->out_scores, out_keys ? h->out_keys : nullptr, stats)))
    return rc;
  cudaStream_t st = eng_stream(h);
  CUDA_TRY(h, cudaMemcpyAsync(h->out_rows_host, h->out_rows, n_out * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaMemcpyAsync(h->out_scores_host, h->out_scores, n_out * 4, cudaMemcpyDeviceToHost, st));
  if (out_keys) CUDA_TRY(h, cudaMemcpyAsync(h->out_keys_host, h->out_keys, n_out * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  memcpy(out_rows, h->out_rows_host, n_out * 8);
  memcpy(out_scores, h->out_scores_host, n_out * 4);
  if (out_keys) memcpy(out_keys, h->out_keys_host, n_out * 8);
  return RASS_OK;
}

extern "C" int rass_merge_topk_dev(rass_engine* h, const double* keys_dev, const int64_t* rows_dev,
                                   int64_t shard_stride, int G, int B, int k, int64_t* out_rows_dev,
                                   float* out_scores_dev, double* out_keys_dev) {
  CHECK_HANDLE(h);
  if (!keys_dev || !rows_dev || !out_rows_dev || !out_scores_dev || G < 1 || B < 1 || k < 1)
    return rass_fail(h, RASS_E_INVALID, "bad merge arguments");
  cudaStream_t st = eng_stream(h);
  int rc = launch_merge_topk(h, keys_dev, rows_dev, shard_stride, G, B, k, out_rows_dev, out_scores_dev,
                             out_keys_dev, st);
  if (rc) return rc;
  return RASS_OK;   // enqueued on the engine stream; the caller synchronises (rass_sync) when it needs the result
}

// the same merge for per-shard FUSED hybrid lists: the keys are raw scores, larger is better whatever the vector metric
extern "C" int rass_merge_scores_dev(rass_engine* h, const double* scores_dev, const int64_t* rows_dev,
                                     int64_t shard_stride, int G, int B, int k, int64_t* out_rows_dev,
                                     float* out_scores_dev, double* out_keys_dev) {
  CHECK_HANDLE(h);
  if (!scores_dev || !rows_dev || !out_rows_dev || !out_scores_dev || G < 1 || B < 1 || k < 1)
    return rass_fail(h, RASS_E_INVALID, "bad merge arguments");
  return launch_merge_topk(h, scores_dev, rows_dev, shard_stride, G, B, k, out_rows_dev, out_scores_dev, out_keys_dev,
                           eng_stream(h), true);
}

// bool.filter of the next hybrid queries as a per-row pass mask (NULL clears it)
extern "C" int rass_set_row_filter(rass_engine* h, const uint8_t* mask_host, int64_t n) {
  SHARDED(h, sharded_set_row_filter(h, mask_host, n));
  CHECK_HANDLE(h);
  cudaStream_t st = eng_stream(h);
  if (!mask_host) {
    CUDA_TRY(h, cudaStreamSynchronize(st));
    cudaFree(h->row_filter);
    h->row_filter = nullptr;
    h->row_filter_rows = 0;
    h->row_filter_cap = 0;
    h->sb_filtered_dirty = true;
    return RASS_OK;
  }
  if (n < 0) return rass_fail(h, RASS_E_INVALID, "bad filter length");
  if ((size_t)n > h->row_filter_cap || !h->row_filter) {
    CUDA_TRY(h, cudaStreamSynchronize(st));
    cudaFree(h->row_filter);
    h->row_filter = nullptr;
    const size_t cap = std::max<size_t>((size_t)n, 1024) * 2;
    CUDA_TRY(h, cudaMalloc(&h->row_filter, cap));
    h->row_filter_cap = cap;
  }
  CUDA_TRY(h, cudaMemcpyAsync(h->row_filter, mask_host, (size_t)n, cudaMemcpyHostToDevice, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  h->row_filter_rows = n;
  h->sb_filtered_dirty = true;
  return RASS_OK;
}

// bool.filter as a list of the rows that pass (term filters select few rows: a patient's documents): the mask is
// zeroed and the listed rows are set on the device, so the host never touches O(rows) bytes per query
__global__ void set_mask_rows_kernel(const int64_t* __restrict__ rows, int64_t n, int64_t total, uint8_t* __restrict__ mask) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && rows[i] >= 0 && rows[i] < total) mask[rows[i]] = 1;
}

extern "C" int rass_set_row_filter_rows(rass_engine* h, const int64_t* rows_host, int64_t n, int64_t total_rows) {
  SHARDED(h, sharded_set_row_filter_rows(h, rows_host, n, total_rows));
  CHECK_HANDLE(h);
  if (n < 0 || total_rows < 0 || (n && !rows_host)) return rass_fail(h, RASS_E_INVALID, "bad filter rows");
  cudaStream_t st = eng_stream(h);
  if ((size_t)total_rows > h->row_filter_cap || !h->row_filter) {
    CUDA_TRY(h, cudaStreamSynchronize(st));
    cudaFree(h->row_filter);
    h->row_filter = nullptr;
    const size_t cap = std::max<size_t>((size_t)total_rows, 1024) * 2;
    CUDA_TRY(h, cudaMalloc(&h->row_filter, cap));
    h->row_filter_cap = cap;
  }
  if ((size_t)n > h->filter_rows_cap) {
    CUDA_TRY(h, cudaStreamSynchronize(st));
    cudaFree(h->filter_rows_dev);
    h->filter_rows_dev = nullptr;
    h->filter_rows_cap = 0;
    const size_t cap = std::max<size_t>((size_t)n * 2, 4096);
    CUDA_TRY(h, cudaMalloc(&h->filter_rows_dev, cap * sizeof(int64_t)));
    h->filter_rows_cap = cap;
  }
  CUDA_TRY(h, cudaMemsetAsync(h->row_filter, 0, (size_t)std::max<int64_t>(total_rows, 1), st));
  if (n) {
    CUDA_TRY(h, cudaMemcpyAsync(h->filter_rows_dev, rows_host, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    set_mask_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h->filter_rows_dev, n, total_rows, h->row_filter);
    CUDA_TRY(h, cudaGetLastError());
  }
  CUDA_TRY(h, cudaStreamSynchronize(st));     // rows_host may be pageable and freed on return
  h->row_filter_rows = total_rows;
  h->sb_filtered_dirty = true;
  return RASS_OK;
}

// stored values of a LIST of rows (the hits of one search) in one gather + one copy: [n, dim] fp32
__global__ void gather_rows_kernel(const float* __restrict__ x32, const __nv_bfloat16* __restrict__ x16, int dim,
                                   int dim_pad, const int64_t* __restrict__ rows, float* __restrict__ out) {
  const int64_t r = rows[blockIdx.x];
  for (int j = threadIdx.x; j < dim; j += blockDim.x)
    out[(size_t)blockIdx.x * dim + j] = x32 ? x32[(size_t)r * dim_pad + j] : __bfloat162float(x16[(size_t)r * dim_pad + j]);
}

extern "C" int rass_read_rows_list(rass_engine* h, const int64_t* rows_host, int64_t n, float* out_host) {
  SHARDED(h, sharded_read_rows_list(h, rows_host, n, out_host));
  CHECK_HANDLE(h);
  if (n < 0 || (n && (!rows_host || !out_host))) return rass_fail(h, RASS_E_INVALID, "bad arguments");
  if (n == 0) return RASS_OK;
  for (int64_t i = 0; i < n; ++i)
    if (rows_host[i] < 0 || rows_host[i] >= h->n_rows)
      return rass_fail(h, RASS_E_NOTFOUND, "row %lld out of range", (long long)rows_host[i]);
  cudaStream_t st = eng_stream(h);
  int rc;
  if ((size_t)n > h->filter_rows_cap) {
    CUDA_TRY(h, cudaStreamSynchronize(st));
    cudaFree(h->filter_rows_dev);
    h->filter_rows_dev = nullptr;
    h->filter_rows_cap = 0;
    const size_t cap = std::max<size_t>((size_t)n * 2, 4096);
    CUDA_TRY(h, cudaMalloc(&h->filter_rows_dev, cap * sizeof(int64_t)));
    h->filter_rows_cap = cap;
  }
  if ((rc = ensure_dev_stage(h, (size_t)n * h->dim * 4))) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(h->filter_rows_dev, rows_host, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  gather_rows_kernel<<<(unsigned)n, 256, 0, st>>>((h->flags & RASS_BF16_ONLY) ? nullptr : h->x32, h->x16, h->dim,
                                                  h->dim_pad, h->filter_rows_dev, h->dev_stage);
  CUDA_TRY(h, cudaGetLastError());
  CUDA_TRY(h, cudaMemcpyAsync(out_host, h->dev_stage, (size_t)n * h->dim * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return RASS_OK;
}

// Debug entry (not part of the reference surface): raw tcgen05 dot products of <= 64 queries against every row,
// out_host [n_rows, 64].  Lets the tests check the TMA/UMMA descriptors in isolation.
extern "C" int rass_debug_gemm_scores(rass_engine* h, const float* q_host, int B, float* out_host) {
  SHARDED(h, rass_fail(h, RASS_E_UNSUPPORTED, "debug entry points take a single-device handle"));
  CHECK_HANDLE(h);
  if (!q_host || !out_host || B < 1 || B > RASS_QPAD) return rass_fail(h, RASS_E_INVALID, "bad arguments");
  if (h->n_rows == 0) return RASS_OK;
  int rc;
  float* q_dev = nullptr;
  SearchWs& ws = h->ws[0];
  if ((rc = ensure_query_workspace(h, ws, B))) return rc;
  if ((rc = stage_queries(h, q_host, B, &q_dev))) return rc;
  cudaStream_t st = eng_stream(h);
  if ((rc = launch_query_prep(h, ws, q_dev, B, st))) return rc;
  if ((rc = select_scan_offsets(h, st))) return rc;
  return gemm_selftest(h, ws, B, out_host, st);
}

extern "C" int rass_debug_umma_scores(rass_engine* h, const float* q_host, int B, float* out_host) {
  SHARDED(h, rass_fail(h, RASS_E_UNSUPPORTED, "debug entry points take a single-device handle"));
  CHECK_HANDLE(h);
  if (!q_host || !out_host || B < 1 || B > RASS_GROUP_Q) return rass_fail(h, RASS_E_INVALID, "bad arguments");
  if (h->n_rows == 0) return RASS_OK;
  int rc;
  float* q_dev = nullptr;
  SearchWs& ws = h->ws[0];
  if ((rc = ensure_query_workspace(h, ws, B))) return rc;
  if ((rc = stage_queries(h, q_host, B, &q_dev))) return rc;
  cudaStream_t st = eng_stream(h);
  if ((rc = launch_query_prep(h, ws, q_dev, B, st))) return rc;
  if ((rc = select_scan_offsets(h, st))) return rc;
  return umma_selftest(h, ws, 0, out_host, st);
}

extern "C" int rass_debug_umma8_scores(rass_engine* h, const float* q_host, int B, int32_t* acc_host, int8_t* x8_host,
                                       int8_t* q8_host) {
  SHARDED(h, rass_fail(h, RASS_E_UNSUPPORTED, "debug entry points take a single-device handle"));
  CHECK_HANDLE(h);
  if (!q_host || !acc_host || B < 1 || B > RASS_GROUP_Q) return rass_fail(h, RASS_E_INVALID, "bad arguments");
  if (!has_int8_shadow(h->flags)) return rass_fail(h, RASS_E_UNSUPPORTED, "the store has no int8 shadow");
  if (h->n_rows == 0) return RASS_OK;
  int rc;
  float* q_dev = nullptr;
  SearchWs& ws = h->ws[0];
  if ((rc = ensure_query_workspace(h, ws, B))) return rc;
  if ((rc = stage_queries(h, q_host, B, &q_dev))) return rc;
  cudaStream_t st = eng_stream(h);
  if ((rc = launch_query_prep(h, ws, q_dev, B, st))) return rc;
  if ((rc = select_scan_offsets(h, st))) return rc;
  if ((rc = umma8_selftest(h, ws, acc_host, st))) return rc;
  const size_t d = (size_t)h->dim_pad;
  if (x8_host) CUDA_TRY(h, cudaMemcpyAsync(x8_host, h->x8, (size_t)h->n_rows * d, cudaMemcpyDeviceToHost, st));
  if (q8_host) CUDA_TRY(h, cudaMemcpyAsync(q8_host, ws.q8, 2 * RASS_GROUP_Q * d, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return RASS_OK;
}
