// Single-process multi-GPU: one engine handle over several devices (rass_create_sharded).
//
// The reference is ONE uvicorn process (app/main.py:3356-3357) that asks OpenSearch for `number_of_shards`
// (app/main.py:357) and lets the coordinator node merge the per-shard hits.  Here the "cluster" is the GPUs of one
// NVSwitch box inside the caller's process: the coordinator handle owns one single-device engine per GPU plus a worker
// thread each (so the G devices are driven in parallel), and every entry point of include/rass_b200.h works on it.
//
//   rows      global row r lives on shard (r >> 10) % G (RowMap, common.cuh): an index that grows by bulk appends stays
//             balanced, and ids stay dense and append-ordered, which is what the "row ascending" tie-break needs.
//   search    queries are copied to every device; each shard runs the ordinary exact search and its finish kernel
//             stores its [B, k] (fp64 key, global row) list STRAIGHT INTO the coordinator device's gather buffer through
//             peer-mapped memory over NVLink -- compute and exchange are one kernel, there is no all-gather; the
//             coordinator then runs merge_topk_kernel over the G lists.  Without peer access the lists travel by
//             cudaMemcpyPeerAsync.
//   hybrid    postings are split by the same row map with corpus-wide statistics (scores are shard-invariant); the
//             merged k nearest are handed to every shard, which fuses its own rows and again stores its fused top-k into
//             the coordinator's buffer; a raw-score merge finishes.
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>

#include "common.cuh"

namespace {

class Worker {
 public:
  explicit Worker(int device) : device_(device), th_([this] { loop(); }) {}
  ~Worker() {
    {
      std::lock_guard<std::mutex> l(m_);
      stop_ = true;
    }
    cv_.notify_all();
    th_.join();
  }
  void post(std::function<int()> fn) {
    {
      std::lock_guard<std::mutex> l(m_);
      job_ = std::move(fn);
      has_job_ = true;
      done_ = false;
    }
    cv_.notify_all();
  }
  int wait() {
    std::unique_lock<std::mutex> l(m_);
    cv_done_.wait(l, [this] { return done_; });
    return rc_;
  }

 private:
  void loop() {
    cudaSetDevice(device_);
    for (;;) {
      std::function<int()> fn;
      {
        std::unique_lock<std::mutex> l(m_);
        cv_.wait(l, [this] { return has_job_ || stop_; });
        if (stop_) return;
        fn = std::move(job_);
        has_job_ = false;
      }
      const int rc = fn();
      {
        std::lock_guard<std::mutex> l(m_);
        rc_ = rc;
        done_ = true;
      }
      cv_done_.notify_all();
    }
  }
  int device_;
  std::mutex m_;
  std::condition_variable cv_, cv_done_;
  std::function<int()> job_;
  bool has_job_ = false, done_ = true, stop_ = false;
  int rc_ = 0;
  std::thread th_;     // last: the thread starts with every other member alive
};

}  // namespace

struct ShardSet {
  int G = 0;
  std::vector<rass_engine*> sh;
  std::vector<int> dev;
  std::vector<std::unique_ptr<Worker>> workers;
  bool peer_ok = true;              // every shard can store into the coordinator device's memory
  // coordinator-device buffers, two sets (async slots); [G][cap] lists + [G] certificate words
  size_t cap = 0;                   // entries per shard list
  double* g_keys[2] = {nullptr, nullptr};
  int64_t* g_rows[2] = {nullptr, nullptr};
  int64_t* g_flag[2] = {nullptr, nullptr};
  // shard-local landing buffers when peer stores are not possible
  std::vector<double*> l_keys;
  std::vector<int64_t*> l_rows;
  // merged lists on the coordinator device and their pinned mirrors
  int64_t* m_rows = nullptr;
  float* m_scores = nullptr;
  double* m_keys = nullptr;
  int64_t* m_rows_host = nullptr;
  float* m_scores_host = nullptr;
  double* m_keys_host = nullptr;
  // per shard: device copies of the (global) knn list for the fusion step, query broadcast buffers of the async path
  std::vector<int64_t*> knn_rows;
  std::vector<float*> knn_scores;
  std::vector<float*> q_bcast[2];
  size_t knn_cap = 0, q_cap = 0;
  cudaEvent_t ev_q[2] = {nullptr, nullptr};             // coordinator: queries of the slot are ready
  std::vector<cudaEvent_t> ev_sh[2];                    // shard g: its list of the slot is in the gather buffer
  cudaEvent_t ev_done[2] = {nullptr, nullptr};
  bool pending[2] = {false, false};
  rass_stats slot_stats[2];
  std::vector<rass_stats> st;
};

rass_engine* sharded_first(rass_engine* h) { return h->shards->sh[0]; }
const std::vector<rass_engine*>& sharded_shards(rass_engine* h) { return h->shards->sh; }

static RowMap shard_map(const rass_engine* h, int g) { return RowMap{h->rmap.base, g, h->shards->G, RASS_SHARD_BLOCK_LOG2}; }
static int shard_of(const rass_engine* h, int64_t row) { return (int)((row >> RASS_SHARD_BLOCK_LOG2) % h->shards->G); }
// number of global rows < total that live on shard g
static int64_t shard_rows_below(const rass_engine* h, int g, int64_t total) {
  const int64_t blk = int64_t(1) << RASS_SHARD_BLOCK_LOG2, G = h->shards->G;
  const int64_t full = total / blk, rem = total % blk;
  int64_t n = (full / G) * blk + ((full % G) > g ? blk : 0);
  if (rem && (full % G) == g) n += rem;
  return n;
}

// cudaMemcpyPeer is asynchronous with respect to the host and is not ordered against cudaStreamNonBlocking streams, which
// is what every engine runs on: copy on the shard's own stream and wait for it.
static cudaError_t peer_copy_sync(void* dst, int dst_dev, const void* src, int src_dev, size_t bytes, cudaStream_t st) {
  cudaError_t e = cudaMemcpyPeerAsync(dst, dst_dev, src, src_dev, bytes, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  return e;
}

static int run_all(rass_engine* h, const std::function<int(int)>& fn) {
  ShardSet* S = h->shards;
  for (int g = 0; g < S->G; ++g) S->workers[g]->post([&fn, g] { return fn(g); });
  int rc = RASS_OK, bad = -1;
  for (int g = 0; g < S->G; ++g) {
    const int r = S->workers[g]->wait();
    if (r && !rc) { rc = r; bad = g; }
  }
  if (rc) h->err = "shard " + std::to_string(bad) + " (device " + std::to_string(S->dev[bad]) + "): " + S->sh[bad]->err;
  cudaSetDevice(h->device);
  return rc;
}

static void free_gather(ShardSet* S) {
  for (int s = 0; s < 2; ++s) {
    cudaFree(S->g_keys[s]); cudaFree(S->g_rows[s]); cudaFree(S->g_flag[s]);
    S->g_keys[s] = nullptr; S->g_rows[s] = nullptr; S->g_flag[s] = nullptr;
  }
  cudaFree(S->m_rows); cudaFree(S->m_scores); cudaFree(S->m_keys);
  cudaFreeHost(S->m_rows_host); cudaFreeHost(S->m_scores_host); cudaFreeHost(S->m_keys_host);
  S->m_rows = nullptr; S->m_scores = nullptr; S->m_keys = nullptr;
  S->m_rows_host = nullptr; S->m_scores_host = nullptr; S->m_keys_host = nullptr;
}

// gather + merged buffers for lists of n = B * k entries
static int ensure_gather(rass_engine* h, size_t n) {
  ShardSet* S = h->shards;
  if (n <= S->cap) return RASS_OK;
  cudaSetDevice(h->device);
  CUDA_TRY(h, cudaDeviceSynchronize());
  free_gather(S);
  const size_t cap = std::max<size_t>(n * 2, 4096);
  for (int s = 0; s < 2; ++s) {
    CUDA_TRY(h, cudaMalloc(&S->g_keys[s], (size_t)S->G * cap * sizeof(double)));
    CUDA_TRY(h, cudaMalloc(&S->g_rows[s], (size_t)S->G * cap * sizeof(int64_t)));
    CUDA_TRY(h, cudaMalloc(&S->g_flag[s], (size_t)S->G * sizeof(int64_t)));
    CUDA_TRY(h, cudaMemset(S->g_flag[s], 0, (size_t)S->G * sizeof(int64_t)));
  }
  CUDA_TRY(h, cudaMalloc(&S->m_rows, cap * sizeof(int64_t)));
  CUDA_TRY(h, cudaMalloc(&S->m_scores, cap * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&S->m_keys, cap * sizeof(double)));
  CUDA_TRY(h, cudaMallocHost(&S->m_rows_host, cap * sizeof(int64_t)));
  CUDA_TRY(h, cudaMallocHost(&S->m_scores_host, cap * sizeof(float)));
  CUDA_TRY(h, cudaMallocHost(&S->m_keys_host, cap * sizeof(double)));
  if (!S->peer_ok) {
    const int rc = run_all(h, [&](int g) {
      rass_engine* sh = S->sh[g];
      cudaFree(S->l_keys[g]); cudaFree(S->l_rows[g]);
      S->l_keys[g] = nullptr; S->l_rows[g] = nullptr;
      CUDA_TRY(sh, cudaMalloc(&S->l_keys[g], cap * sizeof(double)));
      CUDA_TRY(sh, cudaMalloc(&S->l_rows[g], cap * sizeof(int64_t)));
      return (int)RASS_OK;
    });
    if (rc) return rc;
  }
  S->cap = cap;
  return RASS_OK;
}

static int ensure_knn_bufs(rass_engine* h, size_t n) {
  ShardSet* S = h->shards;
  if (n <= S->knn_cap) return RASS_OK;
  const size_t cap = std::max<size_t>(n * 2, 4096);
  const int rc = run_all(h, [&](int g) {
    rass_engine* sh = S->sh[g];
    CUDA_TRY(sh, cudaStreamSynchronize(eng_stream(sh)));
    cudaFree(S->knn_rows[g]); cudaFree(S->knn_scores[g]);
    S->knn_rows[g] = nullptr; S->knn_scores[g] = nullptr;
    CUDA_TRY(sh, cudaMalloc(&S->knn_rows[g], cap * sizeof(int64_t)));
    CUDA_TRY(sh, cudaMalloc(&S->knn_scores[g], cap * sizeof(float)));
    return (int)RASS_OK;
  });
  if (rc) return rc;
  S->knn_cap = cap;
  return RASS_OK;
}

// ---------------------------------------------------------------------------------------------
// lifecycle
// ---------------------------------------------------------------------------------------------
extern "C" int rass_create_sharded(int dim, int metric, int n_devices, const int* device_ids, int64_t capacity_rows,
                                   uint32_t flags, rass_engine** out) {
  if (!out) return rass_fail(nullptr, RASS_E_INVALID, "out is null");
  *out = nullptr;
  if (n_devices < 1 || n_devices > 64 || !device_ids) return rass_fail(nullptr, RASS_E_INVALID, "bad device list");
  // (a device may be listed more than once: several shards then share it -- how the 1-GPU test box runs this file)
  if (n_devices == 1) return rass_create(dim, metric, device_ids[0], capacity_rows, flags, out);
  rass_engine* h = new rass_engine();
  ShardSet* S = new ShardSet();
  h->shards = S;
  h->dim = dim;
  h->dim_pad = (dim + 255) / 256 * 256;
  h->metric = metric;
  h->device = device_ids[0];
  h->flags = (flags & (RASS_KEEP_FP32 | RASS_BF16_ONLY)) ? flags : flags | RASS_KEEP_FP32;
  S->G = n_devices;
  const int64_t per = capacity_rows > 0 ? (capacity_rows + n_devices - 1) / n_devices + (int64_t(1) << RASS_SHARD_BLOCK_LOG2) : 0;
  for (int g = 0; g < n_devices; ++g) {
    rass_engine* sh = nullptr;
    const int rc = rass_create(dim, metric, device_ids[g], per, flags, &sh);
    if (rc) {
      for (rass_engine* e : S->sh) rass_destroy(e);
      delete S;
      delete h;
      return rc;       // g_create_error carries the shard's message
    }
    sh->rmap = RowMap{0, g, n_devices, RASS_SHARD_BLOCK_LOG2};
    S->sh.push_back(sh);
    S->dev.push_back(device_ids[g]);
  }
  // peer access: every shard stores its result lists into the coordinator device's memory
  for (int g = 1; g < n_devices; ++g) {
    int can = 0;
    if (device_ids[g] == device_ids[0]) continue;
    cudaSetDevice(device_ids[g]);
    if (cudaDeviceCanAccessPeer(&can, device_ids[g], device_ids[0]) != cudaSuccess || !can) {
      S->peer_ok = false;
    } else {
      const cudaError_t e = cudaDeviceEnablePeerAccess(device_ids[0], 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) S->peer_ok = false;
    }
    cudaGetLastError();
  }
  if (getenv("RASS_DEBUG_NO_PEER")) S->peer_ok = false;      // exercise the staged-copy exchange on a peer-capable box
  cudaSetDevice(h->device);
  auto bail = [&](const char* what) {
    g_create_error = std::string(what) + ": " + cudaGetErrorString(cudaGetLastError());
    rass_destroy(h);
    return (int)RASS_E_NCCL;
  };
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) return bail("coordinator stream");
  for (int s = 0; s < 2; ++s) {
    if (cudaEventCreateWithFlags(&S->ev_q[s], cudaEventDisableTiming) != cudaSuccess) return bail("event");
    if (cudaEventCreateWithFlags(&S->ev_done[s], cudaEventDisableTiming) != cudaSuccess) return bail("event");
    S->ev_sh[s].assign((size_t)n_devices, nullptr);
    S->q_bcast[s].assign((size_t)n_devices, nullptr);
  }
  S->l_keys.assign((size_t)n_devices, nullptr);
  S->l_rows.assign((size_t)n_devices, nullptr);
  S->knn_rows.assign((size_t)n_devices, nullptr);
  S->knn_scores.assign((size_t)n_devices, nullptr);
  S->st.resize((size_t)n_devices);
  for (int g = 0; g < n_devices; ++g) {
    cudaSetDevice(device_ids[g]);
    for (int s = 0; s < 2; ++s)
      if (cudaEventCreateWithFlags(&S->ev_sh[s][g], cudaEventDisableTiming) != cudaSuccess) return bail("event");
    S->workers.emplace_back(new Worker(device_ids[g]));
  }
  cudaSetDevice(h->device);
  *out = h;
  return RASS_OK;
}

int sharded_destroy(rass_engine* h) {
  ShardSet* S = h->shards;
  S->workers.clear();                     // joins the threads
  for (int g = 0; g < (int)S->sh.size(); ++g) {
    cudaSetDevice(S->dev[g]);
    cudaDeviceSynchronize();
    for (int s = 0; s < 2; ++s) {
      if (g < (int)S->ev_sh[s].size() && S->ev_sh[s][g]) cudaEventDestroy(S->ev_sh[s][g]);
      if (g < (int)S->q_bcast[s].size()) cudaFree(S->q_bcast[s][g]);
    }
    if (g < (int)S->l_keys.size()) { cudaFree(S->l_keys[g]); cudaFree(S->l_rows[g]); }
    if (g < (int)S->knn_rows.size()) { cudaFree(S->knn_rows[g]); cudaFree(S->knn_scores[g]); }
    rass_destroy(S->sh[g]);
  }
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  free_gather(S);
  for (int s = 0; s < 2; ++s) {
    if (S->ev_q[s]) cudaEventDestroy(S->ev_q[s]);
    if (S->ev_done[s]) cudaEventDestroy(S->ev_done[s]);
  }
  if (h->stream) cudaStreamDestroy(h->stream);
  delete S;
  h->shards = nullptr;
  delete h;
  return RASS_OK;
}

int sharded_set_option(rass_engine* h, int opt, int64_t value) {
  ShardSet* S = h->shards;
  if (opt == RASS_OPT_STREAM) {            // the stream the *_dev entry points of the coordinator are ordered on
    if (value == -1) { h->has_user_stream = false; h->user_stream = nullptr; }
    else { h->has_user_stream = true; h->user_stream = reinterpret_cast<cudaStream_t>(value); }
    return RASS_OK;
  }
  for (int g = 0; g < S->G; ++g) {
    const int rc = rass_set_option(S->sh[g], opt, value);
    if (rc) { h->err = S->sh[g]->err; return rc; }
  }
  if (opt == RASS_OPT_PATH) h->path = (int)value;
  if (opt == RASS_OPT_KNN_PREFILTER) h->knn_prefilter = value != 0;
  return RASS_OK;
}

int sharded_set_row_base(rass_engine* h, int64_t base) {
  h->rmap.base = base;
  for (rass_engine* sh : h->shards->sh) sh->rmap.base = base;
  return RASS_OK;
}

int sharded_sync(rass_engine* h) {
  const int rc = run_all(h, [&](int g) { return rass_sync(h->shards->sh[g]); });
  if (rc) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(eng_stream(h)));
  return RASS_OK;
}

// ---------------------------------------------------------------------------------------------
// store
// ---------------------------------------------------------------------------------------------
// global rows [first, first + n) in block runs: fn(g, global_row, run_len)
template <typename F>
static int for_runs_of_shard(const rass_engine* h, int g, int64_t first, int64_t n, F fn) {
  const int64_t blk = int64_t(1) << RASS_SHARD_BLOCK_LOG2;
  for (int64_t r = first; r < first + n;) {
    const int64_t run = std::min(first + n, (r / blk + 1) * blk) - r;
    if (shard_of(h, r) == g) {
      const int rc = fn(r, run);
      if (rc) return rc;
    }
    r += run;
  }
  return RASS_OK;
}

static int sharded_append_impl(rass_engine* h, const float* rows, bool on_device, int64_t n, int64_t* out_first_row) {
  ShardSet* S = h->shards;
  if (n < 0 || (n > 0 && !rows)) return rass_fail(h, RASS_E_INVALID, "bad rows");
  const int64_t first = h->n_rows;
  if (on_device) CUDA_TRY(h, cudaStreamSynchronize(eng_stream(h)));      // the caller's rows are complete
  const int rc = run_all(h, [&](int g) {
    rass_engine* sh = S->sh[g];
    return for_runs_of_shard(h, g, first, n, [&](int64_t r, int64_t run) {
      const float* src = rows + (size_t)(r - first) * h->dim;
      if (!on_device) return rass_append(sh, src, run, nullptr);
      if (S->dev[g] == h->device) return rass_append_dev(sh, src, run, nullptr);
      // device rows of the coordinator -> this shard's device (peer copy), then the ordinary device append
      float* tmp = nullptr;
      CUDA_TRY(sh, cudaMalloc(&tmp, (size_t)run * h->dim * 4));
      cudaError_t e = peer_copy_sync(tmp, S->dev[g], src, h->device, (size_t)run * h->dim * 4, eng_stream(sh));
      int rc2 = e == cudaSuccess ? rass_append_dev(sh, tmp, run, nullptr)
                                 : rass_fail(sh, RASS_E_NCCL, "peer copy of appended rows: %s", cudaGetErrorString(e));
      cudaFree(tmp);
      return rc2;
    });
  });
  if (rc) return rc;
  h->n_rows += n;
  h->n_live += n;
  h->dead.resize((size_t)h->n_rows, 0);
  if (out_first_row) *out_first_row = first;
  return RASS_OK;
}

int sharded_append(rass_engine* h, const float* rows_host, int64_t n, int64_t* out_first_row) {
  return sharded_append_impl(h, rows_host, false, n, out_first_row);
}
int sharded_append_dev(rass_engine* h, const float* rows_dev, int64_t n, int64_t* out_first_row) {
  return sharded_append_impl(h, rows_dev, true, n, out_first_row);
}

int sharded_overwrite(rass_engine* h, int64_t row, const float* v_host) {
  if (row < 0 || row >= h->n_rows || !v_host) return rass_fail(h, RASS_E_NOTFOUND, "row %lld out of range", (long long)row);
  const int g = shard_of(h, row);
  rass_engine* sh = h->shards->sh[g];
  const int rc = rass_overwrite(sh, row_global_to_local(shard_map(h, g), h->rmap.base + row), v_host);
  cudaSetDevice(h->device);
  if (rc) { h->err = sh->err; return rc; }
  if (h->dead[(size_t)row]) { h->dead[(size_t)row] = 0; h->n_live++; }
  return RASS_OK;
}

int sharded_tombstone(rass_engine* h, int64_t row) {
  if (row < 0 || row >= h->n_rows) return rass_fail(h, RASS_E_NOTFOUND, "row %lld out of range", (long long)row);
  if (h->dead[(size_t)row]) return RASS_OK;
  const int g = shard_of(h, row);
  rass_engine* sh = h->shards->sh[g];
  const int rc = rass_tombstone(sh, row_global_to_local(shard_map(h, g), h->rmap.base + row));
  cudaSetDevice(h->device);
  if (rc) { h->err = sh->err; return rc; }
  h->dead[(size_t)row] = 1;
  h->n_live--;
  return RASS_OK;
}

int sharded_read_rows(rass_engine* h, int64_t first_row, int64_t n, float* out_host) {
  if (first_row < 0 || n < 0 || first_row + n > h->n_rows || (n && !out_host))
    return rass_fail(h, RASS_E_NOTFOUND, "rows [%lld, +%lld) out of range", (long long)first_row, (long long)n);
  ShardSet* S = h->shards;
  return run_all(h, [&](int g) {
    return for_runs_of_shard(h, g, first_row, n, [&](int64_t r, int64_t run) {
      return rass_read_rows(S->sh[g], row_global_to_local(shard_map(h, g), h->rmap.base + r), run,
                            out_host + (size_t)(r - first_row) * h->dim);
    });
  });
}

int sharded_read_rows_list(rass_engine* h, const int64_t* rows_host, int64_t n, float* out_host) {
  if (n < 0 || (n && (!rows_host || !out_host))) return rass_fail(h, RASS_E_INVALID, "bad arguments");
  for (int64_t i = 0; i < n; ++i)
    if (rows_host[i] < 0 || rows_host[i] >= h->n_rows)
      return rass_fail(h, RASS_E_NOTFOUND, "row %lld out of range", (long long)rows_host[i]);
  ShardSet* S = h->shards;
  return run_all(h, [&](int g) {
    std::vector<int64_t> local, where;
    for (int64_t i = 0; i < n; ++i)
      if (shard_of(h, rows_host[i]) == g) {
        local.push_back(row_global_to_local(shard_map(h, g), h->rmap.base + rows_host[i]));
        where.push_back(i);
      }
    if (local.empty()) return (int)RASS_OK;
    std::vector<float> tmp(local.size() * (size_t)h->dim);
    const int rc = rass_read_rows_list(S->sh[g], local.data(), (int64_t)local.size(), tmp.data());
    if (rc) return rc;
    for (size_t i = 0; i < local.size(); ++i)
      memcpy(out_host + (size_t)where[i] * h->dim, tmp.data() + i * (size_t)h->dim, (size_t)h->dim * 4);
    return (int)RASS_OK;
  });
}

int sharded_set_row_filter(rass_engine* h, const uint8_t* mask_host, int64_t n) {
  ShardSet* S = h->shards;
  if (mask_host && n < 0) return rass_fail(h, RASS_E_INVALID, "bad filter length");
  return run_all(h, [&](int g) {
    if (!mask_host) return rass_set_row_filter(S->sh[g], nullptr, 0);
    const int64_t n_local = shard_rows_below(h, g, n);
    std::vector<uint8_t> m((size_t)std::max<int64_t>(n_local, 1));
    const RowMap rm = shard_map(h, g);
    for (int64_t l = 0; l < n_local; ++l) m[(size_t)l] = mask_host[row_local_to_global(rm, l) - rm.base];
    return rass_set_row_filter(S->sh[g], m.data(), n_local);
  });
}

int sharded_set_row_filter_rows(rass_engine* h, const int64_t* rows_host, int64_t n, int64_t total_rows) {
  ShardSet* S = h->shards;
  if (n < 0 || total_rows < 0 || (n && !rows_host)) return rass_fail(h, RASS_E_INVALID, "bad filter rows");
  return run_all(h, [&](int g) {
    std::vector<int64_t> local;
    const RowMap rm = shard_map(h, g);
    for (int64_t i = 0; i < n; ++i)
      if (rows_host[i] >= 0 && rows_host[i] < total_rows && shard_of(h, rows_host[i]) == g)
        local.push_back(row_global_to_local(rm, rm.base + rows_host[i]));
    return rass_set_row_filter_rows(S->sh[g], local.data(), (int64_t)local.size(), shard_rows_below(h, g, total_rows));
  });
}

// ---------------------------------------------------------------------------------------------
// search
// ---------------------------------------------------------------------------------------------
static void fold_stats(ShardSet* S, rass_stats* out, int extra_launches) {
  rass_stats s;
  memset(&s, 0, sizeof(s));
  s.n_certified = 1 << 30;
  for (const rass_stats& t : S->st) {
    s.scan_ms = std::max(s.scan_ms, t.scan_ms);
    s.finish_ms = std::max(s.finish_ms, t.finish_ms);
    s.total_ms = std::max(s.total_ms, t.total_ms);
    s.rows_scanned += t.rows_scanned;
    s.bytes_streamed += t.bytes_streamed;
    s.n_queries = t.n_queries;
    s.n_certified = std::min(s.n_certified, t.n_certified);
    s.n_fallback += t.n_fallback;
    s.n_retried += t.n_retried;
    s.path = t.path;
    s.passes = std::max(s.passes, t.passes);
    s.launches += t.launches;
    s.max_candidates = std::max(s.max_candidates, t.max_candidates);
  }
  s.launches += extra_launches;
  *out = s;
}

// Every shard searches its rows and stores its exact [B, k] list into slot 0 of the coordinator's gather buffer; the
// merged list is left in S->m_* on the coordinator device (stream synchronised).  q_host: [B, dim] fp32.
static int knn_to_coordinator(rass_engine* h, const float* q_host, int B, int k, bool want_keys, rass_stats* stats) {
  ShardSet* S = h->shards;
  if (B < 1) return rass_fail(h, RASS_E_INVALID, "B must be >= 1");
  if (k < 1 || k > RASS_MAX_K) return rass_fail(h, RASS_E_INVALID, "k must be in [1, %d], got %d", RASS_MAX_K, k);
  const size_t n = (size_t)B * k;
  int rc;
  if ((rc = ensure_gather(h, n))) return rc;
  rc = run_all(h, [&](int g) {
    rass_engine* sh = S->sh[g];
    float* qd = nullptr;
    int r;
    if ((r = ensure_out_workspace(sh, n))) return r;
    if ((r = stage_queries(sh, q_host, B, &qd))) return r;
    int64_t* o_rows = S->peer_ok || S->dev[g] == h->device ? S->g_rows[0] + (size_t)g * S->cap : S->l_rows[g];
    double* o_keys = S->peer_ok || S->dev[g] == h->device ? S->g_keys[0] + (size_t)g * S->cap : S->l_keys[g];
    // blocking form: certificate failures are retried / re-scanned exactly before it returns (stream synchronised)
    if ((r = search_core(sh, qd, B, k, o_rows, sh->out_scores, o_keys, &S->st[g]))) return r;
    if (o_rows == S->l_rows[g]) {
      cudaError_t e = peer_copy_sync(S->g_rows[0] + (size_t)g * S->cap, h->device, o_rows, S->dev[g], n * 8, eng_stream(sh));
      if (e == cudaSuccess)
        e = peer_copy_sync(S->g_keys[0] + (size_t)g * S->cap, h->device, o_keys, S->dev[g], n * 8, eng_stream(sh));
      if (e != cudaSuccess) return rass_fail(sh, RASS_E_NCCL, "list exchange: %s", cudaGetErrorString(e));
    }
    return (int)RASS_OK;
  });
  if (rc) return rc;
  cudaStream_t st = eng_stream(h);
  if ((rc = launch_merge_topk(h, S->g_keys[0], S->g_rows[0], (int64_t)S->cap, S->G, B, k, S->m_rows, S->m_scores,
                              want_keys ? S->m_keys : nullptr, st)))
    return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  if (stats) fold_stats(S, stats, 1);
  return RASS_OK;
}

int sharded_search_knn(rass_engine* h, const float* q_host, int B, int k, int64_t* out_rows, float* out_scores,
                       double* out_keys, rass_stats* stats) {
  ShardSet* S = h->shards;
  if (!q_host || !out_rows || !out_scores) return rass_fail(h, RASS_E_INVALID, "null buffer");
  rass_stats s;
  int rc = knn_to_coordinator(h, q_host, B, k, out_keys != nullptr, &s);
  if (rc) return rc;
  const size_t n = (size_t)B * k;
  cudaStream_t st = eng_stream(h);
  CUDA_TRY(h, cudaMemcpyAsync(S->m_rows_host, S->m_rows, n * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaMemcpyAsync(S->m_scores_host, S->m_scores, n * 4, cudaMemcpyDeviceToHost, st));
  if (out_keys) CUDA_TRY(h, cudaMemcpyAsync(S->m_keys_host, S->m_keys, n * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  memcpy(out_rows, S->m_rows_host, n * 8);
  memcpy(out_scores, S->m_scores_host, n * 4);
  if (out_keys) memcpy(out_keys, S->m_keys_host, n * 8);
  h->last_stats = s;
  if (stats) *stats = s;
  return RASS_OK;
}

__global__ void sum_flags_kernel(const int64_t* __restrict__ flags, int G, int64_t* __restrict__ out) {
  int64_t s = 0;
  for (int g = 0; g < G; ++g) s += flags[g];
  *out = s;
}

static int ensure_q_bcast(rass_engine* h, size_t n_floats) {
  ShardSet* S = h->shards;
  if (n_floats <= S->q_cap) return RASS_OK;
  const size_t cap = std::max<size_t>(n_floats * 2, (size_t)64 * h->dim);
  const int rc = run_all(h, [&](int g) {
    rass_engine* sh = S->sh[g];
    CUDA_TRY(sh, cudaStreamSynchronize(eng_stream(sh)));
    for (int s = 0; s < 2; ++s) {
      cudaFree(S->q_bcast[s][g]);
      S->q_bcast[s][g] = nullptr;
      CUDA_TRY(sh, cudaMalloc(&S->q_bcast[s][g], cap * 4));
    }
    return (int)RASS_OK;
  });
  if (rc) return rc;
  S->q_cap = cap;
  return RASS_OK;
}

// Enqueue-only search of device queries (q_dev / outputs on the coordinator device, ordered on its stream): the
// queries are broadcast by peer copies behind an event, every shard's finish kernel stores its list and its certificate
// word into the slot's gather buffer, the coordinator stream waits for the G events and merges.  No host synchronisation.
int sharded_search_knn_dev_async(rass_engine* h, const float* q_dev, int B, int k, int64_t* out_rows_dev,
                                 float* out_scores_dev, double* out_keys_dev, int slot, int64_t* flag_out_dev) {
  ShardSet* S = h->shards;
  if (!q_dev || !out_rows_dev || !out_scores_dev) return rass_fail(h, RASS_E_INVALID, "null buffer");
  if (slot < 0 || slot > 1) return rass_fail(h, RASS_E_INVALID, "slot must be 0 or 1");
  if (S->pending[slot]) return rass_fail(h, RASS_E_INVALID, "async slot %d still has a search in flight", slot);
  if (B < 1) return rass_fail(h, RASS_E_INVALID, "B must be >= 1");
  if (k < 1 || k > RASS_MAX_K) return rass_fail(h, RASS_E_INVALID, "k must be in [1, %d], got %d", RASS_MAX_K, k);
  const size_t n = (size_t)B * k;
  int rc;
  if ((rc = ensure_gather(h, n))) return rc;
  if ((rc = ensure_q_bcast(h, (size_t)B * h->dim))) return rc;
  cudaStream_t st = eng_stream(h);
  CUDA_TRY(h, cudaEventRecord(S->ev_q[slot], st));
  rc = run_all(h, [&](int g) {
    rass_engine* sh = S->sh[g];
    cudaStream_t sg = eng_stream(sh);
    int r;
    if ((r = ensure_out_workspace(sh, 2 * n))) return r;
    CUDA_TRY(sh, cudaStreamWaitEvent(sg, S->ev_q[slot], 0));
    const float* qd = q_dev;
    if (S->dev[g] != h->device) {
      CUDA_TRY(sh, cudaMemcpyPeerAsync(S->q_bcast[slot][g], S->dev[g], q_dev, h->device, (size_t)B * h->dim * 4, sg));
      qd = S->q_bcast[slot][g];
    }
    const bool direct = S->peer_ok || S->dev[g] == h->device;
    int64_t* o_rows = direct ? S->g_rows[slot] + (size_t)g * S->cap : S->l_rows[g];
    double* o_keys = direct ? S->g_keys[slot] + (size_t)g * S->cap : S->l_keys[g];
    int64_t* o_flag = S->g_flag[slot] + g;               // 8 bytes: always a peer store or a small copy below
    int64_t* flag_dst = direct ? o_flag : reinterpret_cast<int64_t*>(sh->out_rows + n);   // spare local word
    if ((r = search_core(sh, qd, B, k, o_rows, sh->out_scores, o_keys, nullptr, slot, flag_dst))) return r;
    sg = slot_stream_of(sh, slot);             // RASS_OPT_ASYNC_OVERLAP: the search ran on the slot's own stream
    if (!direct) {
      CUDA_TRY(sh, cudaMemcpyPeerAsync(S->g_rows[slot] + (size_t)g * S->cap, h->device, o_rows, S->dev[g], n * 8, sg));
      CUDA_TRY(sh, cudaMemcpyPeerAsync(S->g_keys[slot] + (size_t)g * S->cap, h->device, o_keys, S->dev[g], n * 8, sg));
      CUDA_TRY(sh, cudaMemcpyPeerAsync(o_flag, h->device, flag_dst, S->dev[g], 8, sg));
    }
    CUDA_TRY(sh, cudaEventRecord(S->ev_sh[slot][g], sg));
    return (int)RASS_OK;
  });
  if (rc) return rc;
  for (int g = 0; g < S->G; ++g) CUDA_TRY(h, cudaStreamWaitEvent(st, S->ev_sh[slot][g], 0));
  if ((rc = launch_merge_topk(h, S->g_keys[slot], S->g_rows[slot], (int64_t)S->cap, S->G, B, k, out_rows_dev,
                              out_scores_dev, out_keys_dev, st)))
    return rc;
  if (flag_out_dev) {
    sum_flags_kernel<<<1, 1, 0, st>>>(S->g_flag[slot], S->G, flag_out_dev);
    CUDA_TRY(h, cudaGetLastError());
  }
  CUDA_TRY(h, cudaEventRecord(S->ev_done[slot], st));
  S->pending[slot] = true;
  return RASS_OK;
}

int sharded_async_join(rass_engine* h, int slot, void* stream) {
  ShardSet* S = h->shards;
  if (slot < 0 || slot > 1) return rass_fail(h, RASS_E_INVALID, "slot must be 0 or 1");
  if (!S->pending[slot]) return rass_fail(h, RASS_E_INVALID, "no search in flight in slot %d", slot);
  CUDA_TRY(h, cudaStreamWaitEvent(reinterpret_cast<cudaStream_t>(stream), S->ev_done[slot], 0));
  return RASS_OK;
}

int sharded_search_knn_dev_wait(rass_engine* h, int slot, rass_stats* stats) {
  ShardSet* S = h->shards;
  if (slot < 0 || slot > 1) return rass_fail(h, RASS_E_INVALID, "slot must be 0 or 1");
  if (!S->pending[slot]) return rass_fail(h, RASS_E_INVALID, "no search in flight in slot %d", slot);
  bool again = false;
  for (int g = 0; g < S->G; ++g) {
    const int rc = rass_search_knn_dev_wait(S->sh[g], slot, &S->st[g]);
    if (rc == RASS_E_AGAIN) again = true;
    else if (rc) { h->err = S->sh[g]->err; cudaSetDevice(h->device); S->pending[slot] = false; return rc; }
  }
  cudaSetDevice(h->device);
  CUDA_TRY(h, cudaEventSynchronize(S->ev_done[slot]));
  S->pending[slot] = false;
  rass_stats s;
  fold_stats(S, &s, 1);
  h->last_stats = s;
  if (stats) *stats = s;
  return again ? RASS_E_AGAIN : RASS_OK;
}

// blocking device-pointer flavour: through the staged host path would defeat its purpose, so it is the async form
// followed by a wait, and -- when some shard's certificate failed -- a host-staged repeat
int sharded_search_knn_dev(rass_engine* h, const float* q_dev, int B, int k, int64_t* out_rows_dev,
                           float* out_scores_dev, double* out_keys_dev, rass_stats* stats) {
  ShardSet* S = h->shards;
  int rc = sharded_search_knn_dev_async(h, q_dev, B, k, out_rows_dev, out_scores_dev, out_keys_dev, 0, nullptr);
  if (rc) return rc;
  rc = sharded_search_knn_dev_wait(h, 0, stats);
  if (rc != RASS_E_AGAIN) return rc;
  std::vector<float> q((size_t)B * h->dim);
  cudaStream_t st = eng_stream(h);
  CUDA_TRY(h, cudaMemcpyAsync(q.data(), q_dev, q.size() * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  rass_stats s;
  if ((rc = knn_to_coordinator(h, q.data(), B, k, out_keys_dev != nullptr, &s))) return rc;
  const size_t n = (size_t)B * k;
  CUDA_TRY(h, cudaMemcpyAsync(out_rows_dev, S->m_rows, n * 8, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(h, cudaMemcpyAsync(out_scores_dev, S->m_scores, n * 4, cudaMemcpyDeviceToDevice, st));
  if (out_keys_dev) CUDA_TRY(h, cudaMemcpyAsync(out_keys_dev, S->m_keys, n * 8, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  h->last_stats = s;
  if (stats) *stats = s;
  return RASS_OK;
}

// ---------------------------------------------------------------------------------------------
// text: postings split by the row map, corpus-wide statistics
// ---------------------------------------------------------------------------------------------
int sharded_bm25_build(rass_engine* h, const int64_t* indptr, const int32_t* doc, const uint16_t* tf,
                       const int32_t* term_field, const uint32_t* doclen, int64_t V, int64_t N, int F) {
  ShardSet* S = h->shards;
  if (V < 0 || N < 0 || F < 1 || F > 255 || !indptr || (N && !doclen)) return rass_fail(h, RASS_E_INVALID, "bad postings");
  const int64_t nnz = indptr[V];
  if (nnz < 0 || (nnz && (!doc || !tf))) return rass_fail(h, RASS_E_INVALID, "bad postings");
  // corpus-wide statistics: scores must not depend on how the rows are spread (deliberately not OpenSearch's
  // per-shard idf, SURVEY.md 8e)
  std::vector<int64_t> doc_count((size_t)F, 0), sum_ttf((size_t)F, 0), df((size_t)V);
  for (int f = 0; f < F; ++f)
    for (int64_t i = 0; i < N; ++i) {
      const uint32_t l = doclen[(size_t)f * N + i];
      doc_count[(size_t)f] += l != 0;
      sum_ttf[(size_t)f] += l;
    }
  for (int64_t t = 0; t < V; ++t) df[(size_t)t] = indptr[t + 1] - indptr[t];
  const int rc = run_all(h, [&](int g) {
    const RowMap rm = shard_map(h, g);
    const int64_t n_local = shard_rows_below(h, g, N);
    std::vector<int64_t> ip((size_t)V + 1, 0);
    std::vector<int32_t> d;
    std::vector<uint16_t> f_;
    d.reserve((size_t)(nnz / S->G + 1024));
    f_.reserve((size_t)(nnz / S->G + 1024));
    for (int64_t t = 0; t < V; ++t) {
      for (int64_t p = indptr[t]; p < indptr[t + 1]; ++p) {
        const int64_t l = row_global_to_local(rm, rm.base + doc[p]);
        if (l >= 0) { d.push_back((int32_t)l); f_.push_back(tf[p]); }
      }
      ip[(size_t)t + 1] = (int64_t)d.size();
    }
    std::vector<uint32_t> dl((size_t)F * std::max<int64_t>(n_local, 1), 0);
    for (int f = 0; f < F; ++f)
      for (int64_t l = 0; l < n_local; ++l)
        dl[(size_t)f * n_local + l] = doclen[(size_t)f * N + (row_local_to_global(rm, l) - rm.base)];
    return bm25_build_impl(S->sh[g], ip.data(), d.data(), f_.data(), term_field, dl.data(), V, n_local, F,
                           doc_count.data(), sum_ttf.data(), df.data());
  });
  if (rc) return rc;
  h->bm25.built = true;
  h->bm25.V = V;
  h->bm25.N = N;
  return RASS_OK;
}

// ---- device-side text ingest on a sharded handle: token streams split by the row map, every shard inverts and merges its
// own rows, the corpus-wide statistics are summed between the merge and the finalisation of the commit ----
int sharded_text_add_rows(rass_engine* h, int field, const int64_t* rows, int64_t n_rows, const int64_t* tok_indptr,
                          const int32_t* tok_terms) {
  ShardSet* S = h->shards;
  if (n_rows < 0 || (n_rows && (!rows || !tok_indptr))) return rass_fail(h, RASS_E_INVALID, "bad token stream");
  if (n_rows == 0) return RASS_OK;
  if (tok_indptr[0] != 0) return rass_fail(h, RASS_E_INVALID, "token offsets start at 0");
  for (int64_t i = 0; i < n_rows; ++i) {
    if (tok_indptr[i + 1] < tok_indptr[i]) return rass_fail(h, RASS_E_INVALID, "token offsets must not decrease");
    if (rows[i] < h->rmap.base || (i && rows[i] <= rows[i - 1]))
      return rass_fail(h, RASS_E_INVALID, "the rows of a bulk must be ascending and distinct");
  }
  if (tok_indptr[n_rows] && !tok_terms) return rass_fail(h, RASS_E_INVALID, "bad token stream");
  return run_all(h, [&](int g) {
    const RowMap rm = shard_map(h, g);
    std::vector<int64_t> lr, ip(1, 0);
    std::vector<int32_t> tk;
    for (int64_t i = 0; i < n_rows; ++i) {
      const int64_t l = row_global_to_local(rm, rows[i]);
      if (l < 0) continue;
      lr.push_back(l);                                        // ascending: the map is monotone inside a shard
      tk.insert(tk.end(), tok_terms + tok_indptr[i], tok_terms + tok_indptr[i + 1]);
      ip.push_back((int64_t)tk.size());
    }
    if (lr.empty()) return (int)RASS_OK;
    return rass_text_add_rows(S->sh[g], field, lr.data(), (int64_t)lr.size(), ip.data(), tk.empty() ? nullptr : tk.data());
  });
}

int sharded_text_commit(rass_engine* h, const int64_t* field_vocab, int F, int64_t N) {
  ShardSet* S = h->shards;
  if (!field_vocab || F < 1 || F > 255 || N < 0) return rass_fail(h, RASS_E_INVALID, "bad commit");
  int64_t V = 0;
  for (int f = 0; f < F; ++f) V += field_vocab[f];
  std::vector<std::vector<int64_t>> dc((size_t)S->G, std::vector<int64_t>((size_t)F, 0)), ttf = dc;
  int rc = run_all(h, [&](int g) {
    rass_engine* sh = S->sh[g];
    const int64_t n_local = shard_rows_below(h, g, N);
    int r = text_commit_merge(sh, field_vocab, F, n_local);
    if (r) return r;
    return text_local_stats(sh, F, n_local, dc[(size_t)g].data(), ttf[(size_t)g].data());
  });
  if (rc) return rc;
  // corpus-wide statistics: scores must not depend on how the rows are spread (SURVEY.md 8e)
  std::vector<int64_t> g_dc((size_t)F, 0), g_ttf((size_t)F, 0), g_df((size_t)V, 0);
  int64_t nnz = 0;
  for (int g = 0; g < S->G; ++g) {
    for (int f = 0; f < F; ++f) { g_dc[(size_t)f] += dc[(size_t)g][(size_t)f]; g_ttf[(size_t)f] += ttf[(size_t)g][(size_t)f]; }
    const std::vector<int64_t>& ip = S->sh[g]->bm25.indptr_host;
    for (int64_t t = 0; t < V; ++t) g_df[(size_t)t] += ip[(size_t)t + 1] - ip[(size_t)t];
    nnz += ip[(size_t)V];
  }
  rc = run_all(h, [&](int g) {
    return text_finalize_global(S->sh[g], shard_rows_below(h, g, N), F, g_dc.data(), g_ttf.data(), g_df.data());
  });
  if (rc) return rc;
  Bm25State& b = h->bm25;
  b.built = true;
  b.V = V; b.N = N; b.F = F; b.nnz = nnz;
  b.indptr_host.assign((size_t)V + 1, 0);                     // corpus-wide document frequencies, as offsets
  for (int64_t t = 0; t < V; ++t) b.indptr_host[(size_t)t + 1] = b.indptr_host[(size_t)t] + g_df[(size_t)t];
  b.field_doc_count = g_dc;
  b.field_sum_ttf = g_ttf;
  return RASS_OK;
}

int sharded_text_size(rass_engine* h, int64_t* V, int64_t* N, int64_t* nnz, int* F) {
  const Bm25State& b = h->bm25;
  const bool have = b.built && !b.indptr_host.empty();
  if (V) *V = have ? b.V : 0;
  if (N) *N = have ? b.N : 0;
  if (nnz) *nnz = have ? b.nnz : 0;
  if (F) *F = have ? b.F : 0;
  return RASS_OK;
}

int sharded_text_stats(rass_engine* h, int64_t* indptr, int64_t* doc_count, int64_t* sum_ttf) {
  const Bm25State& b = h->bm25;
  if (!b.built || b.indptr_host.empty()) return rass_fail(h, RASS_E_NOTFOUND, "no committed text index on this handle");
  if (indptr) memcpy(indptr, b.indptr_host.data(), ((size_t)b.V + 1) * 8);
  for (int f = 0; f < b.F; ++f) {
    if (doc_count) doc_count[f] = b.field_doc_count[(size_t)f];
    if (sum_ttf) sum_ttf[f] = b.field_sum_ttf[(size_t)f];
  }
  return RASS_OK;
}

// knn list (global rows) on the coordinator device -> fused top-k: every shard fuses its own rows against the list and
// stores its fused list into the gather buffer; raw-score merge on the coordinator.  Leaves S->m_rows / m_scores.
static int fuse_on_shards(rass_engine* h, int B, const int32_t* qterm_indptr, const int32_t* qterms,
                          const float* qweights, const uint8_t* qflags, float w_text, const int64_t* knn_rows_c,
                          const float* knn_scores_c, float w_knn, int k, rass_stats* stats) {
  ShardSet* S = h->shards;
  const size_t n = (size_t)B * k;
  int rc;
  if ((rc = ensure_gather(h, n))) return rc;
  if (knn_rows_c && (rc = ensure_knn_bufs(h, n))) return rc;
  rc = run_all(h, [&](int g) {
    rass_engine* sh = S->sh[g];
    int r;
    if ((r = ensure_out_workspace(sh, 2 * n))) return r;
    const int64_t* kr = nullptr;
    const float* ks = nullptr;
    if (knn_rows_c) {
      if (S->dev[g] == h->device) { kr = knn_rows_c; ks = knn_scores_c; }
      else {
        cudaError_t e = peer_copy_sync(S->knn_rows[g], S->dev[g], knn_rows_c, h->device, n * 8, eng_stream(sh));
        if (e == cudaSuccess) e = peer_copy_sync(S->knn_scores[g], S->dev[g], knn_scores_c, h->device, n * 4, eng_stream(sh));
        if (e != cudaSuccess) return rass_fail(sh, RASS_E_NCCL, "knn list broadcast: %s", cudaGetErrorString(e));
        kr = S->knn_rows[g];
        ks = S->knn_scores[g];
      }
    }
    const bool direct = S->peer_ok || S->dev[g] == h->device;
    HybridExt ext = {kr, ks, direct ? S->g_rows[0] + (size_t)g * S->cap : S->l_rows[g], sh->out_scores,
                     direct ? S->g_keys[0] + (size_t)g * S->cap : S->l_keys[g]};
    if ((r = hybrid_core(sh, nullptr, B, qterm_indptr, qterms, qweights, qflags, w_text, w_knn, k, nullptr, nullptr,
                         &S->st[g], &ext)))
      return r;
    if (!direct) {
      cudaError_t e = peer_copy_sync(S->g_rows[0] + (size_t)g * S->cap, h->device, S->l_rows[g], S->dev[g], n * 8, eng_stream(sh));
      if (e == cudaSuccess)
        e = peer_copy_sync(S->g_keys[0] + (size_t)g * S->cap, h->device, S->l_keys[g], S->dev[g], n * 8, eng_stream(sh));
      if (e != cudaSuccess) return rass_fail(sh, RASS_E_NCCL, "fused list exchange: %s", cudaGetErrorString(e));
    }
    return (int)RASS_OK;
  });
  if (rc) return rc;
  cudaStream_t st = eng_stream(h);
  if ((rc = launch_merge_topk(h, S->g_keys[0], S->g_rows[0], (int64_t)S->cap, S->G, B, k, S->m_rows, S->m_scores,
                              nullptr, st, true)))
    return rc;
  CUDA_TRY(h, cudaStreamSynchronize(st));
  if (stats) {
    rass_stats f;
    fold_stats(S, &f, 1);
    stats->finish_ms += f.finish_ms;
    stats->total_ms += f.finish_ms;
    stats->launches += f.launches;
    stats->bytes_streamed += f.bytes_streamed;
    stats->path |= f.path & RASS_PATH_HYBRID_ORDER_FREE;
    stats->n_queries = B;
  }
  return RASS_OK;
}

static int merged_to_host(rass_engine* h, size_t n, int64_t* out_rows, float* out_scores) {
  ShardSet* S = h->shards;
  cudaStream_t st = eng_stream(h);
  CUDA_TRY(h, cudaMemcpyAsync(S->m_rows_host, S->m_rows, n * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaMemcpyAsync(S->m_scores_host, S->m_scores, n * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  memcpy(out_rows, S->m_rows_host, n * 8);
  memcpy(out_scores, S->m_scores_host, n * 4);
  return RASS_OK;
}

int sharded_search_hybrid(rass_engine* h, const float* q_host, int B, const int32_t* qterm_indptr, const int32_t* qterms,
                          const float* qweights, const uint8_t* qflags, float w_text, float w_knn, int k,
                          int64_t* out_rows, float* out_scores, rass_stats* stats) {
  ShardSet* S = h->shards;
  if (B < 1 || !out_rows || !out_scores) return rass_fail(h, RASS_E_INVALID, "bad arguments");
  if (k < 1 || k > RASS_MAX_K) return rass_fail(h, RASS_E_INVALID, "k must be in [1, %d], got %d", RASS_MAX_K, k);
  if (!q_host && !qterm_indptr) return rass_fail(h, RASS_E_INVALID, "neither a vector nor a text clause");
  if (qterm_indptr && (!h->bm25.built || !qterms)) return rass_fail(h, RASS_E_INVALID, "text clause without rass_bm25_build");
  rass_stats s;
  memset(&s, 0, sizeof(s));
  s.n_queries = B;
  int rc;
  const size_t n = (size_t)B * k;
  const bool have_vec = q_host != nullptr && h->n_rows > 0;
  if (have_vec && (rc = knn_to_coordinator(h, q_host, B, k, false, &s))) return rc;
  if (have_vec) {
    // the merged list becomes the knn clause of every shard; it must not alias the buffers the fusion merges into
    if ((rc = ensure_knn_bufs(h, n))) return rc;
    cudaStream_t st = eng_stream(h);
    // shard 0 lives on the coordinator device: its knn buffers double as the coordinator's copy
    CUDA_TRY(h, cudaMemcpyAsync(S->knn_rows[0], S->m_rows, n * 8, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(h, cudaMemcpyAsync(S->knn_scores[0], S->m_scores, n * 4, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
  }
  if ((rc = fuse_on_shards(h, B, qterm_indptr, qterms, qweights, qflags, w_text, have_vec ? S->knn_rows[0] : nullptr,
                           have_vec ? S->knn_scores[0] : nullptr, w_knn, k, &s)))
    return rc;
  if ((rc = merged_to_host(h, n, out_rows, out_scores))) return rc;
  h->last_stats = s;
  if (stats) *stats = s;
  return RASS_OK;
}

int sharded_fuse_hybrid(rass_engine* h, int B, const int32_t* qterm_indptr, const int32_t* qterms,
                        const float* qweights, const uint8_t* qflags, float w_text, const int64_t* knn_rows_host,
                        const float* knn_scores_host, float w_knn, int k, int64_t* out_rows, float* out_scores) {
  ShardSet* S = h->shards;
  if (B < 1 || k < 1 || k > RASS_MAX_K || !out_rows || !out_scores || (knn_rows_host && !knn_scores_host))
    return rass_fail(h, RASS_E_INVALID, "bad arguments");
  if (qterm_indptr && (!h->bm25.built || !qterms)) return rass_fail(h, RASS_E_INVALID, "text clause without rass_bm25_build");
  const size_t n = (size_t)B * k;
  int rc;
  rass_stats s;
  memset(&s, 0, sizeof(s));
  if (knn_rows_host) {
    if ((rc = ensure_knn_bufs(h, n))) return rc;
    if ((rc = ensure_gather(h, n))) return rc;
    cudaStream_t st = eng_stream(h);
    memcpy(S->m_rows_host, knn_rows_host, n * 8);
    memcpy(S->m_scores_host, knn_scores_host, n * 4);
    CUDA_TRY(h, cudaMemcpyAsync(S->knn_rows[0], S->m_rows_host, n * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(h, cudaMemcpyAsync(S->knn_scores[0], S->m_scores_host, n * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
  }
  if ((rc = fuse_on_shards(h, B, qterm_indptr, qterms, qweights, qflags, w_text, knn_rows_host ? S->knn_rows[0] : nullptr,
                           knn_rows_host ? S->knn_scores[0] : nullptr, w_knn, k, &s)))
    return rc;
  h->last_stats = s;
  return merged_to_host(h, n, out_rows, out_scores);
}

// ---------------------------------------------------------------------------------------------
// snapshot / restore: the single-engine file format, rows in global order -- a snapshot restores onto any device count
// ---------------------------------------------------------------------------------------------
int sharded_save(rass_engine* h, const char* path) {
  if (!path) return rass_fail(h, RASS_E_INVALID, "null path");
  FILE* f = fopen(path, "wb");
  if (!f) return rass_fail(h, RASS_E_INVALID, "cannot open %s for writing", path);
  struct { char magic[8]; uint32_t version, dim, metric, flags; int64_t n_rows, n_live; } hd;
  memset(&hd, 0, sizeof(hd));
  memcpy(hd.magic, "RASSB200", 8);
  hd.version = 1; hd.dim = (uint32_t)h->dim; hd.metric = (uint32_t)h->metric; hd.flags = h->flags;
  hd.n_rows = h->n_rows; hd.n_live = h->n_live;
  bool ok = fwrite(&hd, sizeof(hd), 1, f) == 1;
  if (ok && h->n_rows) ok = fwrite(h->dead.data(), 1, (size_t)h->n_rows, f) == (size_t)h->n_rows;
  const int64_t chunk = std::max<int64_t>(1, (int64_t)(((size_t)64 << 20) / ((size_t)h->dim * 4)));
  std::vector<float> buf((size_t)std::min<int64_t>(chunk, std::max<int64_t>(h->n_rows, 1)) * h->dim);
  int rc = RASS_OK;
  for (int64_t off = 0; ok && off < h->n_rows; off += chunk) {
    const int64_t m = std::min<int64_t>(chunk, h->n_rows - off);
    if ((rc = sharded_read_rows(h, off, m, buf.data()))) break;
    ok = fwrite(buf.data(), (size_t)h->dim * 4, (size_t)m, f) == (size_t)m;
  }
  ok = (fclose(f) == 0) && ok;
  if (rc) return rc;
  if (!ok) return rass_fail(h, RASS_E_INVALID, "short write to %s", path);
  return RASS_OK;
}
