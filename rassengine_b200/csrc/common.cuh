// Shared declarations for the engine: handle layout, error plumbing, the per-warp top-list used by the selects.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/rass_b200.h"

#define RASS_WARPS_PER_CTA 8
#define RASS_MAX_K 128
#define RASS_CAND_MAX 2048     // rerank candidate cap per query
#define RASS_GROUP_Q 64        // queries finished per finish launch (= queries per tcgen05 pass)
#define RASS_QPAD 256          // the query workspace is zero padded to a multiple of this (one scan_gemm group)
#define RASS_STREAM_SEG 64     // pool entries per (CTA, query) segment of the streaming scan (32..64 kept)
// pool entries per (CTA, query) segment of the tcgen05 scans: 256 (a compaction keeps 32..64) for k <= 32,
// 512 (keeps 128..256) for larger k
static inline int rass_tc_seg(int k) { return k > 32 ? 512 : 256; }
// entries a compaction of such a segment keeps at least (at most twice as many)
__host__ __device__ constexpr int rass_tc_keep(int seg) { return seg == 512 ? 128 : seg / 8; }
#define RASS_EXACT_NQ 4        // queries per pass of the fp64 scan
#define RASS_FINISH_THREADS 1024

// Where a shard's local rows sit among the global rows.  One shard: global = base + local.  A shard g of G inside a
// single-process sharded handle (sharded.cu) owns every G-th block of 2^blk_log2 consecutive global rows, so an index
// that grows by bulk appends stays balanced: global = base + (((local >> s) * G + g) << s) + (local & (2^s - 1)).
struct RowMap {
  int64_t base;
  int32_t g, G, blk_log2;
};
#define RASS_SHARD_BLOCK_LOG2 10
__host__ __device__ inline int64_t row_local_to_global(const RowMap& m, int64_t local) {
  if (m.G <= 1) return m.base + local;
  const int64_t b = local >> m.blk_log2, in = local & ((int64_t(1) << m.blk_log2) - 1);
  return m.base + (((b * m.G + m.g) << m.blk_log2) | in);
}
// -1: the row belongs to another shard (or lies below the base)
__host__ __device__ inline int64_t row_global_to_local(const RowMap& m, int64_t global) {
  const int64_t r = global - m.base;
  if (r < 0) return -1;
  if (m.G <= 1) return r;
  const int64_t b = r >> m.blk_log2;
  if ((int32_t)(b % m.G) != m.g) return -1;
  return ((b / m.G) << m.blk_log2) | (r & ((int64_t(1) << m.blk_log2) - 1));
}

#define HYB_TILE 4096            // docs per tile of the hybrid kernels: a tile's fused clause sums live in shared memory
#define HYB_TABLE_MIN_DF 512     // terms at least this frequent get a row of per-tile posting offsets

// the postings of one bulk of new rows of one field, sorted by (term, doc): what a commit folds into the CSR (postings.cu)
struct TextSegment {
  int field = 0;
  int64_t n_post = 0, n_uniq = 0;
  int32_t* uterm = nullptr;      // device [n_uniq] distinct local term ids, ascending
  int64_t* uptr = nullptr;       // device [n_uniq + 1] where each one's run starts
  int32_t* doc = nullptr;        // device [n_post]
  uint16_t* tf = nullptr;        // device [n_post]
};

struct Bm25State {
  bool built = false;
  int64_t V = 0, N = 0, nnz = 0;
  int F = 1;                     // analysed fields sharing the CSR
  std::vector<uint8_t> term_field_host;  // term -> field
  int64_t* indptr = nullptr;     // device [V+1]
  int32_t* doc = nullptr;        // device [nnz]
  uint16_t* tf = nullptr;        // device [nnz]
  float* xq = nullptr;           // device [nnz] tf * inv[norm of the doc]: the posting's impact (term_xrange_kernel)
  uint8_t* norm = nullptr;       // device [F][N]  SmallFloat byte4 of the field length of the doc
  float* inv_dev = nullptr;      // device [F][256] 1 / (k1 * ((1-b) + b * len/avgdl))
  int n_tiles = 0;               // tiles of 4096 docs
  uint32_t* tile_off = nullptr;  // device [n_table][n_tiles + 1] postings of a frequent term before each tile
  std::vector<int32_t> table_row_host;   // term -> row of tile_off, -1 for rare terms
  unsigned char* qt_host = nullptr;      // pinned staging of the per-call query-term arrays
  unsigned char* qt_dev = nullptr;
  size_t qt_cap = 0, qt_q_cap = 0, qt_bytes = 0;
  uint32_t* hyb_gthr = nullptr;          // device [qt_q_cap] cross-tile pruning bound of the running hybrid batch
  uint32_t* vocab_blob = nullptr;        // device: the term dictionary as code points, terms back to back (fuzziness: AUTO)
  int64_t* vocab_off = nullptr;          // device [vocab_V + 1], in code points
  int64_t vocab_V = 0;
  int32_t* fz_terms = nullptr;           // device [vocab_V] matches of the running fuzzy scan
  int32_t* fz_edits = nullptr;
  int* fz_n = nullptr;
  float avgdl = 0.f;
  int64_t doc_count = 0;
  std::vector<int64_t> indptr_host;
  std::vector<float> idf_host;   // (float) ln(1 + (docCount - df + .5) / (df + .5))
  std::vector<float> xmin_host, xmax_host;   // per term: range of tf * inv[norm] over its postings (term_xrange_kernel)
  bool force_ordered = false;    // RASS_OPT_HYBRID_ORDERED: always take the ordered tile kernel (tests, A/B)
  bool maxscore = false;         // RASS_OPT_HYBRID_MAXSCORE: essential / non-essential term split in the order-free kernel
  int* sel_fallback = nullptr;   // device [qt_q_cap]: queries hybrid_select_kernel hands to the radix select
  // device-side ingest (postings.cu)
  std::vector<TextSegment> pending;      // segments rass_text_commit has not folded in yet
  uint32_t* doclen_dev = nullptr;        // device [doclen_F][doclen_stride] tokens of the field per row
  uint32_t* gen_dev = nullptr;           // device [doclen_F][doclen_stride] which source owns the (field, row): 0 = the
                                         // committed CSR, s = the s-th pending segment (rewrites, postings.cu)
  bool has_rewrite = false;              // a pending segment rewrites rows the index held: the commit re-sorts
  int doclen_F = 0;
  int64_t doclen_stride = 0;
  std::vector<int64_t> field_vocab;      // terms per field as of the last build / commit (field f owns one block of ids)
  std::vector<int64_t> field_last_row;   // highest row each field holds (segments included)
  bool contiguous_fields = true;
  std::vector<int64_t> field_doc_count, field_sum_ttf;   // per field, as of the last build / commit
  std::vector<uint8_t> field_omit_norms; // rass_text_omit_norms: the field's documents all count as length 1 (`keyword`)
  int64_t pending_V = 0;                 // terms of the CSR text_commit_merge left for the finalisation
  void* scratch = nullptr;               // arena of the segment builds, kept between bulks, released by the commit
  size_t scratch_bytes = 0;
};

// device-resident facts of the store, raised by store_convert_kernel (atomicMax: they only ever grow), read by the
// certificate of every search
struct StoreScalars {
  float rho_x;        // max over rows of ||x - bf16(x)|| / ||x||
  float max_xnorm;    // max over rows of ||x||
  float rho_x8;       // max over rows of ||x - s_x x8|| / ||x|| (the int8 shadow; 0 without one)
};

// device-resident counters of one search, reset by query_prep_kernel
struct SearchScalars {
  int flagged_n;      // queries that failed the certificate in the running search
  int max_cand;       // largest rerank candidate set in the running search
  int n_certified;
  int finish_done;    // CTAs of the running finish launch that are through (the last one publishes flagged_n, resets this)
  int tile_ctr[2];    // scan_umma_kernel's tile scheduler: tiles handed out beyond the first per CTA, CTAs through (the
                      // last one zeroes both)
};

// What one search in flight owns on the device (grows on demand).  The handle holds two: ws[0] serves the blocking
// search and async slot 0, ws[1] async slot 1 under RASS_OPT_ASYNC_OVERLAP (allocated on its first use).
struct SearchWs {
  SearchScalars* scal = nullptr;    // device
  // query workspace
  int q_cap = 0;
  float* q_raw = nullptr;           // [q_cap, dim_pad] fp32 as given (zero padded)
  float* q_hat = nullptr;           // [q_cap, dim_pad] fp32 scan query (unit for cosine)
  __nv_bfloat16* q16 = nullptr;     // [q_cap rounded to 64, dim_pad]
  double* q_norm = nullptr;         // [q_cap]
  float* q_rho = nullptr;           // [q_cap] ||q_hat - bf16(q_hat)|| / ||q_hat||
  // the int8 form of q_hat: q_hat ~ s1 q1 + s2 q2, two int8 parts (the second quantises the first one's residual).
  // Group g of 64 queries is rows [128 g, 128 g + 128): q1 of its queries, then q2
  int8_t* q8 = nullptr;             // [q_cap * 2, dim_pad]
  float* q8_scale = nullptr;        // [q_cap][2] s1, s2
  float* q_rho8 = nullptr;          // [q_cap] ||q_hat - (s1 q1 + s2 q2)|| / ||q_hat||
  uint32_t* q_gthr = nullptr;       // [q_cap] tcgen05 scans: threshold seed, then the largest pivot any CTA published
  // candidate pool of one query group (RASS_GROUP_Q queries)
  size_t pool_entries = 0;          // per query: stride of the running search
  size_t pool_alloc_entries = 0;    // allocated, in entries
  float* pool_key = nullptr;
  uint32_t* pool_row = nullptr;
  size_t pool_segs = 0;             // per query: stride of the running search
  size_t pool_alloc_segs = 0;       // allocated, in segments
  float* pool_thr = nullptr;
  int* pool_cnt = nullptr;
  int* flagged = nullptr;           // device [q_cap]: ids of queries that failed the certificate
  int* flagged_host = nullptr;      // pinned [q_cap]
  void* tmap_q = nullptr;           // host copy of the CUtensorMap over q16, 64-row boxes (scan_umma)
  void* tmap_q2 = nullptr;          // 128-row boxes (scan_gemm: one CTA's half of a 256-query group)
  const void* tmap_qbase = nullptr; // the q16 each map was encoded for
  const void* tmap_q2base = nullptr;
  void* tmap_q8 = nullptr;          // over q8, 128-row boxes (scan_umma, int8 pass)
  const void* tmap_q8base = nullptr;
};

// a device array that grows in place (vmm.cu): reserved address range, physical chunks mapped on demand
struct VmArray {
  void* base = nullptr;
  size_t reserved = 0, mapped = 0, chunk = 0;
  int device = 0;
  std::vector<unsigned long long> handles;   // CUmemGenericAllocationHandle of every mapped chunk
};
bool vm_available();
bool vm_reserve(VmArray* a, int device, size_t max_bytes, size_t chunk_hint);
int vm_grow(VmArray* a, size_t bytes);       // 0 ok, 1 out of memory, 2 other failure
void vm_free(VmArray* a);

struct rass_engine {
  int dim = 0, dim_pad = 0, metric = 0, device = 0;
  uint32_t flags = 0;
  int num_sms = 0;
  int path = RASS_PATH_AUTO;
  int64_t cap = 0, n_rows = 0, n_live = 0;
  RowMap rmap = {0, 0, 1, RASS_SHARD_BLOCK_LOG2};     // local row -> global row (rass_set_row_base, sharded handles)
  struct ShardSet* shards = nullptr;                  // non-null: a coordinator over several single-device engines
  float* x32 = nullptr;             // [cap, dim_pad] fp32 (null when BF16_ONLY)
  __nv_bfloat16* x16 = nullptr;     // [cap, dim_pad] bf16 shadow / corpus
  double* norm64 = nullptr;         // [cap] ||x|| accumulated in fp64 from the stored values
  float* sa = nullptr;              // [cap] scan scale:  cosine 1/||x|| (0 for zero rows), L2 1
  float* sb = nullptr;              // [cap] scan offset: cosine 0, L2 -0.5||x||^2; -inf = tombstone
  int8_t* x8 = nullptr;             // [cap, dim_pad] int8 shadow x ~ s_x x8, s_x = max|x| / 127 (null when BF16_ONLY or
                                    // NO_INT8_SHADOW)
  float* sa8 = nullptr;             // [cap] scan scale of the int8 shadow: s_x * sa
  // the seven arrays above live in growable virtual-memory arrays when the driver offers them (vm[i].base == the
  // pointer); otherwise they are cudaMalloc'ed and grow by copy
  VmArray vm[7];
  bool use_vm = false;
  StoreScalars* store_scal = nullptr;   // device
  StoreScalars store_scal_host = {};    // host copy, refreshed before a search after rows were written
  bool store_scal_stale = false;
  // AUTO takes the int8 64-query pass only for k <= int8_k_max: lowered to k - 1 when an int8 pass AUTO chose left more
  // than a quarter of a search's queries uncertified (each of those needs the bf16 pass as well, so at that k the bf16
  // pass alone is cheaper).  The rerank set grows about linearly in k and with the corpus, so it only ever goes down.
  int int8_k_max = RASS_MAX_K;
  SearchWs ws[2];
  SearchScalars* scal_host = nullptr;   // pinned mirror of ws[0].scal for the blocking search
  cudaStream_t stream = nullptr, user_stream = nullptr, copy_stream = nullptr;
  bool has_user_stream = false;     // user_stream may legitimately be 0 (the legacy default stream)
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t stage_ev[2] = {nullptr, nullptr};
  float* stage[2] = {nullptr, nullptr};  // pinned host staging
  size_t stage_bytes = 0;
  float* dev_stage = nullptr;            // device staging (BF16_ONLY appends, dim != dim_pad appends)
  size_t dev_stage_bytes = 0;
  // exact (fp64) lists
  size_t xlist_entries = 0;
  double* xlist_key = nullptr;
  uint32_t* xlist_row = nullptr;
  int64_t* out_rows = nullptr;      // device result staging for the host-pointer API
  float* out_scores = nullptr;
  double* out_keys = nullptr;
  size_t out_cap = 0;
  int64_t* out_rows_host = nullptr; // pinned
  float* out_scores_host = nullptr;
  double* out_keys_host = nullptr;
  float* q_stage_host = nullptr;    // pinned query staging
  float* q_stage_dev = nullptr;
  size_t q_stage_cap = 0;
  std::vector<uint8_t> dead;        // host mirror of the tombstones
  std::vector<cudaEvent_t> ev_pool; // per-group scan timing
  void* tmap_x = nullptr;           // host copy of the CUtensorMap over x16 (rebuilt on growth)
  int64_t tmap_rows = -1;
  const void* tmap_base = nullptr;
  void* tmap_x8 = nullptr;          // the same over x8
  int64_t tmap8_rows = -1;
  const void* tmap8_base = nullptr;
  // second-chance pass (queries whose certificate failed at k > 32): ids, gathered queries, results
  int* retry_ids = nullptr;
  float* retry_q = nullptr;
  int64_t* retry_rows = nullptr;
  float* retry_scores = nullptr;
  double* retry_keys = nullptr;
  size_t retry_cap = 0;
  int retry_k = 0;
  // RASS_OPT_ASYNC_OVERLAP: each async slot runs on its own stream (forked from the engine stream when the search is
  // enqueued) and slot 1 uses the second search workspace ws[1], so the fixed costs of batch i (query prep, threshold
  // seed, finish) run under the scan of batch i+1.
  bool async_overlap = false;
  int scan_reserve_sms = 0;         // RASS_OPT_SCAN_RESERVE_SMS
  cudaStream_t slot_stream[2] = {nullptr, nullptr};
  cudaEvent_t slot_fork[2] = {nullptr, nullptr};
  // two searches may be in flight through rass_search_knn_dev_async (one slot each)
  struct AsyncSlot {
    bool pending = false, trivial = false;
    int k = 0;
    SearchScalars* scal_host = nullptr;   // pinned: its own copy, a blocking search may reuse ws[0] before the wait
    cudaEvent_t done = nullptr;
    size_t n_ev = 0;
    rass_stats stats;
  } aslot[2];
  int64_t* flist_dev = nullptr;     // per-query filter row lists of the running call (filtered.cu): [B + 1] offsets + rows
  size_t flist_cap = 0;
  uint8_t* row_filter = nullptr;    // device [row_filter_rows] 1 = row passes the bool.filter of the running query
  int64_t* filter_rows_dev = nullptr;   // staging of row lists (rass_set_row_filter_rows, rass_read_rows_list)
  size_t filter_rows_cap = 0;
  bool knn_prefilter = false;       // RASS_OPT_KNN_PREFILTER: rass_search_knn scans only rows passing row_filter
  float* sb_filtered = nullptr;     // [cap] sb with -inf for rows failing the filter (built lazily)
  int64_t sb_filtered_cap = 0;
  bool sb_filtered_dirty = true;
  const float* sb_scan = nullptr;   // the offset array the running search's scans read: sb or sb_filtered
  int64_t row_filter_rows = 0;
  size_t row_filter_cap = 0;
  Bm25State bm25;
  rass_stats last_stats = {};       // of the last search / hybrid / fuse call (rass_last_stats)
  std::string err;
};

extern thread_local std::string g_create_error;

int rass_fail(rass_engine* h, int code, const char* fmt, ...);

#define CUDA_TRY(h, call)                                                                         \
  do {                                                                                            \
    cudaError_t e_ = (call);                                                                      \
    if (e_ != cudaSuccess)                                                                        \
      return rass_fail((h), e_ == cudaErrorMemoryAllocation ? RASS_E_OOM : RASS_E_CUDA,           \
                       "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

static inline cudaStream_t eng_stream(const rass_engine* h) { return h->has_user_stream ? h->user_stream : h->stream; }
// the stream an async slot's search was (or will be) enqueued on
static inline cudaStream_t slot_stream_of(const rass_engine* h, int slot) {
  return h->async_overlap && h->slot_stream[slot] ? h->slot_stream[slot] : eng_stream(h);
}

// fp32 accumulation allowance of a length-d dot product with |x||q| <= 1 (gamma_d, doubled for the tensor
// pipe's unspecified summation order)
static inline float acc_allowance(int dim_pad) { return (float)dim_pad * 1.1920929e-7f; }

// the store keeps the int8 shadow (x8, sa8)
static inline bool has_int8_shadow(uint32_t flags) { return !(flags & (RASS_BF16_ONLY | RASS_NO_INT8_SHADOW)); }

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ float bf16lo(uint32_t p) { return __uint_as_float(p << 16); }
__device__ __forceinline__ float bf16hi(uint32_t p) { return __uint_as_float(p & 0xffff0000u); }

template <typename K>
__device__ __forceinline__ K neg_inf();
template <>
__device__ __forceinline__ float neg_inf<float>() { return __int_as_float(0xff800000); }
template <>
__device__ __forceinline__ double neg_inf<double>() { return __longlong_as_double(0xfff0000000000000ULL); }

template <typename K>
__device__ __forceinline__ bool entry_better(K ka, uint32_t ra, K kb, uint32_t rb) {
  return ka > kb || (ka == kb && ra < rb);
}

__device__ __forceinline__ float shfl_xor_t(float v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
__device__ __forceinline__ double shfl_xor_t(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
__device__ __forceinline__ float shfl_t(float v, int l) { return __shfl_sync(0xffffffffu, v, l); }
__device__ __forceinline__ double shfl_t(double v, int l) { return __shfl_sync(0xffffffffu, v, l); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

// order-preserving float <-> uint32 maps (larger float <-> larger integer); 0 is below every float
__device__ __forceinline__ uint32_t ord32(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float unord32(uint32_t o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

// Warp-cooperative compaction of up to 32*E (ordered key, row) entries held E per lane (ok == 0: empty slot).
// Bisects for a pivot with keep .. 2*keep entries strictly above it, writes those entries densely to
// out_key/out_row and returns their count; every entry not written has key <= unord32(pivot).  Ties can make the
// band unreachable; then the upper end is used (fewer entries kept, the bound still holds).
template <int E>
__device__ __forceinline__ int warp_compact(const uint32_t (&ok)[E], const uint32_t (&rw)[E], int keep,
                                            float* out_key, uint32_t* out_row, uint32_t& pivot) {
  const int lane = threadIdx.x & 31;
  uint32_t kmin = 0xffffffffu, kmax = 0;
#pragma unroll
  for (int i = 0; i < E; ++i)
    if (ok[i]) { kmin = min(kmin, ok[i]); kmax = max(kmax, ok[i]); }
  kmin = __reduce_min_sync(0xffffffffu, kmin);
  kmax = __reduce_max_sync(0xffffffffu, kmax);
  // invariant: count(> lo) > 2*keep (or lo is below everything), count(> hi) < keep
  uint32_t lo = kmin - 1, hi = kmax;
  pivot = kmax;
  int total = 0;
#pragma unroll
  for (int i = 0; i < E; ++i) total += ok[i] != 0;
  total = __reduce_add_sync(0xffffffffu, total);
  if (total <= 2 * keep) {
    pivot = 0x007fffffu;        // ord32(-inf): nothing needs to go, every real entry is above it
  } else {
    bool found = false;
    while (hi - lo > 1) {
      const uint32_t mid = lo + ((hi - lo) >> 1);
      int cgt = 0;
#pragma unroll
      for (int i = 0; i < E; ++i) cgt += ok[i] > mid;
      cgt = __reduce_add_sync(0xffffffffu, cgt);
      if (cgt > 2 * keep) lo = mid;
      else if (cgt < keep) hi = mid;
      else { pivot = mid; found = true; break; }
    }
    if (!found) pivot = hi;
  }
  int kept = 0;
#pragma unroll
  for (int i = 0; i < E; ++i) {
    const bool k = ok[i] > pivot;
    const unsigned bal = __ballot_sync(0xffffffffu, k);
    if (k) {
      const int pos = kept + __popc(bal & ((1u << lane) - 1));
      out_key[pos] = unord32(ok[i]);
      out_row[pos] = rw[i];
    }
    kept += __popc(bal);
  }
  return kept;
}

// Per-warp running top-(32*M) list.  Lane l owns slots key[0..M), row[0..M).  (thr_key, thr_row) is the
// worst kept entry, uniform across the warp.  An entry is better when its key is larger, or equal with a
// smaller row -- the (score desc, row asc) order of the oracle.  All methods must be called by the
// full warp with warp-uniform arguments.
template <typename K, int M>
struct WarpTop {
  K key[M];
  uint32_t row[M];
  K thr_key;
  uint32_t thr_row;

  __device__ __forceinline__ void init() {
#pragma unroll
    for (int i = 0; i < M; ++i) { key[i] = neg_inf<K>(); row[i] = 0xffffffffu; }
    thr_key = neg_inf<K>();
    thr_row = 0xffffffffu;
  }

  // hot-path test for streams that arrive in ascending row order: equal keys can never displace
  __device__ __forceinline__ bool admits_ascending(K k) const { return k > thr_key; }

  __device__ __noinline__ void insert(K k, uint32_t r) {
    if (!entry_better<K>(k, r, thr_key, thr_row)) return;
    const int lane = threadIdx.x & 31;
    // locate the worst entry: first lane (then first slot) that holds (thr_key, thr_row)
    int slot = -1;
#pragma unroll
    for (int i = M - 1; i >= 0; --i)
      if (key[i] == thr_key && row[i] == thr_row) slot = i;
    unsigned holders = __ballot_sync(0xffffffffu, slot >= 0);
    int owner = __ffs(holders) - 1;
    if (lane == owner) {
#pragma unroll
      for (int i = 0; i < M; ++i)
        if (i == slot) { key[i] = k; row[i] = r; }
    }
    // recompute the worst entry
    K wk = key[0];
    uint32_t wr = row[0];
#pragma unroll
    for (int i = 1; i < M; ++i)
      if (entry_better<K>(wk, wr, key[i], row[i])) { wk = key[i]; wr = row[i]; }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
      K ok = shfl_xor_t(wk, m);
      uint32_t orow = __shfl_xor_sync(0xffffffffu, wr, m);
      if (entry_better<K>(wk, wr, ok, orow)) { wk = ok; wr = orow; }
    }
    thr_key = wk;
    thr_row = wr;
  }
};

// The exact key of (row, query): fp64 accumulation of the stored values, the definition the oracle uses
// (oracle/knn.py cos64 / l2sq64).  Called by a full warp; the result is uniform across the warp.
//   cosine: dot64 / (||x||_64 * ||q||_64), 0 when either norm is 0        (larger is better)
//   L2    : -(sum (x - q)^2)                                              (larger is better)
// qs: the raw fp32 query in shared memory, zero padded to dim_pad.
template <bool BF16_ROWS>
__device__ __forceinline__ double exact_key_warp(const float* __restrict__ x32, const __nv_bfloat16* __restrict__ x16,
                                                 const double* __restrict__ norm64, uint32_t row, const float* qs,
                                                 double qnorm, int dim_pad, int metric) {
  const int lane = threadIdx.x & 31;
  double acc = 0.0;
  if (BF16_ROWS) {
    const uint4* p = reinterpret_cast<const uint4*>(x16 + (size_t)row * dim_pad);
    for (int j = lane; j < dim_pad / 8; j += 32) {
      uint4 v = __ldg(p + j);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
      const float* qq = qs + j * 8;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        double a = (double)bf16lo(w[e]), b = (double)bf16hi(w[e]);
        double q0 = (double)qq[2 * e], q1 = (double)qq[2 * e + 1];
        if (metric == RASS_METRIC_COSINE) {
          acc = fma(a, q0, acc);
          acc = fma(b, q1, acc);
        } else {
          double d0 = a - q0, d1 = b - q1;
          acc = fma(d0, d0, acc);
          acc = fma(d1, d1, acc);
        }
      }
    }
  } else {
    const float4* p = reinterpret_cast<const float4*>(x32 + (size_t)row * dim_pad);
    for (int j = lane; j < dim_pad / 4; j += 32) {
      float4 v = __ldg(p + j);
      const float4 q = *reinterpret_cast<const float4*>(qs + j * 4);
      if (metric == RASS_METRIC_COSINE) {
        acc = fma((double)v.x, (double)q.x, acc);
        acc = fma((double)v.y, (double)q.y, acc);
        acc = fma((double)v.z, (double)q.z, acc);
        acc = fma((double)v.w, (double)q.w, acc);
      } else {
        double d0 = (double)v.x - (double)q.x, d1 = (double)v.y - (double)q.y;
        double d2 = (double)v.z - (double)q.z, d3 = (double)v.w - (double)q.w;
        acc = fma(d0, d0, acc);
        acc = fma(d1, d1, acc);
        acc = fma(d2, d2, acc);
        acc = fma(d3, d3, acc);
      }
    }
  }
  acc = warp_sum(acc);
  if (metric == RASS_METRIC_COSINE) {
    double den = norm64[row] * qnorm;
    return den > 0.0 ? acc / den : 0.0;
  }
  return -acc;
}

// Scan key of the int8 pass from the exact integer dots of the row's x8 with the query's two int8 parts: the tcgen05
// epilogue and the threshold seed both compute it with this one expression (explicitly rounded, never contracted
// differently), so a seed T is a pivot in the pass's own key units.  |acc| <= 1024 * 127^2 < 2^24: the conversions
// to float are exact.
__device__ __forceinline__ float int8_key(int32_t acc1, int32_t acc2, float s1, float s2, float sa8, float sb) {
  return __fmaf_rn(__fmaf_rn(s1, __int2float_rn(acc1), __fmul_rn(s2, __int2float_rn(acc2))), sa8, sb);
}

__device__ __forceinline__ float warp_max_nonneg(float v) {
  return __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(v)));
}

// symmetric round-to-nearest int8 code of v at scale s (s = max|.| / 127; 0 codes everything as 0)
__device__ __forceinline__ float int8_code(float v, float s) {
  return s > 0.f ? fminf(fmaxf(rintf(__fdiv_rn(v, s)), -127.f), 127.f) : 0.f;
}

__device__ __forceinline__ float score_from_key(double key, int metric) {
  // OpenSearch k-NN score translation: cosinesimil 1/(2 - cos); l2 1/(1 + d^2)
  return metric == RASS_METRIC_COSINE ? (float)(1.0 / (2.0 - key)) : (float)(1.0 / (1.0 - key));
}

#endif  // __CUDACC__

// ---------------------------------------------------------------------------------------------
// kernel launchers (defined in the .cu files)
// ---------------------------------------------------------------------------------------------
int launch_store_convert(rass_engine* h, const float* src_dev, int64_t src_stride, int64_t first_row, int64_t n,
                         cudaStream_t st);
int launch_query_prep(rass_engine* h, const SearchWs& ws, const float* q_dev, int B, cudaStream_t st);
int launch_seed_thresholds(rass_engine* h, const SearchWs& ws, int B, int seg, size_t n_clear, bool* cleared,
                           cudaStream_t st, bool int8 = false);
// streaming scan of queries [q0, q0+nq) (nq = 1 or 2); their pool slots are q - g0
int launch_scan_stream(rass_engine* h, const SearchWs& ws, int q0, int nq, int g0, cudaStream_t st);
int scan_stream_segs(const rass_engine* h);
// tcgen05 scan of queries [q0, q0+nq) (nq <= 64) into pool slots 0..nq; int8: over x8 with the int8 query parts
int launch_scan_umma(rass_engine* h, SearchWs& ws, int q0, int nq, int seg, cudaStream_t st, bool pool_cleared = false,
                     bool int8 = false);
int scan_umma_segs(const rass_engine* h);
int umma_selftest(rass_engine* h, SearchWs& ws, int n_rows_tile, float* out_host, cudaStream_t st);
// the int8 pass's raw int32 accumulators of the first 64 prepared queries: out_host [n_rows, 128]
int umma8_selftest(rass_engine* h, SearchWs& ws, int32_t* out_host, cudaStream_t st);
// CTA-pair tcgen05 scan of all B prepared queries (groups of 256) into pool slots 0..B
int launch_scan_gemm(rass_engine* h, SearchWs& ws, int B, int seg, cudaStream_t st, bool pool_cleared = false);
int scan_gemm_segs(const rass_engine* h, int B);
int gemm_selftest(rass_engine* h, SearchWs& ws, int B, float* out_host, cudaStream_t st);
// CUtensorMap over a [rows, dim_pad] bf16 (elem_bytes 2) or int8 (1) matrix: boxes of box_rows x 128 bytes, 128B swizzle
int encode_rows_map(rass_engine* h, void* map, const void* base, int64_t rows, int box_rows, int elem_bytes = 2);
// what the scan that filled the pool multiplied: the fp32 query and the stored rows, the bf16 shadows, the int8 ones
enum ScanOperands { SCAN_FP32_Q = 0, SCAN_BF16 = 1, SCAN_INT8 = 2 };
// merge the pool of queries [g0, g0+ng), rerank in fp64, emit top-k, flag uncertified queries
int launch_finish(rass_engine* h, const SearchWs& ws, int g0, int ng, int k, int n_segs, int seg_size, bool has_cnt,
                  ScanOperands ops, int64_t* out_rows, float* out_scores, double* out_keys, cudaStream_t st,
                  int64_t* flag_out = nullptr);
// fp64 scan of the listed queries (qids host array, n_q of them)
int launch_exact(rass_engine* h, const SearchWs& ws, int k, const int* qids_host, int n_q, int64_t* out_rows,
                 float* out_scores, double* out_keys, cudaStream_t st, int* launches);
// raw_score: the keys are fused scores (larger is better whatever the engine's metric), emitted as they are
int launch_merge_topk(rass_engine* h, const double* keys, const int64_t* rows, int64_t shard_stride, int G, int B,
                      int k, int64_t* out_rows, float* out_scores, double* out_keys, cudaStream_t st,
                      bool raw_score = false);
// kNN search of B device queries [B, dim] fp32 into device outputs (engine.cu): blocking (async_slot < 0, the stream
// is synchronised before returning) or enqueue-only into async slot 0 / 1 (rass_search_knn_dev_async)
int search_core(rass_engine* h, const float* q_dev, int B, int k, int64_t* out_rows, float* out_scores,
                double* out_keys, rass_stats* stats, int async_slot = -1, int64_t* async_flag_dev = nullptr);
int stage_queries(rass_engine* h, const float* q_host, int B, float** q_dev_out);
// Row-sharded hybrid: fuse against an EXTERNAL (global) knn list and leave this shard's top-k on the device
struct HybridExt {
  const int64_t* knn_rows_dev;   // [B, k] global rows (-1 = none); rows outside this shard are ignored
  const float* knn_scores_dev;   // [B, k]
  int64_t* out_rows_dev;         // [B, k] global rows
  float* out_scores_dev;         // [B, k] fused float scores
  double* out_keys_dev;          // [B, k] the same as double (what the shard merge ranks by), nullable
};
// device views of a batch's staged query terms (stage_hybrid_terms, bm25.cu)
struct HybridTerms {
  const int32_t* qt_indptr;
  const int64_t* t_lo;
  const uint32_t* t_len;
  const float* t_w;
  const int32_t* t_row;
  const float* t_bound;
  const uint8_t* t_field;
  const uint8_t* t_flag;
  bool multi, order_free;
  size_t n_terms;
  int64_t postings;
};
typedef HybridTerms FilteredTermArrays;
int stage_hybrid_terms(rass_engine* h, int B, const int32_t* qterm_indptr, const int32_t* qterms, const float* qweights,
                       const uint8_t* qflags, float w_text, HybridTerms* out, cudaStream_t st);
int hybrid_core(rass_engine* h, const float* q_host, int B, const int32_t* qterm_indptr, const int32_t* qterms,
                const float* qweights, const uint8_t* qflags, float w_text, float w_knn, int k, int64_t* out_rows,
                float* out_scores, rass_stats* stats, const HybridExt* ext = nullptr);
// g_doc_count / g_sum_ttf: [F] corpus-wide statistics, g_df: [V] (all nullable: taken from the arrays given)
int bm25_build_impl(rass_engine* h, const int64_t* indptr, const int32_t* doc, const uint16_t* tf,
                    const int32_t* term_field, const uint32_t* doclen, int64_t V, int64_t N, int F,
                    const int64_t* g_doc_count, const int64_t* g_sum_ttf, const int64_t* g_df);
// ---- single-process multi-GPU handles (sharded.cu): the public entry points forward to these when h->shards is set ----
int sharded_destroy(rass_engine* h);
int sharded_set_option(rass_engine* h, int opt, int64_t value);
int sharded_set_row_base(rass_engine* h, int64_t base);
int sharded_sync(rass_engine* h);
int sharded_append(rass_engine* h, const float* rows_host, int64_t n, int64_t* out_first_row);
int sharded_append_dev(rass_engine* h, const float* rows_dev, int64_t n, int64_t* out_first_row);
int sharded_overwrite(rass_engine* h, int64_t row, const float* v_host);
int sharded_tombstone(rass_engine* h, int64_t row);
int sharded_read_rows(rass_engine* h, int64_t first_row, int64_t n, float* out_host);
int sharded_read_rows_list(rass_engine* h, const int64_t* rows_host, int64_t n, float* out_host);
int sharded_set_row_filter(rass_engine* h, const uint8_t* mask_host, int64_t n);
int sharded_set_row_filter_rows(rass_engine* h, const int64_t* rows_host, int64_t n, int64_t total_rows);
int sharded_search_knn(rass_engine* h, const float* q_host, int B, int k, int64_t* out_rows, float* out_scores,
                       double* out_keys, rass_stats* stats);
int sharded_search_knn_dev(rass_engine* h, const float* q_dev, int B, int k, int64_t* out_rows_dev,
                           float* out_scores_dev, double* out_keys_dev, rass_stats* stats);
int sharded_search_knn_dev_async(rass_engine* h, const float* q_dev, int B, int k, int64_t* out_rows_dev,
                                 float* out_scores_dev, double* out_keys_dev, int slot, int64_t* flag_out_dev);
int sharded_search_knn_dev_wait(rass_engine* h, int slot, rass_stats* stats);
int sharded_async_join(rass_engine* h, int slot, void* stream);
int sharded_bm25_build(rass_engine* h, const int64_t* indptr, const int32_t* doc, const uint16_t* tf,
                       const int32_t* term_field, const uint32_t* doclen, int64_t V, int64_t N, int F);
int sharded_search_hybrid(rass_engine* h, const float* q_host, int B, const int32_t* qterm_indptr, const int32_t* qterms,
                          const float* qweights, const uint8_t* qflags, float w_text, float w_knn, int k,
                          int64_t* out_rows, float* out_scores, rass_stats* stats);
int sharded_fuse_hybrid(rass_engine* h, int B, const int32_t* qterm_indptr, const int32_t* qterms,
                        const float* qweights, const uint8_t* qflags, float w_text, const int64_t* knn_rows_host,
                        const float* knn_scores_host, float w_knn, int k, int64_t* out_rows, float* out_scores);
int sharded_save(rass_engine* h, const char* path);
int sharded_text_add_rows(rass_engine* h, int field, const int64_t* rows, int64_t n_rows, const int64_t* tok_indptr,
                          const int32_t* tok_terms);
int sharded_text_commit(rass_engine* h, const int64_t* field_vocab, int F, int64_t N);
int sharded_text_size(rass_engine* h, int64_t* V, int64_t* N, int64_t* nnz, int* F);
int sharded_text_stats(rass_engine* h, int64_t* indptr, int64_t* doc_count, int64_t* sum_ttf);
// the two halves of rass_text_commit and the statistics a sharded handle sums in between (postings.cu)
int text_commit_merge(rass_engine* h, const int64_t* field_vocab, int F, int64_t N);
int text_local_stats(rass_engine* h, int F, int64_t N, int64_t* doc_count, int64_t* sum_ttf);
int text_finalize_global(rass_engine* h, int64_t N, int F, const int64_t* g_doc_count, const int64_t* g_sum_ttf,
                         const int64_t* global_df);
const std::vector<rass_engine*>& sharded_shards(rass_engine* h);
rass_engine* sharded_first(rass_engine* h);      // the shard on the coordinator device (dictionary scans run there)
#define SHARDED(h, call)                 \
  do {                                   \
    if ((h) && (h)->shards) return call; \
  } while (0)

int ensure_query_workspace(rass_engine* h, SearchWs& ws, int B);
int ensure_pool(rass_engine* h, SearchWs& ws, size_t entries_per_query, size_t segs_per_query,
                size_t n_queries = RASS_GROUP_Q);
int ensure_xlist_workspace(rass_engine* h, size_t entries);
int ensure_out_workspace(rass_engine* h, size_t n);
