// Large-batch kNN scan: the dense Q . X^T contraction on CTA pairs of the 5th-generation tensor cores.
//
// Replaces the `knn` clause executor (reference app/main.py:1538-1542 -> OpenSearch k-NN plugin / nmslib HNSW)
// when hundreds of queries share the corpus (BASELINE configs[2] batch 8192 top-100, configs[4] batch 1024).
// At 256 queries per pass the scan is tensor-bound (256 flop per corpus byte against a ridge of ~210), so the
// design goal is MMA issue without gaps and no score matrix in HBM.
//
// Work item = (corpus chunk, group of 256 queries).  Items are dealt round-robin to the 74 CTA pairs in group-major
// order, so the pairs that run at the same time sweep the SAME chunk for DIFFERENT query groups: the chunk comes
// from HBM once and from the 126 MB L2 for the other groups.  Inside an item a pair walks the chunk in tiles of
// 256 rows: tcgen05.mma cta_group::2, M = 256 (128 rows per CTA), N = 256 queries, K = 16 per instruction;
// every CTA streams its own 128 corpus rows and its half of the query block (2 x 16 KB per 64-element k-block)
// through a TMA ring whose full-barriers live in the leader CTA; the accumulator (128 lanes x 256 fp32 columns per
// CTA, two stages = all 512 TMEM columns) is drained by four epilogue warps per CTA: thread = corpus row,
// tcgen05.ld, score = acc * sa + sb, one compare against the per-query running threshold, and the survivors are
// appended to the (item, CTA) segment of the candidate pool and compacted exactly as in scan_umma.cu.  The bound
// each segment publishes (every row it dropped or rejected has key <= thr) is what the certificate in finish.cu needs.
#include "tc_ptx.cuh"

#define G2_ROWS 128                        // corpus rows per CTA per tile (256 per pair)
#define G2_NQ 256                          // queries per group (MMA N) of the main instantiation; 128 for 65..128 queries
#define G2_KBLK 64                         // bf16 elements per k-block (128 bytes: one swizzle row)
#define G2_A_BYTES (G2_ROWS * 128)         // 16 KB
#define G2_MAX_STAGES 8
#define G2_MAX_ACC 4
#define G2_TMEM_COLS 512
#define G2_THREADS 256
#define G2_HIT_STRIDE 36                   // floats per epilogue thread in the hit staging area (36: STS.128 conflict-free)

namespace {

// NQ = 256: the contraction regime (tensor-bound).  NQ = 128: 65..128 queries, half the MMA work per corpus byte, so
// the pass is HBM-bound again (~3.1 ms at 10M rows instead of 5.1 ms).
template <int NQ>
struct G2Cfg {
  static constexpr int B_BYTES = (NQ / 2) * 128;                 // this CTA's half of the query block per k-block
  static constexpr int STAGE_BYTES = G2_A_BYTES + B_BYTES;       // 32 KB / 24 KB
  static constexpr int STAGES = NQ == 256 ? 6 : 8;               // 192 KB of ring either way
  static constexpr int ACC = G2_TMEM_COLS / NQ;                  // TMEM accumulator stages of NQ columns
  // kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, N = NQ, M = 256 (pair)
  static constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NQ >> 3) << 17) | ((256u >> 4) << 24);
};

struct GemmSmem {
  uint64_t full[G2_MAX_STAGES];   // used in the leader CTA: both CTAs' TMA bytes of a stage have landed
  uint64_t empty[G2_MAX_STAGES];  // per CTA: the pair's MMAs have read this stage
  uint64_t acc_full[G2_MAX_ACC];  // per CTA: accumulator stage complete
  uint64_t acc_empty[G2_MAX_ACC]; // used in the leader CTA: both CTAs' epilogues have drained the stage
  uint32_t tmem_base;
  uint32_t pad;
  alignas(16) float thr[G2_NQ];
  int cnt[G2_NQ];
  // a thread that finds survivors among its 32 scores parks them here so the append loop can index them (registers
  // cannot be indexed: the alternative is a 32-deep select chain per survivor)
  alignas(16) float hit[128 * G2_HIT_STRIDE];
};

struct GemmPlan {
  int n_ptiles;          // 256-row pair tiles
  int n_groups;          // query groups of 256
  int n_chunks;          // corpus chunks
  int tiles_per_chunk;   // pair tiles per chunk
  int n_items;           // n_chunks * n_groups
};

}  // namespace

template <int SEG, int NQ>      // SEG: pool entries per (item, CTA, query) segment, see scan_umma.cu
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(G2_THREADS, 1)
    scan_gemm_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_q,
                     const float* __restrict__ sa, const float* __restrict__ sb, int64_t n_rows, GemmPlan plan,
                     int k_blocks, int n_queries, float* __restrict__ pool_key, uint32_t* __restrict__ pool_row,
                     float* __restrict__ pool_thr, int* __restrict__ pool_cnt, size_t pool_entries, int n_segs,
                     uint32_t* __restrict__ gthr, float* __restrict__ dbg_out, int dbg_mode) {
  extern __shared__ unsigned char smem_dyn[];
  // 128B-swizzled tiles need 1024-byte alignment: [ stages: G2Cfg<NQ>::STAGES * (A 16 KB | B 16 KB) ][ GemmSmem ]
  // (the dynamic window starts at the same offset in both CTAs, so the pair's operand descriptors agree)
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  GemmSmem* ss = reinterpret_cast<GemmSmem*>(smem + (size_t)G2Cfg<NQ>::STAGES * G2Cfg<NQ>::STAGE_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    for (int i = 0; i < G2Cfg<NQ>::STAGES; ++i) { mbar_init(&ss->full[i], 1); mbar_init(&ss->empty[i], 1); }
    for (int i = 0; i < G2Cfg<NQ>::ACC; ++i) { mbar_init(&ss->acc_full[i], 1); mbar_init(&ss->acc_empty[i], 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&ss->tmem_base)),
                 "r"((uint32_t)G2_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();       // the peer's barriers are initialised before anything of ours can reach them
  tc_fence_after();
  const uint32_t tmem_base = ss->tmem_base;

  if (warp == 0) {
    // ===== TMA producer (both CTAs): own 128 corpus rows + own half of the query block per k-block =====
    if (lane == 0) {
      int stage = 0, n_issued = 0;
      uint32_t phase = 0;
      for (int w = pair; w < plan.n_items; w += n_pairs) {
        const int chunk = w / plan.n_groups, grp = w - chunk * plan.n_groups;
        const int t0 = chunk * plan.tiles_per_chunk, t1 = min(t0 + plan.tiles_per_chunk, plan.n_ptiles);
        const int q_row = grp * NQ + (int)rank * (NQ / 2);
        for (int t = t0; t < t1; ++t) {
          const int x_row = t * 2 * G2_ROWS + (int)rank * G2_ROWS;
          for (int kb = 0; kb < k_blocks; ++kb) {
            mbar_wait_relaxed(&ss->empty[stage], phase ^ 1);
            const uint32_t bar = mapa_u32(smem_u32(&ss->full[stage]), 0);
            const bool warm = dbg_mode >= 3 && n_issued >= G2Cfg<NQ>::STAGES;      // timing experiments only
            const bool skip_b = warm, skip_a = warm && dbg_mode == 4;
            ++n_issued;
            if (rank == 0) {
              const uint32_t bytes = 2 * ((skip_a ? 0 : G2_A_BYTES) + (skip_b ? 0 : G2Cfg<NQ>::B_BYTES));
              if (bytes) mbar_expect_tx(&ss->full[stage], bytes); else mbar_arrive(&ss->full[stage]);
            }
            unsigned char* dst = smem + (size_t)stage * G2Cfg<NQ>::STAGE_BYTES;
            if (!skip_a) tma_load_2d_pair(&map_x, bar, dst, kb * G2_KBLK, x_row, kEvictNormal);
            if (!skip_b) tma_load_2d_pair(&map_q, bar, dst + G2_A_BYTES, kb * G2_KBLK, q_row, kEvictLast);
            if (++stage == G2Cfg<NQ>::STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (leader CTA only) =====
    if (lane == 0 && rank == 0) {
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      const uint32_t s_base = smem_u32(smem);
      for (int w = pair; w < plan.n_items; w += n_pairs) {
        const int chunk = w / plan.n_groups;
        const int t0 = chunk * plan.tiles_per_chunk, t1 = min(t0 + plan.tiles_per_chunk, plan.n_ptiles);
        for (int t = t0; t < t1; ++t) {
          mbar_wait(&ss->acc_empty[acc], acc_phase ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)acc * NQ;
          for (int kb = 0; kb < k_blocks; ++kb) {
            mbar_wait(&ss->full[stage], phase);
            tc_fence_after();
            const uint32_t a_addr = s_base + (uint32_t)stage * G2Cfg<NQ>::STAGE_BYTES;
            const uint32_t b_addr = a_addr + G2_A_BYTES;
#pragma unroll
            for (int k = 0; k < G2_KBLK / 16; ++k)
              umma_bf16_pair(d_tmem, smem_desc_sw128(a_addr + k * 32), smem_desc_sw128(b_addr + k * 32), G2Cfg<NQ>::IDESC,
                             (uint32_t)((kb | k) != 0));
            umma_commit_pair(&ss->empty[stage]);   // frees the stage in both CTAs once these MMAs have read it
            if (++stage == G2Cfg<NQ>::STAGES) { stage = 0; phase ^= 1; }
          }
          umma_commit_pair(&ss->acc_full[acc]);    // accumulator complete, both CTAs' epilogues
          if (++acc == G2Cfg<NQ>::ACC) { acc = 0; acc_phase ^= 1; }
        }
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue (both CTAs): thread = corpus row =====
    const int ew = warp - 4;                 // TMEM lane quadrant (warp % 4)
    const int et = threadIdx.x - 128;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int w = pair; w < plan.n_items; w += n_pairs) {
      const int chunk = w / plan.n_groups, grp = w - chunk * plan.n_groups;
      const int t0 = chunk * plan.tiles_per_chunk, t1 = min(t0 + plan.tiles_per_chunk, plan.n_ptiles);
      const int seg = chunk * 2 + (int)rank;
      const int nq_here = min(NQ, n_queries - grp * NQ);
      // fresh running state of this item's 256 queries; padding queries admit nothing
      for (int q = et; q < NQ; q += 128) {
        const uint32_t g = __ldcg(gthr + (size_t)grp * NQ + q);
        ss->thr[q] = q < nq_here ? (g > 0x007fffffu ? unord32(g) : neg_inf<float>()) : __int_as_float(0x7f800000);
        ss->cnt[q] = 0;
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const size_t slot0 = (size_t)grp * NQ;
      for (int t = t0; t < t1; ++t) {
        const int64_t row = (int64_t)t * 2 * G2_ROWS + rank * G2_ROWS + ew * 32 + lane;
        float a = 0.f, b = neg_inf<float>();
        if (row < n_rows) { a = __ldg(sa + row); b = __ldg(sb + row); }
        // the pivots other CTAs have published for this lane's two queries (used after the tile, latency hidden)
        const uint32_t g0 = __ldcg(gthr + slot0 + 4 * lane + ew);
        const uint32_t g1 = NQ > 128 ? __ldcg(gthr + slot0 + 128 + 4 * lane + ew) : 0u;
        // one lane polls (sleeping between polls: the epilogue is normally far ahead of the tensor pipe), the warp
        // follows through the warp barrier; 127 spinning threads next to the MMAs only cost power
        if (lane == 0) mbar_wait_relaxed(&ss->acc_full[acc], acc_phase);
        __syncwarp();
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)acc * NQ;
#pragma unroll 1
        for (int c = 0; c < (dbg_mode == 1 ? 32 : NQ); c += 32) {
          uint32_t v[32];
          tmem_ld32(taddr + c, v);
          tmem_ld_wait();
          if (dbg_out && grp == 0 && row < n_rows) {
#pragma unroll
            for (int j = 0; j < 32; ++j) dbg_out[(size_t)row * 256 + c + j] = __uint_as_float(v[j]);
          }
          // hot loop: one FMA and one predicate-accumulating compare per score; survivors are rare (a few per
          // warp and tile), so their bit mask is only built when this thread has one
          bool any = false;
#pragma unroll
          for (int j4 = 0; j4 < 32; j4 += 4) {
            const float4 t4 = *reinterpret_cast<const float4*>(&ss->thr[c + j4]);
            const float tt[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float s = fmaf(__uint_as_float(v[j4 + j]), a, b);
              v[j4 + j] = __float_as_uint(s);
              any |= s > tt[j];
            }
          }
          uint32_t m = 0;
          if (any) {
#pragma unroll
            for (int j = 0; j < 32; ++j) m |= (__uint_as_float(v[j]) > ss->thr[c + j]) ? (1u << j) : 0u;
          }
          if (dbg_mode == 2) m = 0;
          // each lane walks its own hits
          if (m) {
            float* mine = ss->hit + (size_t)et * G2_HIT_STRIDE;
#pragma unroll
            for (int u = 0; u < 32; u += 4)
              *reinterpret_cast<uint4*>(mine + u) = make_uint4(v[u], v[u + 1], v[u + 2], v[u + 3]);
            while (m) {
              const int j = __ffs(m) - 1;
              m &= m - 1;
              const float s = mine[j];
              const int pos = atomicAdd(&ss->cnt[c + j], 1);
              if (pos < SEG) {
                const size_t o = (slot0 + c + j) * pool_entries + (size_t)seg * SEG + pos;
                pool_key[o] = s;
                pool_row[o] = (uint32_t)row;
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&ss->acc_empty[acc]), 0));
        if (++acc == G2Cfg<NQ>::ACC) { acc = 0; acc_phase ^= 1; }

        // compaction: all 128 epilogue threads of this CTA have finished the tile's appends
        asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll 1
        for (int qb = 0; qb < NQ; qb += 128) {
          // warp ew owns queries q = ew (mod 4); lane l looks at q = qb + 4 l + ew
          {
            // a pivot any CTA found for this query bounds every row this segment rejects from now on as well:
            // that CTA keeps >= 32 rows above it, and the certificate takes the maximum over segments anyway
            const uint32_t g = qb ? g1 : g0;
            const int q = qb + 4 * lane + ew;
            if (g > 0x007fffffu) ss->thr[q] = fmaxf(ss->thr[q], unord32(g));
          }
          __syncwarp();
          unsigned need = __ballot_sync(0xffffffffu, ss->cnt[qb + 4 * lane + ew] > (SEG / 2));
          while (need) {
            const int q = qb + 4 * (__ffs(need) - 1) + ew;
            need &= need - 1;
            const int n = min(ss->cnt[q], SEG);
            const size_t base = (slot0 + q) * pool_entries + (size_t)seg * SEG;
            uint32_t ok[SEG / 32], rw[SEG / 32];
#pragma unroll
            for (int i = 0; i < SEG / 32; ++i) {
              const int idx = i * 32 + lane;
              ok[i] = idx < n ? ord32(__ldcg(pool_key + base + idx)) : 0u;
              rw[i] = idx < n ? __ldcg(pool_row + base + idx) : 0xffffffffu;
            }
            __syncwarp();
            uint32_t pivot;
            const int kept =
                warp_compact<SEG / 32>(ok, rw, rass_tc_keep(SEG), pool_key + base, pool_row + base, pivot);
            __syncwarp();
            // everything dropped here, and every row rejected from now on, has key <= pivot
            if (lane == 0) {
              ss->cnt[q] = kept;
              ss->thr[q] = fmaxf(ss->thr[q], unord32(pivot));
              atomicMax(gthr + slot0 + q, pivot);
            }
          }
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      // publish the segment sizes and bounds of this item
      for (int q = et; q < nq_here; q += 128) {
        pool_cnt[(slot0 + q) * n_segs + seg] = min(ss->cnt[q], SEG);
        pool_thr[(slot0 + q) * n_segs + seg] = ss->thr[q];
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();       // neither CTA leaves (or frees TMEM) while the pair's MMAs / remote arrives are in flight
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)G2_TMEM_COLS)
                 : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int gcd_int(int a, int b) { return b ? gcd_int(b, a % b) : a; }

static int gemm_nq(int B) { return B <= 128 ? 128 : G2_NQ; }

static GemmPlan make_plan(const rass_engine* h, int B, int n_pairs) {
  GemmPlan p;
  const int nq = gemm_nq(B);
  p.n_ptiles = (int)((h->n_rows + 2 * G2_ROWS - 1) / (2 * G2_ROWS));
  p.n_groups = (B + nq - 1) / nq;
  // items = chunks x groups is a multiple of the pair count, so every pair gets the same number of items
  int chunks = n_pairs / gcd_int(n_pairs, p.n_groups);
  if (chunks > p.n_ptiles) chunks = p.n_ptiles;
  p.tiles_per_chunk = (p.n_ptiles + chunks - 1) / chunks;
  p.n_chunks = (p.n_ptiles + p.tiles_per_chunk - 1) / p.tiles_per_chunk;
  p.n_items = p.n_chunks * p.n_groups;
  return p;
}

static int gemm_pairs(const rass_engine* h) { return h->num_sms / 2; }

int scan_gemm_segs(const rass_engine* h, int B) { return 2 * make_plan(h, B, gemm_pairs(h)).n_chunks; }

static size_t gemm_smem_bytes() { return (size_t)G2Cfg<256>::STAGES * G2Cfg<256>::STAGE_BYTES + sizeof(GemmSmem) + 1024; }
static_assert(G2Cfg<256>::STAGES * G2Cfg<256>::STAGE_BYTES == G2Cfg<128>::STAGES * G2Cfg<128>::STAGE_BYTES, "one smem size");

__global__ void clear_gemm_segs_kernel(float* thr, int* cnt, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  thr[i] = neg_inf<float>();
  cnt[i] = 0;
}

static int gemm_launch(rass_engine* h, SearchWs& ws, int B, int seg, float* dbg_out, cudaStream_t st,
                       bool pool_cleared = false) {
  int rc;
  if (!h->tmap_x) h->tmap_x = calloc(1, sizeof(CUtensorMap));
  if (!ws.tmap_q2) ws.tmap_q2 = calloc(1, sizeof(CUtensorMap));
  if (h->tmap_base != h->x16 || h->tmap_rows != h->cap) {
    if ((rc = encode_rows_map(h, h->tmap_x, h->x16, h->cap, G2_ROWS))) return rc;
    h->tmap_base = h->x16;
    h->tmap_rows = h->cap;
  }
  if (ws.tmap_q2base != ws.q16) {
    if ((rc = encode_rows_map(h, ws.tmap_q2, ws.q16, ws.q_cap, G2_NQ / 2))) return rc;
    ws.tmap_q2base = ws.q16;
  }
  if (!ws.tmap_q) ws.tmap_q = calloc(1, sizeof(CUtensorMap));
  if (ws.tmap_qbase != ws.q16) {          // 64-row query boxes: shared with scan_umma, used by the 128-query form
    if ((rc = encode_rows_map(h, ws.tmap_q, ws.q16, ws.q_cap, 64))) return rc;
    ws.tmap_qbase = ws.q16;
  }
  const int n_pairs = gemm_pairs(h);
  const GemmPlan plan = make_plan(h, B, n_pairs);
  const int n_segs = scan_gemm_segs(h, B);
  const size_t n = (size_t)n_segs * B;
  if (!pool_cleared) {
    clear_gemm_segs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ws.pool_thr, ws.pool_cnt, n);
    CUDA_TRY(h, cudaGetLastError());
  }
  // per-query bound shared between the CTAs (ordered-integer image of a float; 0 = nothing published yet): seeded by
  // launch_seed_thresholds before a search; the self-test has no seed
  if (dbg_out) CUDA_TRY(h, cudaMemsetAsync(ws.q_gthr, 0, (size_t)ws.q_cap * sizeof(uint32_t), st));
  const int grid = 2 * (plan.n_items < n_pairs ? plan.n_items : n_pairs);
  // timing experiments only (results are wrong): 1 = epilogue reads one column block, 2 = epilogue drops every hit
  static const int dbg_mode = getenv("RASS_GEMM_DEBUG_MODE") ? atoi(getenv("RASS_GEMM_DEBUG_MODE")) : 0;
  const size_t smem = gemm_smem_bytes();
#define RASS_GEMM_LAUNCH(S, N, QMAP)                                                                                 \
  do {                                                                                                               \
    CUDA_TRY(h, cudaFuncSetAttribute(scan_gemm_kernel<S, N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    scan_gemm_kernel<S, N><<<grid, G2_THREADS, smem, st>>>(                                                          \
        *(CUtensorMap*)h->tmap_x, *(CUtensorMap*)(QMAP), h->sa, h->sb_scan, h->n_rows, plan, h->dim_pad / G2_KBLK,   \
        B, ws.pool_key, ws.pool_row, ws.pool_thr, ws.pool_cnt, ws.pool_entries, n_segs, ws.q_gthr, dbg_out, dbg_mode); \
  } while (0)
  if (gemm_nq(B) == 128) {
    if (seg == 512) RASS_GEMM_LAUNCH(512, 128, ws.tmap_q); else RASS_GEMM_LAUNCH(256, 128, ws.tmap_q);
  } else {
    if (seg == 512) RASS_GEMM_LAUNCH(512, 256, ws.tmap_q2); else RASS_GEMM_LAUNCH(256, 256, ws.tmap_q2);
  }
#undef RASS_GEMM_LAUNCH
  CUDA_TRY(h, cudaGetLastError());
  return RASS_OK;
}

// all B prepared queries (q16 rows [0, B), padded with zero rows to a multiple of 256) against the whole shard;
// query q's candidates land in pool slot q
int launch_scan_gemm(rass_engine* h, SearchWs& ws, int B, int seg, cudaStream_t st, bool pool_cleared) {
  return gemm_launch(h, ws, B, seg, nullptr, st, pool_cleared);
}

// Debug/self-test entry: raw tensor-core dot products of the first 256 prepared queries against every row.
// out_host: [n_rows, 256] fp32.
int gemm_selftest(rass_engine* h, SearchWs& ws, int B, float* out_host, cudaStream_t st) {
  float* dbg = nullptr;
  const size_t n = (size_t)h->n_rows * G2_NQ;
  CUDA_TRY(h, cudaMalloc(&dbg, n * 4));
  CUDA_TRY(h, cudaMemsetAsync(dbg, 0, n * 4, st));
  const int n_segs = scan_gemm_segs(h, B);
  int rc = ensure_pool(h, ws, (size_t)n_segs * 256, (size_t)n_segs, B);
  if (!rc) rc = gemm_launch(h, ws, B, 256, dbg, st);
  if (!rc) {
    cudaError_t e = cudaMemcpyAsync(out_host, dbg, n * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = rass_fail(h, RASS_E_CUDA, "gemm selftest: %s", cudaGetErrorString(e));
  }
  cudaFree(dbg);
  return rc;
}
