// Batched kNN scan on the 5th-generation tensor cores: up to 64 queries per corpus pass.
//
// Replaces the `knn` clause executor (reference app/main.py:1538-1542 -> OpenSearch k-NN plugin / nmslib HNSW)
// when several queries share one pass over the bf16 shadow matrix.  For <= 64 queries the pass is still
// HBM-bound (64 flop/byte against a ridge of ~210), but only the tensor pipe can keep up with the stream.
//
// One persistent CTA per SM.  A = a 128-row corpus tile (M = 128, K-major, 128B-swizzled, streamed by TMA in
// 64-element k-blocks through a ring of smem stages), B = the 64 queries (N = 64, resident in smem for the
// whole pass), D = 128 x 64 fp32 in TMEM, four accumulator stages so the epilogue of tile i overlaps the MMAs
// of tiles i+1..i+3.  Warp 0 lane 0 issues TMA, warp 1 lane 0 issues tcgen05.mma, warp 2 owns the TMEM
// allocation, warps 4-7 are the epilogue: thread = corpus row (TMEM lane), 64 scores per thread read with
// tcgen05.ld; a score that beats the CTA's running per-query threshold is appended to that query's segment of
// the candidate pool.  When a segment passes 128 entries it is compacted: a warp bisects for a pivot with
// 32..64 entries above it, keeps those and raises the threshold to the pivot; everything dropped or
// rejected is <= that threshold, which is the bound the certificate in finish.cu needs.  The score matrix never reaches HBM.
//
// The int8 instantiation (I8) streams the int8 shadow x8 instead -- half the bytes per row -- with kind::i8 MMAs: B = the
// 64 queries' two int8 parts (N = 128: q1 in columns 0..63, q2 in 64..127), D = 128 x 128 s32 (exact integer dots), all
// 512 TMEM columns over the four stages.  A k-block is still one 128-byte swizzle row (128 int8 elements), so the smem
// ring, its stages and the Q block's size are those of the bf16 pass.  The epilogue combines the two accumulators of a
// query into key = sa8 * (s1 * acc1 + s2 * acc2) + sb (int8_key); everything after that is shared.
#include "tc_ptx.cuh"

#define UMMA_ROWS 128
#define UMMA_NQ 64
#define UMMA_KBLK 64                       // bf16 elements per k-block (128 bytes: one swizzle row; 128 int8 elements)
#define UMMA_STAGE_BYTES (UMMA_ROWS * 128)  // 16 KB
#define UMMA_QBLK_BYTES (UMMA_NQ * 128)     // 8 KB (int8: 16 KB, two parts per query)
#define UMMA_STAGES 6                       // smem stages of the ring (run-time: 2..UMMA_STAGES, see umma_launch)
#define UMMA_ACC 4                          // TMEM accumulator stages (64 columns each; int8: 128)
#define UMMA_THREADS 256
#define UMMA_RING 8                         // tile ids in flight between the producer and the other roles

namespace {

// kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, N = 64, M = 128
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((UMMA_NQ >> 3) << 17) | ((UMMA_ROWS >> 4) << 24);
// kind::i8 instruction descriptor: D = s32, A = B = signed int8, both K-major, N = 128, M = 128
constexpr uint32_t kIdesc8 = (2u << 4) | (1u << 7) | (1u << 10) | (((2 * UMMA_NQ) >> 3) << 17) | ((UMMA_ROWS >> 4) << 24);

// per operand kind: accumulator columns per stage (= B rows), elements per k-block
template <bool I8> constexpr int umma_ncol() { return I8 ? 2 * UMMA_NQ : UMMA_NQ; }
template <bool I8> constexpr int umma_kblk() { return I8 ? 2 * UMMA_KBLK : UMMA_KBLK; }

struct UmmaSmem {
  uint64_t full[UMMA_STAGES];
  uint64_t empty[UMMA_STAGES];
  uint64_t acc_full[UMMA_ACC];
  uint64_t acc_empty[UMMA_ACC];
  uint64_t q_full;
  uint64_t ring_full[UMMA_RING];
  int ring[UMMA_RING];
  uint32_t tmem_base;
  uint32_t pad;
  float thr[UMMA_NQ];
  int cnt[UMMA_NQ];
  float qsc[2][UMMA_NQ];     // int8 pass: the scales s1, s2 of the queries' two parts
};

}  // namespace

// SEG = pool entries per (CTA, query) segment: once SEG/2 is passed a compaction keeps rass_tc_keep(SEG) .. twice
// that many entries.  256 (keeps 32..64) serves k <= 32; 512 (keeps 128..256) keeps at least k entries above every
// pivot for k <= 128, so a cluster of near neighbours inside one segment cannot push the bound past the k-th best.
// I8: map_x over x8, map_q over q8 (q_row0 = the group's first q8 row), sa = sa8, q8_scale = the group's [64][2] scales.
template <int SEG, bool I8>
__global__ void __launch_bounds__(UMMA_THREADS, 1)
    scan_umma_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_q,
                     const float* __restrict__ sa, const float* __restrict__ sb, const float* __restrict__ q8_scale,
                     int64_t n_rows, int n_tiles,
                     int k_blocks, int q_row0, float* __restrict__ pool_key, uint32_t* __restrict__ pool_row,
                     float* __restrict__ pool_thr, int* __restrict__ pool_cnt, size_t pool_entries, int n_segs,
                     uint32_t* __restrict__ gthr, int* __restrict__ tile_ctr, float* __restrict__ dbg_out,
                     int relaxed_wait, unsigned long long* __restrict__ dbg_t, int n_stages) {
  constexpr int NCOL = umma_ncol<I8>(), KBLK = umma_kblk<I8>(), QBLK_BYTES = NCOL * 128;
  constexpr uint32_t TMEM_COLS = UMMA_ACC * NCOL;
  extern __shared__ unsigned char smem_dyn[];
  // 128B-swizzled tiles need 1024-byte alignment: [ Q: k_blocks * QBLK_BYTES ][ stages: UMMA_STAGES * 16 KB ][ UmmaSmem ]
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  unsigned char* q_smem = smem;
  unsigned char* x_smem = smem + (size_t)k_blocks * QBLK_BYTES;
  UmmaSmem* ss = reinterpret_cast<UmmaSmem*>(x_smem + (size_t)n_stages * UMMA_STAGE_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cta = blockIdx.x;
  if (dbg_t && threadIdx.x == 0) dbg_t[cta * 4 + 0] = globaltimer_ns();

  if (threadIdx.x == 0) {
    for (int i = 0; i < UMMA_STAGES; ++i) { mbar_init(&ss->full[i], 1); mbar_init(&ss->empty[i], 1); }
    for (int i = 0; i < UMMA_ACC; ++i) { mbar_init(&ss->acc_full[i], 1); mbar_init(&ss->acc_empty[i], 4); }
    mbar_init(&ss->q_full, 1);
    for (int i = 0; i < UMMA_RING; ++i) mbar_init(&ss->ring_full[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (threadIdx.x < UMMA_NQ) {
    // the seed launch_seed_thresholds left for the query (0 = none): see store.cu
    const uint32_t g = __ldcg(gthr + threadIdx.x);
    ss->thr[threadIdx.x] = g > 0x007fffffu ? unord32(g) : neg_inf<float>();
    ss->cnt[threadIdx.x] = 0;
    if (I8) {
      ss->qsc[0][threadIdx.x] = q8_scale[2 * threadIdx.x];
      ss->qsc[1][threadIdx.x] = q8_scale[2 * threadIdx.x + 1];
    }
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&ss->tmem_base)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = ss->tmem_base;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      mbar_expect_tx(&ss->q_full, (uint32_t)k_blocks * QBLK_BYTES);
      for (int kb = 0; kb < k_blocks; ++kb)
        tma_load_2d(&map_q, &ss->q_full, q_smem + (size_t)kb * QBLK_BYTES, kb * KBLK, q_row0, kEvictLast);
      int stage = 0;
      uint32_t phase = 0;
      // Tiles are drawn from a device-wide counter (the first one is the CTA's own): a CTA that starts late -- the
      // previous batch's finish kernel may still hold its SM -- or meets more compactions simply takes fewer tiles,
      // and all CTAs end within one tile of each other.  The id of the tile after this one is requested before this
      // tile's loads are issued, so the L2 round trip of the atomic is never waited for.  Ids travel to the MMA and
      // epilogue roles through a ring in shared memory; the roles are at most 5 tiles apart (4 accumulator stages +
      // the smem stages), so UMMA_RING slots never wrap onto a live entry.
      int tile = cta;
      for (int it = 0;; ++it) {
        ss->ring[it & (UMMA_RING - 1)] = tile;
        mbar_arrive(&ss->ring_full[it & (UMMA_RING - 1)]);
        if (tile >= n_tiles) break;
        const int next = tile_ctr ? (int)gridDim.x + atomicAdd(tile_ctr, 1) : tile + (int)gridDim.x;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(&ss->empty[stage], phase ^ 1);
          mbar_expect_tx(&ss->full[stage], UMMA_STAGE_BYTES);
          tma_load_2d(&map_x, &ss->full[stage], x_smem + (size_t)stage * UMMA_STAGE_BYTES, kb * KBLK,
                      tile * UMMA_ROWS, kEvictFirst);
          if (++stage == n_stages) { stage = 0; phase ^= 1; }
        }
        tile = next;
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      mbar_wait(&ss->q_full, 0);
      tc_fence_after();
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      const uint32_t q_base = smem_u32(q_smem), x_base = smem_u32(x_smem);
      for (int it = 0;; ++it) {
        mbar_wait(&ss->ring_full[it & (UMMA_RING - 1)], (uint32_t)(it / UMMA_RING) & 1u);
        if (*(volatile int*)&ss->ring[it & (UMMA_RING - 1)] >= n_tiles) break;
        mbar_wait(&ss->acc_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * NCOL;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(&ss->full[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = x_base + (uint32_t)stage * UMMA_STAGE_BYTES;
          const uint32_t b_addr = q_base + (uint32_t)kb * QBLK_BYTES;
          // four MMAs of K = 32 bytes (16 bf16 / 32 int8 elements) per 128-byte k-block
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            if (I8)
              umma_i8(d_tmem, smem_desc_sw128(a_addr + k * 32), smem_desc_sw128(b_addr + k * 32), kIdesc8,
                      (uint32_t)((kb | k) != 0));
            else
              umma_bf16(d_tmem, smem_desc_sw128(a_addr + k * 32), smem_desc_sw128(b_addr + k * 32), kIdesc,
                        (uint32_t)((kb | k) != 0));
          }
          umma_commit(&ss->empty[stage]);   // frees the smem stage once these MMAs have read it
          if (++stage == n_stages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&ss->acc_full[acc]);    // accumulator complete
        if (++acc == UMMA_ACC) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue: thread = corpus row =====
    const int ew = warp - 4;                 // TMEM lane quadrant (warp % 4)
    const int et = threadIdx.x - 128;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int it = 0;; ++it) {
      mbar_wait(&ss->ring_full[it & (UMMA_RING - 1)], (uint32_t)(it / UMMA_RING) & 1u);
      const int tile = *(volatile int*)&ss->ring[it & (UMMA_RING - 1)];
      if (tile >= n_tiles) break;
      const int64_t row = (int64_t)tile * UMMA_ROWS + ew * 32 + lane;
      float a = 0.f, b = neg_inf<float>();
      if (row < n_rows) { a = __ldg(sa + row); b = __ldg(sb + row); }
      // the largest pivot any CTA has published for the query this lane looks after (used after the tile)
      const uint32_t g = lane < UMMA_NQ / 4 ? __ldcg(gthr + 4 * lane + ew) : 0u;
      // one lane polls (sleeping between polls: the epilogue is normally far ahead of the tensor pipe), the warp
      // follows through the warp barrier; 127 spinning threads next to the MMAs only cost power
      // every thread polls: measured ~1 % faster here than one sleeping lane per warp (A/B on the same box, cfg2),
      // unlike in the tensor-bound pair kernel; RASS_DEBUG_RELAXED_WAIT switches for the comparison
      if (!relaxed_wait) mbar_wait(&ss->acc_full[acc], acc_phase);
      else if (lane == 0) mbar_wait_relaxed(&ss->acc_full[acc], acc_phase);
      __syncwarp();
      tc_fence_after();
      if (dbg_t && et == 0 && it == 0) dbg_t[cta * 4 + 1] = globaltimer_ns();
      const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)acc * NCOL;
#pragma unroll
      for (int c = 0; c < UMMA_NQ; c += 16) {
        uint32_t v[16], w[16];     // w: the int8 pass's second-part accumulators of the same queries
        tmem_ld16(taddr + c, v);
        if (I8) tmem_ld16(taddr + c + UMMA_NQ, w);
        tmem_ld_wait();
        if (dbg_out && row < n_rows) {
          // raw accumulators: fp32 [n_rows, 64] (bf16), int32 [n_rows, 128] (int8)
          uint32_t* dbg = reinterpret_cast<uint32_t*>(dbg_out) + (size_t)row * NCOL;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            dbg[c + j] = v[j];
            if (I8) dbg[UMMA_NQ + c + j] = w[j];
          }
        }
        float sc[16];
        uint32_t m = 0;
#pragma unroll
        for (int j4 = 0; j4 < 16; j4 += 4) {
          const float4 t4 = *reinterpret_cast<const float4*>(&ss->thr[c + j4]);
          const float tt[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (I8)
              sc[j4 + j] = int8_key((int32_t)v[j4 + j], (int32_t)w[j4 + j], ss->qsc[0][c + j4 + j],
                                    ss->qsc[1][c + j4 + j], a, b);
            else
              sc[j4 + j] = fmaf(__uint_as_float(v[j4 + j]), a, b);
            m |= (sc[j4 + j] > tt[j]) ? (1u << (j4 + j)) : 0u;
          }
        }
        if (__any_sync(0xffffffffu, m != 0)) {
          // each lane walks its own hits; lanes run their i-th append together
          while (m) {
            const int j = __ffs(m) - 1;
            m &= m - 1;
            float s = sc[0];
#pragma unroll
            for (int t = 1; t < 16; ++t) s = (j == t) ? sc[t] : s;
            const int pos = atomicAdd(&ss->cnt[c + j], 1);
            if (pos < SEG) {
              const size_t o = (size_t)(c + j) * pool_entries + (size_t)cta * SEG + pos;
              pool_key[o] = s;
              pool_row[o] = (uint32_t)row;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&ss->acc_empty[acc]);
      if (++acc == UMMA_ACC) { acc = 0; acc_phase ^= 1; }

      // compaction: all 128 epilogue threads have finished this tile's appends
      asm volatile("bar.sync 1, 128;" ::: "memory");
      // warp ew owns queries q = ew (mod 4).  A pivot found by ANY CTA bounds what this CTA may reject as well: the
      // certificate takes the maximum bound over segments, and this segment publishes the largest threshold it used.
      if (g > 0x007fffffu) ss->thr[4 * lane + ew] = fmaxf(ss->thr[4 * lane + ew], unord32(g));
      __syncwarp();
      // segments past their high-water mark; the loads of the next one are in flight while this one is compacted
      // (a compaction is mostly the L2 round trip of its 2 x SEG/32 loads per lane)
      unsigned need = __ballot_sync(0xffffffffu, lane < UMMA_NQ / 4 && ss->cnt[4 * lane + ew] > (SEG / 2));
      uint32_t ok[SEG / 32], rw[SEG / 32], ok_n[SEG / 32], rw_n[SEG / 32];
      auto load_seg = [&](int q, uint32_t (&k_)[SEG / 32], uint32_t (&r_)[SEG / 32]) {
        const int n = min(ss->cnt[q], SEG);
        const size_t base = (size_t)q * pool_entries + (size_t)cta * SEG;
#pragma unroll
        for (int i = 0; i < SEG / 32; ++i) {
          const int idx = i * 32 + lane;
          // keys as order-preserving integers; empty slots are 0
          k_[i] = idx < n ? ord32(__ldcg(pool_key + base + idx)) : 0u;
          r_[i] = idx < n ? __ldcg(pool_row + base + idx) : 0xffffffffu;
        }
      };
      int q_cur = -1;
      if (need) {
        q_cur = 4 * (__ffs(need) - 1) + ew;
        need &= need - 1;
        load_seg(q_cur, ok, rw);
      }
      while (q_cur >= 0) {
        int q_next = -1;
        if (need) {
          q_next = 4 * (__ffs(need) - 1) + ew;
          need &= need - 1;
          load_seg(q_next, ok_n, rw_n);
        }
        const size_t base = (size_t)q_cur * pool_entries + (size_t)cta * SEG;
        __syncwarp();
        uint32_t pivot;
        const int kept = warp_compact<SEG / 32>(ok, rw, rass_tc_keep(SEG), pool_key + base, pool_row + base, pivot);
        __syncwarp();
        // everything dropped here, and every row rejected from now on, has key <= pivot
        if (lane == 0) {
          ss->cnt[q_cur] = kept;
          ss->thr[q_cur] = fmaxf(ss->thr[q_cur], unord32(pivot));
          atomicMax(gthr + q_cur, pivot);
        }
#pragma unroll
        for (int i = 0; i < SEG / 32; ++i) { ok[i] = ok_n[i]; rw[i] = rw_n[i]; }
        q_cur = q_next;
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (dbg_t && et == 0 && cta == 0 && it < 64) dbg_t[1024 + it] = globaltimer_ns();
    }
    if (dbg_t && et == 0) dbg_t[cta * 4 + 2] = globaltimer_ns();
    // publish the segment sizes and bounds
    if (et < UMMA_NQ) {
      pool_cnt[(size_t)et * n_segs + cta] = min(ss->cnt[et], SEG);
      pool_thr[(size_t)et * n_segs + cta] = ss->thr[et];
    }
  }

  tc_fence_before();
  __syncthreads();
  if (dbg_t && threadIdx.x == 0) dbg_t[cta * 4 + 3] = globaltimer_ns();
  // the last CTA through leaves the tile counter at zero for the next pass (every producer has drawn its last id)
  if (tile_ctr && threadIdx.x == 0 && atomicAdd(tile_ctr + 1, 1) == (int)gridDim.x - 1) {
    tile_ctr[0] = 0;
    tile_ctr[1] = 0;
  }
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS)
                 : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode(rass_engine* h) {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !p) {
    rass_fail(h, RASS_E_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    return nullptr;
  }
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

int encode_rows_map(rass_engine* h, void* map_out, const void* base, int64_t rows, int box_rows, int elem_bytes) {
  CUtensorMap* map = reinterpret_cast<CUtensorMap*>(map_out);
  EncodeTiledFn enc = get_encode(h);
  if (!enc) return RASS_E_CUDA;
  cuuint64_t dims[2] = {(cuuint64_t)h->dim_pad, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)h->dim_pad * elem_bytes};
  cuuint32_t box[2] = {(cuuint32_t)(128 / elem_bytes), (cuuint32_t)box_rows};   // one 128-byte swizzle row
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = elem_bytes == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUresult r = enc(map, dt, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return rass_fail(h, RASS_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return RASS_OK;
}

// stages of the TMA ring: UMMA_STAGES by default; RASS_DEBUG_UMMA_STAGES=n (2..UMMA_STAGES) for the measurement of what
// a smaller ring costs (a ring of 5 would leave room for the seed / finish kernels next to a scan CTA)
static int umma_stages() {
  static const int n = [] {
    const char* e = getenv("RASS_DEBUG_UMMA_STAGES");
    const int v = e ? atoi(e) : UMMA_STAGES;
    return v < 2 ? 2 : (v > UMMA_STAGES ? UMMA_STAGES : v);
  }();
  return n;
}

// (the same for both operand kinds: the int8 Q block is twice the rows of half the k-blocks)
static size_t umma_smem_bytes(const rass_engine* h) {
  return (size_t)(h->dim_pad / UMMA_KBLK) * UMMA_QBLK_BYTES + (size_t)umma_stages() * UMMA_STAGE_BYTES +
         sizeof(UmmaSmem) + 1024;
}

int scan_umma_segs(const rass_engine* h) { return h->num_sms; }

// RASS_DEBUG_TIMES: where a pass spends its fixed cost (start skew, first accumulator, spread of the CTAs' last tile)
static void umma_report_times(rass_engine* h, unsigned long long* dbg_t, int grid, cudaStream_t st) {
  static int n_reports = 0;
  std::vector<unsigned long long> t(1024 + 64);
  if (cudaStreamSynchronize(st) != cudaSuccess) return;
  if (cudaMemcpy(t.data(), dbg_t, t.size() * 8, cudaMemcpyDeviceToHost) != cudaSuccess) return;
  if (++n_reports > 400 || (n_reports % 20) != 0) return;
  fprintf(stderr, "[umma times] CTA 0, epilogue done with tile i (us since start):");
  for (int i = 0; i < 64 && i < (int)((h->n_rows + 127) / 128 + grid - 1) / grid; ++i)
    fprintf(stderr, " %.1f", (double)(t[1024 + i] - t[0]) * 1e-3);
  fprintf(stderr, "\n");
  unsigned long long t0 = ~0ull, s_max = 0, e_min = ~0ull, e_max = 0, x_max = 0;
  double first = 0, first_max = 0, e_mean = 0;
  for (int c = 0; c < grid; ++c) {
    t0 = std::min(t0, t[c * 4]);
    s_max = std::max(s_max, t[c * 4]);
  }
  for (int c = 0; c < grid; ++c) {
    const double f = (double)(t[c * 4 + 1] - t[c * 4]) * 1e-3;
    first += f / grid;
    first_max = std::max(first_max, f);
    e_min = std::min(e_min, t[c * 4 + 2]);
    e_max = std::max(e_max, t[c * 4 + 2]);
    e_mean += (double)(t[c * 4 + 2] - t0) * 1e-3 / grid;
    x_max = std::max(x_max, t[c * 4 + 3]);
  }
  fprintf(stderr, "[umma times] rows %lld grid %d: start skew %.1f us, first accumulator after %.1f us (max %.1f), "
          "last tile done min %.1f mean %.1f max %.1f us, kernel end %.1f us\n", (long long)h->n_rows, grid,
          (double)(s_max - t0) * 1e-3, first, first_max, (double)(e_min - t0) * 1e-3, e_mean, (double)(e_max - t0) * 1e-3,
          (double)(x_max - t0) * 1e-3);
}

static int umma_launch(rass_engine* h, SearchWs& ws, int q0, int64_t n_rows, int seg, float* dbg_out, cudaStream_t st,
                       bool int8) {
  int rc;
  if (int8) {
    if (!h->x8 || !ws.q8) return rass_fail(h, RASS_E_UNSUPPORTED, "the int8 pass needs the int8 shadow");
    if (!h->tmap_x8) h->tmap_x8 = calloc(1, sizeof(CUtensorMap));
    if (!ws.tmap_q8) ws.tmap_q8 = calloc(1, sizeof(CUtensorMap));
    if (h->tmap8_base != h->x8 || h->tmap8_rows != h->cap) {
      if ((rc = encode_rows_map(h, (CUtensorMap*)h->tmap_x8, h->x8, h->cap, UMMA_ROWS, 1))) return rc;
      h->tmap8_base = h->x8;
      h->tmap8_rows = h->cap;
    }
    if (ws.tmap_q8base != ws.q8) {
      if ((rc = encode_rows_map(h, (CUtensorMap*)ws.tmap_q8, ws.q8, (int64_t)ws.q_cap * 2, 2 * UMMA_NQ, 1))) return rc;
      ws.tmap_q8base = ws.q8;
    }
  } else {
    if (!h->tmap_x) h->tmap_x = calloc(1, sizeof(CUtensorMap));
    if (!ws.tmap_q) ws.tmap_q = calloc(1, sizeof(CUtensorMap));
    // the map spans the whole reservation (>= 1024 rows); rows >= n_rows are masked in the epilogue
    if (h->tmap_base != h->x16 || h->tmap_rows != h->cap) {
      if ((rc = encode_rows_map(h, (CUtensorMap*)h->tmap_x, h->x16, h->cap, UMMA_ROWS))) return rc;
      h->tmap_base = h->x16;
      h->tmap_rows = h->cap;
    }
    if (ws.tmap_qbase != ws.q16) {
      if ((rc = encode_rows_map(h, (CUtensorMap*)ws.tmap_q, ws.q16, ws.q_cap, UMMA_NQ))) return rc;
      ws.tmap_qbase = ws.q16;
    }
  }
  const int n_tiles = (int)((n_rows + UMMA_ROWS - 1) / UMMA_ROWS);
  // RASS_OPT_SCAN_RESERVE_SMS: leave a few SMs to the kernels that run beside the pass (the other slot's finish, the
  // NCCL all-gather and the merge of a row-sharded index); the tile counter spreads the tiles over whatever runs
  const int ctas = std::max(1, h->num_sms - h->scan_reserve_sms);
  const int grid = n_tiles < ctas ? n_tiles : ctas;
  // q_gthr[q0 .. q0 + 64) was initialised by launch_seed_thresholds (or cleared by the self-test)
  static const int relaxed_wait = getenv("RASS_DEBUG_RELAXED_WAIT") != nullptr;
  // RASS_DEBUG_STATIC_TILES: tile = cta + i * grid instead of the device-wide counter (the A/B switch of the measurement)
  static const bool static_tiles = getenv("RASS_DEBUG_STATIC_TILES") != nullptr;
  const size_t smem = umma_smem_bytes(h);
  // timing experiment only (RASS_DEBUG_TIMES): per-CTA timestamps, printed after a blocking wait
  static const bool want_times = getenv("RASS_DEBUG_TIMES") != nullptr;
  static unsigned long long* dbg_t = nullptr;
  if (want_times && !dbg_t) CUDA_TRY(h, cudaMalloc(&dbg_t, 4 * 1024 * sizeof(unsigned long long)));
#define RASS_UMMA_LAUNCH(S, I8)                                                                                      \
  do {                                                                                                               \
    CUDA_TRY(h, cudaFuncSetAttribute(scan_umma_kernel<S, I8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    scan_umma_kernel<S, I8><<<grid, UMMA_THREADS, smem, st>>>(                                                       \
        *(CUtensorMap*)(I8 ? h->tmap_x8 : h->tmap_x), *(CUtensorMap*)(I8 ? ws.tmap_q8 : ws.tmap_q),                  \
        I8 ? h->sa8 : h->sa, h->sb_scan, I8 ? ws.q8_scale + 2 * q0 : nullptr, n_rows, n_tiles,                       \
        h->dim_pad / umma_kblk<I8>(), I8 ? 2 * q0 : q0, ws.pool_key, ws.pool_row, ws.pool_thr, ws.pool_cnt,          \
        ws.pool_entries, scan_umma_segs(h), ws.q_gthr + q0, static_tiles ? nullptr : &ws.scal->tile_ctr[0], dbg_out, \
        relaxed_wait, dbg_t, umma_stages());                                                                         \
  } while (0)
  if (int8) {
    if (seg == 512) RASS_UMMA_LAUNCH(512, true); else RASS_UMMA_LAUNCH(256, true);
  } else {
    if (seg == 512) RASS_UMMA_LAUNCH(512, false); else RASS_UMMA_LAUNCH(256, false);
  }
#undef RASS_UMMA_LAUNCH
  CUDA_TRY(h, cudaGetLastError());
  if (dbg_t) umma_report_times(h, dbg_t, grid, st);
  // segments of CTAs that did not launch (fewer tiles than SMs) were cleared by the caller and read as empty
  return RASS_OK;
}

__global__ void clear_segs_kernel(float* thr, int* cnt, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  thr[i] = neg_inf<float>();
  cnt[i] = 0;
}

int launch_scan_umma(rass_engine* h, SearchWs& ws, int q0, int nq, int seg, cudaStream_t st, bool pool_cleared,
                     bool int8) {
  (void)nq;
  if (!pool_cleared) {       // the seed kernel clears for the first group of a search
    const size_t n = (size_t)scan_umma_segs(h) * RASS_GROUP_Q;
    clear_segs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ws.pool_thr, ws.pool_cnt, n);
    CUDA_TRY(h, cudaGetLastError());
  }
  return umma_launch(h, ws, q0, h->n_rows, seg, nullptr, st, int8);
}

// Debug/self-test entry: raw tensor-core dot products of the first 64 prepared queries against every row.
// out_host: [n_rows, 64] fp32.  Used by tests to localise descriptor/layout errors.
int umma_selftest(rass_engine* h, SearchWs& ws, int n_rows_unused, float* out_host, cudaStream_t st) {
  (void)n_rows_unused;
  float* dbg = nullptr;
  const size_t n = (size_t)h->n_rows * UMMA_NQ;
  CUDA_TRY(h, cudaMalloc(&dbg, n * 4));
  CUDA_TRY(h, cudaMemsetAsync(dbg, 0, n * 4, st));
  int rc = ensure_pool(h, ws, (size_t)scan_umma_segs(h) * 256, (size_t)scan_umma_segs(h));
  if (!rc) {
    const size_t ns = (size_t)scan_umma_segs(h) * RASS_GROUP_Q;
    clear_segs_kernel<<<(unsigned)((ns + 255) / 256), 256, 0, st>>>(ws.pool_thr, ws.pool_cnt, ns);
    cudaMemsetAsync(ws.q_gthr, 0, UMMA_NQ * sizeof(uint32_t), st);
    rc = umma_launch(h, ws, 0, h->n_rows, 256, dbg, st, false);
  }
  if (!rc) {
    cudaError_t e = cudaMemcpyAsync(out_host, dbg, n * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = rass_fail(h, RASS_E_CUDA, "umma selftest: %s", cudaGetErrorString(e));
  }
  cudaFree(dbg);
  return rc;
}

// The int8 pass's raw int32 accumulators of the first 64 prepared queries against every row: out_host [n_rows, 128]
// (columns q: first part of query q, 64 + q: its second part).  Lets the tests check the kind::i8 descriptors and the
// UINT8 tensor maps against integer dot products.
int umma8_selftest(rass_engine* h, SearchWs& ws, int32_t* out_host, cudaStream_t st) {
  int32_t* dbg = nullptr;
  const size_t n = (size_t)h->n_rows * 2 * UMMA_NQ;
  CUDA_TRY(h, cudaMalloc(&dbg, n * 4));
  CUDA_TRY(h, cudaMemsetAsync(dbg, 0, n * 4, st));
  int rc = ensure_pool(h, ws, (size_t)scan_umma_segs(h) * 256, (size_t)scan_umma_segs(h));
  if (!rc) {
    const size_t ns = (size_t)scan_umma_segs(h) * RASS_GROUP_Q;
    clear_segs_kernel<<<(unsigned)((ns + 255) / 256), 256, 0, st>>>(ws.pool_thr, ws.pool_cnt, ns);
    cudaMemsetAsync(ws.q_gthr, 0, UMMA_NQ * sizeof(uint32_t), st);
    rc = umma_launch(h, ws, 0, h->n_rows, 256, reinterpret_cast<float*>(dbg), st, true);
  }
  if (!rc) {
    cudaError_t e = cudaMemcpyAsync(out_host, dbg, n * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = rass_fail(h, RASS_E_CUDA, "umma8 selftest: %s", cudaGetErrorString(e));
  }
  cudaFree(dbg);
  return rc;
}
