// Vector-store fill and query preparation kernels.
//
// store_convert replaces what OpenSearch does with `_source["embedding"]` on a bulk "index" action
// (reference app/main.py:1256-1269): it lays one appended row down as the resident fp32 row, its bf16
// shadow, its int8 shadow (the arrays the scans stream), its fp64-accumulated norm and the per-row scan
// scale/offset.
// query_prep is the device half of the query normalisation at app/main.py:1536-1537.
#include <cooperative_groups.h>

#include "common.cuh"

// one warp per row
__global__ void __launch_bounds__(256) store_convert_kernel(const float* __restrict__ src, int64_t src_stride, int dim,
                                                            int dim_pad, int metric, int bf16_only, int write32,
                                                            float* __restrict__ x32, __nv_bfloat16* __restrict__ x16,
                                                            double* __restrict__ norm64, float* __restrict__ sa,
                                                            float* __restrict__ sb, int8_t* __restrict__ x8,
                                                            float* __restrict__ sa8, StoreScalars* scal,
                                                            int64_t first_row, int64_t n) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n) return;
  const int64_t row = first_row + r;
  const float* s = src + r * src_stride;
  double n2 = 0.0, e2 = 0.0;
  float amax = 0.f;
  for (int j = lane * 4; j < dim_pad; j += 128) {
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      v[e] = (j + e < dim) ? s[j + e] : 0.f;
      amax = fmaxf(amax, fabsf(v[e]));
    }
    __nv_bfloat16 b[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      b[e] = __float2bfloat16_rn(v[e]);
      float back = __bfloat162float(b[e]);
      if (bf16_only) {
        n2 = fma((double)back, (double)back, n2);
      } else {
        n2 = fma((double)v[e], (double)v[e], n2);
        double d = (double)v[e] - (double)back;
        e2 = fma(d, d, e2);
      }
    }
    uint2 packed;
    packed.x = (uint32_t)__bfloat16_as_ushort(b[0]) | ((uint32_t)__bfloat16_as_ushort(b[1]) << 16);
    packed.y = (uint32_t)__bfloat16_as_ushort(b[2]) | ((uint32_t)__bfloat16_as_ushort(b[3]) << 16);
    *reinterpret_cast<uint2*>(x16 + (size_t)row * dim_pad + j) = packed;
    if (write32) *reinterpret_cast<float4*>(x32 + (size_t)row * dim_pad + j) = make_float4(v[0], v[1], v[2], v[3]);
  }
  n2 = warp_sum(n2);
  e2 = warp_sum(e2);
  if (lane == 0) {
    double nrm = sqrt(n2);
    norm64[row] = nrm;
    if (metric == RASS_METRIC_COSINE) {
      sa[row] = nrm > 0.0 ? (float)(1.0 / nrm) : 0.f;
      sb[row] = 0.f;
    } else {
      sa[row] = 1.f;
      sb[row] = (float)(-0.5 * n2);
    }
    // round the ratios up so the bound stays a bound after the float conversion
    float rho = nrm > 0.0 ? __double2float_ru(sqrt(e2) / nrm) : 0.f;
    atomicMax(reinterpret_cast<int*>(&scal->rho_x), __float_as_int(rho));
    atomicMax(reinterpret_cast<int*>(&scal->max_xnorm), __float_as_int(__double2float_ru(nrm)));
  }
  if (!x8) return;
  // int8 shadow: x ~ s_x x8 with s_x = max|x| / 127 (a zero row: scale 0, codes 0); its residual in fp64
  const float s_x = warp_max_nonneg(amax) / 127.f;
  double e8 = 0.0;
  for (int j = lane * 4; j < dim_pad; j += 128) {
    uint32_t packed = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float v = (j + e < dim) ? s[j + e] : 0.f;
      const float c = int8_code(v, s_x);
      const double d = (double)v - (double)s_x * (double)c;
      e8 = fma(d, d, e8);
      packed |= (uint32_t)(uint8_t)(int8_t)c << (8 * e);
    }
    *reinterpret_cast<uint32_t*>(x8 + (size_t)row * dim_pad + j) = packed;
  }
  e8 = warp_sum(e8);
  if (lane == 0) {
    const double nrm = sqrt(n2);
    sa8[row] = metric == RASS_METRIC_COSINE ? (nrm > 0.0 ? (float)((double)s_x / nrm) : 0.f) : s_x;
    const float rho = nrm > 0.0 ? __double2float_ru(sqrt(e8) / nrm) : 0.f;
    atomicMax(reinterpret_cast<int*>(&scal->rho_x8), __float_as_int(rho));
  }
}

int launch_store_convert(rass_engine* h, const float* src_dev, int64_t src_stride, int64_t first_row, int64_t n,
                         cudaStream_t st) {
  if (n <= 0) return RASS_OK;
  h->sb_filtered_dirty = true;
  h->store_scal_stale = true;
  const bool bf16_only = (h->flags & RASS_BF16_ONLY) != 0;
  const bool in_place = !bf16_only && src_dev == h->x32 + (size_t)first_row * h->dim_pad;
  const int warps = 8;
  int64_t blocks = (n + warps - 1) / warps;
  store_convert_kernel<<<(unsigned)blocks, warps * 32, 0, st>>>(src_dev, src_stride, h->dim, h->dim_pad, h->metric,
                                                                bf16_only ? 1 : 0, (!bf16_only && !in_place) ? 1 : 0,
                                                                h->x32, h->x16, h->norm64, h->sa, h->sb, h->x8, h->sa8,
                                                                h->store_scal, first_row, n);
  CUDA_TRY(h, cudaGetLastError());
  return RASS_OK;
}

// one warp per query slot; slots >= B (up to the 256-multiple the tcgen05 passes read) are zeroed
__global__ void __launch_bounds__(128) query_prep_kernel(const float* __restrict__ q, int dim, int dim_pad, int metric,
                                                         int B, int B_pad, float* __restrict__ q_raw,
                                                         float* __restrict__ q_hat, __nv_bfloat16* __restrict__ q16,
                                                         double* __restrict__ q_norm, float* __restrict__ q_rho,
                                                         int8_t* __restrict__ q8, float* __restrict__ q8_scale,
                                                         float* __restrict__ q_rho8, SearchScalars* __restrict__ scal) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (blockIdx.x == 0 && threadIdx.x == 0) {      // the per-search counters
    scal->flagged_n = 0;
    scal->max_cand = 0;
    scal->n_certified = 0;
    // (every scan_umma_kernel launch leaves its tile counter at zero; a search starts from zero whatever happened before)
    scal->tile_ctr[0] = 0;
    scal->tile_ctr[1] = 0;
  }
  if (b >= B_pad) return;
  // rows of the query's two int8 parts: group b / 64 holds 128 rows, part 1 then part 2
  const size_t r1 = (size_t)(b / RASS_GROUP_Q) * (2 * RASS_GROUP_Q) + (b % RASS_GROUP_Q), r2 = r1 + RASS_GROUP_Q;
  if (b >= B) {
    for (int j = lane; j < dim_pad; j += 32) q16[(size_t)b * dim_pad + j] = __float2bfloat16_rn(0.f);
    if (q8) {
      for (int j = lane; j < dim_pad; j += 32) { q8[r1 * dim_pad + j] = 0; q8[r2 * dim_pad + j] = 0; }
      if (lane < 2) q8_scale[2 * b + lane] = 0.f;
    }
    return;
  }
  const float* s = q + (size_t)b * dim;
  double n2 = 0.0;
  for (int j = lane; j < dim; j += 32) n2 = fma((double)s[j], (double)s[j], n2);
  n2 = warp_sum(n2);
  const double nrm = sqrt(n2);
  const double inv = (metric == RASS_METRIC_COSINE) ? (nrm > 0.0 ? 1.0 / nrm : 0.0) : 1.0;
  double h2 = 0.0, e2 = 0.0;
  float amax = 0.f;
  for (int j = lane; j < dim_pad; j += 32) {
    float v = j < dim ? s[j] : 0.f;
    float hat = (float)((double)v * inv);
    amax = fmaxf(amax, fabsf(hat));
    __nv_bfloat16 hb = __float2bfloat16_rn(hat);
    double d = (double)hat - (double)__bfloat162float(hb);
    h2 = fma((double)hat, (double)hat, h2);
    e2 = fma(d, d, e2);
    q_raw[(size_t)b * dim_pad + j] = v;
    q_hat[(size_t)b * dim_pad + j] = hat;
    q16[(size_t)b * dim_pad + j] = hb;
  }
  h2 = warp_sum(h2);
  e2 = warp_sum(e2);
  if (lane == 0) {
    q_norm[b] = nrm;
    q_rho[b] = h2 > 0.0 ? __double2float_ru(sqrt(e2 / h2)) : 0.f;
  }
  if (!q8) return;
  // two int8 parts: q_hat ~ s1 q1 + s2 q2, q2 the code of the residual of the first part (one part alone would leave
  // rho_q ~ 0.01, as large as the rows' own residual; two leave ~ 4e-5).  The residual is measured in fp64.
  // (each lane reads back the q_hat / q8 entries it wrote itself)
  const float s1 = warp_max_nonneg(amax) / 127.f;
  float rmax = 0.f;
  for (int j = lane; j < dim_pad; j += 32) {
    const float hat = q_hat[(size_t)b * dim_pad + j];
    const float c1 = int8_code(hat, s1);
    rmax = fmaxf(rmax, fabsf(fmaf(-s1, c1, hat)));
    q8[r1 * dim_pad + j] = (int8_t)c1;
  }
  const float s2 = warp_max_nonneg(rmax) / 127.f;
  double e8 = 0.0;
  for (int j = lane; j < dim_pad; j += 32) {
    const float hat = q_hat[(size_t)b * dim_pad + j];
    const float c1 = (float)q8[r1 * dim_pad + j];
    const float c2 = int8_code(fmaf(-s1, c1, hat), s2);
    q8[r2 * dim_pad + j] = (int8_t)c2;
    const double d = (double)hat - ((double)s1 * (double)c1 + (double)s2 * (double)c2);
    e8 = fma(d, d, e8);
  }
  e8 = warp_sum(e8);
  if (lane == 0) {
    q8_scale[2 * b] = s1;
    q8_scale[2 * b + 1] = s2;
    q_rho8[b] = h2 > 0.0 ? __double2float_ru(sqrt(e8 / h2)) : 0.f;
  }
}

int launch_query_prep(rass_engine* h, const SearchWs& ws, const float* q_dev, int B, cudaStream_t st) {
  const int B_pad = (B + RASS_QPAD - 1) / RASS_QPAD * RASS_QPAD;
  const int warps = 4;
  query_prep_kernel<<<(B_pad + warps - 1) / warps, warps * 32, 0, st>>>(q_dev, h->dim, h->dim_pad, h->metric, B, B_pad,
                                                                        ws.q_raw, ws.q_hat, ws.q16, ws.q_norm,
                                                                        ws.q_rho, ws.q8, ws.q8_scale, ws.q_rho8,
                                                                        ws.scal);
  CUDA_TRY(h, cudaGetLastError());
  return RASS_OK;
}

// ---------------------------------------------------------------------------------------------
// Threshold seed for the tcgen05 scans.
//
// A scan CTA starts with threshold -inf, so every score of its first two tiles is a "hit": measured on the 64-query
// kernel, tile 0 takes 13.6 us and tile 1 (64 first compactions) 45.7 us against 5.5 us in steady state -- a fixed
// 36-48 us per pass (profiles/r1_scan_kernels_ncu.md).  One CTA pair per query scores RASS_SEED_ROWS corpus rows (16 evenly
// spaced runs of 32) with the arithmetic the scan uses (bf16 operands, fp32 accumulate, key = dot * sa + sb_scan) and publishes in
// q_gthr the largest T with at least `rank` sampled keys strictly above it.  T is a legal pivot: those rows are part of
// the corpus, so the scan meets at least `rank` >= (entries a compaction keeps) keys above it -- the same guarantee a
// pivot found by warp_compact carries -- and every scan CTA starts from it.  The accumulation order differs from the
// tensor pipe's, so a sampled key within an ulp of T can land on the other side; `rank` leaves 8 (16) spare rows over
// what the certificate needs, and the certificate in finish.cu is what guarantees exactness in any case.
// The int8 form (I8) scores the sample from x8 and the query's two int8 parts: the integer dots are exact in any order
// and int8_key is the epilogue's own expression, so its keys are bit-identical to the pass's.
// ---------------------------------------------------------------------------------------------
#define RASS_SEED_ROWS 512
#define RASS_SEED_BLOCKS (RASS_SEED_ROWS / 32)
#define RASS_SEED_THREADS 512

// A CTA pair (cluster of 2) per query: reading the 1 MB sample through one SM's L2 port takes ~9 us, so each CTA scores
// half of it and the second one hands its keys over through distributed shared memory.  NVEC = dim_pad / 256 when it is
// known at compile time (all 16-byte loads of four rows are then issued before the first use), 0 = run-time loop.
// I8: x = x8, q = q8 (the 128-row group layout of query_prep_kernel), sa = sa8; a lane loads 8 bytes per 16 of bf16.
template <int NVEC, bool I8>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(RASS_SEED_THREADS, 1) seed_thresholds_kernel(
    const void* __restrict__ x, const float* __restrict__ sa, const float* __restrict__ sb,
    const void* __restrict__ q, const float* __restrict__ q8_scale, int dim_pad, int64_t n_rows, int B, int rank,
    uint32_t* __restrict__ gthr, float* __restrict__ pool_thr, int* __restrict__ pool_cnt, size_t n_clear) {
  namespace cg = cooperative_groups;
  // the segment bounds and sizes of the pass that follows start empty (saves the scans' own clearing launch)
  for (size_t i = (size_t)blockIdx.x * RASS_SEED_THREADS + threadIdx.x; i < n_clear;
       i += (size_t)gridDim.x * RASS_SEED_THREADS) {
    pool_thr[i] = neg_inf<float>();
    pool_cnt[i] = 0;
  }
  const int b = blockIdx.x >> 1;                 // uniform over the pair: both CTAs leave here, or neither
  if (b >= B) {
    if (threadIdx.x == 0 && (blockIdx.x & 1) == 0) gthr[b] = 0u;
    return;
  }
  cg::cluster_group pair = cg::this_cluster();
  const int half = (int)pair.block_rank();
  extern __shared__ float seed_smem[];
  float* qs = seed_smem;                                             // [dim_pad] the bf16 query, widened (I8: q1, q2)
  uint32_t* keys = reinterpret_cast<uint32_t*>(seed_smem + dim_pad);  // [RASS_SEED_ROWS] ordered images (CTA 0's copy is used)
  uint32_t* keys0 = pair.map_shared_rank(keys, 0);
  uint2* q1s = reinterpret_cast<uint2*>(seed_smem);
  uint2* q2s = q1s + (dim_pad >> 3);
  float s1 = 0.f, s2 = 0.f;
  if (I8) {
    const size_t r1 = (size_t)(b / RASS_GROUP_Q) * (2 * RASS_GROUP_Q) + (b % RASS_GROUP_Q);
    const uint2* q1 = reinterpret_cast<const uint2*>(static_cast<const int8_t*>(q) + r1 * dim_pad);
    const uint2* q2 = reinterpret_cast<const uint2*>(static_cast<const int8_t*>(q) + (r1 + RASS_GROUP_Q) * dim_pad);
    for (int j = threadIdx.x; j < (dim_pad >> 3); j += RASS_SEED_THREADS) { q1s[j] = q1[j]; q2s[j] = q2[j]; }
    s1 = q8_scale[2 * b];
    s2 = q8_scale[2 * b + 1];
  } else {
    const __nv_bfloat16* q16 = static_cast<const __nv_bfloat16*>(q);
    for (int j = threadIdx.x; j < dim_pad; j += RASS_SEED_THREADS) qs[j] = __bfloat162float(q16[(size_t)b * dim_pad + j]);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nvec = NVEC ? NVEC : (dim_pad >> 8);                     // 16-byte (I8: 8-byte) loads per lane per row
  // the sample: RASS_SEED_BLOCKS evenly spaced runs of 32 consecutive rows (few distinct pages: 512 scattered rows cost
  // a TLB miss each)
  const int64_t block_stride = n_rows / RASS_SEED_BLOCKS;
  constexpr int ROWS_PER_WARP = RASS_SEED_ROWS / 2 / (RASS_SEED_THREADS / 32);
  static_assert(ROWS_PER_WARP % 4 == 0 && 32 % ROWS_PER_WARP == 0, "a warp scores its rows four at a time, inside one run");
  for (int i0 = 0; i0 < ROWS_PER_WARP; i0 += 4) {
    const int i = half * (RASS_SEED_ROWS / 2) + warp * ROWS_PER_WARP + i0;   // sample index of the first of four rows
    const int64_t row0 = (int64_t)(i >> 5) * block_stride + (i & 31);
    float a = 0.f, off = 0.f;
    if (lane < 4) { a = __ldg(sa + row0 + lane); off = __ldg(sb + row0 + lane); }
    if (I8) {
      int acc1[4] = {0, 0, 0, 0}, acc2[4] = {0, 0, 0, 0};
      auto dp_block = [&](const uint2 (&xv)[4], int v) {
        const uint2 w1 = q1s[v * 32 + lane], w2 = q2s[v * 32 + lane];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          acc1[r] = __dp4a((int)xv[r].x, (int)w1.x, acc1[r]);
          acc1[r] = __dp4a((int)xv[r].y, (int)w1.y, acc1[r]);
          acc2[r] = __dp4a((int)xv[r].x, (int)w2.x, acc2[r]);
          acc2[r] = __dp4a((int)xv[r].y, (int)w2.y, acc2[r]);
        }
      };
      const uint2* p = static_cast<const uint2*>(x) + (size_t)row0 * (dim_pad >> 3) + lane;
      if (NVEC) {
        // all loads before the first use, pinned in order as in the bf16 form below
        uint2 xv[NVEC ? NVEC : 1][4];
#pragma unroll
        for (int v = 0; v < NVEC; ++v)
#pragma unroll
          for (int r = 0; r < 4; ++r)
            asm volatile("ld.global.nc.v2.u32 {%0, %1}, [%2];"
                         : "=r"(xv[v][r].x), "=r"(xv[v][r].y)
                         : "l"(p + (size_t)r * (dim_pad >> 3) + v * 32));
#pragma unroll
        for (int v = 0; v < NVEC; ++v)
#pragma unroll
          for (int r = 0; r < 4; ++r) asm volatile("" : "+r"(xv[v][r].x), "+r"(xv[v][r].y));
#pragma unroll
        for (int v = 0; v < NVEC; ++v) dp_block(xv[v], v);
      } else {
        for (int v = 0; v < nvec; ++v) {
          uint2 xv[4];
#pragma unroll
          for (int r = 0; r < 4; ++r) xv[r] = __ldg(p + (size_t)r * (dim_pad >> 3) + v * 32);
          dp_block(xv, v);
        }
      }
      int m1 = 0, m2 = 0;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int d1 = __reduce_add_sync(0xffffffffu, acc1[r]), d2 = __reduce_add_sync(0xffffffffu, acc2[r]);
        if (lane == r) { m1 = d1; m2 = d2; }
      }
      if (lane < 4) keys0[i + lane] = ord32(int8_key(m1, m2, s1, s2, a, off));
      continue;
    }
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    auto fma_block = [&](const uint4 (&x)[4], int v) {
      const float4 qa = *reinterpret_cast<const float4*>(qs + (v * 32 + lane) * 8);
      const float4 qb = *reinterpret_cast<const float4*>(qs + (v * 32 + lane) * 8 + 4);
      const float qv[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const uint32_t w[4] = {x[r].x, x[r].y, x[r].z, x[r].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          acc[r] = fmaf(__uint_as_float(w[e] << 16), qv[2 * e], acc[r]);
          acc[r] = fmaf(__uint_as_float(w[e] & 0xffff0000u), qv[2 * e + 1], acc[r]);
        }
      }
    };
    const uint4* p = static_cast<const uint4*>(x) + (size_t)row0 * (dim_pad >> 3) + lane;
    if (NVEC) {
      // all 4 * NVEC loads are issued before the first use: the volatile loads keep their order, and the empty
      // volatile statements after them pin every loaded register, so no FMA can be scheduled in between (left to
      // itself the compiler interleaves them, two loads in flight per warp, and the kernel is a chain of round trips)
      uint4 x[NVEC ? NVEC : 1][4];
#pragma unroll
      for (int v = 0; v < NVEC; ++v)
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const uint4* src = p + (size_t)r * (dim_pad >> 3) + v * 32;
          asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];"
                       : "=r"(x[v][r].x), "=r"(x[v][r].y), "=r"(x[v][r].z), "=r"(x[v][r].w)
                       : "l"(src));
        }
#pragma unroll
      for (int v = 0; v < NVEC; ++v)
#pragma unroll
        for (int r = 0; r < 4; ++r)
          asm volatile("" : "+r"(x[v][r].x), "+r"(x[v][r].y), "+r"(x[v][r].z), "+r"(x[v][r].w));
#pragma unroll
      for (int v = 0; v < NVEC; ++v) fma_block(x[v], v);
    } else {
      for (int v = 0; v < nvec; ++v) {
        uint4 x[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) x[r] = __ldg(p + (size_t)r * (dim_pad >> 3) + v * 32);
        fma_block(x, v);
      }
    }
    float mine = 0.f;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      float dot = acc[r];
#pragma unroll
      for (int m = 16; m >= 1; m >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, m);
      if (lane == r) mine = dot;
    }
    if (lane < 4) keys0[i + lane] = ord32(fmaf(mine, a, off));
  }
  pair.sync();                                   // both halves of the keys are in CTA 0's shared memory
  if (half == 0 && warp == 0) {
    uint32_t kk[RASS_SEED_ROWS / 32];
#pragma unroll
    for (int i = 0; i < RASS_SEED_ROWS / 32; ++i) kk[i] = keys[i * 32 + lane];
    // v = the rank-th largest key: the largest value with at least `rank` keys >= it
    uint32_t v = 0;
    for (int bit = 31; bit >= 0; --bit) {
      const uint32_t cand = v | (1u << bit);
      int c = 0;
#pragma unroll
      for (int i = 0; i < RASS_SEED_ROWS / 32; ++i) c += kk[i] >= cand;
      c = __reduce_add_sync(0xffffffffu, c);
      if (c >= rank) v = cand;
    }
    // strictly above v - 1 = at or above v; nothing is published unless `rank` sampled keys are finite (> -inf)
    const uint32_t t = v ? v - 1 : 0u;
    if (lane == 0) gthr[b] = t > 0x007fffffu ? t : 0u;
  }
}

// Initialises q_gthr[0, B_pad) for the scans that follow: a seed per query, or 0 ("nothing published") when the corpus
// is too small to sample or RASS_DEBUG_NO_SEED is set (the A/B switch of the measurement).  When the kernel runs it
// also empties the first n_clear segment bounds / sizes of the candidate pool (*cleared = true).  seg = the segment size the
// scan will use: its compactions keep >= 32 (seg 256) or >= 128 (seg 512) entries above a pivot, and so must the seed.
int launch_seed_thresholds(rass_engine* h, const SearchWs& ws, int B, int seg, size_t n_clear, bool* cleared,
                           cudaStream_t st, bool int8) {
  *cleared = false;
  static const bool no_seed = getenv("RASS_DEBUG_NO_SEED") != nullptr;
  const int B_pad = (B + RASS_QPAD - 1) / RASS_QPAD * RASS_QPAD;
  const int rank = seg == 512 ? 144 : 40;
  if (no_seed || h->n_rows < 16 * RASS_SEED_ROWS) {
    CUDA_TRY(h, cudaMemsetAsync(ws.q_gthr, 0, (size_t)B_pad * sizeof(uint32_t), st));
    return RASS_OK;
  }
  const size_t smem = (size_t)h->dim_pad * sizeof(float) + RASS_SEED_ROWS * sizeof(uint32_t);
  const void* x = int8 ? (const void*)h->x8 : (const void*)h->x16;
  const void* q = int8 ? (const void*)ws.q8 : (const void*)ws.q16;
  const float* sa = int8 ? h->sa8 : h->sa;
#define RASS_SEED_LAUNCH(NV, I8)                                                                                      \
  do {                                                                                                              \
    if (smem > 48 * 1024)                                                                                           \
      CUDA_TRY(h, cudaFuncSetAttribute(seed_thresholds_kernel<NV, I8>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                       (int)smem));                                                                 \
    seed_thresholds_kernel<NV, I8><<<2 * B_pad, RASS_SEED_THREADS, smem, st>>>(                                     \
        x, sa, h->sb_scan, q, ws.q8_scale, h->dim_pad, h->n_rows, B, rank, ws.q_gthr, ws.pool_thr, ws.pool_cnt,     \
        n_clear);                                                                                                   \
  } while (0)
  if (h->dim_pad == 1024) {
    if (int8) RASS_SEED_LAUNCH(4, true); else RASS_SEED_LAUNCH(4, false);
  } else {
    if (int8) RASS_SEED_LAUNCH(0, true); else RASS_SEED_LAUNCH(0, false);
  }
#undef RASS_SEED_LAUNCH
  CUDA_TRY(h, cudaGetLastError());
  *cleared = true;
  return RASS_OK;
}
