// Small-batch kNN scan: a coalesced, 128-bit vectorised streaming GEMV over the bf16 shadow matrix fused with a
// per-warp register top-32 select, so no score vector ever reaches HBM.
//
// Replaces the `knn` clause executor (reference app/main.py:1538-1542 -> OpenSearch k-NN plugin / nmslib HNSW)
// for 1 or 2 queries per corpus pass.  HBM-bound: the algorithmic traffic is n_rows * dim_pad * 2 bytes per pass.
//
// Work split: warp w of W owns row groups g = w, w + W, ... (a group = R consecutive rows, R * NQ = 4), which
// interleaves neighbouring rows over the lists.  Each lane holds its 8-element slices of the query in
// registers, issues all R * VEC 16-byte loads of a group before using them, and the 4 partial dot products
// of a group are reduced with one transposing butterfly (6 shuffles).  At the end of the pass the 8 warp lists of
// a CTA are merged to one segment of 32..64 entries per query (296 segments instead of 2368 for finish.cu to
// read).  Every row a warp dropped has a score <= the final threshold of that warp's list and every entry the
// merge dropped is <= its pivot; the maximum of the two is the bound the certificate in finish.cu relies on.
#include "common.cuh"

template <int NQ, int VEC>
__global__ void __launch_bounds__(RASS_WARPS_PER_CTA * 32, 2)
    scan_stream_kernel(const uint4* __restrict__ x16, const float* __restrict__ sa, const float* __restrict__ sb,
                       const float* __restrict__ q_hat, int64_t n_rows, float* __restrict__ pool_key,
                       uint32_t* __restrict__ pool_row, float* __restrict__ pool_thr, int* __restrict__ pool_cnt,
                       int slot0, int n_segs, size_t pool_entries) {
  constexpr int R = 4 / NQ;             // rows per group
  constexpr int ROW_U4 = VEC * 32;      // uint4 per row
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int gw = blockIdx.x * RASS_WARPS_PER_CTA + warp;
  const int W = gridDim.x * RASS_WARPS_PER_CTA;

  float q[NQ][VEC][8];
#pragma unroll
  for (int qi = 0; qi < NQ; ++qi)
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const float4* p = reinterpret_cast<const float4*>(q_hat + (size_t)qi * (VEC * 256) + (j * 32 + lane) * 8);
      float4 a = p[0], b = p[1];
      q[qi][j][0] = a.x; q[qi][j][1] = a.y; q[qi][j][2] = a.z; q[qi][j][3] = a.w;
      q[qi][j][4] = b.x; q[qi][j][5] = b.y; q[qi][j][6] = b.z; q[qi][j][7] = b.w;
    }

  WarpTop<float, 1> top[NQ];
#pragma unroll
  for (int qi = 0; qi < NQ; ++qi) top[qi].init();

  const int64_t n_groups = (n_rows + R - 1) / R;
  const int vi = lane >> 3;             // which of the 4 reduced values this lane ends up holding
  const int my_r = vi / NQ, my_q = vi % NQ;

  for (int64_t g = gw; g < n_groups; g += W) {
    const int64_t row0 = g * R;
    uint4 v[R][VEC];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      int64_t row = row0 + r;
      if (row >= n_rows) row = n_rows - 1;  // clamped rows are masked below
      const uint4* p = x16 + (size_t)row * ROW_U4 + lane;
#pragma unroll
      for (int j = 0; j < VEC; ++j) v[r][j] = ldg_stream(p + j * 32);
    }
    float acc[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[i] = 0.f;
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const uint32_t w[4] = {v[r][j].x, v[r][j].y, v[r][j].z, v[r][j].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float lo = bf16lo(w[e]), hi = bf16hi(w[e]);
#pragma unroll
          for (int qi = 0; qi < NQ; ++qi) {
            acc[r * NQ + qi] = fmaf(lo, q[qi][j][2 * e], acc[r * NQ + qi]);
            acc[r * NQ + qi] = fmaf(hi, q[qi][j][2 * e + 1], acc[r * NQ + qi]);
          }
        }
      }
    // transposing butterfly: afterwards lanes [8*i, 8*i+8) hold the full sum of value i
    const bool b4 = lane & 16, b3 = lane & 8;
    float a0 = b4 ? acc[2] : acc[0], s0 = b4 ? acc[0] : acc[2];
    float a1 = b4 ? acc[3] : acc[1], s1 = b4 ? acc[1] : acc[3];
    a0 += __shfl_xor_sync(0xffffffffu, s0, 16);
    a1 += __shfl_xor_sync(0xffffffffu, s1, 16);
    float c = b3 ? a1 : a0, d = b3 ? a0 : a1;
    c += __shfl_xor_sync(0xffffffffu, d, 8);
    c += __shfl_xor_sync(0xffffffffu, c, 4);
    c += __shfl_xor_sync(0xffffffffu, c, 2);
    c += __shfl_xor_sync(0xffffffffu, c, 1);

    const int64_t my_row = row0 + my_r;
    float score = neg_inf<float>();
    if (my_row < n_rows) score = fmaf(c, __ldg(sa + my_row), __ldg(sb + my_row));
    float my_thr = top[0].thr_key;
#pragma unroll
    for (int qi = 1; qi < NQ; ++qi)
      if (my_q == qi) my_thr = top[qi].thr_key;
    const unsigned hit = __ballot_sync(0xffffffffu, score > my_thr);
    if (hit) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (hit & (1u << (i * 8))) {
          const float s = __shfl_sync(0xffffffffu, score, i * 8);
          top[i % NQ].insert(s, (uint32_t)(row0 + i / NQ));
        }
      }
    }
  }

  // CTA-level merge: the 8 warp lists of a query (256 entries) are compacted to the best 32..64 by warp qi.
  // The segment bound covers what the merge drops (<= pivot) and what every warp dropped (<= its threshold).
  __shared__ float s_key[NQ][RASS_WARPS_PER_CTA * 32];
  __shared__ uint32_t s_row[NQ][RASS_WARPS_PER_CTA * 32];
  __shared__ float s_thr[NQ][RASS_WARPS_PER_CTA];
#pragma unroll
  for (int qi = 0; qi < NQ; ++qi) {
    s_key[qi][warp * 32 + lane] = top[qi].key[0];
    s_row[qi][warp * 32 + lane] = top[qi].row[0];
    if (lane == 0) s_thr[qi][warp] = top[qi].thr_key;
  }
  __syncthreads();
  if (warp < NQ) {
    const int qi = warp;
    uint32_t ok[RASS_WARPS_PER_CTA], rw[RASS_WARPS_PER_CTA];
#pragma unroll
    for (int i = 0; i < RASS_WARPS_PER_CTA; ++i) {
      rw[i] = s_row[qi][i * 32 + lane];
      ok[i] = rw[i] != 0xffffffffu ? ord32(s_key[qi][i * 32 + lane]) : 0u;
    }
    const size_t base = (size_t)(slot0 + qi) * pool_entries + (size_t)blockIdx.x * RASS_STREAM_SEG;
    uint32_t pivot;
    const int kept = warp_compact<RASS_WARPS_PER_CTA>(ok, rw, RASS_STREAM_SEG / 2, pool_key + base, pool_row + base, pivot);
    if (lane == 0) {
      float bound = unord32(pivot);   // -inf when the merge dropped nothing
#pragma unroll
      for (int w = 0; w < RASS_WARPS_PER_CTA; ++w) bound = fmaxf(bound, s_thr[qi][w]);
      pool_thr[(size_t)(slot0 + qi) * n_segs + blockIdx.x] = bound;
      pool_cnt[(size_t)(slot0 + qi) * n_segs + blockIdx.x] = kept;
    }
  }
}

static int stream_ctas(const rass_engine* h) { return h->num_sms * 2; }

int scan_stream_segs(const rass_engine* h) { return stream_ctas(h); }

template <int NQ>
static int launch_vec(rass_engine* h, const SearchWs& ws, int q0, int slot0, cudaStream_t st) {
  const int grid = stream_ctas(h);
  const int n_segs = scan_stream_segs(h);
  const uint4* x = reinterpret_cast<const uint4*>(h->x16);
  const float* qh = ws.q_hat + (size_t)q0 * h->dim_pad;
#define RASS_LAUNCH(V)                                                                                          \
  scan_stream_kernel<NQ, V><<<grid, RASS_WARPS_PER_CTA * 32, 0, st>>>(x, h->sa, h->sb_scan, qh, h->n_rows, ws.pool_key, \
                                                                      ws.pool_row, ws.pool_thr, ws.pool_cnt, slot0, \
                                                                      n_segs, ws.pool_entries)
  switch (h->dim_pad / 256) {
    case 1: RASS_LAUNCH(1); break;
    case 2: RASS_LAUNCH(2); break;
    case 3: RASS_LAUNCH(3); break;
    case 4: RASS_LAUNCH(4); break;
    default: return rass_fail(h, RASS_E_INVALID, "dim_pad %d unsupported by the streaming scan", h->dim_pad);
  }
#undef RASS_LAUNCH
  CUDA_TRY(h, cudaGetLastError());
  return RASS_OK;
}

int launch_scan_stream(rass_engine* h, const SearchWs& ws, int q0, int nq, int g0, cudaStream_t st) {
  if (nq == 1) return launch_vec<1>(h, ws, q0, q0 - g0, st);
  if (nq == 2) return launch_vec<2>(h, ws, q0, q0 - g0, st);
  return rass_fail(h, RASS_E_INVALID, "streaming scan takes 1 or 2 queries per pass");
}
