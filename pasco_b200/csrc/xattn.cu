// Masked cross-attention of a handful of queries (≤128) over ALL voxels of a scale, sm_100a (tcgen05 + TMEM).
//
//   O[q, h, :] = Σ_v softmax_v( Q[q,h,:]·K[v,h,:]·scale + mask[q,v] ) · V[v,h,:]
//
// (pasco/models/transformer/blocks.py:73-92 with the attention mask of transformer_predictor_v2.py:220-289: 100 queries,
// 8 heads of width 48, P = 25 k … 400 k keys.)  Q is tiny and P huge, so the kernel streams K and V once per pass
// through shared memory and keeps the query operand resident; FLOPs are negligible, the roofline is HBM:
// 2 passes x P x H x D x 4 B (K twice, V once).
//
// Two passes share one kernel template (no online-softmax rescaling of the TMEM accumulator is needed):
//   PASS 0  S = Q_h·K_hᵀ per 64-key tile (tcgen05, M=128 queries, N=64 keys, K=64 padded head dim) → per (chunk, h, q)
//           running max m and Σ exp(s − m); `k_xattn_lse` merges the chunks into lse[h, q].
//   PASS 1  S again, p = exp(s − lse) (already normalised), P → bf16 (hi+lo) K-major smem tile, O_h += P·V_h (tcgen05,
//           V tile as MN-major B operand), accumulated in TMEM over all tiles of the CTA, then stored as the chunk's
//           partial O in the workspace; the chunks are added into O in chunk order (k_add_partials).
// A CTA = (head, key chunk); warps 0-3: one query row per thread (TMEM lane = row; mask, exp, row statistics),
// warps 4-7: K/V tile gather (16 lanes per 256-byte padded row segment, fp32 → bf16 hi/lo split, 128-byte swizzle),
// warp 8: single-thread MMA issue.  Operands are split bf16x3 like the convolution ("fp32" mode).
#include <math_constants.h>
#include "common.cuh"
#include "umma.cuh"

using namespace pasco;
using namespace umma;

namespace {

constexpr int BK = 64;                      // keys per tile
constexpr int QM = 128;                     // query rows (padded) = UMMA M
constexpr int DP = 64;                      // padded head dim = one 128-byte swizzle row of bf16
constexpr int TILE_Q = QM * 128;            // 16 KB: [128 rows][64] bf16
constexpr int TILE_K = BK * 128;            // 8 KB : [64 keys][64] bf16
constexpr int NTHREADS = 9 * 32;
constexpr int MMA_WARP = 8;

struct XParams {
  const float* q;      // [Q, H*D]
  const float* k;      // [P, H*D]
  const float* v;      // [P, H*D]
  const uint32_t* mask; // bit rows [Q, 2*ceil(P/64)]: bit j of word 2t + j/32 = key 64t + j masked; nullptr = none
  const float* lse;    // [H, Q]            (pass 1)
  float* out;          // [Q, H*D] zeroed   (pass 1)
  float* ws;           // [chunks, H, Q, 2] (pass 0), then [chunks, Q, H*D] per-chunk outputs (pass 1)
  int Q, H, D;
  int64_t P;
  int chunks;
  float scale;
};

// smem layout (bytes from a 1024-aligned base)
//   Q_hi | Q_lo                        2 x 16 KB
//   stage s (x2): K_hi | K_lo | V_hi | V_lo     4 x 8 KB
//   P_hi[2 k-blocks? no: 64 keys = 1 block] | P_lo   2 x 16 KB   (pass 1)
constexpr int OFF_Q = 0;
constexpr int OFF_KV = 2 * TILE_Q;
constexpr int KV_STAGE = 4 * TILE_K;
constexpr int OFF_P = OFF_KV + 2 * KV_STAGE;
constexpr int OFF_BAR = OFF_P + 2 * TILE_Q;
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;

__device__ __forceinline__ uint32_t sw_off(uint32_t row, uint32_t chunk16) { return row * 128u + ((chunk16 ^ (row & 7u)) << 4); }

template <int PASS>
__global__ void __launch_bounds__(NTHREADS, 1) k_xattn_fwd(const __grid_constant__ XParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* kv_full = bars;        // [2]
  uint64_t* kv_empty = bars + 2;   // [2]
  uint64_t* s_full = bars + 4;     // [2]
  uint64_t* s_empty = bars + 6;    // [2]
  uint64_t* p_full = bars + 8;     // [1]
  uint64_t* p_empty = bars + 9;    // [1]
  uint64_t* o_full = bars + 10;    // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.x % p.H;
  const int chunk = blockIdx.x / p.H;
  const int64_t n_tiles = (p.P + BK - 1) / BK;
  const int64_t tiles_per_chunk = (n_tiles + p.chunks - 1) / p.chunks;
  const int64_t t0 = (int64_t)chunk * tiles_per_chunk;
  const int64_t t1 = t0 + tiles_per_chunk < n_tiles ? t0 + tiles_per_chunk : n_tiles;
  const int64_t my_tiles = t1 > t0 ? t1 - t0 : 0;
  const int HD = p.H * p.D;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(kv_full + i), 4);
      mbar_init(smem_u32(kv_empty + i), 1);
      mbar_init(smem_u32(s_full + i), 1);
      mbar_init(smem_u32(s_empty + i), 4);
    }
    mbar_init(smem_u32(p_full), 4);
    mbar_init(smem_u32(p_empty), 1);
    mbar_init(smem_u32(o_full), 1);
    fence_barrier_init();
  }
  if (warp == MMA_WARP) tmem_alloc(smem_u32(tmem_slot), 256);
  // ---- resident query operand: Q_h * scale → bf16 hi/lo, rows >= Q and columns >= D are zero ----
  for (int t = threadIdx.x; t < QM * 8; t += NTHREADS) {       // one 16-byte output chunk (8 bf16) per iteration
    const int row = t >> 3, c = t & 7;
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int d = c * 8 + j;
      f[j] = (row < p.Q && d < p.D) ? __ldg(p.q + (int64_t)row * HD + h * p.D + d) * p.scale : 0.f;
    }
    uint2 h0, l0, h1, l1;
    split4(make_float4(f[0], f[1], f[2], f[3]), h0, l0);
    split4(make_float4(f[4], f[5], f[6], f[7]), h1, l1);
    const uint32_t off = sw_off(row, c);
    *reinterpret_cast<uint4*>(smem + OFF_Q + off) = make_uint4(h0.x, h0.y, h1.x, h1.y);
    *reinterpret_cast<uint4*>(smem + OFF_Q + TILE_Q + off) = make_uint4(l0.x, l0.y, l1.x, l1.y);
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t TM_S = tmem_base;          // 2 x 64 columns
  const uint32_t TM_O = tmem_base + 128;    // 64 columns

  if (warp >= 4 && warp < 8) {
    // ===================================== K / V tile gather =====================================
    const int gw = warp - 4;                 // 16 keys per warp
    const int chunk4 = lane & 15, rsub = lane >> 4;
    uint32_t phase = 0;
    for (int64_t it = 0; it < my_tiles; ++it) {
      const int st = (int)(it & 1);
      const int64_t key0 = (t0 + it) * BK;
      // loads first (before the stage is free)
      float4 kv[2][8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = gw * 16 + i * 2 + rsub;
        const int64_t key = key0 + r;
        const bool ok = key < p.P && chunk4 * 4 < p.D;
        kv[0][i] = ok ? __ldg(reinterpret_cast<const float4*>(p.k + key * HD + h * p.D + chunk4 * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (PASS == 1)
          kv[1][i] = ok ? __ldg(reinterpret_cast<const float4*>(p.v + key * HD + h * p.D + chunk4 * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      mbar_wait(smem_u32(kv_empty + st), phase ^ 1);
      uint8_t* base = smem + OFF_KV + st * KV_STAGE;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t r = (uint32_t)(gw * 16 + i * 2 + rsub);
        const uint32_t off = r * 128u + ((((uint32_t)chunk4 >> 1) ^ (r & 7u)) << 4) + (((uint32_t)chunk4 & 1u) << 3);
        uint2 hi, lo;
        split4(kv[0][i], hi, lo);
        *reinterpret_cast<uint2*>(base + off) = hi;
        *reinterpret_cast<uint2*>(base + TILE_K + off) = lo;
        if (PASS == 1) {
          split4(kv[1][i], hi, lo);
          *reinterpret_cast<uint2*>(base + 2 * TILE_K + off) = hi;
          *reinterpret_cast<uint2*>(base + 3 * TILE_K + off) = lo;
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(kv_full + st));
      if (st == 1) phase ^= 1;
    }
  } else if (warp == MMA_WARP) {
    // ===================================== MMA issue =====================================
    if (lane == 0 && my_tiles > 0) {
      const uint32_t idesc_s = make_idesc_bf16(QM, BK, 0, 0);   // S[128 q][64 keys] = Q (K-major) · K (K-major)
      const uint32_t idesc_o = make_idesc_bf16(QM, DP, 0, 1);   // O[128 q][64 d]   = P (K-major) · V (MN-major)
      const uint32_t q_hi = smem_u32(smem + OFF_Q), q_lo = q_hi + TILE_Q;
      const uint32_t p_hi = smem_u32(smem + OFF_P), p_lo = p_hi + TILE_Q;
      auto issue_s = [&](int64_t it) {
        const int st = (int)(it & 1);
        mbar_wait(smem_u32(kv_full + st), (uint32_t)((it >> 1) & 1));
        mbar_wait(smem_u32(s_empty + st), (uint32_t)(((it >> 1) & 1) ^ 1));
        tc_fence_after();
        const uint32_t k_hi = smem_u32(smem + OFF_KV + st * KV_STAGE), k_lo = k_hi + TILE_K;
#pragma unroll
        for (int j = 0; j < DP / 16; ++j) {
          const uint64_t a_hi = make_desc_sw128(q_hi + j * 32, 16, 1024), a_lo = make_desc_sw128(q_lo + j * 32, 16, 1024);
          const uint64_t b_hi = make_desc_sw128(k_hi + j * 32, 16, 1024), b_lo = make_desc_sw128(k_lo + j * 32, 16, 1024);
          mma_bf16(TM_S + st * BK, a_hi, b_hi, idesc_s, j > 0 ? 1u : 0u);
          mma_bf16(TM_S + st * BK, a_lo, b_hi, idesc_s, 1);
          mma_bf16(TM_S + st * BK, a_hi, b_lo, idesc_s, 1);
        }
        mma_commit(smem_u32(s_full + st));
        if (PASS == 0) mma_commit(smem_u32(kv_empty + st));
      };
      issue_s(0);
      for (int64_t it = 0; it < my_tiles; ++it) {
        if (it + 1 < my_tiles) issue_s(it + 1);
        if (PASS == 1) {
          const int st = (int)(it & 1);
          mbar_wait(smem_u32(p_full), (uint32_t)(it & 1));
          tc_fence_after();
          const uint32_t v_hi = smem_u32(smem + OFF_KV + st * KV_STAGE + 2 * TILE_K), v_lo = v_hi + TILE_K;
#pragma unroll
          for (int j = 0; j < BK / 16; ++j) {
            const uint64_t a_hi = make_desc_sw128(p_hi + j * 32, 16, 1024), a_lo = make_desc_sw128(p_lo + j * 32, 16, 1024);
            // V tile: rows = keys (contraction), 128-byte rows of 64 head-dim values → MN-major B, 16 keys = 2 KB
            const uint64_t b_hi = make_desc_sw128(v_hi + j * 2048, TILE_K, 1024), b_lo = make_desc_sw128(v_lo + j * 2048, TILE_K, 1024);
            const uint32_t acc = (it > 0 || j > 0) ? 1u : 0u;
            mma_bf16(TM_O, a_hi, b_hi, idesc_o, acc);
            mma_bf16(TM_O, a_lo, b_hi, idesc_o, 1);
            mma_bf16(TM_O, a_hi, b_lo, idesc_o, 1);
          }
          mma_commit(smem_u32(p_empty));
          mma_commit(smem_u32(kv_empty + st));
        }
      }
      if (PASS == 1) mma_commit(smem_u32(o_full));
    }
  } else {
    // ===================================== softmax rows (warps 0-3) =====================================
    const int qrow = warp * 32 + lane;
    const bool qok = qrow < p.Q;
    float m_run = -CUDART_INF_F, l_run = 0.f;
    const float my_lse = (PASS == 1 && qok) ? __ldg(p.lse + (int64_t)h * p.Q + qrow) : 0.f;
    for (int64_t it = 0; it < my_tiles; ++it) {
      const int st = (int)(it & 1);
      const int64_t key0 = (t0 + it) * BK;
      // mask bytes of this row for the 64 keys of the tile
      uint32_t mbits[2] = {0xffffffffu, 0xffffffffu};
      if (qok) {
        if (p.mask) {
          const uint2 w = __ldg(reinterpret_cast<const uint2*>(p.mask + ((int64_t)qrow * n_tiles + (t0 + it)) * 2));
          mbits[0] = w.x;
          mbits[1] = w.y;
        } else {
          mbits[0] = mbits[1] = 0u;
        }
        const int64_t left = p.P - key0;          // keys beyond P are masked
        if (left < 64) {
          if (left <= 32) {
            mbits[1] = 0xffffffffu;
            if (left < 32) mbits[0] |= ~0u << left;
          } else {
            mbits[1] |= ~0u << (left - 32);
          }
        }
      }
      mbar_wait(smem_u32(s_full + st), (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      float s[BK];
      {
        float a[32], b[32];
        const uint32_t taddr = TM_S + ((uint32_t)(warp * 32) << 16) + (uint32_t)(st * BK);
        tmem_ld32(taddr, a);
        tmem_ld32(taddr + 32, b);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          s[j] = a[j];
          s[32 + j] = b[j];
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(s_empty + st));
      if (PASS == 0) {
        float mx = m_run;
#pragma unroll
        for (int j = 0; j < BK; ++j)
          if (!((mbits[j >> 5] >> (j & 31)) & 1u)) mx = fmaxf(mx, s[j]);
        if (mx > -CUDART_INF_F) {
          float acc = l_run * __expf(m_run - mx);
#pragma unroll
          for (int j = 0; j < BK; ++j)
            if (!((mbits[j >> 5] >> (j & 31)) & 1u)) acc += __expf(s[j] - mx);
          l_run = acc;
          m_run = mx;
        }
      } else {
        mbar_wait(smem_u32(p_empty), (uint32_t)((it & 1) ^ 1));
        uint8_t* ph = smem + OFF_P;
#pragma unroll
        for (int c = 0; c < 8; ++c) {       // 8 probabilities per 16-byte chunk
          float f[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int col = c * 8 + j;
            f[j] = ((mbits[col >> 5] >> (col & 31)) & 1u) ? 0.f : __expf(s[col] - my_lse);
          }
          uint2 h0, l0, h1, l1;
          split4(make_float4(f[0], f[1], f[2], f[3]), h0, l0);
          split4(make_float4(f[4], f[5], f[6], f[7]), h1, l1);
          const uint32_t off = sw_off((uint32_t)qrow, (uint32_t)c);
          *reinterpret_cast<uint4*>(ph + off) = make_uint4(h0.x, h0.y, h1.x, h1.y);
          *reinterpret_cast<uint4*>(ph + TILE_Q + off) = make_uint4(l0.x, l0.y, l1.x, l1.y);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(p_full));
      }
    }
    if (PASS == 0) {
      if (qok) {
        float* w = p.ws + (((int64_t)chunk * p.H + h) * p.Q + qrow) * 2;
        w[0] = m_run;
        w[1] = l_run;
      }
    } else if (my_tiles > 0) {
      mbar_wait(smem_u32(o_full), 0);
      tc_fence_after();
      float a[32], b[32];
      const uint32_t taddr = TM_O + ((uint32_t)(warp * 32) << 16);
      tmem_ld32(taddr, a);
      tmem_ld32(taddr + 32, b);
      tmem_ld_wait();
      if (qok) {
        float* orow = p.ws + (int64_t)p.chunks * p.H * p.Q * 2 + ((int64_t)chunk * p.Q + qrow) * HD + h * p.D;
#pragma unroll
        for (int d = 0; d < 32; ++d)
          if (d < p.D) orow[d] = a[d];
#pragma unroll
        for (int d = 0; d < 32; ++d)
          if (32 + d < p.D) orow[32 + d] = b[d];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

__global__ void k_xattn_lse(const float* __restrict__ ws, int chunks, int HQ, float* __restrict__ lse) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= HQ) return;
  float M = -CUDART_INF_F;
  for (int c = 0; c < chunks; ++c) M = fmaxf(M, ws[((int64_t)c * HQ + i) * 2]);
  float L = 0.f;
  for (int c = 0; c < chunks; ++c) {
    const float m = ws[((int64_t)c * HQ + i) * 2], l = ws[((int64_t)c * HQ + i) * 2 + 1];
    if (m > -CUDART_INF_F) L += l * __expf(m - M);
  }
  lse[i] = M + logf(L);
}

int pick_chunks(int64_t P, int H) {
  int64_t tiles = (P + BK - 1) / BK;
  int c = (num_sms() + H - 1) / H;        // ~one CTA per SM
  if (c > tiles) c = (int)tiles;
  return c < 1 ? 1 : c;
}

// key chunks that own at least one tile (the kernels' split: ceil(tiles / chunks) tiles per chunk); only these write
// their slot of per-chunk partial sums
int live_chunks(int64_t P, int chunks) {
  const int64_t tiles = (P + BK - 1) / BK, per = (tiles + chunks - 1) / chunks;
  return (int)((tiles + per - 1) / per);
}

}  // namespace

extern "C" int64_t pasco_xattn_workspace_bytes(int32_t Q, int64_t P, int32_t H, int32_t D) {
  return (int64_t)pick_chunks(P, H) * (H * Q * 2 + (int64_t)Q * H * D) * sizeof(float);
}

extern "C" int pasco_xattn_forward(const float* q, const float* k, const float* v, const uint32_t* mask, int32_t Q,
                                   int64_t P, int32_t H, int32_t D, float scale, float* out, float* lse, float* workspace,
                                   int64_t workspace_bytes, pasco_stream_t s) {
  PASCO_CHECK_ARG(Q >= 1 && Q <= QM, "pasco_xattn_forward: Q (%d) must be in [1,128]", Q);
  PASCO_CHECK_ARG(D >= 4 && D <= DP && D % 4 == 0, "pasco_xattn_forward: head dim (%d) must be a multiple of 4, <= 64", D);
  PASCO_CHECK_ARG((H * D) % 4 == 0 && P >= 1, "pasco_xattn_forward: bad shape");
  PASCO_CHECK_ARG(workspace_bytes >= pasco_xattn_workspace_bytes(Q, P, H, D), "pasco_xattn_forward: workspace too small");
  PASCO_CHECK_ARG((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)out) & 15) == 0, "pasco_xattn_forward: pointers must be 16-byte aligned");
  XParams p;
  p.q = q; p.k = k; p.v = v; p.mask = mask; p.lse = lse; p.out = out; p.ws = workspace;
  p.Q = Q; p.H = H; p.D = D; p.P = P; p.scale = scale;
  p.chunks = pick_chunks(P, H);
  cudaStream_t st = (cudaStream_t)s;
  const int grid = p.chunks * H;
  cudaError_t e = cudaFuncSetAttribute(k_xattn_fwd<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_xattn_fwd<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  if (e != cudaSuccess) {
    set_error("pasco_xattn_forward: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
    return -1;
  }
  k_xattn_fwd<0><<<grid, NTHREADS, SMEM_BYTES, st>>>(p);
  k_xattn_lse<<<(H * Q + 127) / 128, 128, 0, st>>>(workspace, p.chunks, H * Q, lse);
  k_xattn_fwd<1><<<grid, NTHREADS, SMEM_BYTES, st>>>(p);
  // the chunks' partial outputs summed in chunk order (identical from run to run, unlike float atomics)
  const int64_t n_o = (int64_t)Q * H * D;
  k_add_partials<<<grid_for(n_o, 256), 256, 0, st>>>(workspace + (int64_t)p.chunks * H * Q * 2, live_chunks(P, p.chunks),
                                                     n_o, n_o, out);
  PASCO_CHECK_LAUNCH("pasco_xattn_forward");
  return 0;
}

// ==================================================================================================================
// backward:  given dO, recompute S and P from the saved log-sum-exp and produce dQ, dK, dV
//
//   P = exp(S − lse) (masked → 0),  dP = dO·Vᵀ,  dS = P ∘ (dP − rowsum(dO ∘ O)),
//   dV = Pᵀ·dO,  dK = dSᵀ·Qs,  dQ = scale · dS·K                       (Qs = scale·Q)
//
// Same CTA = (head, key chunk) decomposition and 64-key tiles as the forward.  Five tcgen05 GEMM groups per tile:
//   S  [128q x 64k] = Qs(K-major) · K(K-major)            dP [128q x 64k] = dO(K-major) · V(K-major)
//   dVᵀ[ 64d x 64k] = dOᵀ(MN-major, M padded to 128 with a zero block) · P(MN-major)
//   dKᵀ[ 64d x 64k] = Qsᵀ(MN-major, zero-padded)            · dS(MN-major)
//   dQ [128q x 64d] += dS(K-major) · K(MN-major)              (accumulates in TMEM over the CTA's tiles)
// dVᵀ/dKᵀ land with lane = head-dim index, so one warp store writes 32 consecutive floats of a key's row:
// every dK/dV row is written exactly once (no atomics); each chunk stores its dQ, and the chunks are summed in order.
// ==================================================================================================================
namespace {

struct XBwdParams {
  const float* q; const float* k; const float* v; const uint32_t* mask; const float* lse;
  const float* out; const float* dout;
  float* dq; float* dk; float* dv;
  float* dq_part;      // [chunks, Q, H*D] dQ of each key chunk
  int Q, H, D;
  int64_t P;
  int chunks;
  float scale;
};

constexpr int B_OFF_Q = 0;                          // Qs hi | lo           2 x 16 KB
constexpr int B_OFF_DO = 2 * TILE_Q;                // dO hi | lo           2 x 16 KB
constexpr int B_OFF_ZERO = 4 * TILE_Q;              // zero block           16 KB
constexpr int B_OFF_KV = 5 * TILE_Q;                // 2 stages x (K hi|lo, V hi|lo) = 2 x 32 KB
constexpr int B_OFF_P = B_OFF_KV + 2 * KV_STAGE;    // P hi | lo            2 x 16 KB
constexpr int B_OFF_DS = B_OFF_P + 2 * TILE_Q;      // dS hi | lo           2 x 16 KB
constexpr int B_OFF_BAR = B_OFF_DS + 2 * TILE_Q;
constexpr int B_SMEM_BYTES = B_OFF_BAR + 256 + 1024;

__global__ void __launch_bounds__(NTHREADS, 1) k_xattn_bwd(const __grid_constant__ XBwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + B_OFF_BAR);
  uint64_t* kv_full = bars;         // [2]
  uint64_t* kv_empty = bars + 2;    // [2]
  uint64_t* sdp_full = bars + 4;    // [2]
  uint64_t* sdp_empty = bars + 6;   // [2]
  uint64_t* pds_full = bars + 8;
  uint64_t* pds_empty = bars + 9;
  uint64_t* dvk_full = bars + 10;
  uint64_t* dvk_empty = bars + 11;
  uint64_t* dq_full = bars + 12;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.x % p.H;
  const int chunk = blockIdx.x / p.H;
  const int64_t n_tiles = (p.P + BK - 1) / BK;
  const int64_t tiles_per_chunk = (n_tiles + p.chunks - 1) / p.chunks;
  const int64_t t0 = (int64_t)chunk * tiles_per_chunk;
  const int64_t t1 = t0 + tiles_per_chunk < n_tiles ? t0 + tiles_per_chunk : n_tiles;
  const int64_t my_tiles = t1 > t0 ? t1 - t0 : 0;
  const int HD = p.H * p.D;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(kv_full + i), 4);
      mbar_init(smem_u32(kv_empty + i), 1);
      mbar_init(smem_u32(sdp_full + i), 1);
      mbar_init(smem_u32(sdp_empty + i), 4);
    }
    mbar_init(smem_u32(pds_full), 4);
    mbar_init(smem_u32(pds_empty), 1);
    mbar_init(smem_u32(dvk_full), 1);
    mbar_init(smem_u32(dvk_empty), 4);
    mbar_init(smem_u32(dq_full), 1);
    fence_barrier_init();
  }
  if (warp == MMA_WARP) tmem_alloc(smem_u32(tmem_slot), 512);
  // resident operands: Qs = scale*Q_h and dO_h as bf16 hi/lo [128 rows][64], zero block
  for (int t = threadIdx.x; t < QM * 8; t += NTHREADS) {
    const int row = t >> 3, c = t & 7;
    float f[8], g[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int d = c * 8 + j;
      const bool ok = row < p.Q && d < p.D;
      f[j] = ok ? __ldg(p.q + (int64_t)row * HD + h * p.D + d) * p.scale : 0.f;
      g[j] = ok ? __ldg(p.dout + (int64_t)row * HD + h * p.D + d) : 0.f;
    }
    uint2 h0, l0, h1, l1;
    const uint32_t off = sw_off(row, c);
    split4(make_float4(f[0], f[1], f[2], f[3]), h0, l0);
    split4(make_float4(f[4], f[5], f[6], f[7]), h1, l1);
    *reinterpret_cast<uint4*>(smem + B_OFF_Q + off) = make_uint4(h0.x, h0.y, h1.x, h1.y);
    *reinterpret_cast<uint4*>(smem + B_OFF_Q + TILE_Q + off) = make_uint4(l0.x, l0.y, l1.x, l1.y);
    split4(make_float4(g[0], g[1], g[2], g[3]), h0, l0);
    split4(make_float4(g[4], g[5], g[6], g[7]), h1, l1);
    *reinterpret_cast<uint4*>(smem + B_OFF_DO + off) = make_uint4(h0.x, h0.y, h1.x, h1.y);
    *reinterpret_cast<uint4*>(smem + B_OFF_DO + TILE_Q + off) = make_uint4(l0.x, l0.y, l1.x, l1.y);
    *reinterpret_cast<uint4*>(smem + B_OFF_ZERO + t * 16) = make_uint4(0u, 0u, 0u, 0u);
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t TM_S = tmem_base, TM_DP = tmem_base + 128, TM_DVT = tmem_base + 256, TM_DKT = tmem_base + 320,
                 TM_DQ = tmem_base + 384;

  if (warp >= 4 && warp < 8) {
    // ===================================== K / V tile gather (as forward pass 1) =====================================
    const int gw = warp - 4;
    const int chunk4 = lane & 15, rsub = lane >> 4;
    uint32_t phase = 0;
    for (int64_t it = 0; it < my_tiles; ++it) {
      const int st = (int)(it & 1);
      const int64_t key0 = (t0 + it) * BK;
      float4 kv[2][8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = gw * 16 + i * 2 + rsub;
        const int64_t key = key0 + r;
        const bool ok = key < p.P && chunk4 * 4 < p.D;
        kv[0][i] = ok ? __ldg(reinterpret_cast<const float4*>(p.k + key * HD + h * p.D + chunk4 * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        kv[1][i] = ok ? __ldg(reinterpret_cast<const float4*>(p.v + key * HD + h * p.D + chunk4 * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      mbar_wait(smem_u32(kv_empty + st), phase ^ 1);
      uint8_t* base = smem + B_OFF_KV + st * KV_STAGE;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t r = (uint32_t)(gw * 16 + i * 2 + rsub);
        const uint32_t off = r * 128u + ((((uint32_t)chunk4 >> 1) ^ (r & 7u)) << 4) + (((uint32_t)chunk4 & 1u) << 3);
        uint2 hi, lo;
        split4(kv[0][i], hi, lo);
        *reinterpret_cast<uint2*>(base + off) = hi;
        *reinterpret_cast<uint2*>(base + TILE_K + off) = lo;
        split4(kv[1][i], hi, lo);
        *reinterpret_cast<uint2*>(base + 2 * TILE_K + off) = hi;
        *reinterpret_cast<uint2*>(base + 3 * TILE_K + off) = lo;
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(kv_full + st));
      if (st == 1) phase ^= 1;
    }
  } else if (warp == MMA_WARP) {
    if (lane == 0 && my_tiles > 0) {
      const uint32_t id_kk = make_idesc_bf16(QM, BK, 0, 0);   // K-major x K-major
      const uint32_t id_mm = make_idesc_bf16(QM, BK, 1, 1);   // MN-major x MN-major
      const uint32_t id_km = make_idesc_bf16(QM, DP, 0, 1);   // K-major x MN-major
      const uint32_t q_hi = smem_u32(smem + B_OFF_Q), q_lo = q_hi + TILE_Q;
      const uint32_t o_hi = smem_u32(smem + B_OFF_DO), o_lo = o_hi + TILE_Q;
      const uint32_t zero = smem_u32(smem + B_OFF_ZERO);
      const uint32_t p_hi = smem_u32(smem + B_OFF_P), p_lo = p_hi + TILE_Q;
      const uint32_t s_hi = smem_u32(smem + B_OFF_DS), s_lo = s_hi + TILE_Q;
      auto gemm_kk = [&](uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint64_t ah = make_desc_sw128(a_hi + j * 32, 16, 1024), al = make_desc_sw128(a_lo + j * 32, 16, 1024);
          const uint64_t bh = make_desc_sw128(b_hi + j * 32, 16, 1024), bl = make_desc_sw128(b_lo + j * 32, 16, 1024);
          mma_bf16(d, ah, bh, id_kk, j > 0 ? 1u : 0u);
          mma_bf16(d, al, bh, id_kk, 1);
          mma_bf16(d, ah, bl, id_kk, 1);
        }
      };
      // D[128 (64 real + zero block)][64 keys] = Aᵀ·B with A, B tiles of [128 q rows][128 B]: contraction over the q rows
      auto gemm_mm = [&](uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo) {
#pragma unroll
        for (int j = 0; j < QM / 16; ++j) {
          const uint64_t ah = make_desc_sw128(a_hi + j * 2048, zero - a_hi, 1024), al = make_desc_sw128(a_lo + j * 2048, zero - a_lo, 1024);
          const uint64_t bh = make_desc_sw128(b_hi + j * 2048, 16, 1024), bl = make_desc_sw128(b_lo + j * 2048, 16, 1024);
          mma_bf16(d, ah, bh, id_mm, j > 0 ? 1u : 0u);
          mma_bf16(d, al, bh, id_mm, 1);
          mma_bf16(d, ah, bl, id_mm, 1);
        }
      };
      auto issue_a = [&](int64_t it) {
        const int st = (int)(it & 1);
        mbar_wait(smem_u32(kv_full + st), (uint32_t)((it >> 1) & 1));
        mbar_wait(smem_u32(sdp_empty + st), (uint32_t)(((it >> 1) & 1) ^ 1));
        tc_fence_after();
        const uint32_t k_hi = smem_u32(smem + B_OFF_KV + st * KV_STAGE), k_lo = k_hi + TILE_K;
        const uint32_t v_hi = k_hi + 2 * TILE_K, v_lo = v_hi + TILE_K;
        gemm_kk(TM_S + st * BK, q_hi, q_lo, k_hi, k_lo);
        gemm_kk(TM_DP + st * BK, o_hi, o_lo, v_hi, v_lo);
        mma_commit(smem_u32(sdp_full + st));
      };
      issue_a(0);
      for (int64_t it = 0; it < my_tiles; ++it) {
        if (it + 1 < my_tiles) issue_a(it + 1);
        const int st = (int)(it & 1);
        mbar_wait(smem_u32(pds_full), (uint32_t)(it & 1));
        mbar_wait(smem_u32(dvk_empty), (uint32_t)((it & 1) ^ 1));
        tc_fence_after();
        gemm_mm(TM_DVT, o_hi, o_lo, p_hi, p_lo);     // dVᵀ = dOᵀ · P
        gemm_mm(TM_DKT, q_hi, q_lo, s_hi, s_lo);     // dKᵀ = Qsᵀ · dS
        {                                            // dQ += dS · K   (K tile as MN-major B: 16 keys = 2 KB)
          const uint32_t k_hi = smem_u32(smem + B_OFF_KV + st * KV_STAGE), k_lo = k_hi + TILE_K;
#pragma unroll
          for (int j = 0; j < BK / 16; ++j) {
            const uint64_t ah = make_desc_sw128(s_hi + j * 32, 16, 1024), al = make_desc_sw128(s_lo + j * 32, 16, 1024);
            const uint64_t bh = make_desc_sw128(k_hi + j * 2048, TILE_K, 1024), bl = make_desc_sw128(k_lo + j * 2048, TILE_K, 1024);
            mma_bf16(TM_DQ, ah, bh, id_km, (it > 0 || j > 0) ? 1u : 0u);
            mma_bf16(TM_DQ, al, bh, id_km, 1);
            mma_bf16(TM_DQ, ah, bl, id_km, 1);
          }
        }
        mma_commit(smem_u32(dvk_full));
        mma_commit(smem_u32(pds_empty));
        mma_commit(smem_u32(kv_empty + st));
      }
      mma_commit(smem_u32(dq_full));
    }
  } else {
    // ===================================== query rows: P / dS, then the dK/dV epilogue of the previous tile ==========
    const int qrow = warp * 32 + lane;
    const bool qok = qrow < p.Q;
    float my_lse = 0.f, my_delta = 0.f;
    if (qok) {
      my_lse = __ldg(p.lse + (int64_t)h * p.Q + qrow);
      for (int d = 0; d < p.D; ++d)
        my_delta += __ldg(p.dout + (int64_t)qrow * HD + h * p.D + d) * __ldg(p.out + (int64_t)qrow * HD + h * p.D + d);
    }
    // write-out of dVᵀ/dKᵀ of tile e: lane = head-dim index (warps 0,1 hold d = 0..63), column = key
    auto epilogue = [&](int64_t e) {
      mbar_wait(smem_u32(dvk_full), (uint32_t)(e & 1));
      tc_fence_after();
      const int d = warp * 32 + lane;
      if (warp < 2) {
        const int64_t key0 = (t0 + e) * BK;
#pragma unroll
        for (int which = 0; which < 2; ++which) {
          float* dst = which == 0 ? p.dv : p.dk;
          const uint32_t taddr = (which == 0 ? TM_DVT : TM_DKT) + ((uint32_t)(warp * 32) << 16);
          float a[32], b[32];
          tmem_ld32(taddr, a);
          tmem_ld32(taddr + 32, b);
          tmem_ld_wait();
          if (d < p.D) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (key0 + j < p.P) dst[(key0 + j) * HD + h * p.D + d] = a[j];
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (key0 + 32 + j < p.P) dst[(key0 + 32 + j) * HD + h * p.D + d] = b[j];
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(dvk_empty));
    };
    for (int64_t it = 0; it < my_tiles; ++it) {
      const int st = (int)(it & 1);
      const int64_t key0 = (t0 + it) * BK;
      uint32_t mbits[2] = {0xffffffffu, 0xffffffffu};
      if (qok) {
        if (p.mask) {
          const uint2 w = __ldg(reinterpret_cast<const uint2*>(p.mask + ((int64_t)qrow * n_tiles + (t0 + it)) * 2));
          mbits[0] = w.x;
          mbits[1] = w.y;
        } else {
          mbits[0] = mbits[1] = 0u;
        }
        const int64_t left = p.P - key0;
        if (left < 64) {
          if (left <= 32) {
            mbits[1] = 0xffffffffu;
            if (left < 32) mbits[0] |= ~0u << left;
          } else {
            mbits[1] |= ~0u << (left - 32);
          }
        }
      }
      mbar_wait(smem_u32(sdp_full + st), (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      float pr[BK], ds[BK];
      {
        float a[32], b[32];
        const uint32_t ts = TM_S + ((uint32_t)(warp * 32) << 16) + (uint32_t)(st * BK);
        tmem_ld32(ts, a);
        tmem_ld32(ts + 32, b);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          pr[j] = ((mbits[0] >> j) & 1u) ? 0.f : __expf(a[j] - my_lse);
          pr[32 + j] = ((mbits[1] >> j) & 1u) ? 0.f : __expf(b[j] - my_lse);
        }
        const uint32_t td = TM_DP + ((uint32_t)(warp * 32) << 16) + (uint32_t)(st * BK);
        tmem_ld32(td, a);
        tmem_ld32(td + 32, b);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          ds[j] = pr[j] * (a[j] - my_delta);
          ds[32 + j] = pr[32 + j] * (b[j] - my_delta);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(sdp_empty + st));
      mbar_wait(smem_u32(pds_empty), (uint32_t)((it & 1) ^ 1));
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        uint2 h0, l0, h1, l1;
        const uint32_t off = sw_off((uint32_t)qrow, (uint32_t)c);
        split4(make_float4(pr[c * 8], pr[c * 8 + 1], pr[c * 8 + 2], pr[c * 8 + 3]), h0, l0);
        split4(make_float4(pr[c * 8 + 4], pr[c * 8 + 5], pr[c * 8 + 6], pr[c * 8 + 7]), h1, l1);
        *reinterpret_cast<uint4*>(smem + B_OFF_P + off) = make_uint4(h0.x, h0.y, h1.x, h1.y);
        *reinterpret_cast<uint4*>(smem + B_OFF_P + TILE_Q + off) = make_uint4(l0.x, l0.y, l1.x, l1.y);
        split4(make_float4(ds[c * 8], ds[c * 8 + 1], ds[c * 8 + 2], ds[c * 8 + 3]), h0, l0);
        split4(make_float4(ds[c * 8 + 4], ds[c * 8 + 5], ds[c * 8 + 6], ds[c * 8 + 7]), h1, l1);
        *reinterpret_cast<uint4*>(smem + B_OFF_DS + off) = make_uint4(h0.x, h0.y, h1.x, h1.y);
        *reinterpret_cast<uint4*>(smem + B_OFF_DS + TILE_Q + off) = make_uint4(l0.x, l0.y, l1.x, l1.y);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(pds_full));
      if (it > 0) epilogue(it - 1);
    }
    if (my_tiles > 0) {
      epilogue(my_tiles - 1);
      mbar_wait(smem_u32(dq_full), 0);
      tc_fence_after();
      float a[32], b[32];
      const uint32_t taddr = TM_DQ + ((uint32_t)(warp * 32) << 16);
      tmem_ld32(taddr, a);
      tmem_ld32(taddr + 32, b);
      tmem_ld_wait();
      if (qok) {
        float* row = p.dq_part + ((int64_t)chunk * p.Q + qrow) * HD + h * p.D;
#pragma unroll
        for (int d = 0; d < 32; ++d)
          if (d < p.D) row[d] = a[d] * p.scale;
#pragma unroll
        for (int d = 0; d < 32; ++d)
          if (32 + d < p.D) row[32 + d] = b[d] * p.scale;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

extern "C" int pasco_xattn_backward(const float* q, const float* k, const float* v, const uint32_t* mask, const float* lse,
                                    const float* out, const float* dout, int32_t Q, int64_t P, int32_t H, int32_t D,
                                    float scale, float* dq, float* dk, float* dv, float* workspace,
                                    int64_t workspace_bytes, pasco_stream_t s) {
  PASCO_CHECK_ARG(Q >= 1 && Q <= QM, "pasco_xattn_backward: Q (%d) must be in [1,128]", Q);
  PASCO_CHECK_ARG(D >= 4 && D <= DP && D % 4 == 0, "pasco_xattn_backward: head dim (%d) must be a multiple of 4, <= 64", D);
  PASCO_CHECK_ARG((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)dq | (uintptr_t)dk | (uintptr_t)dv) & 15) == 0,
                  "pasco_xattn_backward: pointers must be 16-byte aligned");
  XBwdParams p;
  p.q = q; p.k = k; p.v = v; p.mask = mask; p.lse = lse; p.out = out; p.dout = dout;
  p.dq = dq; p.dk = dk; p.dv = dv;
  p.Q = Q; p.H = H; p.D = D; p.P = P; p.scale = scale;
  p.chunks = pick_chunks(P, H);
  const int64_t n_q = (int64_t)Q * H * D;
  const int n_live = live_chunks(P, p.chunks);
  PASCO_CHECK_ARG(workspace && workspace_bytes >= (int64_t)n_live * n_q * (int64_t)sizeof(float),
                  "pasco_xattn_backward: workspace smaller than pasco_xattn_workspace_bytes");
  p.dq_part = workspace;
  cudaError_t e = cudaFuncSetAttribute(k_xattn_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM_BYTES);
  if (e != cudaSuccess) {
    set_error("pasco_xattn_backward: cudaFuncSetAttribute(%d) failed: %s", B_SMEM_BYTES, cudaGetErrorString(e));
    return -1;
  }
  k_xattn_bwd<<<p.chunks * H, NTHREADS, B_SMEM_BYTES, (cudaStream_t)s>>>(p);
  k_add_partials<<<grid_for(n_q, 256), 256, 0, (cudaStream_t)s>>>(p.dq_part, n_live, n_q, n_q, dq);
  PASCO_CHECK_LAUNCH("pasco_xattn_backward");
  return 0;
}
