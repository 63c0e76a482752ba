// Weight gradient of the sparse convolution on tcgen05 (sm_100a).
//
//   dW[k] = Σ_o in[nbr[k,o], :]^T @ gout[o, :]
//
// UMMA view: D[M = 128 input channels][N = Cout] += A^T · G with the voxel rows as the contraction dimension, so
// both operands are MN-major: the very same gathered [rows][64 ch] swizzled tiles the forward kernel builds serve as
// A (LBO = distance between two 64-channel sub-tiles) and the gout tile as B (LBO = distance between 64-col blocks).
// "sub-tile" s = (offset k, 64-channel block cb); a unit = two consecutive sub-tiles = one M=128 accumulator of
// Cout TMEM columns; a CTA keeps 512/Cout units resident in TMEM, walks its share of 64-row tiles, and finally
// stores its partial dW in its own workspace slot; the slots are then added in a fixed order (k_add_partials), so dW
// is the same from run to run (float atomics would round differently each time).
#include <stdlib.h>
#include "common.cuh"
#include "umma.cuh"

using namespace pasco;
using namespace umma;

namespace {

constexpr int NUM_GATHER_WARPS = 8;                 // 8 tile rows each
constexpr int MMA_WARP = NUM_GATHER_WARPS;           // 8 (gather warps 0-3 also run the epilogue: TMEM quadrant = warp % 4)
constexpr int NUM_THREADS = (MMA_WARP + 1) * 32;     // 288
constexpr int WROWS = 64 / NUM_GATHER_WARPS;         // rows of a 64-row tile per gather warp
constexpr int WLOADS = WROWS / 2;                    // float4 loads per lane per sub-tile
constexpr int MAX_STAGES = 8;
constexpr int WG_R = 64;                  // voxel rows per tile (contraction block)
constexpr int WG_SUB_BYTES = WG_R * 128;  // one [64 rows][64 ch] bf16 tile = 8 KB

struct WgradParams {
  const float* in;
  const int32_t* nbr;
  const float* gout;
  const float* in_scale;
  const float* in_shift;
  float* dW;
  int64_t n_out;
  int64_t in_pitch, gout_pitch;   // row strides (floats)
  int K, Cin, Cout, in_act;
  int stages, tmem_cols;
  int units_per_pass, num_units, num_subs, passes, ctas_per_pass;
  float* part;  // [ctas_per_pass][K][Cin][Cout] partial dW of each CTA of a pass
};

constexpr int IDX_RING = 16;   // unit slots are short: fetch neighbour indices 15 slots ahead (HBM-latency bound otherwise)

__device__ __forceinline__ void cp_async4(uint32_t dst_smem, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ float act_apply(float z, int act) {
  if (act == 1) return fmaxf(z, 0.f);
  if (act == 2) return z > 0.f ? z : 0.01f * z;
  return z;
}

// One [WG_R rows][64 ch] sub-tile is gathered by 8 warps x 8 rows; lanes (l & 7) of a warp hold the source row of
// tile row w*8 + (l & 7).  Loads and the convert+store are separate so several sub-tiles can be in flight.
struct SubRegs {
  float4 v[WLOADS];
  uint32_t valid;
};

__device__ __forceinline__ void sub_load(SubRegs& r, const float* __restrict__ src, int ld, int cbase_blk, int idx, int lane) {
  const int chunk = lane & 15, rsub = lane >> 4;
  const int cbase = cbase_blk + chunk * 4;
  r.valid = 0;
#pragma unroll
  for (int i = 0; i < WLOADS; ++i) {
    const int s = __shfl_sync(0xffffffffu, idx, i * 2 + rsub);
    r.v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (s >= 0) {
      r.v[i] = __ldg(reinterpret_cast<const float4*>(src + (int64_t)s * ld + cbase));
      r.valid |= 1u << i;
    }
  }
}

template <int NSPLIT, bool AFFINE_OK>
__device__ __forceinline__ void sub_store(const SubRegs& r, uint8_t* dst_hi, uint8_t* dst_lo, int cbase_blk, int warp, int lane,
                                          const float* scale, const float* shift, int act) {
  const int chunk = lane & 15, rsub = lane >> 4;
  float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
  const bool affine = AFFINE_OK && scale != nullptr;
  if (affine) {
    sc = __ldg(reinterpret_cast<const float4*>(scale + cbase_blk + chunk * 4));
    sh = __ldg(reinterpret_cast<const float4*>(shift + cbase_blk + chunk * 4));
  }
#pragma unroll
  for (int i = 0; i < WLOADS; ++i) {
    float4 x = r.v[i];
    if (AFFINE_OK && (affine || act) && ((r.valid >> i) & 1u)) {
      x.x = act_apply(fmaf(x.x, sc.x, sh.x), act);
      x.y = act_apply(fmaf(x.y, sc.y, sh.y), act);
      x.z = act_apply(fmaf(x.z, sc.z, sh.z), act);
      x.w = act_apply(fmaf(x.w, sc.w, sh.w), act);
    }
    const uint32_t trow = (uint32_t)(warp * WROWS + i * 2 + rsub);
    const uint32_t off = trow * 128u + ((((uint32_t)chunk >> 1) ^ (trow & 7u)) << 4) + (((uint32_t)chunk & 1u) << 3);
    if (NSPLIT == 3) {
      uint2 hi, lo;
      split4(x, hi, lo);
      *reinterpret_cast<uint2*>(dst_hi + off) = hi;
      *reinterpret_cast<uint2*>(dst_lo + off) = lo;
    } else {
      *reinterpret_cast<uint2*>(dst_hi + off) = to_bf16x4(x);
    }
  }
}

template <int NSPLIT>
__global__ void __launch_bounds__(NUM_THREADS, 1) k_wgrad_tc(const __grid_constant__ WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int n_op = (NSPLIT == 3) ? 2 : 1;
  const int NB = p.Cout / 64;                    // 64-column blocks of gout
  const int g_bytes = n_op * NB * WG_SUB_BYTES;  // one gout tile (hi [+ lo])
  const int a_bytes = n_op * 2 * WG_SUB_BYTES;   // one stage: two sub-tiles (hi [+ lo])
  uint8_t* g_smem = smem;                        // [2][g_bytes]
  uint8_t* a_smem = smem + 2 * (size_t)g_bytes;  // [stages][a_bytes]
  uint64_t* bars = reinterpret_cast<uint64_t*>(a_smem + (size_t)p.stages * a_bytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + MAX_STAGES;
  uint64_t* gfull_bar = bars + 2 * MAX_STAGES;       // [2]
  uint64_t* gempty_bar = bars + 2 * MAX_STAGES + 2;  // [2]
  uint64_t* done_bar = bars + 2 * MAX_STAGES + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_STAGES + 5);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int CB = p.Cin / 64;
  const int pass = blockIdx.x % p.passes;
  const int cta_in_pass = blockIdx.x / p.passes;
  const int unit0 = pass * p.units_per_pass;
  const int nunits = min(p.units_per_pass, p.num_units - unit0);
  const int64_t num_rt = (p.n_out + WG_R - 1) / WG_R;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(full_bar + s), NUM_GATHER_WARPS);
      mbar_init(smem_u32(empty_bar + s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(gfull_bar + b), NUM_GATHER_WARPS);
      mbar_init(smem_u32(gempty_bar + b), 1);
    }
    mbar_init(smem_u32(done_bar), 1);
    fence_barrier_init();
  }
  // slot descriptor table: [j][0]=type (0 gout, 1 unit), [1],[2]=column bases of the two sub-tiles (-1 = none),
  // [3],[4]=kernel offset of the two sub-tiles (-1 = padding)
  int* idx_ring = reinterpret_cast<int*>(tmem_slot + 4);            // [IDX_RING][2][WG_R]
  int* desc = idx_ring + IDX_RING * 2 * WG_R;                        // [<=16][8]
  {
    const int GSd = (NB + 1) / 2;
    for (int j = threadIdx.x; j < GSd + nunits; j += NUM_THREADS) {
      int* dj = desc + j * 8;
      if (j < GSd) {
        dj[0] = 0; dj[1] = j * 2 * 64; dj[2] = (j * 2 + 1 < NB) ? (j * 2 + 1) * 64 : -1; dj[3] = -1; dj[4] = -1;
      } else {
        dj[0] = 1;
        for (int h = 0; h < 2; ++h) {
          const int sub = (unit0 + (j - GSd)) * 2 + h;
          const bool ok = sub < p.num_subs;
          dj[1 + h] = ok ? (sub % CB) * 64 : 0;
          dj[3 + h] = ok ? sub / CB : -1;
        }
      }
    }
  }
  if (warp == MMA_WARP) tmem_alloc(smem_u32(tmem_slot), (uint32_t)p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int GS = (NB + 1) / 2;
  const int spr = GS + nunits;               // slots per row tile

  if (warp < NUM_GATHER_WARPS) {
    // Flat slot sequence per row tile:  GS gout slots (two 64-column blocks each), then one slot per unit (two
    // gathered sub-tiles).  Every slot = 2 x WLOADS float4 loads per lane; the loads of slot s+1 are in flight in
    // registers while slot s is converted and stored; neighbour indices arrive through a cp.async ring PF_DIST slots
    // ahead.  Slot geometry comes from a small descriptor table in shared memory (no divisions in the loop).
    const int my_r = warp * WROWS + (lane & (WROWS - 1));          // this lane's row inside the 64-row tile
    const int64_t stride_rt = p.ctas_per_pass;
    constexpr int PF_DIST = 12;

    auto prefetch = [&](int64_t rt, int j, int g) {              // indices of slot (rt, j) → ring entry g
      if (lane < 16) {
        const int h = lane >> 3;
        const int k = desc[j * 8 + 3 + h];
        int* d = idx_ring + ((g & (IDX_RING - 1)) * 2 + h) * WG_R + warp * WROWS + (lane & 7);
        const int64_t row = rt * WG_R + warp * WROWS + (lane & 7);
        if (p.nbr && k >= 0 && rt < num_rt && row < p.n_out) cp_async4(smem_u32(d), p.nbr + (int64_t)k * p.n_out + row);
        else *d = (k >= 0 && rt < num_rt && row < p.n_out) ? (int)row : -1;
      }
      cp_async_commit();
    };
    auto issue = [&](int64_t rt, int j, int g, SubRegs (&r)[2]) {
      cp_async_wait<PF_DIST - 1>();
      __syncwarp();
      const int* dj = desc + j * 8;
      const int64_t row = rt * WG_R + my_r;
      if (dj[0] == 0) {                                            // gout slot: identity rows
        int gidx = row < p.n_out ? (int)row : -1;
        sub_load(r[0], p.gout, (int)p.gout_pitch, dj[1], gidx, lane);
        if (dj[2] >= 0) sub_load(r[1], p.gout, (int)p.gout_pitch, dj[2], gidx, lane);
      } else {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          int idx = idx_ring[((g & (IDX_RING - 1)) * 2 + h) * WG_R + my_r];
          if (!p.nbr && idx >= 0) idx = (int)row;
          sub_load(r[h], p.in, (int)p.in_pitch, dj[1 + h], idx, lane);
        }
      }
    };
    int stage = 0;
    uint32_t phase = 0;
    auto store = [&](int j, int git, SubRegs (&r)[2]) {
      const int* dj = desc + j * 8;
      if (dj[0] == 0) {
        const int gb = git & 1;
        if (j == 0) mbar_wait(smem_u32(gempty_bar + gb), ((git >> 1) & 1) ^ 1);
        uint8_t* g = g_smem + (size_t)gb * g_bytes;
        const int nb = j * 2;
        sub_store<NSPLIT, false>(r[0], g + (size_t)nb * WG_SUB_BYTES, g + (size_t)(NB + nb) * WG_SUB_BYTES, 0, warp, lane,
                                 nullptr, nullptr, 0);
        if (dj[2] >= 0)
          sub_store<NSPLIT, false>(r[1], g + (size_t)(nb + 1) * WG_SUB_BYTES, g + (size_t)(NB + nb + 1) * WG_SUB_BYTES, 0,
                                   warp, lane, nullptr, nullptr, 0);
        if (j == GS - 1) {
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_u32(gfull_bar + gb));
        }
      } else {
        mbar_wait(smem_u32(empty_bar + stage), phase ^ 1);
        uint8_t* a = a_smem + (size_t)stage * a_bytes;
#pragma unroll
        for (int h = 0; h < 2; ++h)
          sub_store<NSPLIT, true>(r[h], a + (size_t)h * WG_SUB_BYTES, a + (size_t)(2 + h) * WG_SUB_BYTES, dj[1 + h], warp, lane,
                                  p.in_scale, p.in_shift, p.in_act);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(full_bar + stage));
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    };

    // three cursors over the same slot sequence: prefetch (PF_DIST ahead), load, store
    int64_t p_rt = cta_in_pass, l_rt = cta_in_pass, s_rt = cta_in_pass;
    int p_j = 0, l_j = 0, s_j = 0, p_g = 0, l_g = 0, s_git = 0;
#define WG_ADV(rt, j) do { if (++(j) == spr) { (j) = 0; (rt) += stride_rt; } } while (0)
    if (l_rt < num_rt) {
      for (int a = 0; a < PF_DIST; ++a) {
        prefetch(p_rt, p_j, p_g);
        ++p_g;
        WG_ADV(p_rt, p_j);
      }
      SubRegs ra[2], rb[2];
      auto issue_next = [&](SubRegs (&r)[2]) {
        issue(l_rt, l_j, l_g, r);
        prefetch(p_rt, p_j, p_g);
        ++p_g;
        WG_ADV(p_rt, p_j);
        ++l_g;
        WG_ADV(l_rt, l_j);
      };
      auto store_next = [&](SubRegs (&r)[2]) {
        store(s_j, s_git, r);
        if (++s_j == spr) {
          s_j = 0;
          s_rt += stride_rt;
          ++s_git;
        }
      };
      issue_next(ra);
      while (s_rt < num_rt) {
        if (l_rt < num_rt) issue_next(rb);
        store_next(ra);
        if (s_rt >= num_rt) break;
        if (l_rt < num_rt) issue_next(ra);
        store_next(rb);
      }
    }
#undef WG_ADV
    cp_async_wait<0>();
    // epilogue (gather warps 0-3, after their last slot): once the CTA's last MMA has retired, store the partial dW
    if (warp < 4) {
    const int q = warp;
    const bool any_work = cta_in_pass < num_rt;
    if (any_work) {
      mbar_wait(smem_u32(done_bar), 0);
      tc_fence_after();
      const int L = q * 32 + lane;  // accumulator row = channel within the unit
      for (int u = 0; u < nunits; ++u) {
        const int sub = (unit0 + u) * 2 + (L >> 6);
        const bool ok = sub < p.num_subs;
        const int k = ok ? sub / CB : 0;
        const int cb = ok ? sub - k * CB : 0;
        float* drow = p.part + ((int64_t)cta_in_pass * p.K * p.Cin + (int64_t)k * p.Cin + cb * 64 + (L & 63)) * p.Cout;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(u * p.Cout);
        for (int c0 = 0; c0 < p.Cout; c0 += 32) {
          float v[32];
          tmem_ld32(taddr + c0, v);
          tmem_ld_wait();
          if (ok) {
#pragma unroll
            for (int j = 0; j < 32; ++j) drow[c0 + j] = v[j];
          }
        }
      }
    }
  }
  } else if (warp == MMA_WARP) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(128, p.Cout, 1, 1);
      int stage = 0;
      uint32_t phase = 0;
      int git = 0;
      for (int64_t rt = cta_in_pass; rt < num_rt; rt += p.ctas_per_pass, ++git) {
        const int gb = git & 1;
        mbar_wait(smem_u32(gfull_bar + gb), (git >> 1) & 1);
        tc_fence_after();
        const uint32_t g_hi = smem_u32(g_smem + (size_t)gb * g_bytes);
        const uint32_t g_lo = g_hi + NB * WG_SUB_BYTES;
        for (int u = 0; u < nunits; ++u) {
          mbar_wait(smem_u32(full_bar + stage), phase);
          tc_fence_after();
          const uint32_t a_hi = smem_u32(a_smem + (size_t)stage * a_bytes);
          const uint32_t a_lo = a_hi + 2 * WG_SUB_BYTES;
          const uint32_t d_tmem = tmem_base + (uint32_t)(u * p.Cout);
#pragma unroll
          for (int j = 0; j < WG_R / 16; ++j) {
            const uint32_t acc = (git > 0 || j > 0) ? 1u : 0u;
            const uint64_t da_hi = make_desc_sw128(a_hi + j * 2048, WG_SUB_BYTES, 1024);
            const uint64_t db_hi = make_desc_sw128(g_hi + j * 2048, WG_SUB_BYTES, 1024);
            mma_bf16(d_tmem, da_hi, db_hi, idesc, acc);
            if (NSPLIT == 3) {
              const uint64_t da_lo = make_desc_sw128(a_lo + j * 2048, WG_SUB_BYTES, 1024);
              const uint64_t db_lo = make_desc_sw128(g_lo + j * 2048, WG_SUB_BYTES, 1024);
              mma_bf16(d_tmem, da_lo, db_hi, idesc, 1);
              mma_bf16(d_tmem, da_hi, db_lo, idesc, 1);
            }
          }
          mma_commit(smem_u32(empty_bar + stage));
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        mma_commit(smem_u32(gempty_bar + gb));
      }
      mma_commit(smem_u32(done_bar));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------------------
// Plane-gather variant of the weight gradient: both operands arrive as pre-split bf16 planes
// ------------------------------------------------------------------------------------------------------------
// Same UMMA view, TMEM residency, passes and epilogue as k_wgrad_tc; the producers only move bytes: 16-byte cp.async
// copies from the `in` planes (gathered rows; a missing neighbour is a zero-fill copy that touches no memory) and from
// the `gout` planes (contiguous rows) straight into the 128-byte-swizzled tiles.  Slot 0 of a row tile = the whole gout
// tile, slots 1.. = one unit of two gathered sub-tiles each; every producer thread arrives on the slot's "full" barrier
// with cp.async.mbarrier.arrive.noinc (count = 256 threads), so the hardware completes it when the last copy has landed
// and the producers run a whole ring ahead of the MMA.  Round-1 k_wgrad_tc spent ~600 gather / convert / store
// instructions per sub-tile and ran at 15 % tensor-pipe utilisation, 2.4x slower than the forward.
struct WgradPlParams {
  const uint16_t* in_hi;
  const uint16_t* in_lo;
  const uint16_t* g_hi;
  const uint16_t* g_lo;
  const int32_t* nbr;
  float* dW;
  int64_t n_out;
  int64_t in_pitch, gout_pitch;   // row strides (bf16 elements)
  int K, Cin, Cout;
  int stages, tmem_cols, depth;
  int units_per_pass, num_units, num_subs, passes, ctas_per_pass;
  float* part;  // [ctas_per_pass][K][Cin][Cout] partial dW of each CTA of a pass
};

__device__ __forceinline__ void cp_async16_zfill(uint32_t dst_smem, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}

constexpr int WG_MMA_WARPS = 4;                                   // tcgen05.mma issuers of k_wgrad_pl (warps 8..11)
constexpr int NUM_THREADS_WPL = (MMA_WARP + WG_MMA_WARPS) * 32;   // 384

template <int NSPLIT>
__global__ void __launch_bounds__(NUM_THREADS_WPL, 1) k_wgrad_pl(const __grid_constant__ WgradPlParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int n_op = (NSPLIT == 3) ? 2 : 1;
  const int NB = p.Cout / 64;                    // 64-column blocks of gout
  const int g_bytes = n_op * NB * WG_SUB_BYTES;  // one gout tile (hi blocks [+ lo blocks])
  const int a_bytes = n_op * 2 * WG_SUB_BYTES;   // one stage: two sub-tiles (hi, hi [, lo, lo])
  uint8_t* g_smem = smem;                        // [2][g_bytes]
  uint8_t* a_smem = smem + 2 * (size_t)g_bytes;  // [stages][a_bytes]
  uint64_t* bars = reinterpret_cast<uint64_t*>(a_smem + (size_t)p.stages * a_bytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + MAX_STAGES;
  uint64_t* gfull_bar = bars + 2 * MAX_STAGES;       // [2]
  uint64_t* gempty_bar = bars + 2 * MAX_STAGES + 2;  // [2]
  uint64_t* done_bar = bars + 2 * MAX_STAGES + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_STAGES + 5);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int CB = p.Cin / 64;
  const int pass = blockIdx.x % p.passes;
  const int cta_in_pass = blockIdx.x / p.passes;
  const int unit0 = pass * p.units_per_pass;
  const int nunits = min(p.units_per_pass, p.num_units - unit0);
  const int64_t num_rt = (p.n_out + WG_R - 1) / WG_R;

  // MMA issuers: the units of a row tile accumulate into different TMEM columns, so issuer `mid` (one thread of warp
  // 8 + mid) owns the units u ≡ mid (mod n_mma); one issuer alone needs ~100 cycles of descriptor work per tcgen05.mma
  // that executes in 32 (N = 64) and left the tensor pipe at 33 %
  // A parity wait is only sound for a waiter that sees every phase of the barrier, so a stage of the unit ring must
  // always be consumed by the same issuer: unit slot `ord` holds unit ord % nunits and sits in stage ord % stages, hence
  // n_mma must divide both nunits and stages (the host picks `stages` and the pass split accordingly).
  int n_mma = 1;
  for (int c = 2; c <= WG_MMA_WARPS && c <= p.depth; ++c)
    if (nunits % c == 0 && p.stages % c == 0) n_mma = c;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(full_bar + s), 32);    // one cp.async arrival per lane of the warp that fills the slot
      mbar_init(smem_u32(empty_bar + s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(gfull_bar + b), 32);
      mbar_init(smem_u32(gempty_bar + b), n_mma);     // one commit per MMA issuer
    }
    mbar_init(smem_u32(done_bar), n_mma);
    fence_barrier_init();
  }
  if (warp == MMA_WARP) tmem_alloc(smem_u32(tmem_slot), (uint32_t)p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < NUM_GATHER_WARPS) {
    // ONE WARP PER SLOT, ownership split by resource:
    //   * warp 7 fills every gout tile (double buffer; consecutive fills by the same warp, so its parity wait on the
    //     "gout empty" barrier is never more than one phase away from the barrier);
    //   * warps 0 .. Wu-1 (Wu = min(7, stages)) fill the unit slots ord = w, w + Wu, ... of the CTA's unit sequence
    //     (row tile major): the stride Wu <= stages keeps a warp within one revolution of the unit ring.
    // A warp waits only on barriers of slots it owns.  (Letting all 8 warps take slots round-robin across both rings, or
    // letting every warp observe every barrier, deadlocks: a parity wait is only sound when the waiter is neither two
    // revolutions ahead of nor one revolution behind the barrier — tools/pipeline_sim.py replays the three schemes.)
    // lane = (row sub-index 0..3, 16-byte chunk 0..7): one copy instruction moves 4 tile rows.  For a unit slot lane l
    // holds the neighbour indices of rows l and l+32 of both sub-tiles (four coalesced 128-byte loads, fetched one of
    // the warp's slots ahead), distributed by one shuffle per instruction.
    const int ch = lane & 7, sub = lane >> 3;
    const int64_t stride_rt = p.ctas_per_pass;
    const int64_t my_rts = cta_in_pass < num_rt ? (num_rt - cta_in_pass + stride_rt - 1) / stride_rt : 0;   // row tiles of this CTA
    const uint8_t* in_hi = reinterpret_cast<const uint8_t*>(p.in_hi);
    const uint8_t* in_lo = reinterpret_cast<const uint8_t*>(p.in_lo);
    const uint8_t* gp_hi = reinterpret_cast<const uint8_t*>(p.g_hi);
    const uint8_t* gp_lo = reinterpret_cast<const uint8_t*>(p.g_lo);
    // unit producers: Wu = the largest divisor of `stages` that is <= 7, so that warp w always fills the same stages
    // (w, w + Wu, ...) and sees every phase of their "empty" barriers — with several MMA issuers stages are not freed in
    // slot order, and a producer that skipped a revolution of a stage could pass its parity wait one use early
    int Wu = 1;
    for (int c = 2; c <= NUM_GATHER_WARPS - 1; ++c)
      if (p.stages % c == 0) Wu = c;
    if (warp == NUM_GATHER_WARPS - 1) {
      // ---- gout tiles: [64 rows][Cout] per plane, contiguous rows ----
      for (int64_t rti = 0; rti < my_rts; ++rti) {
        const int64_t rt = cta_in_pass + rti * stride_rt;
        const int gb = (int)(rti & 1);
        mbar_wait(smem_u32(gempty_bar + gb), (uint32_t)(((rti >> 1) & 1) ^ 1));
        const uint32_t g0 = smem_u32(g_smem + (size_t)gb * g_bytes) + (uint32_t)sub * 128u;
#pragma unroll 4
        for (int i = 0; i < WG_R / 4; ++i) {
          const int64_t row = rt * WG_R + i * 4 + sub;
          const uint32_t nbytes = row < p.n_out ? 16u : 0u;
          const int64_t boff = ((row < p.n_out ? row : 0) * p.gout_pitch + ch * 8) * 2;
          const uint32_t off = (uint32_t)i * 512u + (((uint32_t)ch ^ (((uint32_t)(i & 1) << 2) + (uint32_t)sub)) << 4);
          for (int nb = 0; nb < NB; ++nb) {
            cp_async16_zfill(g0 + (uint32_t)nb * WG_SUB_BYTES + off, gp_hi + boff + nb * 128, nbytes);
            if (NSPLIT == 3) cp_async16_zfill(g0 + (uint32_t)(NB + nb) * WG_SUB_BYTES + off, gp_lo + boff + nb * 128, nbytes);
          }
        }
        cp_async_mbar_arrive_noinc(smem_u32(gfull_bar + gb));
      }
    } else if (warp < Wu) {
      // ---- units: two gathered [64 rows][64 ch] sub-tiles each ----
      const int64_t total_units = my_rts * nunits;
      struct Idx4 { int v[4]; };                    // [sub-tile h][row half]
      auto load_idx = [&](int64_t ord) -> Idx4 {
        Idx4 r;
        r.v[0] = r.v[1] = r.v[2] = r.v[3] = -1;
        if (ord < total_units) {
          const int64_t rt = cta_in_pass + (ord / nunits) * stride_rt;
          const int u = (int)(ord % nunits);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int sbi = (unit0 + u) * 2 + h;
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const int64_t row = rt * WG_R + q * 32 + lane;
              if (sbi < p.num_subs && row < p.n_out)
                r.v[h * 2 + q] = p.nbr ? __ldg(p.nbr + (int64_t)(sbi / CB) * p.n_out + row) : (int)row;
            }
          }
        }
        return r;
      };
      int stage = warp;                             // warp < Wu <= stages
      uint32_t phase = 0;
      Idx4 q0 = load_idx(warp);
      for (int64_t ord = warp; ord < total_units; ord += Wu) {
        const Idx4 q1 = load_idx(ord + Wu);         // indices of this warp's next unit
        const int u = (int)(ord % nunits);
        mbar_wait(smem_u32(empty_bar + stage), phase ^ 1);
        const uint32_t a0 = smem_u32(a_smem + (size_t)stage * a_bytes) + (uint32_t)sub * 128u;
        const int sb0 = (unit0 + u) * 2;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int sbi = sb0 + h;
          const int64_t coff_b = ((int64_t)(sbi < p.num_subs ? sbi % CB : 0) * 64 + ch * 8) * 2;
#pragma unroll
          for (int i = 0; i < WG_R / 4; ++i) {
            const int idx = __shfl_sync(0xffffffffu, q0.v[h * 2 + (i >> 3)], ((i & 7) << 2) + sub);
            const uint32_t nbytes = idx >= 0 ? 16u : 0u;
            const int64_t boff = (int64_t)(idx >= 0 ? idx : 0) * p.in_pitch * 2 + coff_b;
            const uint32_t off = (uint32_t)i * 512u + (((uint32_t)ch ^ (((uint32_t)(i & 1) << 2) + (uint32_t)sub)) << 4);
            cp_async16_zfill(a0 + (uint32_t)h * WG_SUB_BYTES + off, in_hi + boff, nbytes);
            if (NSPLIT == 3) cp_async16_zfill(a0 + (uint32_t)(2 + h) * WG_SUB_BYTES + off, in_lo + boff, nbytes);
          }
        }
        cp_async_mbar_arrive_noinc(smem_u32(full_bar + stage));
        stage += Wu;                                // at most one wrap: Wu <= stages
        if (stage >= p.stages) {
          stage -= p.stages;
          phase ^= 1;
        }
        q0 = q1;
      }
    }
    cp_async_commit();
    cp_async_wait<0>();
    // epilogue (gather warps 0-3): once the CTA's last MMA has retired, store the partial dW
    if (warp < 4) {
      const int qd = warp;
      if (cta_in_pass < num_rt) {
        mbar_wait(smem_u32(done_bar), 0);
        tc_fence_after();
        const int L = qd * 32 + lane;  // accumulator row = channel within the unit
        for (int u = 0; u < nunits; ++u) {
          const int sbi = (unit0 + u) * 2 + (L >> 6);
          const bool ok = sbi < p.num_subs;
          const int k = ok ? sbi / CB : 0;
          const int cb = ok ? sbi - k * CB : 0;
          float* drow = p.part + ((int64_t)cta_in_pass * p.K * p.Cin + (int64_t)k * p.Cin + cb * 64 + (L & 63)) * p.Cout;
          const uint32_t taddr = tmem_base + ((uint32_t)(qd * 32) << 16) + (uint32_t)(u * p.Cout);
          for (int c0 = 0; c0 < p.Cout; c0 += 32) {
            float v[32];
            tmem_ld32(taddr + c0, v);
            tmem_ld_wait();
            if (ok) {
#pragma unroll
              for (int j = 0; j < 32; ++j) drow[c0 + j] = v[j];
            }
          }
        }
      }
    }
  } else if (warp >= MMA_WARP && warp - MMA_WARP < n_mma) {
    // whole warp, warp-uniform loop; the elected lane issues tcgen05.mma / tcgen05.commit (descriptors stay in uniform
    // registers instead of ~13 ELECT / R2UR instructions per MMA)
    const int mid = warp - MMA_WARP;
    const bool lead = elect_one();
    {
      const uint32_t idesc = make_idesc_bf16(128, p.Cout, 1, 1);
      int stage = 0;
      uint32_t phase = 0;
      int git = 0;
      for (int64_t rt = cta_in_pass; rt < num_rt; rt += p.ctas_per_pass, ++git) {
        const int gb = git & 1;
        mbar_wait(smem_u32(gfull_bar + gb), (git >> 1) & 1);
        fence_proxy_async_smem();                  // tiles were written by cp.async copies (generic proxy)
        tc_fence_after();
        const uint32_t g_hi = smem_u32(g_smem + (size_t)gb * g_bytes);
        const uint32_t g_lo = g_hi + NB * WG_SUB_BYTES;
        const uint64_t db_hi0 = make_desc_sw128(g_hi, WG_SUB_BYTES, 1024), db_lo0 = make_desc_sw128(g_lo, WG_SUB_BYTES, 1024);
        for (int u = 0; u < nunits; ++u) {
          if (u % n_mma == mid) {
            mbar_wait(smem_u32(full_bar + stage), phase);
            fence_proxy_async_smem();
            tc_fence_after();
            const uint32_t a_hi = smem_u32(a_smem + (size_t)stage * a_bytes);
            const uint32_t a_lo = a_hi + 2 * WG_SUB_BYTES;
            const uint32_t d_tmem = tmem_base + (uint32_t)(u * p.Cout);
            const uint64_t da_hi0 = make_desc_sw128(a_hi, WG_SUB_BYTES, 1024), da_lo0 = make_desc_sw128(a_lo, WG_SUB_BYTES, 1024);
            if (lead) {
#pragma unroll
              for (int j = 0; j < WG_R / 16; ++j) {             // 16 rows = 2048 bytes = 128 address units per k-step
                const uint32_t acc = (git > 0 || j > 0) ? 1u : 0u;
                mma_bf16(d_tmem, da_hi0 + 128 * j, db_hi0 + 128 * j, idesc, acc);
                if (NSPLIT == 3) {
                  mma_bf16(d_tmem, da_lo0 + 128 * j, db_hi0 + 128 * j, idesc, 1);
                  mma_bf16(d_tmem, da_hi0 + 128 * j, db_lo0 + 128 * j, idesc, 1);
                }
              }
              mma_commit(smem_u32(empty_bar + stage));
            }
            __syncwarp();
          }
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (lead) mma_commit(smem_u32(gempty_bar + gb));
        __syncwarp();
      }
      if (lead) mma_commit(smem_u32(done_bar));
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

int pow2_cols(int c) {
  int v = 32;
  while (v < c) v <<= 1;
  return v;
}

// CTAs that share one pass (one set of accumulator units) of either weight-gradient kernel: one partial dW slot each
int wgrad_ctas_per_pass(int K, int64_t n_out, int Cin, int Cout) {
  const int num_units = (K * (Cin / 64) + 1) / 2;
  const int upp = 512 / Cout < num_units ? 512 / Cout : num_units;
  const int passes = (num_units + upp - 1) / upp;
  const int64_t num_rt = (n_out + WG_R - 1) / WG_R;
  int cpp = num_sms() / passes;
  if (cpp < 1) cpp = 1;
  if (cpp > num_rt) cpp = (int)num_rt;
  return cpp;
}

}  // namespace

extern "C" int64_t pasco_conv_wgrad_workspace_bytes(int32_t K, int64_t n_out, int32_t Cin, int32_t Cout) {
  if (n_out <= 0 || K <= 0 || Cin < 64 || Cout < 64) return 0;
  return (int64_t)wgrad_ctas_per_pass(K, n_out, Cin, Cout) * K * Cin * Cout * sizeof(float);
}

extern "C" int pasco_conv_wgrad_tc(const float* in, int64_t n_in, const int32_t* nbr, int32_t K, int64_t n_out,
                                   int32_t Cin, int32_t Cout, const float* gout, const float* in_scale,
                                   const float* in_shift, int32_t in_act, float* dW, int32_t precision,
                                   int64_t in_pitch, int64_t gout_pitch, float* workspace, int64_t workspace_bytes,
                                   pasco_stream_t s) {
  PASCO_CHECK_ARG(precision == 1 || precision == 3, "pasco_conv_wgrad_tc: precision must be 1 or 3");
  PASCO_CHECK_ARG(Cin % 64 == 0 && Cout % 64 == 0 && Cout <= 256,
                  "pasco_conv_wgrad_tc: Cin (%d) and Cout (%d) must be multiples of 64, Cout <= 256", Cin, Cout);
  (void)n_in;
  if (n_out == 0) return 0;
  int dev = 0, smem_optin = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  const int n_op = precision == 3 ? 2 : 1;
  const int g_bytes = n_op * (Cout / 64) * WG_SUB_BYTES;
  const int a_bytes = n_op * 2 * WG_SUB_BYTES;
  const int fixed = 1024 + (2 * MAX_STAGES + 6) * 8 + 32 + IDX_RING * 2 * WG_R * 4 + 16 * 8 * 4;
  int stages = (smem_optin - fixed - 2 * g_bytes) / a_bytes;
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  PASCO_CHECK_ARG(stages >= 2, "pasco_conv_wgrad_tc: not enough shared memory");
  WgradParams p;
  p.in = in; p.nbr = nbr; p.gout = gout; p.in_scale = in_scale; p.in_shift = in_shift; p.dW = dW;
  p.n_out = n_out; p.K = K; p.Cin = Cin; p.Cout = Cout; p.in_act = in_act;
  p.in_pitch = in_pitch > 0 ? in_pitch : Cin;
  p.gout_pitch = gout_pitch > 0 ? gout_pitch : Cout;
  p.stages = stages;
  p.num_subs = K * (Cin / 64);
  p.num_units = (p.num_subs + 1) / 2;
  p.units_per_pass = 512 / Cout;
  if (p.units_per_pass > p.num_units) p.units_per_pass = p.num_units;
  p.tmem_cols = pow2_cols(p.units_per_pass * Cout);
  p.passes = (p.num_units + p.units_per_pass - 1) / p.units_per_pass;
  p.units_per_pass = (p.num_units + p.passes - 1) / p.passes;   // balance the passes (8+6 → 7+7)
  int64_t num_rt = (n_out + WG_R - 1) / WG_R;
  int cpp = num_sms() / p.passes;
  if (cpp < 1) cpp = 1;
  if (cpp > num_rt) cpp = (int)num_rt;
  p.ctas_per_pass = cpp;
  // each CTA stores its partial dW in its own slot (cpp <= num_rt: every CTA has a row tile, so every slot is written in
  // full); the slots are then summed in a fixed order, which keeps dW identical from run to run
  const int64_t n_w = (int64_t)K * Cin * Cout;
  PASCO_CHECK_ARG(cpp == wgrad_ctas_per_pass(K, n_out, Cin, Cout) && workspace &&
                  workspace_bytes >= (int64_t)cpp * n_w * (int64_t)sizeof(float),
                  "pasco_conv_wgrad_tc: workspace smaller than pasco_conv_wgrad_workspace_bytes");
  p.part = workspace;
  const size_t smem = (size_t)2 * g_bytes + (size_t)stages * a_bytes + fixed;
  const int grid = p.passes * cpp;
  cudaError_t e;
  if (precision == 3) {
    e = cudaFuncSetAttribute(k_wgrad_tc<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) k_wgrad_tc<3><<<grid, NUM_THREADS, smem, (cudaStream_t)s>>>(p);
  } else {
    e = cudaFuncSetAttribute(k_wgrad_tc<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) k_wgrad_tc<1><<<grid, NUM_THREADS, smem, (cudaStream_t)s>>>(p);
  }
  if (e != cudaSuccess) {
    set_error("pasco_conv_wgrad_tc: cudaFuncSetAttribute(%zu bytes) failed: %s", smem, cudaGetErrorString(e));
    return -1;
  }
  k_add_partials<<<grid_for(n_w, 256), 256, 0, (cudaStream_t)s>>>(p.part, cpp, n_w, n_w, dW);
  PASCO_CHECK_LAUNCH("pasco_conv_wgrad_tc");
  return 0;
}

extern "C" int pasco_conv_wgrad_planes(const void* in_hi, const void* in_lo, int64_t n_in, const int32_t* nbr, int32_t K,
                                       int64_t n_out, int32_t Cin, int32_t Cout, const void* g_hi, const void* g_lo,
                                       float* dW, int32_t precision, int64_t in_pitch, int64_t gout_pitch, float* workspace,
                                       int64_t workspace_bytes, pasco_stream_t s) {
  PASCO_CHECK_ARG(precision == 1 || precision == 3, "pasco_conv_wgrad_planes: precision must be 1 or 3");
  PASCO_CHECK_ARG(in_hi && g_hi && (precision == 1 || (in_lo && g_lo)), "pasco_conv_wgrad_planes: missing plane");
  PASCO_CHECK_ARG(Cin % 64 == 0 && Cout % 64 == 0 && Cout <= 256,
                  "pasco_conv_wgrad_planes: Cin (%d) and Cout (%d) must be multiples of 64, Cout <= 256", Cin, Cout);
  (void)n_in;
  if (n_out == 0) return 0;
  int dev = 0, smem_optin = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  const int n_op = precision == 3 ? 2 : 1;
  const int g_bytes = n_op * (Cout / 64) * WG_SUB_BYTES;
  const int a_bytes = n_op * 2 * WG_SUB_BYTES;
  const int fixed = 1024 + (2 * MAX_STAGES + 6) * 8 + 32;
  int stages = (smem_optin - fixed - 2 * g_bytes) / a_bytes;
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  PASCO_CHECK_ARG(stages >= 2, "pasco_conv_wgrad_planes: not enough shared memory");
  WgradPlParams p;
  p.in_hi = (const uint16_t*)in_hi; p.in_lo = (const uint16_t*)in_lo; p.g_hi = (const uint16_t*)g_hi; p.g_lo = (const uint16_t*)g_lo;
  p.nbr = nbr; p.dW = dW;
  p.n_out = n_out; p.K = K; p.Cin = Cin; p.Cout = Cout;
  p.in_pitch = in_pitch > 0 ? in_pitch : Cin;
  p.gout_pitch = gout_pitch > 0 ? gout_pitch : Cout;
  PASCO_CHECK_ARG(p.in_pitch % 8 == 0 && p.gout_pitch % 8 == 0 &&
                  (((uintptr_t)in_hi | (uintptr_t)in_lo | (uintptr_t)g_hi | (uintptr_t)g_lo) & 15) == 0,
                  "pasco_conv_wgrad_planes: planes must be 16-byte aligned with pitches multiple of 8 elements");
  p.stages = stages;
  p.depth = stages - 1 > 7 ? 7 : stages - 1;
  static const int depth_env = [] { const char* e = getenv("PASCO_PL_DEPTH"); return e ? atoi(e) : 0; }();
  if (depth_env > 0 && depth_env < p.depth) p.depth = depth_env;
  p.num_subs = K * (Cin / 64);
  p.num_units = (p.num_subs + 1) / 2;
  const int units_cap = 512 / Cout;                             // accumulators that fit TMEM
  p.units_per_pass = units_cap;
  if (p.units_per_pass > p.num_units) p.units_per_pass = p.num_units;
  p.tmem_cols = pow2_cols(p.units_per_pass * Cout);
  p.passes = (p.num_units + p.units_per_pass - 1) / p.units_per_pass;
  p.units_per_pass = (p.num_units + p.passes - 1) / p.passes;   // balance the passes (8+6 → 7+7) ...
  // ... unless that makes the unit count odd: several MMA issuers need a common divisor of units and stages (kernel
  // comment), so 14 units run as 8 + 6 rather than 7 + 7
  if ((p.units_per_pass & 1) && p.units_per_pass + 1 <= units_cap && p.units_per_pass > 1) p.units_per_pass += 1;
  {
    static const int nm_env = [] { const char* e = getenv("PASCO_WG_NM"); return e ? atoi(e) : 0; }();
    const int nm_max = nm_env >= 1 && nm_env <= WG_MMA_WARPS ? nm_env : WG_MMA_WARPS;
    int best = 1;
    for (int c = 2; c <= nm_max; ++c)
      if (p.units_per_pass % c == 0 && stages / c >= 1 && (stages / c) * c >= 2) best = c;
    // stages: a multiple of the issuer count, and with a large divisor <= 7 (= the number of producer warps, see kernel)
    {
      int pick = 0, pick_w = 0;
      for (int st = stages; st >= 2; --st) {
        if (st % best) continue;
        int w = 1;
        for (int c = 2; c <= 7; ++c)
          if (st % c == 0) w = c;
        if (w > pick_w) { pick_w = w; pick = st; }
      }
      if (pick) stages = pick;
    }
    p.stages = stages;
    p.depth = nm_max;                                           // most issuers a CTA may use
  }
  const int64_t num_rt = (n_out + WG_R - 1) / WG_R;
  int cpp = num_sms() / p.passes;
  if (cpp < 1) cpp = 1;
  if (cpp > num_rt) cpp = (int)num_rt;
  p.ctas_per_pass = cpp;
  // each CTA stores its partial dW in its own slot (cpp <= num_rt: every CTA has a row tile, so every slot is written in
  // full); the slots are then summed in a fixed order, which keeps dW identical from run to run
  const int64_t n_w = (int64_t)K * Cin * Cout;
  PASCO_CHECK_ARG(cpp == wgrad_ctas_per_pass(K, n_out, Cin, Cout) && workspace &&
                  workspace_bytes >= (int64_t)cpp * n_w * (int64_t)sizeof(float),
                  "pasco_conv_wgrad_planes: workspace smaller than pasco_conv_wgrad_workspace_bytes");
  p.part = workspace;
  const size_t smem = (size_t)2 * g_bytes + (size_t)stages * a_bytes + fixed;
  const int grid = p.passes * cpp;
  cudaError_t e;
  if (precision == 3) {
    e = cudaFuncSetAttribute(k_wgrad_pl<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) k_wgrad_pl<3><<<grid, NUM_THREADS_WPL, smem, (cudaStream_t)s>>>(p);
  } else {
    e = cudaFuncSetAttribute(k_wgrad_pl<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) k_wgrad_pl<1><<<grid, NUM_THREADS_WPL, smem, (cudaStream_t)s>>>(p);
  }
  if (e != cudaSuccess) {
    set_error("pasco_conv_wgrad_planes: cudaFuncSetAttribute(%zu bytes) failed: %s", smem, cudaGetErrorString(e));
    return -1;
  }
  k_add_partials<<<grid_for(n_w, 256), 256, 0, (cudaStream_t)s>>>(p.part, cpp, n_w, n_w, dW);
  PASCO_CHECK_LAUNCH("pasco_conv_wgrad_planes");
  return 0;
}
