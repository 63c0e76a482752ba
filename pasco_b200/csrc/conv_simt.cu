// CUDA-core fp32 path of the sparse-conv contraction  out[o,:] = Σ_k in[nbr[k,o],:] @ W[k].
// Any Cin/Cout.  This is the in-library cross-check for the tcgen05 path (conv_tc.cu) and serves the
// shapes the tensor-core kernel does not take (channel counts that are not multiples of 64/16).
#include "common.cuh"

using namespace pasco;

constexpr int TR = 16;  // output rows per block
struct KoffMap {
  int v[256];
};

// W layout: transposed==0 → W[k][ci][co] ; transposed==1 → W[k][co][ci] (used for dgrad: "Cin" here is the
// gradient's channel count = forward Cout)
__global__ void __launch_bounds__(256)
k_conv_simt(const float* __restrict__ in, const int32_t* __restrict__ nbr, int K, int64_t n_out, int Cin, int Cout,
            const float* __restrict__ W, int w_transposed, const __grid_constant__ KoffMap koff, const float* __restrict__ bias,
            float* __restrict__ out) {
  extern __shared__ float sA[];  // [TR][Cin]
  __shared__ int sIdx[TR];
  int64_t row0 = (int64_t)blockIdx.x * TR;
  // each thread owns output columns co = threadIdx.x + j*256, all TR rows
  constexpr int MAXJ = 2;  // Cout <= 512
  float acc[MAXJ][TR];
#pragma unroll
  for (int j = 0; j < MAXJ; ++j)
#pragma unroll
    for (int r = 0; r < TR; ++r) acc[j][r] = 0.f;

  for (int k = 0; k < K; ++k) {
    if (threadIdx.x < TR) {
      int64_t o = row0 + threadIdx.x;
      sIdx[threadIdx.x] = o < n_out ? __ldg(nbr + (int64_t)k * n_out + o) : -1;
    }
    __syncthreads();
    int any = 0;
#pragma unroll
    for (int r = 0; r < TR; ++r) any |= (sIdx[r] >= 0);
    if (any) {
      for (int t = threadIdx.x; t < TR * Cin; t += blockDim.x) {
        int r = t / Cin, c = t - r * Cin;
        int src = sIdx[r];
        sA[t] = src >= 0 ? __ldg(in + (int64_t)src * Cin + c) : 0.f;
      }
      __syncthreads();
      int kw = koff.v[k];
      const float* Wk = W + (int64_t)kw * Cin * Cout;
#pragma unroll
      for (int j = 0; j < MAXJ; ++j) {
        int co = threadIdx.x + j * 256;
        if (co < Cout) {
          for (int ci = 0; ci < Cin; ++ci) {
            float w = w_transposed ? __ldg(Wk + (int64_t)co * Cin + ci) : __ldg(Wk + (int64_t)ci * Cout + co);
#pragma unroll
            for (int r = 0; r < TR; ++r) acc[j][r] = fmaf(sA[r * Cin + ci], w, acc[j][r]);
          }
        }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < MAXJ; ++j) {
    int co = threadIdx.x + j * 256;
    if (co < Cout) {
      float b = bias ? __ldg(bias + co) : 0.f;
#pragma unroll
      for (int r = 0; r < TR; ++r) {
        int64_t o = row0 + r;
        if (o < n_out) out[o * Cout + co] = acc[j][r] + b;
      }
    }
  }
}

extern "C" int pasco_conv_forward_simt(const float* in, const int32_t* nbr, int32_t K, int64_t n_out, int32_t Cin,
                                       int32_t Cout, const float* W, int32_t w_transposed, const int32_t* koff_map,
                                       const float* bias, float* out, pasco_stream_t s) {
  PASCO_CHECK_ARG(Cout <= 512 && Cin <= 2048, "pasco_conv_forward_simt: channel count too large");
  PASCO_CHECK_ARG(K <= 256, "pasco_conv_forward_simt: K too large");
  if (n_out == 0) return 0;
  cudaStream_t st = (cudaStream_t)s;
  KoffMap km;
  for (int k = 0; k < K; ++k) km.v[k] = koff_map ? koff_map[k] : k;
  int64_t nb = (n_out + TR - 1) / TR;
  size_t smem = (size_t)TR * Cin * sizeof(float);
  if (smem > 48 * 1024) cudaFuncSetAttribute(k_conv_simt, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_conv_simt<<<(unsigned)nb, 256, smem, st>>>(in, nbr, K, n_out, Cin, Cout, W, w_transposed, km, bias, out);
  PASCO_CHECK_LAUNCH("pasco_conv_forward_simt");
  return 0;
}

// dW[k][ci][co] = Σ_o in[nbr[k,o]][ci] * gout[o][co];  grid = (row chunks, K); each row chunk stores its partial dW in
// part[chunk][k][ci][co], and the host sums the chunks in order (identical from run to run, unlike float atomics)
constexpr int WG_ROWS = 2048;  // rows per block (at least)
constexpr int WG_TILE = 16;    // rows staged per iteration

__global__ void __launch_bounds__(256)
k_wgrad_simt(const float* __restrict__ in, const int32_t* __restrict__ nbr, int64_t n_out, int Cin, int Cout,
             const float* __restrict__ gout, int64_t rows_per_block, float* __restrict__ part) {
  extern __shared__ float sm[];  // sA[WG_TILE][Cin], sG[WG_TILE][Cout]
  float* sA = sm;
  float* sG = sm + WG_TILE * Cin;
  __shared__ int sIdx[WG_TILE];
  int k = blockIdx.y;
  int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  int64_t r1 = r0 + rows_per_block < n_out ? r0 + rows_per_block : n_out;
  int total = Cin * Cout;
  // each thread owns outputs e = threadIdx.x + j*256 (ci = e / Cout, co = e % Cout)
  constexpr int MAXE = 16;  // up to 4096 outputs per pass
  for (int e0 = 0; e0 < total; e0 += 256 * MAXE) {
    float acc[MAXE];
#pragma unroll
    for (int j = 0; j < MAXE; ++j) acc[j] = 0.f;
    for (int64_t rr = r0; rr < r1; rr += WG_TILE) {
      if (threadIdx.x < WG_TILE) {
        int64_t o = rr + threadIdx.x;
        sIdx[threadIdx.x] = o < r1 ? __ldg(nbr + (int64_t)k * n_out + o) : -1;
      }
      __syncthreads();
      int any = 0;
#pragma unroll
      for (int r = 0; r < WG_TILE; ++r) any |= (sIdx[r] >= 0);
      if (any) {
        for (int t = threadIdx.x; t < WG_TILE * Cin; t += 256) {
          int r = t / Cin, c = t - r * Cin;
          int src = sIdx[r];
          sA[t] = src >= 0 ? __ldg(in + (int64_t)src * Cin + c) : 0.f;
        }
        for (int t = threadIdx.x; t < WG_TILE * Cout; t += 256) {
          int r = t / Cout, c = t - r * Cout;
          sG[t] = (sIdx[r] >= 0) ? __ldg(gout + (rr + r) * Cout + c) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < MAXE; ++j) {
          int e = e0 + threadIdx.x + j * 256;
          if (e < total) {
            int ci = e / Cout, co = e - ci * Cout;
#pragma unroll
            for (int r = 0; r < WG_TILE; ++r) acc[j] = fmaf(sA[r * Cin + ci], sG[r * Cout + co], acc[j]);
          }
        }
      }
      __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < MAXE; ++j) {
      int e = e0 + threadIdx.x + j * 256;
      if (e < total) part[((int64_t)blockIdx.x * gridDim.y + k) * total + e] = acc[j];
    }
  }
}

namespace {
// row chunks of the weight gradient: WG_ROWS rows per block or more, at most about one full wave of blocks in all
// (8 resident 256-thread blocks per SM) and at most 64 MB of partial dW slots
int64_t wgrad_simt_chunks(int K, int64_t n_out, int Cin, int Cout) {
  int64_t chunks = (n_out + WG_ROWS - 1) / WG_ROWS;
  const int64_t wave = (8 * (int64_t)num_sms() + K - 1) / K;
  const int64_t mem = (64ll << 20) / ((int64_t)K * Cin * Cout * (int64_t)sizeof(float));
  if (chunks > wave) chunks = wave;
  if (chunks > mem) chunks = mem;
  if (chunks < 1) chunks = 1;
  const int64_t rows_per_block = (n_out + chunks - 1) / chunks;
  return (n_out + rows_per_block - 1) / rows_per_block;
}
}  // namespace

extern "C" int64_t pasco_conv_wgrad_simt_workspace_bytes(int32_t K, int64_t n_out, int32_t Cin, int32_t Cout) {
  if (n_out <= 0 || K <= 0 || Cin <= 0 || Cout <= 0) return 0;
  return wgrad_simt_chunks(K, n_out, Cin, Cout) * K * Cin * Cout * (int64_t)sizeof(float);
}

extern "C" int pasco_conv_wgrad_simt(const float* in, const int32_t* nbr, int32_t K, int64_t n_out, int32_t Cin,
                                     int32_t Cout, const float* gout, float* dW, float* workspace, int64_t workspace_bytes,
                                     pasco_stream_t s) {
  if (n_out == 0) return 0;
  size_t smem = (size_t)WG_TILE * (Cin + Cout) * sizeof(float);
  PASCO_CHECK_ARG(smem <= 200 * 1024, "pasco_conv_wgrad_simt: channels too large");
  if (smem > 48 * 1024) cudaFuncSetAttribute(k_wgrad_simt, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const int64_t chunks = wgrad_simt_chunks(K, n_out, Cin, Cout);
  const int64_t rows_per_block = (n_out + chunks - 1) / chunks;
  const int64_t n_w = (int64_t)K * Cin * Cout;
  PASCO_CHECK_ARG(workspace && workspace_bytes >= chunks * n_w * (int64_t)sizeof(float),
                  "pasco_conv_wgrad_simt: workspace smaller than pasco_conv_wgrad_simt_workspace_bytes");
  dim3 grid((unsigned)chunks, K);
  k_wgrad_simt<<<grid, 256, smem, (cudaStream_t)s>>>(in, nbr, n_out, Cin, Cout, gout, rows_per_block, workspace);
  k_add_partials<<<grid_for(n_w, 256), 256, 0, (cudaStream_t)s>>>(workspace, (int)chunks, n_w, n_w, dW);
  PASCO_CHECK_LAUNCH("pasco_conv_wgrad_simt");
  return 0;
}
