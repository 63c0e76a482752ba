// Evaluation sweeps: the per-cell and per-row work behind PaSCo's SSC, panoptic-quality and uncertainty metrics
// (pasco/models/metrics.py:480-547,618-690 SSCMetrics, 98-166 UncertaintyMetrics.compute_ece_panop;
// pasco/loss/panoptic_quality.py:96-261 find_matched_segment / pq_compute_single_core).
//
// Integer counts go through shared-memory atomics (warp-aggregated over equal keys) and one global atomic per non-zero
// entry per CTA.  Float sums are run-to-run deterministic: every thread owns its own fp64 accumulators in shared memory,
// the CTA adds them in thread order into its own workspace slot, and k_add_partials_f64 adds the slots in CTA order.
#include "common.cuh"

namespace pasco {
namespace {

constexpr int kEvalThreads = 128;
constexpr int kMaxBins = 64;
constexpr int kMaxClasses = 64;
constexpr int kErrEvalId = 3;   // err_flag code: a class, label or segment id outside the table it indexes

// torchmetrics' binning: slot = bucketize(conf, bounds, right=True) - 1 = #{b : bounds[b] <= conf} - 1, over
// n_bins + 1 slots (conf == 1.0 has its own).  bounds = torch.linspace(0, 1, n_bins + 1) in fp32, passed by the caller.
__device__ __forceinline__ int calib_slot(float conf, const float* s_bounds, int n_bounds) {
  int s = 0;
  for (int b = 0; b < n_bounds; ++b) s += s_bounds[b] <= conf;
  return s > 0 ? s - 1 : 0;
}

// add `v` to the shared int counter `key`, once per distinct key in the warp
__device__ __forceinline__ void warp_count(int* s_cnt, int key, bool active, int v = 1) {
  const unsigned act = __ballot_sync(0xffffffffu, active);
  if (!active) return;
  const unsigned peers = __match_any_sync(act, key);
  const int leader = __ffs(peers) - 1;
  if ((int)(threadIdx.x & 31) == leader) atomicAdd(s_cnt + key, v * __popc(peers));
}

__device__ __forceinline__ void flush_counts(const int* s_cnt, int n, int64_t* out) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    int v = s_cnt[i];
    if (v) atomicAdd(reinterpret_cast<unsigned long long*>(out + i), (unsigned long long)(long long)v);
  }
}

// per-thread fp64 accumulators s_f[slot * blockDim + tid]  →  part[blockIdx * n_slots + slot], summed in thread order
__device__ __forceinline__ void store_partials(const double* s_f, int n_slots, double* part) {
  __syncthreads();
  for (int j = threadIdx.x; j < n_slots; j += blockDim.x) {
    double acc = 0.0;
    for (int t = 0; t < (int)blockDim.x; ++t) acc += s_f[j * blockDim.x + t];
    part[(int64_t)blockIdx.x * n_slots + j] = acc;
  }
}

__global__ void k_add_partials_f64(const double* __restrict__ part, int n_part, int n_slots, double* __restrict__ out) {
  for (int j = threadIdx.x; j < n_slots; j += blockDim.x) {
    double s = 0.0;
    for (int c = 0; c < n_part; ++c) s += part[(int64_t)c * n_slots + j];
    out[j] += s;
  }
}

// One sweep over the cells of a scene.
// Unknown cells (label 255) count nowhere: SSCMetrics.add_batch rewrites them to (0, 0) and then drops them through
// its `nonempty` mask (metrics.py:527-543, 640-680).
//   counts (+=): [K*K] confusion (target, prediction)
//                [2*NB] calibration count, [2*NB] calibration correct     (split 0: pred == 0, 1: pred != 0)
//   partial sums: [2*NB] Σ confidence, [2] Σ -log(p[label] + 1e-12)        (known cells, same split)
__global__ void __launch_bounds__(kEvalThreads) k_eval_ssc(const float* __restrict__ prob, const uint8_t* __restrict__ label,
                                                          int64_t cells, int K, const float* __restrict__ bounds, int n_bounds,
                                                          int64_t* __restrict__ counts, double* __restrict__ part,
                                                          int32_t* err_flag) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int NB = n_bounds;                        // calibration slots = n_bins + 1
  const int n_cnt = K * K + 4 * NB;
  const int n_f = 2 * NB + 2;
  double* s_f = reinterpret_cast<double*>(smem);
  int* s_cnt = reinterpret_cast<int*>(s_f + (size_t)n_f * blockDim.x);
  float* s_bounds = reinterpret_cast<float*>(s_cnt + n_cnt);
  for (int i = threadIdx.x; i < n_f * (int)blockDim.x; i += blockDim.x) s_f[i] = 0.0;
  for (int i = threadIdx.x; i < n_cnt; i += blockDim.x) s_cnt[i] = 0;
  for (int i = threadIdx.x; i < NB; i += blockDim.x) s_bounds[i] = bounds[i];
  __syncthreads();
  double* my_f = s_f + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t n_iter = (cells + stride - 1) / stride;             // every lane runs the same count (warp collectives)
  int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  for (int64_t it = 0; it < n_iter; ++it, c += stride) {
    const bool in = c < cells;
    int pred = 0, lab = 255;
    float best = 0.f, p_lab = 0.f;
    if (in) {
      lab = __ldg(label + c);
      if (lab != 255 && lab >= K) {
        atomicMax(err_flag, kErrEvalId);
        lab = 255;
      }
      best = -INFINITY;
      for (int k0 = 0; k0 < K; k0 += 8) {                             // 8 loads in flight per thread
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = k0 + j < K ? __ldg(prob + (int64_t)(k0 + j) * cells + c) : -INFINITY;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (v[j] > best) { best = v[j]; pred = k0 + j; }            // first maximum, as torch.argmax
          if (k0 + j == lab) p_lab = v[j];
        }
      }
    }
    const bool known = in && lab != 255;
    warp_count(s_cnt, lab * K + pred, known);
    const int split = pred != 0;
    const int slot = split * NB + calib_slot(best, s_bounds, NB);
    warp_count(s_cnt, K * K + slot, known);
    warp_count(s_cnt, K * K + 2 * NB + slot, known && pred == lab);
    if (known) {
      my_f[(size_t)slot * blockDim.x] += (double)best;
      my_f[(size_t)(2 * NB + split) * blockDim.x] += (double)(-logf(p_lab + 1e-12f));
    }
  }
  __syncthreads();
  flush_counts(s_cnt, n_cnt, counts);
  store_partials(s_f, n_f, part);
}

// Intersection table over known cells: table[(n_gt+1) * (n_pred+1)] (+=) with table[g][p] = #{known cells with GT id g
// and predicted id p}.  Cells without a row have predicted id 0: every known cell first counts as (g, 0), then each
// row moves its cell from (g, 0) to (g, p).
__global__ void __launch_bounds__(kEvalThreads) k_eval_pairs(const int32_t* __restrict__ pred_id,
                                                            const int64_t* __restrict__ row_cell, int64_t n_rows,
                                                            const int32_t* __restrict__ gt_id,
                                                            const uint8_t* __restrict__ label, int64_t cells, int n_gt,
                                                            int n_pred, int64_t* __restrict__ table, int32_t* err_flag) {
  extern __shared__ __align__(16) unsigned char smem[];
  int* s_cnt = reinterpret_cast<int*>(smem);
  const int W = n_pred + 1;
  const int n_cnt = (n_gt + 1) * W;
  for (int i = threadIdx.x; i < n_cnt; i += blockDim.x) s_cnt[i] = 0;
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t base = blockIdx.x * (int64_t)blockDim.x; base < cells; base += stride) {
    const int64_t c = base + threadIdx.x;
    bool ok = c < cells && __ldg(label + c) != 255;
    const int g = ok ? __ldg(gt_id + c) : 0;
    if (ok && (g < 0 || g > n_gt)) {
      atomicMax(err_flag, kErrEvalId);
      ok = false;
    }
    warp_count(s_cnt, ok ? g * W : 0, ok);
  }
  for (int64_t base = blockIdx.x * (int64_t)blockDim.x; base < n_rows; base += stride) {
    const int64_t r = base + threadIdx.x;
    bool ok = false;
    int g = 0, p = 0;
    if (r < n_rows) {
      const int64_t c = __ldg(row_cell + r);
      p = __ldg(pred_id + r);
      if (c < 0 || c >= cells || p < 0 || p > n_pred) {
        atomicMax(err_flag, kErrEvalId);
      } else if (__ldg(label + c) != 255) {
        g = __ldg(gt_id + c);
        ok = g >= 0 && g <= n_gt && p != 0;        // an out-of-range g was flagged by the cell sweep
      }
    }
    warp_count(s_cnt, g * W + p, ok);
    warp_count(s_cnt, g * W, ok, -1);
  }
  __syncthreads();
  flush_counts(s_cnt, n_cnt, table);
}

// Binned calibration of the rows' mask confidences (compute_ece_panop): a row is valid when its cell is known, its GT
// id is non-zero and its confidence is non-zero; it is correct when match[pred_id] (the GT id matched to its
// predicted segment, 0 = none) equals its GT id.
//   counts (+=): [NB] count, [NB] correct;   partial sums: [NB] Σ confidence
__global__ void __launch_bounds__(kEvalThreads) k_eval_calib(const float* __restrict__ conf,
                                                            const int32_t* __restrict__ pred_id,
                                                            const int64_t* __restrict__ row_cell, int64_t n_rows,
                                                            const int32_t* __restrict__ gt_id,
                                                            const uint8_t* __restrict__ label, int64_t cells,
                                                            const int32_t* __restrict__ match, int n_pred,
                                                            const float* __restrict__ bounds, int n_bounds,
                                                            int64_t* __restrict__ counts, double* __restrict__ part,
                                                            int32_t* err_flag) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int NB = n_bounds;
  double* s_f = reinterpret_cast<double*>(smem);
  int* s_cnt = reinterpret_cast<int*>(s_f + (size_t)NB * blockDim.x);
  float* s_bounds = reinterpret_cast<float*>(s_cnt + 2 * NB);
  for (int i = threadIdx.x; i < NB * (int)blockDim.x; i += blockDim.x) s_f[i] = 0.0;
  for (int i = threadIdx.x; i < 2 * NB; i += blockDim.x) s_cnt[i] = 0;
  for (int i = threadIdx.x; i < NB; i += blockDim.x) s_bounds[i] = bounds[i];
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t base = blockIdx.x * (int64_t)blockDim.x; base < n_rows; base += stride) {
    const int64_t r = base + threadIdx.x;
    bool valid = false, correct = false;
    float v = 0.f;
    if (r < n_rows) {
      const int64_t c = __ldg(row_cell + r);
      const int p = __ldg(pred_id + r);
      if (c < 0 || c >= cells || p < 0 || p > n_pred) {
        atomicMax(err_flag, kErrEvalId);
      } else if (__ldg(label + c) != 255) {
        const int g = __ldg(gt_id + c);
        v = __ldg(conf + r);
        valid = g != 0 && v != 0.f;
        correct = __ldg(match + p) == g;
      }
    }
    const int slot = calib_slot(v, s_bounds, NB);
    warp_count(s_cnt, slot, valid);
    warp_count(s_cnt, NB + slot, valid && correct);
    if (valid) s_f[(size_t)slot * blockDim.x + threadIdx.x] += (double)v;
  }
  __syncthreads();
  flush_counts(s_cnt, 2 * NB, counts);
  store_partials(s_f, NB, part);
}

int eval_grid(int64_t work) { return grid_for(work, kEvalThreads, 4); }

size_t ssc_smem(int K, int n_bounds) {
  return (size_t)(2 * n_bounds + 2) * kEvalThreads * sizeof(double) + (size_t)(K * K + 4 * n_bounds) * sizeof(int) +
         (size_t)n_bounds * sizeof(float);
}

size_t calib_smem(int n_bounds) {
  return (size_t)n_bounds * kEvalThreads * sizeof(double) + (size_t)2 * n_bounds * sizeof(int) +
         (size_t)n_bounds * sizeof(float);
}

int smem_optin() {
  int dev = 0, v = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  return v;
}

}  // namespace
}  // namespace pasco

using namespace pasco;

extern "C" int64_t pasco_eval_ssc_workspace_bytes(int64_t cells, int32_t n_bins) {
  return (int64_t)eval_grid(cells) * (2 * (n_bins + 1) + 2) * (int64_t)sizeof(double);
}

extern "C" int pasco_eval_ssc(const float* prob, const uint8_t* label, int64_t cells, int32_t K, const float* bounds,
                              int32_t n_bins, int64_t* counts, double* sums, double* workspace, int64_t workspace_bytes,
                              int32_t* err_flag, pasco_stream_t s) {
  PASCO_CHECK_ARG(K >= 1 && K <= kMaxClasses, "pasco_eval_ssc: K=%d outside [1, %d]", K, kMaxClasses);
  PASCO_CHECK_ARG(n_bins >= 1 && n_bins + 1 <= kMaxBins, "pasco_eval_ssc: n_bins=%d outside [1, %d]", n_bins, kMaxBins - 1);
  PASCO_CHECK_ARG(cells >= 1, "pasco_eval_ssc: no cells");
  PASCO_CHECK_ARG(err_flag != nullptr, "pasco_eval_ssc: err_flag is required");
  PASCO_CHECK_ARG(workspace_bytes >= pasco_eval_ssc_workspace_bytes(cells, n_bins),
                  "pasco_eval_ssc: workspace of %lld bytes, %lld needed", (long long)workspace_bytes,
                  (long long)pasco_eval_ssc_workspace_bytes(cells, n_bins));
  const int nb = n_bins + 1, grid = eval_grid(cells);
  const size_t smem = ssc_smem(K, nb);
  cudaStream_t st = (cudaStream_t)s;
  cudaFuncSetAttribute(k_eval_ssc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_eval_ssc<<<grid, kEvalThreads, smem, st>>>(prob, label, cells, K, bounds, nb, counts, workspace, err_flag);
  PASCO_CHECK_LAUNCH("k_eval_ssc");
  k_add_partials_f64<<<1, 64, 0, st>>>(workspace, grid, 2 * nb + 2, sums);
  PASCO_CHECK_LAUNCH("k_add_partials_f64");
  return 0;
}

extern "C" int pasco_eval_pairs(const int32_t* pred_id, const int64_t* row_cell, int64_t n_rows, const int32_t* gt_id,
                                const uint8_t* label, int64_t cells, int32_t n_gt, int32_t n_pred, int64_t* table,
                                int32_t* err_flag, pasco_stream_t s) {
  PASCO_CHECK_ARG(n_gt >= 0 && n_pred >= 0 && cells >= 1 && n_rows >= 0, "pasco_eval_pairs: bad sizes");
  PASCO_CHECK_ARG(err_flag != nullptr, "pasco_eval_pairs: err_flag is required");
  const size_t smem = (size_t)(n_gt + 1) * (n_pred + 1) * sizeof(int);
  PASCO_CHECK_ARG((int64_t)smem <= smem_optin(), "pasco_eval_pairs: a %d x %d table does not fit in shared memory",
                  n_gt + 1, n_pred + 1);
  cudaStream_t st = (cudaStream_t)s;
  cudaFuncSetAttribute(k_eval_pairs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_eval_pairs<<<eval_grid(cells > n_rows ? cells : n_rows), kEvalThreads, smem, st>>>(
      pred_id, row_cell, n_rows, gt_id, label, cells, n_gt, n_pred, table, err_flag);
  PASCO_CHECK_LAUNCH("k_eval_pairs");
  return 0;
}

extern "C" int64_t pasco_eval_calib_workspace_bytes(int64_t n_rows, int32_t n_bins) {
  return (int64_t)eval_grid(n_rows) * (n_bins + 1) * (int64_t)sizeof(double);
}

extern "C" int pasco_eval_calib(const float* conf, const int32_t* pred_id, const int64_t* row_cell, int64_t n_rows,
                                const int32_t* gt_id, const uint8_t* label, int64_t cells, const int32_t* match,
                                int32_t n_pred, const float* bounds, int32_t n_bins, int64_t* counts, double* sums,
                                double* workspace, int64_t workspace_bytes, int32_t* err_flag, pasco_stream_t s) {
  PASCO_CHECK_ARG(n_bins >= 1 && n_bins + 1 <= kMaxBins, "pasco_eval_calib: n_bins=%d outside [1, %d]", n_bins,
                  kMaxBins - 1);
  PASCO_CHECK_ARG(n_rows >= 0 && n_pred >= 0 && cells >= 1, "pasco_eval_calib: bad sizes");
  PASCO_CHECK_ARG(err_flag != nullptr, "pasco_eval_calib: err_flag is required");
  PASCO_CHECK_ARG(workspace_bytes >= pasco_eval_calib_workspace_bytes(n_rows, n_bins),
                  "pasco_eval_calib: workspace of %lld bytes, %lld needed", (long long)workspace_bytes,
                  (long long)pasco_eval_calib_workspace_bytes(n_rows, n_bins));
  const int nb = n_bins + 1, grid = eval_grid(n_rows);
  const size_t smem = calib_smem(nb);
  cudaStream_t st = (cudaStream_t)s;
  cudaFuncSetAttribute(k_eval_calib, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_eval_calib<<<grid, kEvalThreads, smem, st>>>(conf, pred_id, row_cell, n_rows, gt_id, label, cells, match, n_pred,
                                                 bounds, nb, counts, workspace, err_flag);
  PASCO_CHECK_LAUNCH("k_eval_calib");
  k_add_partials_f64<<<1, 64, 0, st>>>(workspace, grid, nb, sums);
  PASCO_CHECK_LAUNCH("k_add_partials_f64");
  return 0;
}
