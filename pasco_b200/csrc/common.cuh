// Shared helpers for libpasco_sm100 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/pasco_sm100.h"

namespace pasco {

void set_error(const char* fmt, ...);

#define PASCO_CHECK_ARG(cond, ...)            \
  do {                                        \
    if (!(cond)) {                            \
      ::pasco::set_error(__VA_ARGS__);        \
      return -2;                              \
    }                                         \
  } while (0)

#define PASCO_CHECK_LAUNCH(name)                                                         \
  do {                                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                \
    if (e__ != cudaSuccess) {                                                            \
      ::pasco::set_error("%s: CUDA launch failed: %s", name, cudaGetErrorString(e__));   \
      return -1;                                                                         \
    }                                                                                    \
  } while (0)

constexpr int kCoordBias = 32768;
constexpr uint64_t kEmptyKey = 0xFFFFFFFFFFFFFFFFull;

__host__ __device__ __forceinline__ uint64_t pack_key(int b, int x, int y, int z) {
  return ((uint64_t)(uint16_t)(b + kCoordBias) << 48) | ((uint64_t)(uint16_t)(x + kCoordBias) << 32) |
         ((uint64_t)(uint16_t)(y + kCoordBias) << 16) | (uint64_t)(uint16_t)(z + kCoordBias);
}

__device__ __forceinline__ uint32_t hash_key(uint64_t k) {  // murmur3 finaliser
  k ^= k >> 33;
  k *= 0xff51afd7ed558ccdull;
  k ^= k >> 33;
  k *= 0xc4ceb9fe1a85ec53ull;
  k ^= k >> 33;
  return (uint32_t)k;
}

__device__ __forceinline__ int table_find(const uint64_t* __restrict__ keys, const int32_t* __restrict__ vals,
                                          uint32_t mask, uint64_t key) {
  uint32_t slot = hash_key(key) & mask;
  while (true) {
    uint64_t k = __ldg(keys + slot);
    if (k == key) return __ldg(vals + slot);
    if (k == kEmptyKey) return -1;
    slot = (slot + 1) & mask;
  }
}

__host__ __device__ __forceinline__ int floor_div(int a, int s) {
  int q = a / s;
  return (a % s != 0 && ((a < 0) != (s < 0))) ? q - 1 : q;
}

inline int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// out[i] += Σ_{c < n_part} part[c * stride + i], summed in slot order: a reduction whose result does not depend on which
// CTA finished first (float atomics would make every run round differently).
static __global__ void k_add_partials(const float* __restrict__ part, int n_part, int64_t stride, int64_t n,
                                      float* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int c = 0; c < n_part; ++c) s += __ldg(part + (int64_t)c * stride + i);
    out[i] += s;
  }
}

inline int grid_for(int64_t work, int block, int waves = 8) {
  int64_t g = (work + block - 1) / block;
  int64_t cap = (int64_t)num_sms() * waves;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace pasco
