// Host-side helpers shared between the translation units of libsimba_b200.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstring>

#include "../../include/simba_b200.h"

namespace simba {
// records the message behind simba_last_error() and returns `code`
int set_error(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
const simba_model_config_t* model_config(const simba_model_t* m);

// Host side of the bf16 weight images. bf16_bits rounds to nearest even and keeps a NaN a (quiet) NaN.
inline uint16_t bf16_bits(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
inline float bf16_value(uint16_t h) {
  const uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
// (hi, lo) split of a bias, hi = bf16(v), lo = bf16(v - hi): the kernels multiply both by a constant 1
inline void bf16_split(float v, uint16_t& hi, uint16_t& lo) {
  hi = bf16_bits(v);
  lo = bf16_bits(v - bf16_value(hi));
}
// byte offset of element (n, k), 0 <= k < 64, in a K-major SWIZZLE_128B tile: row n is 128 bytes, and its
// 16-byte chunk c is stored at chunk c ^ (n & 7)
inline int64_t sw128_offset(int n, int k) { return (int64_t)n * 128 + ((k / 8) ^ (n & 7)) * 16 + (k % 8) * 2; }
// the tcgen05 rollout images pre-scale the raw-variance head by log2(e): the kernels evaluate softplus as
// ln2 * lg2(1 + ex2(x log2 e)) and get x log2 e out of the GEMM
constexpr float kLog2e = 1.4426950408889634f;

// Launches `kernel` on `grid` CTAs of `threads` with `smem` bytes of dynamic shared memory, in clusters of `cluster`
// CTAs (1: no cluster), as a programmatic dependent launch when `pdl` is set. The shared-memory limit is set on every
// launch: it is per device and per function, and these launches happen only at graph capture or in the non-graph
// entry points, never on the replayed hot path.
template <typename Kernel, typename... Args>
static cudaError_t launch_kernel(Kernel kernel, int grid, int threads, size_t smem, cudaStream_t stream, int cluster,
                                 bool pdl, Args... args) {
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (cluster > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = cluster;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}
}   // namespace simba

#define SIMBA_CUDA_TRY(expr)                                                                   \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return simba::set_error(SIMBA_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                  \
                              cudaGetErrorString(_e), __FILE__, __LINE__);                     \
  } while (0)
