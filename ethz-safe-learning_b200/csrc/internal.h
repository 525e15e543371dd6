// Host-side helpers shared between the translation units of libsimba_b200.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>

#include "../../include/simba_b200.h"

namespace simba {
// records the message behind simba_last_error() and returns `code`
int set_error(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
const simba_model_config_t* model_config(const simba_model_t* m);

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
