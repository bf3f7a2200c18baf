// Kernel launch helper: cudaLaunchKernelEx with a plain stream-ordered configuration.  No programmatic dependent launch:
// measured in one call (r2m) it changed nothing at batch 8 (95.05 / 96.21 ms with, 94.98 ms without) and cost 1-2 % at
// batch 1 (384^2 .. 1024^2: 8.99 / 10.65 / 15.68 / 26.71 ms with, 8.84 / 10.45 / 15.59 / 26.54 ms without) — inside a CUDA
// graph the launch gaps are already ~1 us and the early-resident CTAs only add scheduling work.
#pragma once
#include <cuda_runtime.h>

namespace gp {

template <typename... P, typename... A>
inline cudaError_t launch(void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, A&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<P>(args)...);
}

}  // namespace gp
