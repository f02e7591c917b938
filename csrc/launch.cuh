// Launch helper: every kernel of the decode step is launched with Programmatic Dependent
// Launch (PDL) so that kernel N+1 becomes resident while kernel N drains.  Each kernel
// calls pdl_launch_dependents() right after its set-up and pdl_wait() before the first
// access to memory produced by an earlier kernel; a GEMM prefetches its weight tiles
// (which no kernel writes) into shared memory *before* pdl_wait().
#pragma once
#include <cuda_runtime.h>

#include <cstdlib>

namespace b2b {

inline int g_pdl_mode = -1;     // -1: read B2B_PDL from the environment on first use; 0 off; 1 on

inline bool pdl_enabled() {
  if (g_pdl_mode < 0) {
    const char* e = std::getenv("B2B_PDL");
    g_pdl_mode = (e && e[0] == '0') ? 0 : 1;
  }
  return g_pdl_mode == 1;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                 unsigned cluster_z, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster_z > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = 1;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = cluster_z;
    ++n;
  }
  if (pdl_enabled()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

}  // namespace b2b
