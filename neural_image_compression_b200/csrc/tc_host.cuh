// Host-side helpers shared by the tensor-core translation units (conv_tc.cu defines them).
#pragma once
#include <cuda.h>
#include <stdlib.h>

#include <mutex>
#include <utility>
#include <vector>

#include "common.cuh"

namespace nic {

// cuTensorMapEncodeTiled wrappers (driver entry point fetched through the runtime; no -lcuda link dependency)
int encode_2d(CUtensorMap* m, const void* base, uint64_t inner, uint64_t rows, uint32_t box_inner, uint32_t box_rows);   // bf16
int encode_2d_ex(CUtensorMap* m, const void* base, int elem_bytes, uint64_t inner, uint64_t rows, uint32_t box_inner, uint32_t box_rows);
int encode_nhwc(CUtensorMap* m, const void* base, int n, int h, int w, int c, int box_w, int box_h, int stride, int elem_bytes);   // bf16 / f32
int encode_2d_c32(CUtensorMap* m, const void* base, uint64_t inner, uint64_t rows, uint32_t box_rows);   // bf16, 32-column SWIZZLE_64B boxes
int encode_nhwc_c32(CUtensorMap* m, const void* base, int n, int h, int w, int c, int box_w, int box_h, int stride = 1);   // bf16, SWIZZLE_64B
int encode_image_patch(CUtensorMap* m, const void* base, int n, int c, int h, int w, int box_w, int box_h);              // f32 NCHW
// one device int per process: the kernels' "a bounded wait expired" flag (nic_pipeline_status)
int* status_word();
extern void* g_trace_buffer;

// cudaFuncAttributeMaxDynamicSharedMemorySize once per (kernel, device): function attributes belong to a device's context, so a
// process that drives several GPUs needs it on each of them (a plain `static bool` was right only for one process per GPU)
inline int ensure_dyn_smem(const void* kernel, int bytes) {
  static std::mutex m;
  static std::vector<std::pair<const void*, int>> done;
  int dev = 0;
  if (int rc = check_cuda(cudaGetDevice(&dev), "cudaGetDevice")) return rc;
  std::lock_guard<std::mutex> g(m);
  for (const auto& e : done) if (e.first == kernel && e.second == dev) return 0;
  if (int rc = check_cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes), "cudaFuncSetAttribute")) return rc;
  done.emplace_back(kernel, dev);
  return 0;
}

// Launch with the programmatic-stream-serialization attribute when NIC_PDL=1 (see tc_primitives.cuh: pdl_wait /
// pdl_launch_dependents).  Measured inside the CUDA-graph replay of the forward pass: no difference beyond run-to-run noise
// (3.98 / 4.07 ms with, 4.07 / 3.97 ms without) - the graph already hides the launch latency and the next kernel cannot
// use an SM before the previous CTA has left it (one 220 KB CTA per SM) - so it is OFF by default.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl_cluster(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t st, int cluster, Args... args) {
  static const bool pdl = [] { const char* e = getenv("NIC_PDL"); return e && atoi(e) != 0; }();
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (cluster > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = cluster; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr; cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t st, Args... args) {
  return launch_pdl_cluster(kernel, grid, block, smem, st, 1, args...);
}

}  // namespace nic
