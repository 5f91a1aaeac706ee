// Image window of the any-size coders (DESIGN.md section 12): dst[p, i, j] = src[p, min(i, h_src - 1), min(j, w_src - 1)] on
// contiguous fp32 planes.  With a larger dst it is the encoder's pad (the image continued down and to the right by repeating its
// last row and column); with a smaller dst it is the decoder's crop.  A pure copy, so the result is exact.
//
// One block covers kCols consecutive columns of up to gridDim.y-strided dst rows; consecutive threads read and write consecutive
// j (coalesced for any row length, no vector width assumed).  Offsets are 64-bit: 16 x 3 x 3072 x 4032 floats pass 2^31 bytes.
#include "common.cuh"

namespace nic {

constexpr int kWinThreads = 256;
constexpr int kWinPerThread = 4;
constexpr int kCols = kWinThreads * kWinPerThread;

__global__ void __launch_bounds__(kWinThreads)
image_window_kernel(const float* __restrict__ src, int h_src, int w_src, float* __restrict__ dst, int h_dst, int w_dst, long rows) {
  const int j0 = blockIdx.x * kCols + threadIdx.x;
  for (long r = blockIdx.y; r < rows; r += gridDim.y) {
    const long p = r / h_dst;
    const int i = static_cast<int>(r - p * h_dst);
    const float* s = src + (p * h_src + min(i, h_src - 1)) * static_cast<long>(w_src);
    float* d = dst + r * static_cast<long>(w_dst);
#pragma unroll
    for (int k = 0; k < kWinPerThread; ++k) {
      const int j = j0 + k * kWinThreads;
      if (j < w_dst) d[j] = __ldg(s + min(j, w_src - 1));
    }
  }
}

}  // namespace nic

using namespace nic;

extern "C" {

int nic_image_window(const float* src, int32_t planes, int32_t h_src, int32_t w_src, float* dst, int32_t h_dst, int32_t w_dst,
                     void* stream) {
  if (planes < 1 || h_src < 1 || w_src < 1 || h_dst < 1 || w_dst < 1)
    return fail(NIC_E_BADSHAPE, "image_window: planes=%d src %dx%d dst %dx%d", planes, h_src, w_src, h_dst, w_dst);
  if (!src || !dst) return fail(NIC_E_BADSHAPE, "image_window: null pointer");
  if (int rc = nic_check_device()) return rc;
  const long rows = static_cast<long>(planes) * h_dst;
  const unsigned col_blocks = static_cast<unsigned>((w_dst + kCols - 1) / kCols);
  const unsigned row_blocks = static_cast<unsigned>(rows < 65535 ? rows : 65535);
  image_window_kernel<<<dim3(col_blocks, row_blocks), kWinThreads, 0, as_stream(stream)>>>(src, h_src, w_src, dst, h_dst, w_dst, rows);
  return check_launch("image_window_kernel");
}

}  // extern "C"
