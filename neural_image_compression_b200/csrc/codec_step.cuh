// The wavefront order of the y decode (DESIGN.md section 9), shared by the coder (codec.cu) and the step-local entropy parameters
// (codec_params.cu).
#pragma once

namespace nic {

// Pixel rows of wavefront step t (pixel (i, j) is decoded at step 3 i + j): i in [i0, i0 + cnt), j = t - 3 i.
__host__ __device__ __forceinline__ void step_rows(int t, int h, int w, int& i0, int& cnt) {
  const int i1 = min(h - 1, t / 3);
  i0 = t - w + 1 > 0 ? (t - w + 3) / 3 : 0;
  cnt = i1 - i0 + 1;
}

}  // namespace nic
