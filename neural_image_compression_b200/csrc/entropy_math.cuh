// Scalar pieces of the entropy models shared by the likelihood kernels (likelihood.cu) and the entropy coder (codec.cu).
#pragma once
#include "common.cuh"

namespace nic {

__device__ __forceinline__ float softplus_torch(float x) {   // F.softplus defaults: beta 1, threshold 20
  return x > 20.f ? x : log1pf(expf(x));
}

// logits of the cumulative, EntropyModels.py:88-111, for one scalar and one channel's parameters
__device__ __forceinline__ float factorized_logit(float v, const float* __restrict__ q) {
  float h[3], g[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float t = q[i] * v + q[3 + i];
    h[i] = t + q[6 + i] * tanhf(t);
  }
#pragma unroll
  for (int l = 0; l < 2; ++l) {
    const float* w = q + 9 + l * 15;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      float t = w[i * 3 + 0] * h[0];
      t += w[i * 3 + 1] * h[1];
      t += w[i * 3 + 2] * h[2];
      t += w[9 + i];
      g[i] = t + w[12 + i] * tanhf(t);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) h[i] = g[i];
  }
  float t = q[39] * h[0];
  t += q[40] * h[1];
  t += q[41] * h[2];
  return t + q[42];
}

__device__ __forceinline__ float sigmoid_torch(float x) { return 1.0f / (1.0f + expf(-x)); }

}  // namespace nic
