// Step-local entropy parameters of the scalable coder (DESIGN.md section 10): the masked context conv and the 1x1 stack of one or
// two heads, evaluated only at the pixels of one launch (every pixel for the encoder, one wavefront step for the decoder).
//
//   codec_params_kernel<L>   L = 0: context conv (12 live taps of the 5x5 mask 'A') -> phi
//                            L = 1: [phi | psi] -> 640, LeakyReLU(0.01)
//                            L = 2: 640 -> 640, LeakyReLU(0.01)
//                            L = 3: 640 -> (2m | 3Km), written into the NCHW raw tensor at the launch's pixels
//
// Determinism: an output element is computed by ONE thread as acc = bias; acc = fmaf(w_k, x_k, acc) for k = 0 .. cin - 1 in the
// order of the packed weight rows.  The chunking of k through shared memory only changes when inputs are loaded, not the order of
// the chain, and no sum is split across threads, so the bits at a pixel do not depend on the batch, on how many pixels share the
// launch, or on the grid.  The context conv reads only taps of earlier wavefront steps; taps outside the latent read 0.
#include "codec_step.cuh"
#include "common.cuh"

namespace nic {

constexpr int kHidden = 640;      // width of the entropy-parameter stack (ParametersModels.py)
constexpr int kPix = 8;           // pixels per CTA: every weight read from L2 feeds kPix FMAs
constexpr int kOuts = 128;        // output channels per CTA, one per thread
constexpr int kChunk = 64;        // inputs per pixel staged in shared memory per pass

struct ParamsArgs {
  nic_codec_head head[2];
  const float* psi;
  long n;                         // pixels of the launch (all images)
  int M, np, h, w, t, i0, cnt;    // np: raw planes per channel (2 or 3K)
};

template <int L>
__device__ __forceinline__ void layer_shape(const ParamsArgs& a, int m, int& cin, int& cout) {
  if (L == 0) { cin = 12 * m; cout = 2 * m; }
  else if (L == 1) { cin = 2 * m + 2 * a.M; cout = kHidden; }
  else if (L == 2) { cin = kHidden; cout = kHidden; }
  else { cin = kHidden; cout = a.np * m; }
}

// Input k of pixel q (image img, position (i, j)) of layer L.
template <int L>
__device__ __forceinline__ float gather(const ParamsArgs& a, const nic_codec_head& hd, int img, int i, int j, long q, int k) {
  const int m = hd.m;
  if (L == 0) {
    const int s = k / m, c = k - s * m;
    const int di = s < 10 ? s / 5 - 2 : 0, dj = s < 10 ? s % 5 - 2 : s - 12;
    const int ii = i + di, jj = j + dj;
    if (ii < 0 || jj < 0 || jj >= a.w) return 0.f;                       // ii <= i < h always
    return __ldg(hd.sym + ((static_cast<long>(img) * a.h + ii) * a.w + jj) * m + c);
  }
  const float* phi = hd.work;
  if (L == 1) {
    if (k < 2 * m) return phi[q * 2 * m + k];
    return __ldg(a.psi + ((static_cast<long>(img) * a.h + i) * a.w + j) * 2 * a.M + (k - 2 * m));
  }
  const float* hid = phi + a.n * 2 * m + (L == 3 ? a.n * kHidden : 0);
  return hid[q * kHidden + k];
}

template <int L>
__global__ void __launch_bounds__(kOuts) codec_params_kernel(const ParamsArgs a) {
  const nic_codec_head& hd = a.head[blockIdx.z];
  const int m = hd.m;
  int cin, cout;
  layer_shape<L>(a, m, cin, cout);
  if (static_cast<int>(blockIdx.y) * kOuts >= cout) return;           // the other head is wider
  const float* W = L == 0 ? hd.w_ctx : (L == 1 ? hd.w1 : (L == 2 ? hd.w2 : hd.w3));
  const float* bias = L == 0 ? hd.b_ctx : (L == 1 ? hd.b1 : (L == 2 ? hd.b2 : hd.b3));
  const int o = blockIdx.y * kOuts + threadIdx.x;
  const bool live = o < cout;
  const long q0 = static_cast<long>(blockIdx.x) * kPix;

  __shared__ int s_img[kPix], s_i[kPix], s_j[kPix];
  __shared__ __align__(16) float s_in[kPix][kChunk];
  if (threadIdx.x < kPix) {
    const long q = q0 + threadIdx.x;
    int img = -1, i = 0, j = 0;
    if (q < a.n) {
      if (a.t < 0) {
        const long hw = static_cast<long>(a.h) * a.w, r = q % hw;
        img = static_cast<int>(q / hw); i = static_cast<int>(r / a.w); j = static_cast<int>(r % a.w);
      } else {
        img = static_cast<int>(q / a.cnt); i = a.i0 + static_cast<int>(q % a.cnt); j = a.t - 3 * i;
      }
    }
    s_img[threadIdx.x] = img; s_i[threadIdx.x] = i; s_j[threadIdx.x] = j;
  }

  float acc[kPix];
  const float b0 = live ? __ldg(bias + o) : 0.f;
#pragma unroll
  for (int p = 0; p < kPix; ++p) acc[p] = b0;
  for (int k0 = 0; k0 < cin; k0 += kChunk) {
    const int kc = min(kChunk, cin - k0);
    const float* wp = W + static_cast<long>(k0) * cout + o;
    // A step launch holds few CTAs, so the chain is bound by the latency of its weight loads: a full chunk's loads are issued
    // together, before the inputs are staged, and are in flight while that happens.
    float wr[kChunk];
    if (live && kc == kChunk) {
#pragma unroll
      for (int u = 0; u < kChunk; ++u) wr[u] = __ldg(wp + static_cast<long>(u) * cout);
    }
    __syncthreads();                                                    // pixel coordinates written / previous chunk consumed
    for (int e = threadIdx.x; e < kPix * kChunk; e += kOuts) {
      const int p = e / kChunk, kk = e - p * kChunk;
      float v = 0.f;
      if (kk < kc && s_img[p] >= 0) v = gather<L>(a, hd, s_img[p], s_i[p], s_j[p], q0 + p, k0 + kk);
      s_in[p][kk] = v;
    }
    __syncthreads();
    if (!live) continue;
    if (kc == kChunk) {
#pragma unroll
      for (int u = 0; u < kChunk; u += 4) {
#pragma unroll
        for (int p = 0; p < kPix; ++p) {
          const float4 v = *reinterpret_cast<const float4*>(&s_in[p][u]);
          acc[p] = __fmaf_rn(wr[u], v.x, acc[p]);
          acc[p] = __fmaf_rn(wr[u + 1], v.y, acc[p]);
          acc[p] = __fmaf_rn(wr[u + 2], v.z, acc[p]);
          acc[p] = __fmaf_rn(wr[u + 3], v.w, acc[p]);
        }
      }
    } else {
      for (int kk = 0; kk < kc; ++kk) {
        const float wk = __ldg(wp + static_cast<long>(kk) * cout);
#pragma unroll
        for (int p = 0; p < kPix; ++p) acc[p] = __fmaf_rn(wk, s_in[p][kk], acc[p]);
      }
    }
  }
  if (!live) return;
#pragma unroll
  for (int p = 0; p < kPix; ++p) {
    if (s_img[p] < 0) continue;
    const long q = q0 + p;
    if (L == 0) {
      hd.work[q * 2 * m + o] = acc[p];
    } else if (L < 3) {
      const float v = acc[p] > 0.f ? acc[p] : acc[p] * 0.01f;
      hd.work[a.n * 2 * m + (L == 2 ? a.n * kHidden : 0) + q * kHidden + o] = v;
    } else {
      hd.raw[((static_cast<long>(s_img[p]) * cout + o) * a.h + s_i[p]) * a.w + s_j[p]] = acc[p];
    }
  }
}

}  // namespace nic

using namespace nic;

extern "C" int nic_codec_params(const nic_codec_head* heads, int32_t n_heads, const float* psi, int32_t b, int32_t M, int32_t k,
                                int32_t h, int32_t w, int32_t t, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (!heads || n_heads < 1 || n_heads > 2 || !psi) return fail(NIC_E_BADSHAPE, "codec_params: heads=%d psi=%p", n_heads, psi);
  if (b < 1 || M < 1 || k < 1 || k > 5 || h < 1 || w < 3)
    return fail(NIC_E_BADSHAPE, "codec_params: b=%d M=%d k=%d h=%d w=%d", b, M, k, h, w);
  if (t < -1 || t >= 3 * h + w - 3) return fail(NIC_E_BADSHAPE, "codec_params: step %d of %d", t, 3 * h + w - 3);
  ParamsArgs a{};
  a.psi = psi; a.M = M; a.np = k == 1 ? 2 : 3 * k; a.h = h; a.w = w; a.t = t;
  if (t >= 0) step_rows(t, h, w, a.i0, a.cnt);
  a.n = t < 0 ? static_cast<long>(b) * h * w : static_cast<long>(b) * a.cnt;
  int widest = kHidden;
  for (int i = 0; i < n_heads; ++i) {
    const nic_codec_head& hd = heads[i];
    if (hd.m < 1 || !hd.sym || !hd.w_ctx || !hd.b_ctx || !hd.w1 || !hd.b1 || !hd.w2 || !hd.b2 || !hd.w3 || !hd.b3 || !hd.raw || !hd.work)
      return fail(NIC_E_BADSHAPE, "codec_params: head %d: m=%d or a null pointer", i, hd.m);
    if (hd.work_floats < a.n * (2L * hd.m + 2L * kHidden))
      return fail(NIC_E_WORKSPACE, "codec_params: head %d: work of %lld floats, need %lld", i, static_cast<long long>(hd.work_floats),
                  static_cast<long long>(a.n * (2L * hd.m + 2L * kHidden)));
    a.head[i] = hd;
    widest = max(widest, max(2 * hd.m, a.np * hd.m));
  }
  const dim3 grid(static_cast<unsigned>((a.n + kPix - 1) / kPix), static_cast<unsigned>((widest + kOuts - 1) / kOuts), n_heads);
  cudaStream_t st = as_stream(stream);
  codec_params_kernel<0><<<grid, kOuts, 0, st>>>(a);
  if (int rc = check_launch("codec_params_kernel<0>")) return rc;
  codec_params_kernel<1><<<grid, kOuts, 0, st>>>(a);
  if (int rc = check_launch("codec_params_kernel<1>")) return rc;
  codec_params_kernel<2><<<grid, kOuts, 0, st>>>(a);
  if (int rc = check_launch("codec_params_kernel<2>")) return rc;
  codec_params_kernel<3><<<grid, kOuts, 0, st>>>(a);
  return check_launch("codec_params_kernel<3>");
}
