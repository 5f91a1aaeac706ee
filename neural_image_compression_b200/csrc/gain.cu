// Gain units of GainedCheckerboardHierarchical (DESIGN.md section 15): per-image gain vectors from the learned log-gain tables, the
// gained latent hand-off, the gain backward and the fold of the per-image gain gradients into the tables.
//
// Determinism: no float atomics anywhere.  The gain vectors are one expf per element.  nic_gain_bwd gives each (image, 32-channel
// group) to one block whose threads sum fixed pixel strides in double and combine in a fixed order, so the result does not depend
// on the batch or the launch.  The fold walks the images in order, one thread per (table, channel).
#include "common.cuh"

namespace nic {

constexpr int kQuantum = 1024;                     // quality codes are round(1024 q)

__device__ __forceinline__ void quality_split(int qc, int L, int* l0, int* l1, float* t) {
  int l = qc / kQuantum;
  l = l < 0 ? 0 : (l > L - 1 ? L - 1 : l);
  *l0 = l;
  *l1 = l + 1 < L ? l + 1 : L - 1;
  *t = static_cast<float>(qc - l * kQuantum) * (1.f / kQuantum);
}

__global__ void __launch_bounds__(256)
gain_vectors_kernel(const float* __restrict__ t0, const float* __restrict__ t1, const float* __restrict__ t2,
                    const float* __restrict__ t3, int L, int M, const int* __restrict__ q_code, int B, float* __restrict__ out) {
  const long total = 4L * B * M;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int m = static_cast<int>(i % M);
    const int b = static_cast<int>((i / M) % B);
    const int k = static_cast<int>(i / (static_cast<long>(M) * B));
    const float* tab = k == 0 ? t0 : (k == 1 ? t1 : (k == 2 ? t2 : t3));
    int l0, l1;
    float t;
    quality_split(q_code[b], L, &l0, &l1, &t);
    // no contraction into an fma: the interpolated log is the separately rounded (1 - t) a + t b of the reference
    const float s = __fadd_rn(__fmul_rn(1.f - t, tab[l0 * M + m]), __fmul_rn(t, tab[l1 * M + m]));
    out[i] = expf(s);
  }
}

__device__ __forceinline__ void store_nhwc(void* p, int dtype, long pix, int c, int ch, float v, int* lo_nonzero) {
  if (dtype == NIC_DT_BF16) {
    static_cast<__nv_bfloat16*>(p)[pix * c + ch] = __float2bfloat16_rn(v);
  } else if (dtype == NIC_DT_BF16X2) {
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const float lo = v - __bfloat162float(hi);
    static_cast<__nv_bfloat16*>(p)[pix * 2 * c + ch] = hi;
    static_cast<__nv_bfloat16*>(p)[pix * 2 * c + c + ch] = __float2bfloat16_rn(lo);
    if (lo_nonzero && lo != 0.f) *lo_nonzero = 1;
  } else {
    static_cast<float*>(p)[pix * c + ch] = v;
  }
}

// latent_handoff_kernel (conv_simt.cu) with a per-(image, channel) gain before the quantiser and an optional inverse gain on a
// second NHWC output of the quantised values
__global__ void __launch_bounds__(256)
latent_handoff_gain_kernel(const float* __restrict__ v, int n, int c, int h, int w, int qmode, const float* __restrict__ noise,
                           const float* __restrict__ gain, float* __restrict__ v_nchw, float* __restrict__ vin_nchw,
                           void* __restrict__ vin_nhwc, int out_dtype, int* __restrict__ lo_nonzero, void* __restrict__ v_src,
                           int src_dtype, const float* __restrict__ inv_gain, void* __restrict__ scaled, int scaled_dtype) {
  __shared__ float tile[32][33];
  __shared__ float tile_q[32][33];
  __shared__ float g_s[32], gi_s[32];
  const int hw = h * w;
  const int img = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, tyy = threadIdx.x >> 5;
  if (threadIdx.x < 32) {
    const int ch = c0 + threadIdx.x;
    g_s[threadIdx.x] = (gain && ch < c) ? gain[static_cast<long>(img) * c + ch] : 1.f;
    gi_s[threadIdx.x] = (inv_gain && ch < c) ? inv_gain[static_cast<long>(img) * c + ch] : 1.f;
  }
  __syncthreads();
  for (int r = tyy; r < 32; r += 8) {
    const int pix = p0 + r, ch = c0 + tx;
    float val = 0.f;
    if (pix < hw && ch < c) {
      val = v[(static_cast<long>(img) * hw + pix) * c + ch];
      if (gain) val *= g_s[tx];
      if (v_src) store_nhwc(v_src, src_dtype, static_cast<long>(img) * hw + pix, c, ch, val, nullptr);
    }
    tile[r][tx] = val;
  }
  __syncthreads();
  for (int r = tyy; r < 32; r += 8) {
    const int ch = c0 + r, pix = p0 + tx;
    if (pix < hw && ch < c) {
      const long o = (static_cast<long>(img) * c + ch) * hw + pix;
      const float val = tile[tx][r];
      float q = val;
      if (qmode == NIC_Q_ROUND) q = rintf(val);
      else if (qmode == NIC_Q_NOISE) q = val + noise[o];
      if (v_nchw) v_nchw[o] = val;
      if (vin_nchw) vin_nchw[o] = q;
      tile_q[tx][r] = q;
    }
  }
  __syncthreads();
  for (int r = tyy; r < 32; r += 8) {
    const int pix = p0 + r, ch = c0 + tx;
    if (pix < hw && ch < c) {
      const long p = static_cast<long>(img) * hw + pix;
      const float q = tile_q[r][tx];
      if (vin_nhwc) store_nhwc(vin_nhwc, out_dtype, p, c, ch, q, lo_nonzero);
      if (scaled) store_nhwc(scaled, scaled_dtype, p, c, ch, gi_s[tx] * q, nullptr);
    }
  }
}

// dst = factor (.) grad (+ dst; dst may alias grad, so neither is __restrict__), dgain = sum over pixels of grad (.) other, per (image, channel); one block per (32 channels, image)
__global__ void __launch_bounds__(256)
gain_bwd_kernel(const float* grad, const float* __restrict__ factor, const float* __restrict__ other, int c, long hw,
                float* dst, int accumulate, float* __restrict__ dgain) {
  __shared__ double red[8][32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int ch = blockIdx.x * 32 + tx, img = blockIdx.y;
  double acc = 0.0;
  if (ch < c) {
    const float f = factor ? factor[static_cast<long>(img) * c + ch] : 1.f;
    for (long pix = ty; pix < hw; pix += 8) {
      const long o = (static_cast<long>(img) * hw + pix) * c + ch;
      const float gv = grad[o];
      if (other) acc = fma(static_cast<double>(gv), static_cast<double>(other[o]), acc);
      if (dst) dst[o] = accumulate ? __fadd_rn(dst[o], __fmul_rn(f, gv)) : f * gv;     // no fma: the product is rounded first
    }
  }
  red[ty][tx] = acc;
  __syncthreads();
  if (ty == 0 && ch < c && dgain) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i][tx];
    dgain[static_cast<long>(img) * c + ch] = static_cast<float>(s);
  }
}

// d table[k][l] = sum over images b in order of the interpolation weight of row l times g (.) dg of image b
__global__ void __launch_bounds__(256)
gain_fold_kernel(const float* __restrict__ g, const float* __restrict__ dg, const int* __restrict__ q_code, int B, int L, int M,
                 float* __restrict__ dtab) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 4 * M) return;
  const int k = i / M, m = i % M;
  float* d = dtab + static_cast<long>(k) * L * M + m;
  for (int l = 0; l < L; ++l) d[l * M] = 0.f;
  for (int b = 0; b < B; ++b) {
    int l0, l1;
    float t;
    quality_split(q_code[b], L, &l0, &l1, &t);
    const long e = (static_cast<long>(k) * B + b) * M + m;
    const float s = g[e] * dg[e];
    d[l0 * M] += (1.f - t) * s;
    d[l1 * M] += t * s;
  }
}

static bool nhwc_dtype_ok(int dt) { return dt == NIC_DT_F32 || dt == NIC_DT_BF16 || dt == NIC_DT_BF16X2; }

}  // namespace nic

using namespace nic;

extern "C" {

int nic_gain_vectors(const float* y_log_gain, const float* y_log_inv_gain, const float* z_log_gain, const float* z_log_inv_gain,
                     int32_t L, int32_t M, const int32_t* q_code, int32_t B, float* out, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (L < 1 || M < 1 || B < 0) return fail(NIC_E_BADSHAPE, "gain_vectors: L=%d M=%d B=%d", L, M, B);
  if (B == 0) return NIC_OK;
  if (!y_log_gain || !y_log_inv_gain || !z_log_gain || !z_log_inv_gain || !q_code || !out)
    return fail(NIC_E_BADSHAPE, "gain_vectors: null pointer");
  const long total = 4L * B * M;
  const int blocks = static_cast<int>((total + 255) / 256 < kNumSMs * 8 ? (total + 255) / 256 : kNumSMs * 8);
  gain_vectors_kernel<<<blocks, 256, 0, as_stream(stream)>>>(y_log_gain, y_log_inv_gain, z_log_gain, z_log_inv_gain, L, M, q_code,
                                                             B, out);
  return check_launch("gain_vectors_kernel");
}

int nic_latent_handoff_gain(const float* v_nhwc, int32_t n, int32_t c, int32_t h, int32_t w, int32_t qmode, const float* noise_nchw,
                            const float* gain, float* v_nchw, float* v_in_nchw, void* v_in_nhwc, int32_t out_dtype,
                            int32_t* in_lo_nonzero, void* v_src_nhwc, int32_t src_dtype, const float* inv_gain, void* scaled_nhwc,
                            int32_t scaled_dtype, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || c < 1 || h < 1 || w < 1) return fail(NIC_E_BADSHAPE, "latent_handoff_gain: n=%d c=%d h=%d w=%d", n, c, h, w);
  if (qmode != NIC_Q_ROUND && qmode != NIC_Q_NOISE && qmode != NIC_Q_PASSTHRU)
    return fail(NIC_E_BADSHAPE, "latent_handoff_gain: qmode %d", qmode);
  if (qmode == NIC_Q_NOISE && !noise_nchw) return fail(NIC_E_BADSHAPE, "latent_handoff_gain: NIC_Q_NOISE needs noise");
  if (!nhwc_dtype_ok(out_dtype) || !nhwc_dtype_ok(src_dtype) || !nhwc_dtype_ok(scaled_dtype))
    return fail(NIC_E_BADSHAPE, "latent_handoff_gain: dtypes %d / %d / %d", out_dtype, src_dtype, scaled_dtype);
  if (n == 0) return NIC_OK;
  if (n > 65535) return fail(NIC_E_BADSHAPE, "latent_handoff_gain: n=%d > 65535", n);
  if (!v_nhwc) return fail(NIC_E_BADSHAPE, "latent_handoff_gain: null input");
  if (in_lo_nonzero) {
    if (int rc = check_cuda(cudaMemsetAsync(in_lo_nonzero, 0, sizeof(int32_t), as_stream(stream)), "cudaMemsetAsync")) return rc;
  }
  dim3 grid((h * w + 31) / 32, (c + 31) / 32, n);
  latent_handoff_gain_kernel<<<grid, 256, 0, as_stream(stream)>>>(v_nhwc, n, c, h, w, qmode, noise_nchw, gain, v_nchw, v_in_nchw,
                                                                  v_in_nhwc, out_dtype, in_lo_nonzero, v_src_nhwc, src_dtype,
                                                                  inv_gain, scaled_nhwc, scaled_dtype);
  return check_launch("latent_handoff_gain_kernel");
}

int nic_gain_bwd(const float* grad, const float* factor, const float* other, int32_t n, int32_t c, int64_t hw, float* dst,
                 int32_t accumulate, float* dgain, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || c < 1 || hw < 1 || n > 65535) return fail(NIC_E_BADSHAPE, "gain_bwd: n=%d c=%d hw=%ld", n, c, static_cast<long>(hw));
  if (n == 0) return NIC_OK;
  if (!grad || (dst && !factor) || (dgain && !other)) return fail(NIC_E_BADSHAPE, "gain_bwd: null pointer");
  gain_bwd_kernel<<<dim3((c + 31) / 32, n), 256, 0, as_stream(stream)>>>(grad, factor, other, c, hw, dst, accumulate, dgain);
  return check_launch("gain_bwd_kernel");
}

int nic_gain_fold(const float* gains, const float* d_gains, const int32_t* q_code, int32_t B, int32_t L, int32_t M, float* d_tables,
                  void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (B < 0 || L < 1 || M < 1) return fail(NIC_E_BADSHAPE, "gain_fold: B=%d L=%d M=%d", B, L, M);
  if (!d_tables || (B > 0 && (!gains || !d_gains || !q_code))) return fail(NIC_E_BADSHAPE, "gain_fold: null pointer");
  gain_fold_kernel<<<(4 * M + 255) / 256, 256, 0, as_stream(stream)>>>(gains, d_gains, q_code, B, L, M, d_tables);
  return check_launch("gain_fold_kernel");
}

}  // extern "C"
