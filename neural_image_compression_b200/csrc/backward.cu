// Backward kernels of the training step (fp32, CUDA cores): what torch autograd derives from the reference forward
// (Models.py:49-106 + RateDistortionLoss.py:5-49, Trainer.py:85-86), written out by hand.
//
//   wgrad_kernel (+ wgrad_fold_kernel)   dLoss/dW of every Conv2d / ConvTranspose2d (Components.py:9-17, 38-46, 68-74, 98-104,
//                                        ContextModels.py:18-20 - all 25 taps, the reference masks the data not the graph -,
//                                        ParametersModels.py:29-35); split-K over pixels, fixed-order fold (deterministic)
//   colsum kernels                       bias gradients
//   lrelu_bwd / gdn_* kernels            LeakyReLU(0.01) and compressai GDN / IGDN backward incl. the LowerBound gradient rule
//   sse_bwd, layout / add helpers, adam  RateDistortionLoss.py:26-34 backward; torch.optim.Adam(lr) update (Main.ipynb:133)
//
// The data gradient of a conv is the adjoint conv and runs through nic_conv_fwd itself (the host builds the mirrored
// descriptor: Conv2d <-> ConvTranspose2d over the same weight tensor).
#include "conv_common.cuh"

namespace nic {

// wgrad_tc.cu
bool wgrad_tc_supported(const nic_conv_desc* d);
size_t wgrad_tc_workspace_bytes(const nic_conv_desc* d);
int wgrad_tc_launch(const nic_conv_desc* d, const void* x_pair, const void* g_pair, float* part, int* splits_out, cudaStream_t st);

int conv1x1_fp32(const float* x, long pixels, int cin, int cout, const float* w, const float* bias, float* y, int a_square,
                 int epilogue, cudaStream_t st);

// ---------------------------------------------------------------------------------------------------------------
// weight gradient
//   part[split][tap * cb + j][i] = sum over the split's pixels (n, y, x) of SMALL
//        BIG[n, y * s + dy_tap, x * s + dx_tap, j] * SMALL[n, y, x, i]
// Conv2d:          BIG = layer input,  SMALL = output gradient  -> dW[c_out = i][c_in = j][kh][kw]
// ConvTranspose2d: BIG = output gradient, SMALL = layer input   -> dW[c_in = i][c_out = j][kh][kw]
// (dy, dx) = (kh - pad, kw - pad), s = stride in both cases, and both reference layouts are [i][j][kh][kw].
// ---------------------------------------------------------------------------------------------------------------

constexpr int WBK = 16;      // pixels per K step
constexpr int WT = 128;      // tile edge (both operands)

struct WgradParams {
  const float* big; const float* small; float* part;
  int n, hs, ws, hb, wb, cb, cs;
  long bs_n, bs_c, bs_h, bs_w;
  int stride, ntaps, a_square;
  int8_t dy[kMaxTaps], dx[kMaxTaps];
  int P, pix_per_split;        // pixel counts fit 32 bits (checked by the host): the per-load index arithmetic stays 32-bit
  int mtiles_per_tap;          // vector path: ceil(cb / 128)
};

template <bool GATHER>
__global__ void __launch_bounds__(256, 2)
wgrad_kernel(const WgradParams p) {
  __shared__ __align__(16) float As[2][WBK][WT];
  __shared__ __align__(16) float Bs[2][WBK][WT];
  const int tid = threadIdx.x;
  const int p_begin = blockIdx.z * p.pix_per_split;
  int p_end = p_begin + p.pix_per_split;
  if (p_end > p.P) p_end = p.P;
  const int hw_s = p.hs * p.ws;
  const int n0 = blockIdx.y * WT;
  const int mtot = p.ntaps * p.cb;
  // M tile: vector path = 128 channels of one tap; gather path = 128 rows of the flattened (tap, channel) index
  int tap = 0, cb0 = 0;
  if (!GATHER) { tap = blockIdx.x / p.mtiles_per_tap; cb0 = (blockIdx.x % p.mtiles_per_tap) * WT; }
  const int mrow0 = GATHER ? blockIdx.x * WT : tap * p.cb + cb0;      // row of `part` of tile row 0
  const int mvalid = GATHER ? (mtot - mrow0 < WT ? mtot - mrow0 : WT) : (p.cb - cb0 < WT ? p.cb - cb0 : WT);

  // gather path: this thread always loads tile row tid % 128
  int g_dy = 0, g_dx = 0; long g_coff = 0; bool g_ok = false;
  if (GATHER) {
    const int m = mrow0 + (tid & (WT - 1));
    if (m < mtot) { const int t = m / p.cb; g_dy = p.dy[t]; g_dx = p.dx[t]; g_coff = static_cast<long>(m % p.cb) * p.bs_c; g_ok = true; }
  }
  const int v_dy = p.dy[tap], v_dx = p.dx[tap];

  float4 a4[2], b4[2];
  float ag[8];
  auto load_global = [&](int pk0) {
    if (GATHER) {
      // this thread's eight pixels are pk, pk + 2, ...: decode the first one, then step (x, y, img) instead of dividing again
      int pk = pk0 + (tid >> 7);
      int img = pk / hw_s, rem = pk - img * hw_s;
      int y = rem / p.ws, x = rem - y * p.ws;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float v = 0.f;
        if (g_ok && pk < p_end) {
          const int by = y * p.stride + g_dy, bx = x * p.stride + g_dx;
          if (by >= 0 && by < p.hb && bx >= 0 && bx < p.wb) v = __ldg(p.big + img * p.bs_n + by * p.bs_h + bx * p.bs_w + g_coff);
        }
        ag[j] = p.a_square ? v * v : v;
        pk += 2; x += 2;
        while (x >= p.ws) { x -= p.ws; if (++y >= p.hs) { y = 0; ++img; } }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int pk = pk0 + (tid >> 5) + 8 * j;
        const int c = cb0 + (tid & 31) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (pk < p_end && c < p.cb) {
          const int img = pk / hw_s, rem = pk - img * hw_s;
          const int y = rem / p.ws, x = rem - y * p.ws;
          const int by = y * p.stride + v_dy, bx = x * p.stride + v_dx;
          if (by >= 0 && by < p.hb && bx >= 0 && bx < p.wb)
            v = __ldg(reinterpret_cast<const float4*>(p.big + img * p.bs_n + by * p.bs_h + bx * p.bs_w + c));
        }
        if (p.a_square) { v.x *= v.x; v.y *= v.y; v.z *= v.z; v.w *= v.w; }
        a4[j] = v;
      }
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int pk = pk0 + (tid >> 5) + 8 * j;
      const int c = n0 + (tid & 31) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (pk < p_end && c < p.cs) v = __ldg(reinterpret_cast<const float4*>(p.small + static_cast<long>(pk) * p.cs + c));
      b4[j] = v;
    }
  };
  auto store_smem = [&](int buf) {
    if (GATHER) {
#pragma unroll
      for (int j = 0; j < 8; ++j) As[buf][(tid >> 7) + 2 * j][tid & (WT - 1)] = ag[j];
    } else {
#pragma unroll
      for (int j = 0; j < 2; ++j) *reinterpret_cast<float4*>(&As[buf][(tid >> 5) + 8 * j][(tid & 31) * 4]) = a4[j];
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) *reinterpret_cast<float4*>(&Bs[buf][(tid >> 5) + 8 * j][(tid & 31) * 4]) = b4[j];
  };

  const int ty = tid >> 4, tx = tid & 15;           // 16 x 16 threads, 8 x 8 micro-tile as two 4-wide halves per side
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  const int npix = p_end > p_begin ? p_end - p_begin : 0;
  const int steps = (npix + WBK - 1) / WBK;
  if (steps > 0) {
    load_global(p_begin);
    store_smem(0);
  }
  __syncthreads();
  for (int step = 0; step < steps; ++step) {
    const int buf = step & 1;
    if (step + 1 < steps) load_global(p_begin + (step + 1) * WBK);
#pragma unroll
    for (int k = 0; k < WBK; ++k) {
      float a[8], b[8];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 va = *reinterpret_cast<const float4*>(&As[buf][k][h * 64 + ty * 4]);
        a[h * 4 + 0] = va.x; a[h * 4 + 1] = va.y; a[h * 4 + 2] = va.z; a[h * 4 + 3] = va.w;
        const float4 vb = *reinterpret_cast<const float4*>(&Bs[buf][k][h * 64 + tx * 4]);
        b[h * 4 + 0] = vb.x; b[h * 4 + 1] = vb.y; b[h * 4 + 2] = vb.z; b[h * 4 + 3] = vb.w;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (step + 1 < steps) store_smem(buf ^ 1);
    __syncthreads();
  }

  float* out = p.part + static_cast<long>(blockIdx.z) * mtot * p.cs;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = (i >> 2) * 64 + ty * 4 + (i & 3);
    if (r >= mvalid) continue;
    float* row = out + static_cast<long>(mrow0 + r) * p.cs;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int c = n0 + h * 64 + tx * 4;
      if (c + 3 < p.cs) *reinterpret_cast<float4*>(row + c) = make_float4(acc[i][h * 4], acc[i][h * 4 + 1], acc[i][h * 4 + 2], acc[i][h * 4 + 3]);
      else
        for (int j = 0; j < 4; ++j) if (c + j < p.cs) row[c + j] = acc[i][h * 4 + j];
    }
  }
}

// dw[i][j][kh][kw] = sum_split part[split][tap * cb + j][i]   (fixed order)
__global__ void wgrad_fold_kernel(const float* __restrict__ part, int splits, int ntaps, int cb, int cs, int kh, int kw,
                                  TapTable tt, float* __restrict__ dw) {
  const long total = static_cast<long>(ntaps) * cb * cs;
  for (long e = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += static_cast<long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(e % cs);
    const int j = static_cast<int>((e / cs) % cb);
    const int t = static_cast<int>(e / (static_cast<long>(cs) * cb));
    float s = 0.f;
    for (int q = 0; q < splits; ++q) s += part[q * total + e];
    dw[((static_cast<long>(i) * cb + j) * kh + tt.kh[t]) * kw + tt.kw[t]] = s;
  }
}

// ---- bias gradient: column sums -------------------------------------------------------------------------------------
// NHWC rows: part[split][c]
__global__ void __launch_bounds__(256)
colsum_nhwc_kernel(const float* __restrict__ g, long rows, int c, long rows_per_split, float* __restrict__ part) {
  __shared__ float sm[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int ch = blockIdx.x * 32 + cx;
  const long r0 = static_cast<long>(blockIdx.y) * rows_per_split;
  long r1 = r0 + rows_per_split;
  if (r1 > rows) r1 = rows;
  float acc = 0.f;
  if (ch < c)
    for (long r = r0 + ry; r < r1; r += 8) acc += __ldg(g + r * c + ch);
  sm[ry][cx] = acc;
  __syncthreads();
  if (ry == 0 && ch < c) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += sm[i][cx];
    part[static_cast<long>(blockIdx.y) * c + ch] = s;
  }
}
// NCHW [b][c][hw]: part[split][c], split = (image, chunk of the plane)
__global__ void __launch_bounds__(256)
colsum_nchw_kernel(const float* __restrict__ g, int c, long hw, int chunks, float* __restrict__ part) {
  __shared__ float red[8];
  const int ch = blockIdx.x, img = blockIdx.y / chunks, chunk = blockIdx.y % chunks;
  const long per = (hw + chunks - 1) / chunks;
  const long i0 = chunk * per;
  long i1 = i0 + per;
  if (i1 > hw) i1 = hw;
  const float* src = g + (static_cast<long>(img) * c + ch) * hw;
  float acc = 0.f;
  for (long i = i0 + threadIdx.x; i < i1; i += 256) acc += __ldg(src + i);
  const float tot = block_sum_256(acc, red);
  if (threadIdx.x == 0) part[static_cast<long>(blockIdx.y) * c + ch] = tot;
}
__global__ void colsum_fold_kernel(const float* __restrict__ part, int splits, int c, float* __restrict__ out) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  float s = 0.f;
  for (int q = 0; q < splits; ++q) s += part[static_cast<long>(q) * c + ch];
  out[ch] = s;
}

// ---- elementwise ----------------------------------------------------------------------------------------------------------
// LeakyReLU(0.01) backward from the saved OUTPUT (slope > 0: sign(out) = sign(pre-activation)); may run in place on g
__global__ void lrelu_bwd_kernel(const float* __restrict__ g, const float* __restrict__ out, float* __restrict__ gp, long n) {
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x)
    gp[i] = out[i] > 0.f ? g[i] : g[i] * 0.01f;
}

// GDN:  out = u n^-1/2 : t = -1/2 g u n^-3/2, s = g n^-1/2;   IGDN: out = u n^1/2 : t = 1/2 g u n^-1/2, s = g n^1/2
// writes t and du = s (the 2 u (gamma^T t) term is added by gdn_bwd_finish_kernel)
__global__ void gdn_bwd_prep_kernel(const float* __restrict__ g, const float* __restrict__ u, const float* __restrict__ nrm,
                                    int inverse, float* __restrict__ t, float* __restrict__ du, long n) {
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const float gv = g[i], uv = u[i], nv = nrm[i];
    const float rs = 1.0f / sqrtf(nv);
    if (inverse) { t[i] = 0.5f * gv * uv * rs; du[i] = gv * sqrtf(nv); }
    else { t[i] = -0.5f * gv * uv * rs / nv; du[i] = gv * rs; }
  }
}
// out = u * rsqrt(norm)  (inverse: u * sqrt(norm)) - the GDN once its norm = beta + gamma . u^2 is known
__global__ void gdn_apply_kernel(const float* __restrict__ u, const float* __restrict__ nrm, int inverse, float* __restrict__ out, long n) {
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const float nv = nrm[i];
    out[i] = inverse ? u[i] * sqrtf(nv) : u[i] * (1.0f / sqrtf(nv));
  }
}
// the same followed by the residual sum of the 3x3 blocks (Layers.py:58-60, 85-87): out = gdn(u) + addend.  The product is rounded
// before the sum (no FMA contraction): bit-identical to nic_gdn_apply followed by nic_add_inplace, one pass over memory instead of two
__global__ void gdn_apply_add_kernel(const float* __restrict__ u, const float* __restrict__ nrm, const float* __restrict__ addend, int inverse,
                                     float* __restrict__ out, long n) {
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const float nv = nrm[i];
    const float y = inverse ? __fmul_rn(u[i], sqrtf(nv)) : __fmul_rn(u[i], 1.0f / sqrtf(nv));
    out[i] = __fadd_rn(y, addend[i]);
  }
}
__global__ void gdn_bwd_finish_kernel(const float* __restrict__ u, const float* __restrict__ r, float* __restrict__ du, long n) {
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x)
    du[i] = fmaf(2.0f * u[i], r[i], du[i]);
}
// compressai NonNegativeParametrizer: eff = max(raw, bound)^2 - pedestal; natural [i][j] and transposed [j][i] gamma
__global__ void gdn_reparam_kernel(int c, float beta_bound, float gamma_bound, float pedestal, const float* __restrict__ beta,
                                   const float* __restrict__ gamma, float* __restrict__ beta_eff, float* __restrict__ gamma_eff,
                                   float* __restrict__ gamma_t) {
  const int total = c * c;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int row = i / c, col = i % c;
    const float g = fmaxf(gamma[i], gamma_bound);
    const float e = g * g - pedestal;
    gamma_eff[i] = e;
    gamma_t[col * c + row] = e;
    if (i < c) { const float b = fmaxf(beta[i], beta_bound); beta_eff[i] = b * b - pedestal; }
  }
}
// chain rule through eff = LowerBound(raw)^2 - pedestal: G = d_eff * 2 max(raw, bound); passes iff raw >= bound or G < 0
__global__ void gdn_reparam_bwd_kernel(int c, float beta_bound, float gamma_bound, const float* __restrict__ beta,
                                       const float* __restrict__ gamma, const float* __restrict__ dbeta_eff,
                                       const float* __restrict__ dgamma_eff, float* __restrict__ dbeta, float* __restrict__ dgamma) {
  const int total = c * c;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const float raw = gamma[i];
    const float G = dgamma_eff[i] * 2.0f * fmaxf(raw, gamma_bound);
    dgamma[i] = (raw >= gamma_bound || G < 0.f) ? G : 0.f;
    if (i < c) {
      const float rb = beta[i];
      const float Gb = dbeta_eff[i] * 2.0f * fmaxf(rb, beta_bound);
      dbeta[i] = (rb >= beta_bound || Gb < 0.f) ? Gb : 0.f;
    }
  }
}

__global__ void sse_bwd_kernel(const float* __restrict__ x_hat, const float* __restrict__ x, float coef, float* __restrict__ g, long n) {
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x)
    g[i] = coef * (x_hat[i] - x[i]);
}
__global__ void sse_bwd_per_image_kernel(const float* __restrict__ x_hat, const float* __restrict__ x, const float* __restrict__ coef,
                                         long per_image, float* __restrict__ g, long n) {
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x)
    g[i] = coef[i / per_image] * (x_hat[i] - x[i]);
}
__global__ void add_inplace_kernel(float* __restrict__ dst, const float* __restrict__ src, long n) {
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x)
    dst[i] += src[i];
}
// [n][c][hw] <-> [n][hw][c] through 32 x 32 shared-memory tiles; accumulate: dst += transposed(src)
__global__ void __launch_bounds__(256)
layout_convert_kernel(const float* __restrict__ src, float* __restrict__ dst, int c, int hw, int to_nhwc, int accumulate) {
  __shared__ float tile[32][33];
  const int img = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long base = static_cast<long>(img) * c * hw;
  for (int r = ty; r < 32; r += 8) {
    // read coalesced along the source's fast axis
    const int ch = to_nhwc ? c0 + r : c0 + tx, pix = to_nhwc ? p0 + tx : p0 + r;
    float v = 0.f;
    if (ch < c && pix < hw) v = to_nhwc ? src[base + static_cast<long>(ch) * hw + pix] : src[base + static_cast<long>(pix) * c + ch];
    tile[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int ch = to_nhwc ? c0 + tx : c0 + r, pix = to_nhwc ? p0 + r : p0 + tx;
    if (ch < c && pix < hw) {
      const long o = to_nhwc ? base + static_cast<long>(pix) * c + ch : base + static_cast<long>(ch) * hw + pix;
      const float v = tile[tx][r];
      dst[o] = accumulate ? dst[o] + v : v;
    }
  }
}

// f32 [rows][c] -> bf16 pairs [rows][2c] = [hi(c) | lo(c)] (NIC_DT_BF16X2): feeds fp32 activations / gradients to the bf16x3 convs
__global__ void __launch_bounds__(256)
to_pair_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long rows, int c, int square) {
  const int c4 = c >> 2;
  const long total = rows * c4;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const long r = i / c4;
    const int q = static_cast<int>(i - r * c4) * 4;
    float4 v = __ldg(reinterpret_cast<const float4*>(src + r * c + q));
    if (square) { v.x *= v.x; v.y *= v.y; v.z *= v.z; v.w *= v.w; }
    const __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
    const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
    const __nv_bfloat162 l0 = __floats2bfloat162_rn(v.x - f0.x, v.y - f0.y), l1 = __floats2bfloat162_rn(v.z - f1.x, v.w - f1.y);
    __nv_bfloat16* d = dst + r * 2 * c + q;
    uint2 hi, lo;
    hi.x = *reinterpret_cast<const uint32_t*>(&h0); hi.y = *reinterpret_cast<const uint32_t*>(&h1);
    lo.x = *reinterpret_cast<const uint32_t*>(&l0); lo.y = *reinterpret_cast<const uint32_t*>(&l1);
    *reinterpret_cast<uint2*>(d) = hi;
    *reinterpret_cast<uint2*>(d + c) = lo;
  }
}

// torch.optim.Adam (no weight decay, no amsgrad): m, v moments; t = step count after the increment
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long n,
                            float beta1, float beta2, float step_size, float sqrt_bc2, float eps) {
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const float gv = g[i];
    const float mv = m[i] + (gv - m[i]) * (1.0f - beta1);          // exp_avg.lerp_(grad, 1 - beta1)
    const float vv = v[i] * beta2 + (1.0f - beta2) * gv * gv;      // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    m[i] = mv; v[i] = vv;
    const float denom = sqrtf(vv) / sqrt_bc2 + eps;
    p[i] -= step_size * (mv / denom);
  }
}

// many tensors in ONE launch: the pointers travel as kernel arguments (no table upload, no host synchronisation);
// block b works on chunk (b - blk_start[t]) of the tensor t whose block range contains b
constexpr int kAdamMaxTensors = 64;
constexpr int kAdamChunk = 256 * 16;
struct AdamArgs {
  float* p[kAdamMaxTensors]; const float* g[kAdamMaxTensors]; float* m[kAdamMaxTensors]; float* v[kAdamMaxTensors];
  long n[kAdamMaxTensors];
  int blk_start[kAdamMaxTensors + 1];
  int count;
};
__global__ void counter_increment_kernel(int* c) { if (threadIdx.x == 0 && blockIdx.x == 0) *c += 1; }

// step_dev != NULL: the step count lives on the device (a CUDA-graph replay of the launch must see a new t every time)
__global__ void __launch_bounds__(256)
adam_multi_kernel(const __grid_constant__ AdamArgs a, float beta1, float beta2, float lr, float step_size, float sqrt_bc2, float eps,
                  const int* __restrict__ step_dev, const float* __restrict__ lr_dev, float gscale) {
  if (lr_dev) lr = *lr_dev;                  // learning rate on the device: a scheduler's change reaches a CUDA-graph replay
  if (step_dev || lr_dev) {
    const int t = step_dev ? *step_dev : 0;
    if (!step_dev) {                           // host step count: only the learning rate is re-read
      step_size = lr * step_size;              // step_size carries 1 / bc1 in this case (see nic_adam_multi_step_ex)
    } else {
    step_size = static_cast<float>(static_cast<double>(lr) / (1.0 - pow(static_cast<double>(beta1), t)));
    sqrt_bc2 = static_cast<float>(sqrt(1.0 - pow(static_cast<double>(beta2), t)));
    }
  }
  int lo = 0, hi = a.count;                                   // largest t with blk_start[t] <= blockIdx.x
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (a.blk_start[mid] <= static_cast<int>(blockIdx.x)) lo = mid; else hi = mid; }
  const int t = lo;
  float* __restrict__ p = a.p[t]; const float* __restrict__ g = a.g[t]; float* __restrict__ m = a.m[t]; float* __restrict__ v = a.v[t];
  const long n = a.n[t];
  const long i0 = static_cast<long>(blockIdx.x - a.blk_start[t]) * kAdamChunk;
  long i1 = i0 + kAdamChunk;
  if (i1 > n) i1 = n;
  for (long i = i0 + threadIdx.x; i < i1; i += 256) {
    const float gv = g[i] * gscale;                             // gscale = 1 / world: the all-reduced SUM becomes the mean here
    const float mv = m[i] + (gv - m[i]) * (1.0f - beta1);
    const float vv = v[i] * beta2 + (1.0f - beta2) * gv * gv;
    m[i] = mv; v[i] = vv;
    p[i] -= step_size * (mv / (sqrtf(vv) / sqrt_bc2 + eps));
  }
}

static inline int ew_blocks(long n) {
  long b = (n + 255) / 256;
  const long cap = static_cast<long>(kNumSMs) * 8;
  return static_cast<int>(b < 1 ? 1 : (b > cap ? cap : b));
}

static void big_strides(int layout, long c, long h, long w, long* sn, long* sc, long* sh, long* sw) {
  if (layout == NIC_LAYOUT_NCHW) { *sn = c * h * w; *sc = h * w; *sh = w; *sw = 1; }
  else { *sn = h * w * c; *sh = w * c; *sw = c; *sc = 1; }
}

struct WgradPlan { int splits; long pix_per_split; bool gather; int mtiles, ntiles, mtiles_per_tap; long P; int ntaps; };

static WgradPlan plan_wgrad(int ntaps, int cb, int cs, long P, bool gather) {
  WgradPlan w{};
  w.gather = gather; w.P = P; w.ntaps = ntaps;
  w.mtiles_per_tap = (cb + WT - 1) / WT;
  w.mtiles = gather ? (ntaps * cb + WT - 1) / WT : ntaps * w.mtiles_per_tap;
  w.ntiles = (cs + WT - 1) / WT;
  const long base = static_cast<long>(w.mtiles) * w.ntiles;
  long splits = (4L * kNumSMs + base - 1) / base;                  // about two waves of 2 CTAs / SM
  const long max_splits = (P + 255) / 256;                           // >= 256 pixels per split
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  if (splits > 128) splits = 128;                                  // the fold walks the splits serially: keep it short
  long per = (P + splits - 1) / splits;
  per = (per + WBK - 1) / WBK * WBK;
  w.pix_per_split = per;
  w.splits = static_cast<int>((P + per - 1) / per);
  if (w.splits < 1) w.splits = 1;
  return w;
}

// big / small of the forward conv `d`
struct WgradShape { int cb, cs, hb, wb, hs, ws, big_layout; bool big_is_input; };
static WgradShape wgrad_shape(const nic_conv_desc* d) {
  WgradShape s{};
  if (!d->transposed) { s.big_is_input = true; s.cb = d->c_in; s.hb = d->h_in; s.wb = d->w_in; s.cs = d->c_out; s.hs = d->h_out; s.ws = d->w_out; s.big_layout = d->in_layout; }
  else { s.big_is_input = false; s.cb = d->c_out; s.hb = d->h_out; s.wb = d->w_out; s.cs = d->c_in; s.hs = d->h_in; s.ws = d->w_in; s.big_layout = d->out_layout; }
  return s;
}

static size_t align256(size_t v) { return (v + 255) / 256 * 256; }

static int run_wgrad(const float* big, const float* small, int n, const WgradShape& s, int stride, int pad, int kh, int kw, int a_square,
                     float* dw, float* part, cudaStream_t st) {
  nic_conv_desc full{};                 // all kh*kw taps of a plain conv: positions (kh, kw), offsets (kh - pad, kw - pad)
  full.n = 1; full.c_in = full.c_out = 1; full.kh = kh; full.kw = kw; full.stride = 1; full.pad = pad;
  full.h_in = full.w_in = 64; full.h_out = full.w_out = 64 + 2 * pad - kh + 1;
  TapTable tt;
  if (int rc = build_tap_table(&full, &tt)) return rc;
  const long P = static_cast<long>(n) * s.hs * s.ws;
  long bn, bc, bh, bw;
  big_strides(s.big_layout, s.cb, s.hb, s.wb, &bn, &bc, &bh, &bw);
  const bool gather = (bc != 1) || (s.cb % 4 != 0);
  if (s.cs % 4 != 0) return fail(NIC_E_UNSUPPORTED, "wgrad: the small operand needs c %% 4 == 0 (got %d)", s.cs);
  if ((reinterpret_cast<uintptr_t>(small) & 15) || (!gather && (reinterpret_cast<uintptr_t>(big) & 15)))
    return fail(NIC_E_BADALIGN, "wgrad: tensors must be 16-byte aligned");
  const WgradPlan w = plan_wgrad(tt.ntaps, s.cb, s.cs, P, gather);
  WgradParams p{};
  p.big = big; p.small = small; p.part = part;
  p.n = n; p.hs = s.hs; p.ws = s.ws; p.hb = s.hb; p.wb = s.wb; p.cb = s.cb; p.cs = s.cs;
  p.bs_n = bn; p.bs_c = bc; p.bs_h = bh; p.bs_w = bw;
  p.stride = stride; p.ntaps = tt.ntaps; p.a_square = a_square;
  for (int t = 0; t < tt.ntaps; ++t) { p.dy[t] = tt.dy[t]; p.dx[t] = tt.dx[t]; }
  if (P + w.pix_per_split > 0x7fffffffL) return fail(NIC_E_BADSHAPE, "wgrad: %ld pixels", P);
  p.P = static_cast<int>(P); p.pix_per_split = static_cast<int>(w.pix_per_split); p.mtiles_per_tap = w.mtiles_per_tap;
  dim3 grid(w.mtiles, w.ntiles, w.splits);
  if (gather) wgrad_kernel<true><<<grid, 256, 0, st>>>(p);
  else wgrad_kernel<false><<<grid, 256, 0, st>>>(p);
  if (int rc = check_launch("wgrad_kernel")) return rc;
  const long total = static_cast<long>(tt.ntaps) * s.cb * s.cs;
  wgrad_fold_kernel<<<ew_blocks(total), 256, 0, st>>>(part, w.splits, tt.ntaps, s.cb, s.cs, kh, kw, tt, dw);
  return check_launch("wgrad_fold_kernel");
}

static size_t wgrad_part_bytes(int ntaps, const WgradShape& s, int n, bool gather) {
  const WgradPlan w = plan_wgrad(ntaps, s.cb, s.cs, static_cast<long>(n) * s.hs * s.ws, gather);
  return align256(static_cast<size_t>(w.splits) * ntaps * s.cb * s.cs * sizeof(float));
}

constexpr int kColsumSplits = 64;
static int run_colsum_nhwc(const float* g, long rows, int c, float* out, float* part, cudaStream_t st) {
  long per = (rows + kColsumSplits - 1) / kColsumSplits;
  if (per < 8) per = 8;
  const int splits = static_cast<int>((rows + per - 1) / per);
  colsum_nhwc_kernel<<<dim3((c + 31) / 32, splits), 256, 0, st>>>(g, rows, c, per, part);
  if (int rc = check_launch("colsum_nhwc_kernel")) return rc;
  colsum_fold_kernel<<<(c + 127) / 128, 128, 0, st>>>(part, splits, c, out);
  return check_launch("colsum_fold_kernel");
}
static int run_colsum_nchw(const float* g, int n, int c, long hw, float* out, float* part, cudaStream_t st) {
  int chunks = kColsumSplits / (n < 1 ? 1 : n);
  if (chunks < 1) chunks = 1;
  while (chunks > 1 && hw / chunks < 256) chunks >>= 1;
  if (static_cast<long>(n) * chunks > 4096) return fail(NIC_E_BADSHAPE, "colsum: batch %d too large", n);
  colsum_nchw_kernel<<<dim3(c, n * chunks), 256, 0, st>>>(g, c, hw, chunks, part);
  if (int rc = check_launch("colsum_nchw_kernel")) return rc;
  colsum_fold_kernel<<<(c + 127) / 128, 128, 0, st>>>(part, n * chunks, c, out);
  return check_launch("colsum_fold_kernel");
}
static size_t colsum_part_bytes(int n, int c) {
  const int s = (n > kColsumSplits ? n : kColsumSplits);
  return align256(static_cast<size_t>(s) * c * sizeof(float));
}

}  // namespace nic

using namespace nic;

extern "C" {

size_t nic_conv_wgrad_workspace_bytes(const nic_conv_desc* d) {
  if (!d || validate_conv_desc(d)) return 0;
  const WgradShape s = wgrad_shape(d);
  const bool gather = (s.big_layout == NIC_LAYOUT_NCHW) || (s.cb % 4 != 0);
  return wgrad_part_bytes(d->kh * d->kw, s, d->n, gather) + colsum_part_bytes(d->n, d->c_out) + 256;
}

int nic_conv_wgrad(const nic_conv_desc* d, const float* x, const float* g, float* dw, float* db,
                   void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (int rc = validate_conv_desc(d)) return rc;
  if (!x || !g || !dw) return fail(NIC_E_BADSHAPE, "conv_wgrad: null pointer");
  if (d->in_dtype != NIC_DT_F32 || d->out_dtype != NIC_DT_F32) return fail(NIC_E_UNSUPPORTED, "conv_wgrad: f32 tensors only");
  if (d->out_c_total != 0) return fail(NIC_E_UNSUPPORTED, "conv_wgrad: channel windows are not supported (pass a contiguous gradient)");
  const size_t need = nic_conv_wgrad_workspace_bytes(d);
  if (!workspace || workspace_bytes < need) return fail(NIC_E_WORKSPACE, "conv_wgrad: workspace %zu < %zu bytes", workspace_bytes, need);
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(NIC_E_BADALIGN, "conv_wgrad: workspace must be 256-byte aligned");
  cudaStream_t st = as_stream(stream);
  const WgradShape s = wgrad_shape(d);
  const float* big = s.big_is_input ? x : g;
  const float* small = s.big_is_input ? g : x;
  const int small_layout = s.big_is_input ? d->out_layout : d->in_layout;
  if (small_layout != NIC_LAYOUT_NHWC) return fail(NIC_E_UNSUPPORTED, "conv_wgrad: the %s must be NHWC", s.big_is_input ? "output gradient" : "layer input");
  if (d->n == 0) {
    cudaMemsetAsync(dw, 0, sizeof(float) * d->c_in * d->c_out * d->kh * d->kw, st);
    if (db) cudaMemsetAsync(db, 0, sizeof(float) * d->c_out, st);
    return NIC_OK;
  }
  const bool gather = (s.big_layout == NIC_LAYOUT_NCHW) || (s.cb % 4 != 0);
  char* ws = static_cast<char*>(workspace);
  float* part = reinterpret_cast<float*>(ws);
  float* cpart = reinterpret_cast<float*>(ws + wgrad_part_bytes(d->kh * d->kw, s, d->n, gather));
  if (int rc = run_wgrad(big, small, d->n, s, d->stride, d->pad, d->kh, d->kw, 0, dw, part, st)) return rc;
  if (db) {
    const long hw = static_cast<long>(d->h_out) * d->w_out;
    if (d->out_layout == NIC_LAYOUT_NHWC) return run_colsum_nhwc(g, static_cast<long>(d->n) * hw, d->c_out, db, cpart, st);
    return run_colsum_nchw(g, d->n, d->c_out, hw, db, cpart, st);
  }
  return NIC_OK;
}

size_t nic_conv_wgrad_tc_workspace_bytes(const nic_conv_desc* d) {
  if (!d || validate_conv_desc(d) || !wgrad_tc_supported(d)) return 0;
  return wgrad_tc_workspace_bytes(d) + colsum_part_bytes(d->n, d->c_out) + 256;
}

int nic_conv_wgrad_tc(const nic_conv_desc* d, const void* x_pair, const void* g_pair, const float* g, float* dw, float* db,
                      void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (int rc = validate_conv_desc(d)) return rc;
  if (!wgrad_tc_supported(d)) return fail(NIC_E_UNSUPPORTED, "conv_wgrad_tc: layer shape not built for the tensor-core path");
  if (!x_pair || !g_pair || !dw || (db && !g)) return fail(NIC_E_BADSHAPE, "conv_wgrad_tc: null pointer");
  const size_t need = nic_conv_wgrad_tc_workspace_bytes(d);
  if (!workspace || workspace_bytes < need) return fail(NIC_E_WORKSPACE, "conv_wgrad_tc: workspace %zu < %zu bytes", workspace_bytes, need);
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(NIC_E_BADALIGN, "conv_wgrad_tc: workspace must be 256-byte aligned");
  cudaStream_t st = as_stream(stream);
  if (d->n == 0) {
    cudaMemsetAsync(dw, 0, sizeof(float) * d->c_in * d->c_out * d->kh * d->kw, st);
    if (db) cudaMemsetAsync(db, 0, sizeof(float) * d->c_out, st);
    return NIC_OK;
  }
  char* ws = static_cast<char*>(workspace);
  float* part = reinterpret_cast<float*>(ws);
  float* cpart = reinterpret_cast<float*>(ws + wgrad_tc_workspace_bytes(d));
  int splits = 0;
  if (int rc = wgrad_tc_launch(d, x_pair, g_pair, part, &splits, st)) return rc;
  nic_conv_desc full{};
  full.n = 1; full.c_in = full.c_out = 1; full.kh = d->kh; full.kw = d->kw; full.stride = 1; full.pad = d->pad;
  full.h_in = full.w_in = 64; full.h_out = full.w_out = 64 + 2 * d->pad - d->kh + 1;
  TapTable tt;
  if (int rc = build_tap_table(&full, &tt)) return rc;
  const WgradShape s = wgrad_shape(d);
  const long total = static_cast<long>(tt.ntaps) * s.cb * s.cs;
  wgrad_fold_kernel<<<ew_blocks(total), 256, 0, st>>>(part, splits, tt.ntaps, s.cb, s.cs, d->kh, d->kw, tt, dw);
  if (int rc = check_launch("wgrad_fold_kernel")) return rc;
  if (db) return run_colsum_nhwc(g, static_cast<long>(d->n) * d->h_out * d->w_out, d->c_out, db, cpart, st);
  return NIC_OK;
}

int nic_lrelu_bwd(const float* g, const float* out, float* g_pre, int64_t n, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || (n > 0 && (!g || !out || !g_pre))) return fail(NIC_E_BADSHAPE, "lrelu_bwd: bad arguments");
  if (n == 0) return NIC_OK;
  lrelu_bwd_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(g, out, g_pre, n);
  return check_launch("lrelu_bwd_kernel");
}

size_t nic_gdn_bwd_workspace_bytes(int32_t n, int32_t c, int32_t h, int32_t w) {
  if (n < 0 || c < 1 || h < 1 || w < 1) return 0;
  const size_t act = align256(static_cast<size_t>(n) * h * w * c * sizeof(float));
  WgradShape s{}; s.cb = s.cs = c; s.hb = s.hs = 1; s.wb = s.ws = 1;
  const long P = static_cast<long>(n) * h * w;
  const WgradPlan wp = plan_wgrad(1, c, c, P, false);
  return 3 * act + 4 * align256(static_cast<size_t>(c) * c * sizeof(float)) + 3 * align256(c * sizeof(float)) +
         align256(static_cast<size_t>(wp.splits) * c * c * sizeof(float)) + colsum_part_bytes(1, c) + 256;
}

int nic_gdn_bwd(const float* u, const float* g, int32_t n, int32_t c, int32_t h, int32_t w, int32_t inverse, float beta_min,
                const float* beta_raw, const float* gamma_raw, float* du, float* dbeta_raw, float* dgamma_raw,
                void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || c < 1 || h < 1 || w < 1 || c % 4) return fail(NIC_E_BADSHAPE, "gdn_bwd: n=%d c=%d h=%d w=%d (c %% 4 == 0)", n, c, h, w);
  if (!u || !g || !beta_raw || !gamma_raw || !du || !dbeta_raw || !dgamma_raw) return fail(NIC_E_BADSHAPE, "gdn_bwd: null pointer");
  const size_t need = nic_gdn_bwd_workspace_bytes(n, c, h, w);
  if (!workspace || workspace_bytes < need) return fail(NIC_E_WORKSPACE, "gdn_bwd: workspace %zu < %zu bytes", workspace_bytes, need);
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(NIC_E_BADALIGN, "gdn_bwd: workspace must be 256-byte aligned");
  cudaStream_t st = as_stream(stream);
  if (n == 0) {
    cudaMemsetAsync(dbeta_raw, 0, sizeof(float) * c, st);
    cudaMemsetAsync(dgamma_raw, 0, sizeof(float) * c * c, st);
    return NIC_OK;
  }
  const long P = static_cast<long>(n) * h * w, elems = P * c;
  const size_t act = align256(static_cast<size_t>(elems) * sizeof(float)), cc = align256(static_cast<size_t>(c) * c * sizeof(float)),
               c1 = align256(c * sizeof(float));
  char* ws = static_cast<char*>(workspace);
  float* nrm = reinterpret_cast<float*>(ws); ws += act;
  float* t = reinterpret_cast<float*>(ws); ws += act;
  float* r = reinterpret_cast<float*>(ws); ws += act;
  float* gamma_eff = reinterpret_cast<float*>(ws); ws += cc;
  float* gamma_t = reinterpret_cast<float*>(ws); ws += cc;
  float* dgamma_eff = reinterpret_cast<float*>(ws); ws += cc;
  ws += cc;                                                     // spare
  float* beta_eff = reinterpret_cast<float*>(ws); ws += c1;
  float* dbeta_eff = reinterpret_cast<float*>(ws); ws += c1;
  float* zero = reinterpret_cast<float*>(ws); ws += c1;
  const WgradPlan wp = plan_wgrad(1, c, c, P, false);
  float* wpart = reinterpret_cast<float*>(ws); ws += align256(static_cast<size_t>(wp.splits) * c * c * sizeof(float));
  float* cpart = reinterpret_cast<float*>(ws);

  const float pedestal = static_cast<float>(3.814697265625e-06 * 3.814697265625e-06);
  const float beta_bound = static_cast<float>(sqrt(static_cast<double>(beta_min) + static_cast<double>(pedestal)));
  const float gamma_bound = static_cast<float>(sqrt(static_cast<double>(pedestal)));
  gdn_reparam_kernel<<<(c * c + 255) / 256, 256, 0, st>>>(c, beta_bound, gamma_bound, pedestal, beta_raw, gamma_raw, beta_eff, gamma_eff, gamma_t);
  if (int rc = check_launch("gdn_reparam_kernel")) return rc;
  cudaMemsetAsync(zero, 0, sizeof(float) * c, st);
  // norm = beta + gamma . u^2
  if (int rc = conv1x1_fp32(u, P, c, c, gamma_t, beta_eff, nrm, 1, NIC_EPI_BIAS, st)) return rc;
  gdn_bwd_prep_kernel<<<ew_blocks(elems), 256, 0, st>>>(g, u, nrm, inverse, t, du, elems);
  if (int rc = check_launch("gdn_bwd_prep_kernel")) return rc;
  // r_j = sum_i gamma[i][j] t_i : a 1x1 conv with weight [c_in = i][c_out = j] = gamma in its natural layout
  if (int rc = conv1x1_fp32(t, P, c, c, gamma_eff, zero, r, 0, NIC_EPI_BIAS, st)) return rc;
  gdn_bwd_finish_kernel<<<ew_blocks(elems), 256, 0, st>>>(u, r, du, elems);
  if (int rc = check_launch("gdn_bwd_finish_kernel")) return rc;
  // dgamma_eff[i][j] = sum_pix t_i u_j^2 ; dbeta_eff[i] = sum_pix t_i
  WgradShape s{}; s.cb = c; s.cs = c; s.hb = s.hs = 1; s.wb = s.ws = static_cast<int>(P); s.big_layout = NIC_LAYOUT_NHWC; s.big_is_input = true;
  if (P > 0x7fffffffL) return fail(NIC_E_BADSHAPE, "gdn_bwd: %ld pixels", P);
  if (int rc = run_wgrad(u, t, 1, s, 1, 0, 1, 1, 1, dgamma_eff, wpart, st)) return rc;
  if (int rc = run_colsum_nhwc(t, P, c, dbeta_eff, cpart, st)) return rc;
  gdn_reparam_bwd_kernel<<<(c * c + 255) / 256, 256, 0, st>>>(c, beta_bound, gamma_bound, beta_raw, gamma_raw, dbeta_eff, dgamma_eff, dbeta_raw, dgamma_raw);
  return check_launch("gdn_reparam_bwd_kernel");
}

/* ---- the same backward in three calls, for callers that run the two channel-mixing contractions elsewhere (tensor cores) ---- */

int nic_gdn_reparam(int32_t c, float beta_min, const float* beta_raw, const float* gamma_raw, float* beta_eff, float* gamma_eff,
                    float* gamma_eff_t, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (c < 1 || !beta_raw || !gamma_raw || !beta_eff || !gamma_eff || !gamma_eff_t) return fail(NIC_E_BADSHAPE, "gdn_reparam: bad arguments");
  const float pedestal = static_cast<float>(3.814697265625e-06 * 3.814697265625e-06);
  const float beta_bound = static_cast<float>(sqrt(static_cast<double>(beta_min) + static_cast<double>(pedestal)));
  const float gamma_bound = static_cast<float>(sqrt(static_cast<double>(pedestal)));
  gdn_reparam_kernel<<<(c * c + 255) / 256, 256, 0, as_stream(stream)>>>(c, beta_bound, gamma_bound, pedestal, beta_raw, gamma_raw, beta_eff, gamma_eff, gamma_eff_t);
  return check_launch("gdn_reparam_kernel");
}

int nic_gdn_apply(const float* u, const float* norm, int64_t n, int32_t inverse, float* out, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || (n > 0 && (!u || !norm || !out))) return fail(NIC_E_BADSHAPE, "gdn_apply: bad arguments");
  if (n == 0) return NIC_OK;
  gdn_apply_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(u, norm, inverse, out, n);
  return check_launch("gdn_apply_kernel");
}

int nic_gdn_apply_add(const float* u, const float* norm, const float* addend, int64_t n, int32_t inverse, float* out, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || (n > 0 && (!u || !norm || !addend || !out))) return fail(NIC_E_BADSHAPE, "gdn_apply_add: bad arguments");
  if (n == 0) return NIC_OK;
  gdn_apply_add_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(u, norm, addend, inverse, out, n);
  return check_launch("gdn_apply_add_kernel");
}

int nic_gdn_bwd_prep(const float* u, const float* g, const float* norm, int64_t n, int32_t inverse, float* t, float* du, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || (n > 0 && (!u || !g || !norm || !t || !du))) return fail(NIC_E_BADSHAPE, "gdn_bwd_prep: bad arguments");
  if (n == 0) return NIC_OK;
  gdn_bwd_prep_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(g, u, norm, inverse, t, du, n);
  return check_launch("gdn_bwd_prep_kernel");
}

size_t nic_gdn_bwd_finish_workspace_bytes(int64_t pixels, int32_t c) {
  if (pixels < 0 || c < 1) return 0;
  const WgradPlan wp = plan_wgrad(1, c, c, pixels, false);
  return 2 * align256(static_cast<size_t>(c) * c * sizeof(float)) + 2 * align256(c * sizeof(float)) +
         align256(static_cast<size_t>(wp.splits) * c * c * sizeof(float)) + colsum_part_bytes(1, c) + 256;
}

int nic_gdn_bwd_finish(const float* u, const float* t, const float* r, int64_t pixels, int32_t c, float beta_min,
                       const float* beta_raw, const float* gamma_raw, const float* dgamma_eff_in, const float* dbeta_eff_in,
                       float* du, float* dbeta_raw, float* dgamma_raw, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (pixels < 1 || pixels > 0x7fffffffL || c < 4 || c % 4) return fail(NIC_E_BADSHAPE, "gdn_bwd_finish: pixels=%lld c=%d", static_cast<long long>(pixels), c);
  if (!u || !t || !r || !beta_raw || !gamma_raw || !du || !dbeta_raw || !dgamma_raw) return fail(NIC_E_BADSHAPE, "gdn_bwd_finish: null pointer");
  const size_t need = nic_gdn_bwd_finish_workspace_bytes(pixels, c);
  if (!workspace || workspace_bytes < need) return fail(NIC_E_WORKSPACE, "gdn_bwd_finish: workspace %zu < %zu bytes", workspace_bytes, need);
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(NIC_E_BADALIGN, "gdn_bwd_finish: workspace must be 256-byte aligned");
  cudaStream_t st = as_stream(stream);
  const size_t cc = align256(static_cast<size_t>(c) * c * sizeof(float)), c1 = align256(c * sizeof(float));
  char* ws = static_cast<char*>(workspace);
  float* dgamma_eff = reinterpret_cast<float*>(ws); ws += 2 * cc;
  float* dbeta_eff = reinterpret_cast<float*>(ws); ws += 2 * c1;
  const WgradPlan wp = plan_wgrad(1, c, c, pixels, false);
  float* wpart = reinterpret_cast<float*>(ws); ws += align256(static_cast<size_t>(wp.splits) * c * c * sizeof(float));
  float* cpart = reinterpret_cast<float*>(ws);
  const long elems = pixels * c;
  gdn_bwd_finish_kernel<<<ew_blocks(elems), 256, 0, st>>>(u, r, du, elems);
  if (int rc = check_launch("gdn_bwd_finish_kernel")) return rc;
  if (dgamma_eff_in && dbeta_eff_in) {          // the caller ran the (u^2, t) weight gradient elsewhere (nic_conv_wgrad_tc on a 1x1 descriptor)
    dgamma_eff = const_cast<float*>(dgamma_eff_in); dbeta_eff = const_cast<float*>(dbeta_eff_in);
  } else {
    WgradShape s{}; s.cb = c; s.cs = c; s.hb = s.hs = 1; s.wb = s.ws = static_cast<int>(pixels); s.big_layout = NIC_LAYOUT_NHWC; s.big_is_input = true;
    if (int rc = run_wgrad(u, t, 1, s, 1, 0, 1, 1, 1, dgamma_eff, wpart, st)) return rc;
    if (int rc = run_colsum_nhwc(t, pixels, c, dbeta_eff, cpart, st)) return rc;
  }
  const float pedestal = static_cast<float>(3.814697265625e-06 * 3.814697265625e-06);
  const float beta_bound = static_cast<float>(sqrt(static_cast<double>(beta_min) + static_cast<double>(pedestal)));
  const float gamma_bound = static_cast<float>(sqrt(static_cast<double>(pedestal)));
  gdn_reparam_bwd_kernel<<<(c * c + 255) / 256, 256, 0, st>>>(c, beta_bound, gamma_bound, beta_raw, gamma_raw, dbeta_eff, dgamma_eff, dbeta_raw, dgamma_raw);
  return check_launch("gdn_reparam_bwd_kernel");
}

int nic_gdn_bwd_du(const float* u, const float* r, float* du, int64_t n, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || (n > 0 && (!u || !r || !du))) return fail(NIC_E_BADSHAPE, "gdn_bwd_du: bad arguments");
  if (n == 0) return NIC_OK;
  gdn_bwd_finish_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(u, r, du, n);
  return check_launch("gdn_bwd_finish_kernel");
}

int nic_gdn_reparam_bwd(int32_t c, float beta_min, const float* beta_raw, const float* gamma_raw, const float* dbeta_eff,
                        const float* dgamma_eff, float* dbeta_raw, float* dgamma_raw, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (c < 1 || !beta_raw || !gamma_raw || !dbeta_eff || !dgamma_eff || !dbeta_raw || !dgamma_raw) return fail(NIC_E_BADSHAPE, "gdn_reparam_bwd: bad arguments");
  const float pedestal = static_cast<float>(3.814697265625e-06 * 3.814697265625e-06);
  const float beta_bound = static_cast<float>(sqrt(static_cast<double>(beta_min) + static_cast<double>(pedestal)));
  const float gamma_bound = static_cast<float>(sqrt(static_cast<double>(pedestal)));
  gdn_reparam_bwd_kernel<<<(c * c + 255) / 256, 256, 0, as_stream(stream)>>>(c, beta_bound, gamma_bound, beta_raw, gamma_raw, dbeta_eff, dgamma_eff,
                                                                            dbeta_raw, dgamma_raw);
  return check_launch("gdn_reparam_bwd_kernel");
}

int nic_sse_bwd(const float* x_hat, const float* x, int64_t n, float coef, float* g_x_hat, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || (n > 0 && (!x_hat || !x || !g_x_hat))) return fail(NIC_E_BADSHAPE, "sse_bwd: bad arguments");
  if (n == 0) return NIC_OK;
  sse_bwd_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(x_hat, x, coef, g_x_hat, n);
  return check_launch("sse_bwd_kernel");
}

int nic_sse_bwd_per_image(const float* x_hat, const float* x, int32_t b, int64_t per_image, const float* coef, float* g_x_hat,
                          void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (b < 0 || per_image < 1 || (b > 0 && (!x_hat || !x || !coef || !g_x_hat))) return fail(NIC_E_BADSHAPE, "sse_bwd_per_image: bad arguments");
  if (b == 0) return NIC_OK;
  const long n = static_cast<long>(b) * per_image;
  sse_bwd_per_image_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(x_hat, x, coef, per_image, g_x_hat, n);
  return check_launch("sse_bwd_per_image_kernel");
}

int nic_add_inplace(float* dst, const float* src, int64_t n, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || (n > 0 && (!dst || !src))) return fail(NIC_E_BADSHAPE, "add_inplace: bad arguments");
  if (n == 0) return NIC_OK;
  add_inplace_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(dst, src, n);
  return check_launch("add_inplace_kernel");
}

int nic_layout_convert(const float* src, float* dst, int32_t n, int32_t c, int32_t hw, int32_t to_nhwc, int32_t accumulate, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || c < 1 || hw < 1 || n > 65535) return fail(NIC_E_BADSHAPE, "layout_convert: n=%d c=%d hw=%d", n, c, hw);
  if (n == 0) return NIC_OK;
  if (!src || !dst) return fail(NIC_E_BADSHAPE, "layout_convert: null pointer");
  layout_convert_kernel<<<dim3((hw + 31) / 32, (c + 31) / 32, n), 256, 0, as_stream(stream)>>>(src, dst, c, hw, to_nhwc, accumulate);
  return check_launch("layout_convert_kernel");
}

int nic_counter_increment(int32_t* counter, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (!counter) return fail(NIC_E_BADSHAPE, "counter_increment: null pointer");
  counter_increment_kernel<<<1, 32, 0, as_stream(stream)>>>(counter);
  return check_launch("counter_increment_kernel");
}

int nic_adam_multi_step(float* const* p_host, const float* const* g_host, float* const* m_host, float* const* v_host,
                        const int64_t* n_host, int32_t count, float lr, float beta1, float beta2, float eps, int32_t step,
                        const int32_t* step_dev, void* stream) {
  return nic_adam_multi_step_ex(p_host, g_host, m_host, v_host, n_host, count, lr, nullptr, 1.0f, beta1, beta2, eps, step, step_dev, stream);
}

int nic_adam_multi_step_ex(float* const* p_host, const float* const* g_host, float* const* m_host, float* const* v_host,
                           const int64_t* n_host, int32_t count, float lr, const float* lr_dev, float grad_scale, float beta1, float beta2,
                           float eps, int32_t step, const int32_t* step_dev, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (step_dev) step = 1;                       // unused: the kernel reads the device counter
  if (count < 0 || step < 1 || (count > 0 && (!p_host || !g_host || !m_host || !v_host || !n_host))) return fail(NIC_E_BADSHAPE, "adam_multi_step: bad arguments");
  const double bc1 = 1.0 - pow(static_cast<double>(beta1), step), bc2 = 1.0 - pow(static_cast<double>(beta2), step);
  for (int base = 0; base < count; base += kAdamMaxTensors) {
    AdamArgs a{};
    const int cnt = count - base < kAdamMaxTensors ? count - base : kAdamMaxTensors;
    long blocks = 0;
    for (int i = 0; i < cnt; ++i) {
      a.p[i] = p_host[base + i]; a.g[i] = g_host[base + i]; a.m[i] = m_host[base + i]; a.v[i] = v_host[base + i]; a.n[i] = n_host[base + i];
      if (a.n[i] < 0 || (a.n[i] > 0 && (!a.p[i] || !a.g[i] || !a.m[i] || !a.v[i]))) return fail(NIC_E_BADSHAPE, "adam_multi_step: tensor %d", base + i);
      a.blk_start[i] = static_cast<int>(blocks);
      blocks += (a.n[i] + kAdamChunk - 1) / kAdamChunk;
      if (blocks > 0x7fffffffL) return fail(NIC_E_BADSHAPE, "adam_multi_step: too many elements");
    }
    a.blk_start[cnt] = static_cast<int>(blocks);
    a.count = cnt;
    if (blocks == 0) continue;
    // device learning rate with a HOST step count: the kernel forms step_size = lr_dev / bc1 from the 1 / bc1 passed here
    const float step_size = (lr_dev && !step_dev) ? static_cast<float>(1.0 / bc1) : static_cast<float>(lr / bc1);
    adam_multi_kernel<<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(a, beta1, beta2, lr, step_size,
                                                                                  static_cast<float>(sqrt(bc2)), eps, step_dev, lr_dev, grad_scale);
    if (int rc = check_launch("adam_multi_kernel")) return rc;
  }
  return NIC_OK;
}

int nic_to_pair(const float* src, void* dst, int64_t rows, int32_t c, int32_t square, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (rows < 0 || c < 4 || c % 4) return fail(NIC_E_BADSHAPE, "to_pair: rows=%lld c=%d (c %% 4 == 0)", static_cast<long long>(rows), c);
  if (rows == 0) return NIC_OK;
  if (!src || !dst) return fail(NIC_E_BADSHAPE, "to_pair: null pointer");
  if ((reinterpret_cast<uintptr_t>(src) & 15) || (reinterpret_cast<uintptr_t>(dst) & 7)) return fail(NIC_E_BADALIGN, "to_pair: alignment");
  to_pair_kernel<<<ew_blocks(rows * (c / 4)), 256, 0, as_stream(stream)>>>(src, static_cast<__nv_bfloat16*>(dst), rows, c, square);
  return check_launch("to_pair_kernel");
}

int nic_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                  int32_t step, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || step < 1 || (n > 0 && (!p || !g || !m || !v))) return fail(NIC_E_BADSHAPE, "adam_step: bad arguments");
  if (n == 0) return NIC_OK;
  const double bc1 = 1.0 - pow(static_cast<double>(beta1), step), bc2 = 1.0 - pow(static_cast<double>(beta2), step);
  adam_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(p, g, m, v, n, beta1, beta2, static_cast<float>(lr / bc1),
                                                           static_cast<float>(sqrt(bc2)), eps);
  return check_launch("adam_kernel");
}

}  // extern "C"
