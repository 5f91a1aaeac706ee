// Evaluator-side distortion metrics on the device (SURVEY.md section 8 row f3): what CompressionEvaluator.compute_metrics
// (/root/reference/Evaluator.py:26-53) evaluates per image on `imgs` and `x_hat.clamp(0, 1)`:
//   mean squared error over RGB and over luma Y = 0.299 R + 0.587 G + 0.114 B (Evaluator.py:27-30, 34, 41-43)
//   MS-SSIM of the RGB planes and of the luma plane (Evaluator.py:38, 45): `pytorch_msssim.ms_ssim(recon, orig, data_range=1,
//   size_average=True)` - a third-party package absent from /root/reference and from this image (parity unpinned; the algorithm
//   restated here and in oracle/metrics.py is the published one of pytorch_msssim 0.2.x): 11-tap Gaussian (sigma 1.5), separable,
//   VALID convolution of x, y, x^2, y^2, xy; cs = (2 s12 + C2) / (s1 + s2 + C2), ssim = (2 m1 m2 + C1) / (m1^2 + m2^2 + C1) * cs,
//   C1 = (0.01 L)^2, C2 = (0.03 L)^2; five scales with 2x2 average pooling (padding = size % 2, zeros counted) between them;
//   result = prod_i relu(cs_i)^w_i * relu(ssim_5)^w_5 per (image, channel), weights (0.0448, 0.2856, 0.3001, 0.2363, 0.1333).
// Reductions are per-block partial sums folded in a fixed order (deterministic).
#include "tc_host.cuh"

namespace nic {

constexpr int kWin = 11;
constexpr int kTile = 32;                       // output pixels per block edge
constexpr int kIn = kTile + kWin - 1;           // 42

__constant__ float c_gauss[kWin];

// planes: [np][h][w] f32.  One block = one 32 x 32 tile of the VALID output of one plane; writes (sum ssim, sum cs) of its tile.
__global__ void __launch_bounds__(256)
ssim_tile_kernel(const float* __restrict__ xs, const float* __restrict__ ys, int h, int w, float c1, float c2, int clamp_y,
                 float* __restrict__ part /* [np][tiles][2] */) {
  __shared__ float sx[kIn][kIn + 1], sy[kIn][kIn + 1];
  __shared__ float hbuf[5][kIn][kTile + 1];
  __shared__ float red[2][8];
  const int plane = blockIdx.z;
  const int ho = h - kWin + 1, wo = w - kWin + 1;
  const int ty0 = blockIdx.y * kTile, tx0 = blockIdx.x * kTile;
  const float* xp = xs + static_cast<long>(plane) * h * w;
  const float* yp = ys + static_cast<long>(plane) * h * w;
  for (int i = threadIdx.x; i < kIn * kIn; i += 256) {
    const int r = i / kIn, c = i % kIn;
    const int gy = ty0 + r, gx = tx0 + c;
    float a = 0.f, b = 0.f;
    if (gy < h && gx < w) {
      a = xp[static_cast<long>(gy) * w + gx];
      b = yp[static_cast<long>(gy) * w + gx];
      if (clamp_y) b = fminf(fmaxf(b, 0.f), 1.f);
    }
    sx[r][c] = a; sy[r][c] = b;
  }
  __syncthreads();
  // horizontal pass: 42 rows x 32 columns, five maps
  for (int i = threadIdx.x; i < kIn * kTile; i += 256) {
    const int r = i / kTile, c = i % kTile;
    float m1 = 0.f, m2 = 0.f, xx = 0.f, yy = 0.f, xy = 0.f;
#pragma unroll
    for (int k = 0; k < kWin; ++k) {
      const float g = c_gauss[k], a = sx[r][c + k], b = sy[r][c + k];
      m1 += g * a; m2 += g * b; xx += g * a * a; yy += g * b * b; xy += g * a * b;
    }
    hbuf[0][r][c] = m1; hbuf[1][r][c] = m2; hbuf[2][r][c] = xx; hbuf[3][r][c] = yy; hbuf[4][r][c] = xy;
  }
  __syncthreads();
  float s_ssim = 0.f, s_cs = 0.f;
  for (int i = threadIdx.x; i < kTile * kTile; i += 256) {
    const int r = i / kTile, c = i % kTile;
    if (ty0 + r < ho && tx0 + c < wo) {
      float m1 = 0.f, m2 = 0.f, xx = 0.f, yy = 0.f, xy = 0.f;
#pragma unroll
      for (int k = 0; k < kWin; ++k) {
        const float g = c_gauss[k];
        m1 += g * hbuf[0][r + k][c]; m2 += g * hbuf[1][r + k][c]; xx += g * hbuf[2][r + k][c];
        yy += g * hbuf[3][r + k][c]; xy += g * hbuf[4][r + k][c];
      }
      const float m11 = m1 * m1, m22 = m2 * m2, m12 = m1 * m2;
      const float s1 = xx - m11, s2 = yy - m22, s12 = xy - m12;
      const float cs = (2.f * s12 + c2) / (s1 + s2 + c2);
      s_cs += cs;
      s_ssim += (2.f * m12 + c1) / (m11 + m22 + c1) * cs;
    }
  }
  s_ssim = warp_sum(s_ssim); s_cs = warp_sum(s_cs);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { red[0][wid] = s_ssim; red[1][wid] = s_cs; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { a += red[0][i]; b += red[1][i]; }
    const long tiles = static_cast<long>(gridDim.x) * gridDim.y;
    float* o = part + (static_cast<long>(plane) * tiles + static_cast<long>(blockIdx.y) * gridDim.x + blockIdx.x) * 2;
    o[0] = a; o[1] = b;
  }
}

// out[plane][0 | 1] = mean over the valid output of ssim | cs (fixed-order fold of the tile sums)
__global__ void ssim_fold_kernel(const float* __restrict__ part, int tiles, float inv_count, float* __restrict__ out) {
  const int plane = blockIdx.x;
  if (threadIdx.x < 2) {
    double s = 0.0;
    for (int t = 0; t < tiles; ++t) s += static_cast<double>(part[(static_cast<long>(plane) * tiles + t) * 2 + threadIdx.x]);
    out[plane * 2 + threadIdx.x] = static_cast<float>(s * inv_count);
  }
}

// F.avg_pool2d(kernel 2, stride 2, padding (h % 2, w % 2), count_include_pad): out[i][j] = sum of the 2 x 2 window / 4
__global__ void avgpool2_kernel(const float* __restrict__ in, float* __restrict__ out, int np, int h, int w, int ph, int pw, int ho, int wo,
                                int clamp_in) {
  const long total = static_cast<long>(np) * ho * wo;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(i % wo), y = static_cast<int>((i / wo) % ho);
    const long p = i / (static_cast<long>(wo) * ho);
    float s = 0.f;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int iy = 2 * y + dy - ph, ix = 2 * x + dx - pw;
        if (iy >= 0 && iy < h && ix >= 0 && ix < w) {
          float v = in[(p * h + iy) * w + ix];
          if (clamp_in) v = fminf(fmaxf(v, 0.f), 1.f);
          s += v;
        }
      }
    out[i] = 0.25f * s;
  }
}

// luma planes of an NCHW RGB batch (Evaluator.py:26-30); clamp_in: clamp to [0, 1] first (the reconstruction)
__global__ void luma_kernel(const float* __restrict__ rgb, float* __restrict__ y, int b, long hw, int clamp_in) {
  const long total = static_cast<long>(b) * hw;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const long img = i / hw, p = i - img * hw;
    float r = rgb[(img * 3 + 0) * hw + p], g = rgb[(img * 3 + 1) * hw + p], bl = rgb[(img * 3 + 2) * hw + p];
    if (clamp_in) { r = fminf(fmaxf(r, 0.f), 1.f); g = fminf(fmaxf(g, 0.f), 1.f); bl = fminf(fmaxf(bl, 0.f), 1.f); }
    y[i] = 0.299f * r + 0.587f * g + 0.114f * bl;
  }
}

// per-image partial sums of (orig - clamp(recon))^2 over RGB and of the squared luma difference: partials [b][kPartials][2]
__global__ void __launch_bounds__(256)
eval_sse_kernel(const float* __restrict__ orig, const float* __restrict__ recon, long hw, int clamp01, float* __restrict__ partials) {
  __shared__ float red[2][8];
  const int img = blockIdx.y;
  const float* o = orig + static_cast<long>(img) * 3 * hw;
  const float* r = recon + static_cast<long>(img) * 3 * hw;
  float s_rgb = 0.f, s_y = 0.f;
  for (long p = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; p < hw; p += static_cast<long>(gridDim.x) * blockDim.x) {
    float dy = 0.f;
    const float wgt[3] = {0.299f, 0.587f, 0.114f};
    float yo = 0.f, yr = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float b = r[c * hw + p];
      if (clamp01) b = fminf(fmaxf(b, 0.f), 1.f);
      const float a = o[c * hw + p];
      const float d = a - b;
      s_rgb += d * d;
      yo += wgt[c] * a; yr += wgt[c] * b;
    }
    dy = yo - yr;
    s_y += dy * dy;
  }
  s_rgb = warp_sum(s_rgb); s_y = warp_sum(s_y);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { red[0][wid] = s_rgb; red[1][wid] = s_y; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { a += red[0][i]; b += red[1][i]; }
    partials[(static_cast<long>(img) * kPartials + blockIdx.x) * 2 + 0] = a;
    partials[(static_cast<long>(img) * kPartials + blockIdx.x) * 2 + 1] = b;
  }
}
__global__ void eval_sse_fold_kernel(const float* __restrict__ partials, int parts, long hw, float* __restrict__ out /* [b][2] */) {
  const int img = blockIdx.x;
  if (threadIdx.x < 2) {
    double s = 0.0;
    for (int i = 0; i < parts; ++i) s += static_cast<double>(partials[(static_cast<long>(img) * kPartials + i) * 2 + threadIdx.x]);
    out[img * 2 + threadIdx.x] = static_cast<float>(s / (threadIdx.x == 0 ? 3.0 * hw : static_cast<double>(hw)));
  }
}

// ---- backward of the per-level means (the MS-SSIM loss, DESIGN.md section 13; oracle/ms_ssim_bwd.py restates it) ----------------
constexpr int kBT = 32;                         // level-input pixels per tile edge (one CTA)
constexpr int kBO = kBT + kWin - 1;             // 42: VALID output pixels whose window touches the tile
constexpr int kBI = kBO + kWin - 1;             // 52: input pixels those outputs read
constexpr int kBwdSmemFloats = 2 * kBI * (kBI + 1) + 6 * kBI * kBO + 3 * kBO * (kBO + 1);
constexpr int kBwdSmemBytes = kBwdSmemFloats * 4;

/*
 * One 32 x 32 tile of level l's input gradient of one plane:
 *   g[i][j] = (G^T a + 2 x (G^T b) + 2 (x - y) (G^T e))[i][j] + g_coarse[(i + ph) / 2][(j + pw) / 2] / 4
 * with a, b, e the derivatives of the level's cs map (ssim map at the last level) with respect to m1 = G x, exx = G x^2 and
 * euu = G (x - y)^2 at every VALID output pixel, times g_level[plane] / (ho wo), and zero outside the VALID output.
 * The CTA stages 52 x 52 of x and y, recomputes the six moment maps over the 42 x 42 output pixels that touch the tile, forms
 * a / b / e there and applies the transposed filter.  Every output element is written by one thread, from sums in a fixed order.
 */
__global__ void __launch_bounds__(256)
ms_ssim_bwd_tile_kernel(const float* __restrict__ xs, const float* __restrict__ ys, int h, int w, float c1, float c2, int last,
                        const float* __restrict__ g_level, const float* __restrict__ g_coarse, int hc, int wc, int ph, int pw,
                        float* __restrict__ g_out) {
  extern __shared__ float smem[];
  float (*sx)[kBI + 1] = reinterpret_cast<float (*)[kBI + 1]>(smem);
  float (*sy)[kBI + 1] = reinterpret_cast<float (*)[kBI + 1]>(smem + kBI * (kBI + 1));
  float* hb = smem + 2 * kBI * (kBI + 1);                       // [6][kBI][kBO] moment rows; later [3][kBO][kBT] filtered rows
  float* ab = hb + 6 * kBI * kBO;                               // [3][kBO][kBO + 1]: a, b, e
  const int plane = blockIdx.z;
  const int ho = h - kWin + 1, wo = w - kWin + 1;
  const int ty0 = blockIdx.y * kBT, tx0 = blockIdx.x * kBT;
  const int oy0 = ty0 - (kWin - 1), ox0 = tx0 - (kWin - 1);     // first output row / column (and first staged input row / column)
  const long plane_off = static_cast<long>(plane) * h * w;
  const float* xp = xs + plane_off;
  const float* yp = ys + plane_off;
  for (int i = threadIdx.x; i < kBI * kBI; i += 256) {
    const int r = i / kBI, c = i % kBI;
    const int gy = oy0 + r, gx = ox0 + c;
    float a = 0.f, b = 0.f;
    if (gy >= 0 && gy < h && gx >= 0 && gx < w) { a = xp[static_cast<long>(gy) * w + gx]; b = yp[static_cast<long>(gy) * w + gx]; }
    sx[r][c] = a; sy[r][c] = b;
  }
  __syncthreads();
  // moments along the rows: 52 rows x 42 output columns, six maps
  for (int i = threadIdx.x; i < kBI * kBO; i += 256) {
    const int r = i / kBO, c = i % kBO;
    float m1 = 0.f, m2 = 0.f, xx = 0.f, yy = 0.f, mu = 0.f, uu = 0.f;
#pragma unroll
    for (int k = 0; k < kWin; ++k) {
      const float g = c_gauss[k], a = sx[r][c + k], b = sy[r][c + k], u = a - b;
      m1 += g * a; m2 += g * b; xx += g * a * a; yy += g * b * b; mu += g * u; uu += g * u * u;
    }
    hb[0 * kBI * kBO + i] = m1; hb[1 * kBI * kBO + i] = m2; hb[2 * kBI * kBO + i] = xx;
    hb[3 * kBI * kBO + i] = yy; hb[4 * kBI * kBO + i] = mu; hb[5 * kBI * kBO + i] = uu;
  }
  __syncthreads();
  const float scale = g_level[plane] / (static_cast<float>(ho) * static_cast<float>(wo));
  for (int i = threadIdx.x; i < kBO * kBO; i += 256) {
    const int r = i / kBO, c = i % kBO;
    const int p = oy0 + r, q = ox0 + c;
    float a = 0.f, b = 0.f, e = 0.f;
    if (p >= 0 && p < ho && q >= 0 && q < wo) {
      float mom[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int k = 0; k < kWin; ++k) {
        const float g = c_gauss[k];
#pragma unroll
        for (int m = 0; m < 6; ++m) mom[m] += g * hb[m * kBI * kBO + (r + k) * kBO + c];
      }
      const float m1 = mom[0], m2 = mom[1], mu = mom[4];
      const float d = mom[2] - m1 * m1 + mom[3] - m2 * m2 + c2;
      const float v = mom[5] - mu * mu;
      const float inv_d = 1.f / d, vd = v * inv_d;
      a = 2.f * (mu - m1 * vd) * inv_d;
      b = vd * inv_d;
      e = -inv_d;
      if (last) {
        const float inv_b = 1.f / (m1 * m1 + m2 * m2 + c1);
        const float mu2b = mu * mu * inv_b;
        const float lum = 1.f - mu2b, cs = 1.f - vd;
        a = 2.f * (m1 * mu2b - mu) * inv_b * cs + lum * a;
        b *= lum; e *= lum;
      }
      a *= scale; b *= scale; e *= scale;
    }
    ab[(0 * kBO + r) * (kBO + 1) + c] = a; ab[(1 * kBO + r) * (kBO + 1) + c] = b; ab[(2 * kBO + r) * (kBO + 1) + c] = e;
  }
  __syncthreads();
  // transposed filter along the rows: output column c = jj + 10 - k feeds input column jj with tap k
  for (int i = threadIdx.x; i < 3 * kBO * kBT; i += 256) {
    const int m = i / (kBO * kBT), r = (i / kBT) % kBO, jj = i % kBT;
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < kWin; ++k) t += c_gauss[k] * ab[(m * kBO + r) * (kBO + 1) + jj + (kWin - 1) - k];
    hb[i] = t;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kBT * kBT; i += 256) {
    const int ii = i / kBT, jj = i % kBT;
    const int gi = ty0 + ii, gj = tx0 + jj;
    if (gi >= h || gj >= w) continue;
    float t0 = 0.f, t1 = 0.f, t2 = 0.f;
#pragma unroll
    for (int k = 0; k < kWin; ++k) {
      const float g = c_gauss[k];
      const int r = ii + (kWin - 1) - k;
      t0 += g * hb[(0 * kBO + r) * kBT + jj]; t1 += g * hb[(1 * kBO + r) * kBT + jj]; t2 += g * hb[(2 * kBO + r) * kBT + jj];
    }
    const float xv = sx[ii + kWin - 1][jj + kWin - 1], uv = xv - sy[ii + kWin - 1][jj + kWin - 1];
    float gv = t0 + 2.f * xv * t1 + 2.f * uv * t2;
    if (g_coarse) gv += 0.25f * g_coarse[(static_cast<long>(plane) * hc + (gi + ph) / 2) * wc + (gj + pw) / 2];
    g_out[plane_off + static_cast<long>(gi) * w + gj] = gv;
  }
}

// The constant-memory window is per device: uploaded once on each by the first nic_ms_ssim_levels / nic_ms_ssim_bwd call there
// (cudaMemcpyToSymbol, which a CUDA-graph capture cannot record), so that first call must run outside any capture - as the
// warm-up step of parallel.ShardedTrainer(graph=True) does before it captures.
static int ensure_gauss() {
  static bool done_dev[64] = {};
  int dev = 0;
  if (int rc = check_cuda(cudaGetDevice(&dev), "cudaGetDevice")) return rc;
  if (dev < 0 || dev >= 64) return fail(NIC_E_CUDA, "ms_ssim: device index %d", dev);
  bool& done = done_dev[dev];
  if (done) return NIC_OK;
  // pytorch_msssim._fspecial_gauss_1d(11, 1.5): exp(-(i - 5)^2 / (2 sigma^2)) normalised, in float32
  float g[kWin]; float s = 0.f;
  for (int i = 0; i < kWin; ++i) { const float c = static_cast<float>(i - kWin / 2); g[i] = expf(-(c * c) / (2.f * 1.5f * 1.5f)); s += g[i]; }
  for (int i = 0; i < kWin; ++i) g[i] /= s;
  if (int rc = check_cuda(cudaMemcpyToSymbol(c_gauss, g, sizeof(g)), "cudaMemcpyToSymbol(gauss)")) return rc;
  done = true;
  return NIC_OK;
}

}  // namespace nic

using namespace nic;

extern "C" {

int nic_eval_mse(const float* orig, const float* recon, int32_t b, int32_t h, int32_t w, int32_t clamp01, float* mse_rgb_y, float* partials,
                 void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (b < 0 || h < 1 || w < 1) return fail(NIC_E_BADSHAPE, "eval_mse: b=%d h=%d w=%d", b, h, w);
  if (b == 0) return NIC_OK;
  if (!orig || !recon || !mse_rgb_y || !partials) return fail(NIC_E_BADSHAPE, "eval_mse: null pointer");
  const long hw = static_cast<long>(h) * w;
  int parts = static_cast<int>((hw + 255) / 256);
  if (parts > kPartials) parts = kPartials;
  eval_sse_kernel<<<dim3(parts, b), 256, 0, as_stream(stream)>>>(orig, recon, hw, clamp01, partials);
  if (int rc = check_launch("eval_sse_kernel")) return rc;
  eval_sse_fold_kernel<<<b, 32, 0, as_stream(stream)>>>(partials, parts, hw, mse_rgb_y);
  return check_launch("eval_sse_fold_kernel");
}

int nic_luma(const float* rgb, float* y, int32_t b, int32_t h, int32_t w, int32_t clamp01, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (b < 0 || h < 1 || w < 1) return fail(NIC_E_BADSHAPE, "luma: b=%d h=%d w=%d", b, h, w);
  if (b == 0) return NIC_OK;
  if (!rgb || !y) return fail(NIC_E_BADSHAPE, "luma: null pointer");
  const long total = static_cast<long>(b) * h * w;
  long blocks = (total + 255) / 256;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  luma_kernel<<<static_cast<int>(blocks), 256, 0, as_stream(stream)>>>(rgb, y, b, static_cast<long>(h) * w, clamp01);
  return check_launch("luma_kernel");
}

size_t nic_ms_ssim_workspace_bytes(int32_t planes, int32_t h, int32_t w) {
  if (planes < 1 || h < 1 || w < 1) return 0;
  // two ping-pong pyramids (x and y) of the pooled planes + tile partials of the largest level + per-level means
  size_t pooled = 0;
  int hh = h, ww = w;
  for (int l = 1; l < 5; ++l) { hh = (hh + 2 * (hh % 2) - 2) / 2 + 1; ww = (ww + 2 * (ww % 2) - 2) / 2 + 1; pooled += static_cast<size_t>(hh) * ww; }
  const size_t tiles = static_cast<size_t>((h + kTile - 1) / kTile) * ((w + kTile - 1) / kTile);
  return (2 * pooled * planes + tiles * planes * 2 + static_cast<size_t>(planes) * 5 * 2 + 64) * sizeof(float) + 1024;
}

size_t nic_ms_ssim_bwd_workspace_bytes(int32_t planes, int32_t h, int32_t w) {
  if (planes < 1 || h < 1 || w < 1) return 0;
  // the forward's workspace (its pooled pyramids are read back) + the gradients of the pooled levels 1-4
  size_t pooled = 0;
  int hh = h, ww = w;
  for (int l = 1; l < 5; ++l) { hh = (hh + 2 * (hh % 2) - 2) / 2 + 1; ww = (ww + 2 * (ww % 2) - 2) / 2 + 1; pooled += static_cast<size_t>(hh) * ww; }
  return nic_ms_ssim_workspace_bytes(planes, h, w) + pooled * planes * sizeof(float);
}

/*
 * level_means [5][planes][2] = (mean ssim, mean cs) of every scale; the caller combines them (prod relu(.)^w, mean over channels).
 */
int nic_ms_ssim_levels(const float* x, const float* y, int32_t planes, int32_t h, int32_t w, float data_range, int32_t clamp_y,
                       float* level_means, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (planes < 1 || h < 1 || w < 1) return fail(NIC_E_BADSHAPE, "ms_ssim: planes=%d h=%d w=%d", planes, h, w);
  if ((h < w ? h : w) <= (kWin - 1) * 16) return fail(NIC_E_BADSHAPE, "ms_ssim: the smaller side must exceed %d pixels (five scales of an 11-tap window)", (kWin - 1) * 16);
  if (!x || !y || !level_means) return fail(NIC_E_BADSHAPE, "ms_ssim: null pointer");
  const size_t need = nic_ms_ssim_workspace_bytes(planes, h, w);
  if (!workspace || workspace_bytes < need) return fail(NIC_E_WORKSPACE, "ms_ssim: workspace %zu < %zu bytes", workspace_bytes, need);
  if (int rc = ensure_gauss()) return rc;
  cudaStream_t st = as_stream(stream);
  const float c1 = (0.01f * data_range) * (0.01f * data_range), c2 = (0.03f * data_range) * (0.03f * data_range);
  float* ws = static_cast<float*>(workspace);
  const size_t tiles0 = static_cast<size_t>((h + kTile - 1) / kTile) * ((w + kTile - 1) / kTile);
  float* part = ws; ws += tiles0 * planes * 2;
  const float* cx = x; const float* cy = y;
  int ch = h, cw = w, clamp = clamp_y;
  for (int l = 0; l < 5; ++l) {
    const int ho = ch - kWin + 1, wo = cw - kWin + 1;
    dim3 grid((wo + kTile - 1) / kTile, (ho + kTile - 1) / kTile, planes);
    ssim_tile_kernel<<<grid, 256, 0, st>>>(cx, cy, ch, cw, c1, c2, clamp, part);
    if (int rc = check_launch("ssim_tile_kernel")) return rc;
    ssim_fold_kernel<<<planes, 32, 0, st>>>(part, static_cast<int>(grid.x * grid.y), 1.0f / (static_cast<float>(ho) * wo), level_means + static_cast<long>(l) * planes * 2);
    if (int rc = check_launch("ssim_fold_kernel")) return rc;
    if (l == 4) break;
    const int ph = ch % 2, pw = cw % 2;
    const int nh = (ch + 2 * ph - 2) / 2 + 1, nw = (cw + 2 * pw - 2) / 2 + 1;
    float* nx = ws; ws += static_cast<size_t>(planes) * nh * nw;
    float* ny = ws; ws += static_cast<size_t>(planes) * nh * nw;
    const long total = static_cast<long>(planes) * nh * nw;
    long blocks = (total + 255) / 256;
    if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
    avgpool2_kernel<<<static_cast<int>(blocks), 256, 0, st>>>(cx, nx, planes, ch, cw, ph, pw, nh, nw, 0);
    if (int rc = check_launch("avgpool2_kernel")) return rc;
    avgpool2_kernel<<<static_cast<int>(blocks), 256, 0, st>>>(cy, ny, planes, ch, cw, ph, pw, nh, nw, clamp);
    if (int rc = check_launch("avgpool2_kernel")) return rc;
    cx = nx; cy = ny; ch = nh; cw = nw; clamp = 0;
  }
  return NIC_OK;
}

/*
 * g_x [planes][h][w] = d loss / d x from g_level [5][planes] = d loss / d (mean cs of levels 0-3 | mean ssim of level 4).  The
 * workspace is the one nic_ms_ssim_levels(x, y, ..., clamp_y = 0) filled (same x, y, sizes, data_range), at least
 * nic_ms_ssim_bwd_workspace_bytes long: its pooled pyramids are read back, the level gradients go behind them.
 */
int nic_ms_ssim_bwd(const float* x, const float* y, int32_t planes, int32_t h, int32_t w, float data_range, const float* g_level,
                    float* g_x, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (planes < 1 || h < 1 || w < 1) return fail(NIC_E_BADSHAPE, "ms_ssim_bwd: planes=%d h=%d w=%d", planes, h, w);
  if ((h < w ? h : w) <= (kWin - 1) * 16) return fail(NIC_E_BADSHAPE, "ms_ssim_bwd: the smaller side must exceed %d pixels (five scales of an 11-tap window)", (kWin - 1) * 16);
  if (!x || !y || !g_level || !g_x) return fail(NIC_E_BADSHAPE, "ms_ssim_bwd: null pointer");
  const size_t need = nic_ms_ssim_bwd_workspace_bytes(planes, h, w);
  if (!workspace || workspace_bytes < need) return fail(NIC_E_WORKSPACE, "ms_ssim_bwd: workspace %zu < %zu bytes", workspace_bytes, need);
  if (int rc = ensure_gauss()) return rc;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(ms_ssim_bwd_tile_kernel), kBwdSmemBytes)) return rc;
  cudaStream_t st = as_stream(stream);
  const float c1 = (0.01f * data_range) * (0.01f * data_range), c2 = (0.03f * data_range) * (0.03f * data_range);
  // the forward's layout: tile partials, then (x_l, y_l) for l = 1..4; the level gradients start at the forward's size
  float* ws = static_cast<float*>(workspace);
  const size_t tiles0 = static_cast<size_t>((h + kTile - 1) / kTile) * ((w + kTile - 1) / kTile);
  const float* lx[5] = {x}; const float* ly[5] = {y};
  int lh[5] = {h}, lw[5] = {w};
  float* lg[5] = {g_x};
  float* pyr = ws + tiles0 * planes * 2;
  float* grad = reinterpret_cast<float*>(static_cast<char*>(workspace) + nic_ms_ssim_workspace_bytes(planes, h, w));
  for (int l = 1; l < 5; ++l) {
    lh[l] = (lh[l - 1] + 2 * (lh[l - 1] % 2) - 2) / 2 + 1; lw[l] = (lw[l - 1] + 2 * (lw[l - 1] % 2) - 2) / 2 + 1;
    const size_t n = static_cast<size_t>(planes) * lh[l] * lw[l];
    lx[l] = pyr; ly[l] = pyr + n; pyr += 2 * n;
    lg[l] = grad; grad += n;
  }
  for (int l = 4; l >= 0; --l) {
    dim3 grid((lw[l] + kBT - 1) / kBT, (lh[l] + kBT - 1) / kBT, planes);
    const float* gc = l < 4 ? lg[l + 1] : nullptr;
    const int hc = l < 4 ? lh[l + 1] : 0, wc = l < 4 ? lw[l + 1] : 0;
    ms_ssim_bwd_tile_kernel<<<grid, 256, kBwdSmemBytes, st>>>(lx[l], ly[l], lh[l], lw[l], c1, c2, l == 4, g_level + static_cast<long>(l) * planes,
                                                              gc, hc, wc, lh[l] % 2, lw[l] % 2, lg[l]);
    if (int rc = check_launch("ms_ssim_bwd_tile_kernel")) return rc;
  }
  return NIC_OK;
}

}  // extern "C"
