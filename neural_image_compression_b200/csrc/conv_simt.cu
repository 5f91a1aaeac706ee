// fp32 CUDA-core convolution engine (NIC_PREC_FP32): the parity-grade arm of nic_conv_fwd.
//
// One implicit-GEMM kernel over the tap-list formulation of conv_common.cuh:
//   C[M = pixels of one output phase, N = c_out] = sum over (tap, c_in) A . W
// CTA tile BM x BN with BK = 16, 256 threads, register micro-tiles, double-buffered shared memory
// (global loads for step i+1 are issued before the FFMAs of step i).  fp32 operands, fp32 FFMA
// accumulation, so results track the reference's CPU fp32 convolution to accumulation-order rounding.
// The tcgen05 arm (conv_tc.cu) is validated against this kernel on the GPU.
//
// Reference ops served: Components.py:10-16, 39-45, 69-73, 99-103; ContextModels.py:18-20;
// ParametersModels.py:29-35; GDN (compressai) as a 1x1 tap over x^2 with the x * rsqrt / sqrt epilogue.
#include <stdlib.h>
#include "conv_common.cuh"

namespace nic {

int validate_conv_desc(const nic_conv_desc* d) {
  if (!d) return fail(NIC_E_BADSHAPE, "conv: null descriptor");
  if (d->n < 0 || d->c_in < 1 || d->c_out < 1 || d->h_in < 1 || d->w_in < 1)
    return fail(NIC_E_BADSHAPE, "conv: bad extents n=%d c_in=%d c_out=%d h_in=%d w_in=%d", d->n, d->c_in, d->c_out, d->h_in, d->w_in);
  if (d->kh < 1 || d->kw < 1 || d->kh * d->kw > kMaxTaps) return fail(NIC_E_UNSUPPORTED, "conv: kernel %dx%d (max 25 taps)", d->kh, d->kw);
  if (d->stride != 1 && d->stride != 2) return fail(NIC_E_UNSUPPORTED, "conv: stride %d (1 or 2)", d->stride);
  if (d->pad < 0 || d->pad >= d->kh || d->pad >= d->kw) return fail(NIC_E_BADSHAPE, "conv: pad %d", d->pad);
  int ho, wo;
  if (d->transposed) {
    if (d->output_padding < 0 || d->output_padding >= d->stride + (d->stride == 1)) return fail(NIC_E_BADSHAPE, "conv: output_padding %d", d->output_padding);
    ho = (d->h_in - 1) * d->stride - 2 * d->pad + d->kh + d->output_padding;
    wo = (d->w_in - 1) * d->stride - 2 * d->pad + d->kw + d->output_padding;
    if (d->mask_a) return fail(NIC_E_UNSUPPORTED, "conv: masked transposed conv");
  } else {
    ho = (d->h_in + 2 * d->pad - d->kh) / d->stride + 1;
    wo = (d->w_in + 2 * d->pad - d->kw) / d->stride + 1;
  }
  if (ho != d->h_out || wo != d->w_out)
    return fail(NIC_E_BADSHAPE, "conv: output %dx%d does not match %dx%d implied by the input", d->h_out, d->w_out, ho, wo);
  if (d->out_c_total != 0 && (d->out_c_offset < 0 || d->out_c_offset + d->c_out > d->out_c_total))
    return fail(NIC_E_BADSHAPE, "conv: channel window [%d,+%d) outside %d", d->out_c_offset, d->c_out, d->out_c_total);
  if (d->epilogue < NIC_EPI_BIAS || d->epilogue > NIC_EPI_IGDN) return fail(NIC_E_BADSHAPE, "conv: epilogue %d", d->epilogue);
  if (d->mask_a == NIC_MASK_CHECKERBOARD && (d->stride != 1 || d->epilogue != NIC_EPI_BIAS))
    return fail(NIC_E_UNSUPPORTED, "conv: the checkerboard context needs stride 1 and the bias epilogue");
  return NIC_OK;
}

int build_tap_table(const nic_conv_desc* d, TapTable* t) {
  if (int rc = validate_conv_desc(d)) return rc;
  *t = TapTable{};
  int q = 0;
  if (!d->transposed) {
    t->nphases = 1; t->in_stride = d->stride; t->out_stride = 1;
    t->py[0] = t->px[0] = 0; t->phase_begin[0] = 0;
    for (int kh = 0; kh < d->kh; ++kh)
      for (int kw = 0; kw < d->kw; ++kw) {
        if (d->mask_a == NIC_MASK_CHECKERBOARD) {
          if (!((kh + kw) & 1)) continue;                      // checkerboard: only the odd-parity taps, which read anchors
        } else if (d->mask_a && !(kh < d->kh / 2 || (kh == d->kh / 2 && kw < d->kw / 2 + (d->mask_a == 2 ? 1 : 0)))) {
          continue;                                            // 'A'; 2 = 'B': centre tap kept
        }
        t->dy[q] = kh - d->pad; t->dx[q] = kw - d->pad; t->kh[q] = kh; t->kw[q] = kw; ++q;
      }
    t->phase_begin[1] = q;
  } else {
    const int s = d->stride;
    t->nphases = s * s; t->in_stride = 1; t->out_stride = s;
    int ph = 0;
    for (int py = 0; py < s; ++py)
      for (int px = 0; px < s; ++px, ++ph) {
        t->py[ph] = py; t->px[ph] = px; t->phase_begin[ph] = q;
        for (int kh = 0; kh < d->kh; ++kh) {
          const int ny = py + d->pad - kh;
          if (((ny % s) + s) % s != 0) continue;
          for (int kw = 0; kw < d->kw; ++kw) {
            const int nx = px + d->pad - kw;
            if (((nx % s) + s) % s != 0) continue;
            // exact division (numerator is a multiple of s, possibly negative)
            t->dy[q] = (ny >= 0) ? ny / s : -((-ny) / s);
            t->dx[q] = (nx >= 0) ? nx / s : -((-nx) / s);
            t->kh[q] = kh; t->kw[q] = kw; ++q;
          }
        }
      }
    t->phase_begin[ph] = q;
  }
  t->ntaps = q;
  return NIC_OK;
}

// ---------------------------------------------------------------------------------------------
// weight packing
// ---------------------------------------------------------------------------------------------

// fp32: [tap][c_in][c_out]
__global__ void pack_weight_f32_kernel(const float* __restrict__ w, float* __restrict__ out, int cin, int cout,
                                       int kh, int kw, int transposed, TapTable tt) {
  const long total = static_cast<long>(tt.ntaps) * cin * cout;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int co = static_cast<int>(i % cout);
    const int ci = static_cast<int>((i / cout) % cin);
    const int t = static_cast<int>(i / (static_cast<long>(cout) * cin));
    const int a = tt.kh[t], b = tt.kw[t];
    const long src = transposed ? ((static_cast<long>(ci) * cout + co) * kh + a) * kw + b
                                : ((static_cast<long>(co) * cin + ci) * kh + a) * kw + b;
    out[i] = w[src];
  }
}

// GDN reparametrisation (oracle/gdn.py); gamma transposed to [j (input channel)][i (output channel)]
__global__ void pack_gdn_f32_kernel(int c, float beta_bound, float gamma_bound, float pedestal,
                                    const float* __restrict__ beta, const float* __restrict__ gamma,
                                    float* __restrict__ beta_eff, float* __restrict__ gamma_t) {
  const int total = c * c;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int row = i / c, col = i % c;             // gamma[row = out i][col = in j]
    const float g = fmaxf(gamma[i], gamma_bound);
    gamma_t[col * c + row] = g * g - pedestal;
    if (i < c) { const float b = fmaxf(beta[i], beta_bound); beta_eff[i] = b * b - pedestal; }
  }
}

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------

struct SimtParams {
  const float* x; const float* w; const float* bias; float* y;
  int n, cin, hin, win, cout, hout, wout;
  long xs_n, xs_c, xs_h, xs_w;
  long ys_n, ys_c, ys_h, ys_w;
  int epilogue;       // NIC_EPI_*; GDN / IGDN here mean "x * rsqrt/sqrt(acc + bias)" with x read back from the input
  int a_square;       // square the A operand on load (GDN's x^2)
  int out_bf16;       // 1: store the result as bf16 (hand-off to the tensor-core arm); strides are still in elements
                      // 2: store it as a bf16 pair, hi at channel c and lo at channel c + split_off (NIC_DT_BF16X2)
  long split_off;     // element offset of the lo half (= c_out * ys_c)
  TapTable tt;
};

constexpr int BK = 16;

template <int BM, int BN, int TM, int TN, bool GATHER>
__global__ void __launch_bounds__(256, 2)
conv_simt_kernel(const SimtParams p) {
  constexpr int HM = TM / 2, HN = TN / 2;          // each micro-tile is two half-tiles BM/2 (BN/2) apart
  constexpr int TX = BN / TN;                      // threads along N
  static_assert((BM / TM) * (BN / TN) == 256, "256 threads");
  __shared__ __align__(16) float As[2][BK][BM];
  __shared__ __align__(16) float Bs[2][BK][BN];

  const int tid = threadIdx.x;
  const int phase = blockIdx.z;
  const int is = p.tt.in_stride, os = p.tt.out_stride;
  const int py = p.tt.py[phase], px = p.tt.px[phase];
  const int hp = (p.hout - py + os - 1) / os, wp = (p.wout - px + os - 1) / os;
  const long P = static_cast<long>(p.n) * hp * wp;
  const long m0 = static_cast<long>(blockIdx.x) * BM;
  if (m0 >= P) return;
  const int n0 = blockIdx.y * BN;
  const int tap0 = p.tt.phase_begin[phase], tap1 = p.tt.phase_begin[phase + 1];
  const int ktotal = (tap1 - tap0) * p.cin;        // flattened K of this phase
  const long krow0 = static_cast<long>(tap0) * p.cin;
  const int steps = (ktotal + BK - 1) / BK;

  // ---- A loader state -----------------------------------------------------------------------
  // vector path: 2 (BM=128) rows per thread, float4 along c_in (NHWC, c_in % 16 == 0)
  // gather path: rows m = tid % BM, k = tid / BM + (256/BM) * j, scalar loads with arbitrary strides
  constexpr int AV_ROWS = BM * BK / 4 / 256;       // float4 per thread
  constexpr int AG_PER = BM * BK / 256;            // scalars per thread
  int a_img[GATHER ? 1 : AV_ROWS], a_oy[GATHER ? 1 : AV_ROWS], a_ox[GATHER ? 1 : AV_ROWS];
  if (GATHER) {
    const long m = m0 + (tid % BM);
    if (m < P) { a_ox[0] = static_cast<int>(m % wp); a_oy[0] = static_cast<int>((m / wp) % hp); a_img[0] = static_cast<int>(m / (static_cast<long>(wp) * hp)); }
    else a_img[0] = -1;
  } else {
#pragma unroll
    for (int j = 0; j < AV_ROWS; ++j) {
      const long m = m0 + (tid >> 2) + 64 * j;
      if (m < P) { a_ox[j] = static_cast<int>(m % wp); a_oy[j] = static_cast<int>((m / wp) % hp); a_img[j] = static_cast<int>(m / (static_cast<long>(wp) * hp)); }
      else a_img[j] = -1;
    }
  }
  float4 a_reg4[GATHER ? 1 : AV_ROWS];
  float a_reg[GATHER ? AG_PER : 1];
  constexpr int BV = (BN % 4 == 0 && BN >= 128) ? BK * BN / 4 / 256 : 0;   // float4 per thread for B (BN = 128)
  constexpr int BS = (BV == 0) ? BK * BN / 256 : 0;                         // scalars per thread for B (BN = 16)
  float4 b_reg4[BV ? BV : 1];
  float b_reg[BS ? BS : 1];

  auto load_global = [&](int step) {
    const int kbase = step * BK;
    if (GATHER) {
#pragma unroll
      for (int j = 0; j < AG_PER; ++j) {
        const int kk = kbase + (tid / BM) + (256 / BM) * j;
        float v = 0.f;
        if (kk < ktotal && a_img[0] >= 0) {
          const int t = tap0 + kk / p.cin, c = kk % p.cin;
          const int iy = a_oy[0] * is + p.tt.dy[t], ix = a_ox[0] * is + p.tt.dx[t];
          if (iy >= 0 && iy < p.hin && ix >= 0 && ix < p.win)
            v = __ldg(p.x + a_img[0] * p.xs_n + c * p.xs_c + iy * p.xs_h + ix * p.xs_w);
        }
        a_reg[j] = p.a_square ? v * v : v;
      }
    } else {
      const int t = tap0 + kbase / p.cin, c0 = kbase % p.cin + (tid & 3) * 4;
#pragma unroll
      for (int j = 0; j < AV_ROWS; ++j) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a_img[j] >= 0) {
          const int iy = a_oy[j] * is + p.tt.dy[t], ix = a_ox[j] * is + p.tt.dx[t];
          if (iy >= 0 && iy < p.hin && ix >= 0 && ix < p.win)
            v = __ldg(reinterpret_cast<const float4*>(p.x + a_img[j] * p.xs_n + iy * p.xs_h + ix * p.xs_w + c0));
        }
        if (p.a_square) { v.x *= v.x; v.y *= v.y; v.z *= v.z; v.w *= v.w; }
        a_reg4[j] = v;
      }
    }
    if (BV) {
#pragma unroll
      for (int j = 0; j < BV; ++j) {
        const int k = kbase + (tid >> 5) + 8 * j, col = n0 + (tid & 31) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < ktotal && col < p.cout) v = __ldg(reinterpret_cast<const float4*>(p.w + (krow0 + k) * p.cout + col));
        b_reg4[j] = v;
      }
    } else {
#pragma unroll
      for (int j = 0; j < BS; ++j) {
        const int e = tid + 256 * j;
        const int k = kbase + e / BN, col = n0 + e % BN;
        b_reg[j] = (k < ktotal && col < p.cout) ? __ldg(p.w + (krow0 + k) * p.cout + col) : 0.f;
      }
    }
  };
  auto store_smem = [&](int buf) {
    if (GATHER) {
#pragma unroll
      for (int j = 0; j < AG_PER; ++j) As[buf][(tid / BM) + (256 / BM) * j][tid % BM] = a_reg[j];
    } else {
#pragma unroll
      for (int j = 0; j < AV_ROWS; ++j) {
        const int m = (tid >> 2) + 64 * j, k = (tid & 3) * 4;
        As[buf][k + 0][m] = a_reg4[j].x; As[buf][k + 1][m] = a_reg4[j].y;
        As[buf][k + 2][m] = a_reg4[j].z; As[buf][k + 3][m] = a_reg4[j].w;
      }
    }
    if (BV) {
#pragma unroll
      for (int j = 0; j < BV; ++j)
        *reinterpret_cast<float4*>(&Bs[buf][(tid >> 5) + 8 * j][(tid & 31) * 4]) = b_reg4[j];
    } else {
#pragma unroll
      for (int j = 0; j < BS; ++j) { const int e = tid + 256 * j; Bs[buf][e / BN][e % BN] = b_reg[j]; }
    }
  };

  const int ty = tid / TX, tx = tid % TX;
  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  load_global(0);
  store_smem(0);
  __syncthreads();
  for (int step = 0; step < steps; ++step) {
    const int buf = step & 1;
    if (step + 1 < steps) load_global(step + 1);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[TM], b[TN];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (HM == 4) {
          const float4 v = *reinterpret_cast<const float4*>(&As[buf][k][h * (BM / 2) + ty * HM]);
          a[h * HM + 0] = v.x; a[h * HM + 1] = v.y; a[h * HM + 2] = v.z; a[h * HM + 3] = v.w;
        } else {
#pragma unroll
          for (int i = 0; i < HM; ++i) a[h * HM + i] = As[buf][k][h * (BM / 2) + ty * HM + i];
        }
        if (HN == 4) {
          const float4 v = *reinterpret_cast<const float4*>(&Bs[buf][k][h * (BN / 2) + tx * HN]);
          b[h * HN + 0] = v.x; b[h * HN + 1] = v.y; b[h * HN + 2] = v.z; b[h * HN + 3] = v.w;
        } else {
#pragma unroll
          for (int i = 0; i < HN; ++i) b[h * HN + i] = Bs[buf][k][h * (BN / 2) + tx * HN + i];
        }
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (step + 1 < steps) store_smem(buf ^ 1);
    __syncthreads();
  }

  // ---- epilogue -------------------------------------------------------------------------------
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int r = (i / HM) * (BM / 2) + ty * HM + (i % HM);
    const long m = m0 + r;
    if (m >= P) continue;
    const int ox = static_cast<int>(m % wp), oy = static_cast<int>((m / wp) % hp);
    const int img = static_cast<int>(m / (static_cast<long>(wp) * hp));
    const long yoff = img * p.ys_n + static_cast<long>(oy * os + py) * p.ys_h + static_cast<long>(ox * os + px) * p.ys_w;
    float* yrow = p.y + yoff;
    __nv_bfloat16* yrow_b = reinterpret_cast<__nv_bfloat16*>(p.y) + yoff;
    const float* xrow = p.x + img * p.xs_n + static_cast<long>(oy) * p.xs_h + static_cast<long>(ox) * p.xs_w;  // GDN: same pixel
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int cbase = n0 + h * (BN / 2) + tx * HN;
      float v[HN];
#pragma unroll
      for (int j = 0; j < HN; ++j) {
        const int c = cbase + j;
        float t = acc[i][h * HN + j];
        if (c < p.cout) {
          t += __ldg(p.bias + c);
          if (p.epilogue == NIC_EPI_LRELU) t = t > 0.f ? t : t * 0.01f;
          else if (p.epilogue == NIC_EPI_GDN) t = __ldg(xrow + c * p.xs_c) * (1.0f / sqrtf(t));
          else if (p.epilogue == NIC_EPI_IGDN) t = __ldg(xrow + c * p.xs_c) * sqrtf(t);
        }
        v[j] = t;
      }
      if (p.out_bf16) {
#pragma unroll
        for (int j = 0; j < HN; ++j)
          if (cbase + j < p.cout) {
            const __nv_bfloat16 hi = __float2bfloat16_rn(v[j]);
            yrow_b[(cbase + j) * p.ys_c] = hi;
            if (p.out_bf16 == 2) yrow_b[(cbase + j) * p.ys_c + p.split_off] = __float2bfloat16_rn(v[j] - __bfloat162float(hi));
          }
      } else if (HN == 4 && p.ys_c == 1 && cbase + 3 < p.cout && ((reinterpret_cast<uintptr_t>(yrow + cbase) & 15) == 0)) {
        *reinterpret_cast<float4*>(yrow + cbase) = make_float4(v[0], v[1], v[2], v[3]);
      } else {
#pragma unroll
        for (int j = 0; j < HN; ++j) if (cbase + j < p.cout) yrow[(cbase + j) * p.ys_c] = v[j];
      }
    }
  }
}

// Few-input-channel convs to 128 output channels (the RGB-input convs of the 3x3 residual family's first block: Conv2d(3, 128, 3, s2)
// and its 1x1 stride-2 skip, Layers.py:38-47).  The register-tiled kernel above spends its time gathering K = 27 (or 3) operands per
// pixel into 16-deep K slabs: 396 + 339 us for 4 x 512 x 768 images against an output-write floor of ~40 us each.  Here a warp owns
// one output pixel at a time, lane l its channels 4 l .. 4 l + 3 with their KT x 4 weights in registers; the KT inputs of the pixel
// are fetched by lanes 0 .. KT - 1 with one load instruction and handed round by shuffles, the result leaves as one 512-byte row.
// fp32 FMAs in ascending k, bias last - the same sum.
template <int KT>
__global__ void __launch_bounds__(128)
conv_smallcin_kernel(const SimtParams p) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const int cin = p.cin, kt = p.tt.ntaps * cin;
  float4 w[KT];
#pragma unroll
  for (int k = 0; k < KT; ++k)
    w[k] = k < kt ? __ldg(reinterpret_cast<const float4*>(p.w + static_cast<long>(k) * p.cout) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
  const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias) + lane);
  // lane k fetches operand k = (tap, input channel) of the pixel: ONE load instruction per pixel and warp, issued a pixel ahead;
  // the FMA loop takes the operands by shuffle
  const int my_t = lane < kt ? lane / cin : 0, my_c = lane < kt ? lane - my_t * cin : 0;
  const int my_dy = p.tt.dy[my_t], my_dx = p.tt.dx[my_t];
  const long my_coff = my_c * p.xs_c;
  const int is = p.tt.in_stride;
  const int pixels = p.n * p.hout * p.wout, hw = p.wout * p.hout;       // host: < 2^31 (32-bit index arithmetic: no emulated divisions)
  auto fetch = [&](int pix) -> float {
    if (pix >= pixels || lane >= kt) return 0.f;
    const int img = pix / hw, r = pix - img * hw, oy = r / p.wout, ox = r - oy * p.wout;
    const int iy = oy * is + my_dy, ix = ox * is + my_dx;
    return (iy >= 0 && iy < p.hin && ix >= 0 && ix < p.win) ? __ldg(p.x + img * p.xs_n + my_coff + iy * p.xs_h + ix * p.xs_w) : 0.f;
  };
  // PB consecutive pixels per warp and round: their PB loads are in flight together (one load a pixel ahead left every round
  // waiting out a full memory latency: 271 us at K = 27; the arithmetic of a pixel is ~150 issue slots)
  constexpr int PB = 8;
  for (int base = warp * PB; base < pixels; base += nwarps * PB) {
    float v[PB];
#pragma unroll
    for (int j = 0; j < PB; ++j) v[j] = fetch(base + j);
#pragma unroll
    for (int j = 0; j < PB; ++j) {
      const int pix = base + j;
      if (pix >= pixels) break;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int k = 0; k < KT; ++k) {
        const float a = __shfl_sync(0xffffffffu, v[j], k);
        acc.x = fmaf(a, w[k].x, acc.x); acc.y = fmaf(a, w[k].y, acc.y); acc.z = fmaf(a, w[k].z, acc.z); acc.w = fmaf(a, w[k].w, acc.w);
      }
      acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w;
      if (p.epilogue == NIC_EPI_LRELU) {
        acc.x = acc.x > 0.f ? acc.x : acc.x * 0.01f; acc.y = acc.y > 0.f ? acc.y : acc.y * 0.01f;
        acc.z = acc.z > 0.f ? acc.z : acc.z * 0.01f; acc.w = acc.w > 0.f ? acc.w : acc.w * 0.01f;
      }
      const int img = pix / hw, r = pix - img * hw, oy = r / p.wout, ox = r - oy * p.wout;
      __stcs(reinterpret_cast<float4*>(p.y + img * p.ys_n + oy * p.ys_h + ox * p.ys_w + lane * 4), acc);
    }
  }
}

static int launch_simt(const SimtParams& p, cudaStream_t st);
static void set_strides(int layout, long c, long h, long w, long* sn, long* sc, long* sh, long* sw) {
  if (layout == NIC_LAYOUT_NCHW) { *sn = c * h * w; *sc = h * w; *sh = w; *sw = 1; }
  else { *sn = h * w * c; *sh = w * c; *sw = c; *sc = 1; }
}

static int launch_simt(const SimtParams& p, cudaStream_t st) {
  long maxP = 0;
  for (int ph = 0; ph < p.tt.nphases; ++ph) {
    const int os = p.tt.out_stride;
    const long hp = (p.hout - p.tt.py[ph] + os - 1) / os, wp = (p.wout - p.tt.px[ph] + os - 1) / os;
    const long P = static_cast<long>(p.n) * hp * wp;
    if (P > maxP) maxP = P;
  }
  if (maxP == 0) return NIC_OK;
  const int kt = p.tt.ntaps * p.cin;
  const char* sc_env = getenv("NIC_SMALLCIN");                       // A/B switch: 0 = the register-tiled kernel for these layers too
  if (p.tt.nphases == 1 && p.tt.out_stride == 1 && p.cin <= 4 && p.cout == 128 && kt <= 27 && !p.a_square && !p.out_bf16 &&
      (p.epilogue == NIC_EPI_BIAS || p.epilogue == NIC_EPI_LRELU) && p.ys_c == 1 && p.ys_w % 4 == 0 && p.ys_h % 4 == 0 && p.ys_n % 4 == 0 &&
      ((reinterpret_cast<uintptr_t>(p.y) | reinterpret_cast<uintptr_t>(p.w) | reinterpret_cast<uintptr_t>(p.bias)) & 15) == 0 &&
      !(sc_env && atoi(sc_env) == 0)) {
    const long pixels = static_cast<long>(p.n) * p.hout * p.wout;
    if (pixels + kNumSMs * 12L * 4 >= 0x7fffffffL) return fail(NIC_E_BADSHAPE, "conv fp32: %ld output pixels", pixels);
    long blocks = (pixels + 31) / 32;                                 // 4 warps per block (142 registers: 3 blocks per SM), one pixel per warp and iteration
    if (blocks > kNumSMs * 12) blocks = kNumSMs * 12;
    if (kt <= 3) conv_smallcin_kernel<3><<<static_cast<unsigned>(blocks), 128, 0, st>>>(p);
    else if (kt <= 12) conv_smallcin_kernel<12><<<static_cast<unsigned>(blocks), 128, 0, st>>>(p);
    else conv_smallcin_kernel<27><<<static_cast<unsigned>(blocks), 128, 0, st>>>(p);
    return check_launch("conv_smallcin_kernel");
  }
  const bool gather = (p.xs_c != 1) || (p.cin % BK != 0) || ((reinterpret_cast<uintptr_t>(p.x) & 15) != 0) ||
                      (p.xs_w % 4 != 0) || (p.xs_h % 4 != 0) || (p.xs_n % 4 != 0);
  const bool small_n = p.cout <= 16;
  const bool wvec = (p.cout % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.w) & 15) == 0);
  if (!small_n && !wvec) return fail(NIC_E_UNSUPPORTED, "conv fp32: c_out=%d must be <= 16 or a multiple of 4", p.cout);
  dim3 block(256);
  if (small_n) {
    dim3 grid(static_cast<unsigned>((maxP + 127) / 128), 1, p.tt.nphases);
    if (gather) conv_simt_kernel<128, 16, 2, 4, true><<<grid, block, 0, st>>>(p);
    else conv_simt_kernel<128, 16, 2, 4, false><<<grid, block, 0, st>>>(p);
  } else {
    dim3 grid(static_cast<unsigned>((maxP + 127) / 128), (p.cout + 127) / 128, p.tt.nphases);
    if (gather) conv_simt_kernel<128, 128, 8, 8, true><<<grid, block, 0, st>>>(p);
    else conv_simt_kernel<128, 128, 8, 8, false><<<grid, block, 0, st>>>(p);
  }
  return check_launch("conv_simt_kernel");
}

// conv + bias (+ LeakyReLU) with f32 input, optional bf16 NHWC output: used by the tensor-core arm for the 3-channel first layer
int conv_fwd_fp32_ex(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias, void* y, int out_bf16_nhwc,
                     cudaStream_t st) {
  SimtParams p{};
  if (int rc = build_tap_table(d, &p.tt)) return rc;
  p.n = d->n; p.cin = d->c_in; p.hin = d->h_in; p.win = d->w_in; p.cout = d->c_out; p.hout = d->h_out; p.wout = d->w_out;
  p.x = static_cast<const float*>(x); p.w = static_cast<const float*>(w_packed); p.bias = bias; p.y = static_cast<float*>(y);
  set_strides(d->in_layout, d->c_in, d->h_in, d->w_in, &p.xs_n, &p.xs_c, &p.xs_h, &p.xs_w);
  set_strides(out_bf16_nhwc ? NIC_LAYOUT_NHWC : d->out_layout, d->c_out, d->h_out, d->w_out, &p.ys_n, &p.ys_c, &p.ys_h, &p.ys_w);
  p.epilogue = d->epilogue; p.a_square = 0; p.out_bf16 = out_bf16_nhwc;
  return launch_simt(p, st);
}

// fp32 arm of nic_conv_fwd
int conv_fwd_fp32(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias,
                  const void* gdn_gamma, const float* gdn_beta, void* y, void* workspace, size_t workspace_bytes,
                  cudaStream_t st) {
  const bool split_out = d->out_dtype == NIC_DT_BF16X2;
  if (d->in_dtype != NIC_DT_F32 || (d->out_dtype != NIC_DT_F32 && !split_out)) return fail(NIC_E_UNSUPPORTED, "conv fp32: f32 in, f32 or bf16-pair out");
  if (split_out && (d->out_layout != NIC_LAYOUT_NHWC || d->out_c_total != 0)) return fail(NIC_E_UNSUPPORTED, "conv fp32: bf16-pair output is plain NHWC");
  SimtParams p{};
  if (int rc = build_tap_table(d, &p.tt)) return rc;
  p.n = d->n; p.cin = d->c_in; p.hin = d->h_in; p.win = d->w_in; p.cout = d->c_out; p.hout = d->h_out; p.wout = d->w_out;
  p.x = static_cast<const float*>(x); p.w = static_cast<const float*>(w_packed); p.bias = bias;
  set_strides(d->in_layout, d->c_in, d->h_in, d->w_in, &p.xs_n, &p.xs_c, &p.xs_h, &p.xs_w);
  const int ctot = split_out ? 2 * d->c_out : (d->out_c_total ? d->out_c_total : d->c_out);
  long ys_n, ys_c, ys_h, ys_w;
  set_strides(d->out_layout, ctot, d->h_out, d->w_out, &ys_n, &ys_c, &ys_h, &ys_w);
  float* yout = static_cast<float*>(y) + d->out_c_offset * ys_c;
  const bool gdn = d->epilogue == NIC_EPI_GDN || d->epilogue == NIC_EPI_IGDN;
  if (!gdn) {
    p.y = yout; p.ys_n = ys_n; p.ys_c = ys_c; p.ys_h = ys_h; p.ys_w = ys_w;
    p.epilogue = d->epilogue; p.a_square = 0;
    if (split_out) { p.out_bf16 = 2; p.split_off = d->c_out; }
    return launch_simt(p, st);
  }
  // conv + bias into the workspace (NHWC f32), then the GDN contraction as a 1x1 tap over its squares
  const size_t need = static_cast<size_t>(d->n) * d->h_out * d->w_out * d->c_out * sizeof(float);
  if (!workspace || workspace_bytes < need) return fail(NIC_E_WORKSPACE, "conv fp32 + GDN: workspace %zu < %zu bytes", workspace_bytes, need);
  if (!gdn_gamma || !gdn_beta) return fail(NIC_E_BADSHAPE, "conv: GDN epilogue without gamma/beta");
  float* tmp = static_cast<float*>(workspace);
  p.y = tmp; set_strides(NIC_LAYOUT_NHWC, d->c_out, d->h_out, d->w_out, &p.ys_n, &p.ys_c, &p.ys_h, &p.ys_w);
  p.epilogue = NIC_EPI_BIAS; p.a_square = 0;
  if (int rc = launch_simt(p, st)) return rc;
  SimtParams g{};
  nic_conv_desc gd{};
  gd.n = d->n; gd.c_in = gd.c_out = d->c_out; gd.h_in = gd.h_out = d->h_out; gd.w_in = gd.w_out = d->w_out;
  gd.kh = gd.kw = 1; gd.stride = 1;
  if (int rc = build_tap_table(&gd, &g.tt)) return rc;
  g.n = d->n; g.cin = g.cout = d->c_out; g.hin = g.hout = d->h_out; g.win = g.wout = d->w_out;
  g.x = tmp; g.w = static_cast<const float*>(gdn_gamma); g.bias = gdn_beta; g.y = yout;
  g.xs_n = p.ys_n; g.xs_c = p.ys_c; g.xs_h = p.ys_h; g.xs_w = p.ys_w;
  g.ys_n = ys_n; g.ys_c = ys_c; g.ys_h = ys_h; g.ys_w = ys_w;
  g.epilogue = d->epilogue; g.a_square = 1;
  if (split_out) { g.out_bf16 = 2; g.split_off = d->c_out; }
  return launch_simt(g, st);
}

// GDN / IGDN of an fp32 NHWC tensor into a bf16-pair NHWC tensor (second half of a bf16x3 GDN layer)
int gdn_fwd_fp32_split(const float* x, int n, int c, int h, int w, int inverse, const float* gamma, const float* beta, void* y,
                       cudaStream_t st) {
  SimtParams g{};
  nic_conv_desc gd{};
  gd.n = n; gd.c_in = gd.c_out = c; gd.h_in = gd.h_out = h; gd.w_in = gd.w_out = w; gd.kh = gd.kw = 1; gd.stride = 1;
  if (int rc = build_tap_table(&gd, &g.tt)) return rc;
  g.n = n; g.cin = g.cout = c; g.hin = g.hout = h; g.win = g.wout = w;
  g.x = x; g.w = gamma; g.bias = beta; g.y = static_cast<float*>(y);
  set_strides(NIC_LAYOUT_NHWC, c, h, w, &g.xs_n, &g.xs_c, &g.xs_h, &g.xs_w);
  set_strides(NIC_LAYOUT_NHWC, 2 * c, h, w, &g.ys_n, &g.ys_c, &g.ys_h, &g.ys_w);
  g.epilogue = inverse ? NIC_EPI_IGDN : NIC_EPI_GDN; g.a_square = 1; g.out_bf16 = 2; g.split_off = c;
  return launch_simt(g, st);
}

int gdn_fwd_fp32(const float* x, int n, int c, int h, int w, int layout, int inverse, const float* gamma, const float* beta,
                 float* y, cudaStream_t st) {
  SimtParams g{};
  nic_conv_desc gd{};
  gd.n = n; gd.c_in = gd.c_out = c; gd.h_in = gd.h_out = h; gd.w_in = gd.w_out = w; gd.kh = gd.kw = 1; gd.stride = 1;
  if (int rc = build_tap_table(&gd, &g.tt)) return rc;
  g.n = n; g.cin = g.cout = c; g.hin = g.hout = h; g.win = g.wout = w;
  g.x = x; g.w = gamma; g.bias = beta; g.y = y;
  set_strides(layout, c, h, w, &g.xs_n, &g.xs_c, &g.xs_h, &g.xs_w);
  g.ys_n = g.xs_n; g.ys_c = g.xs_c; g.ys_h = g.xs_h; g.ys_w = g.xs_w;
  g.epilogue = inverse ? NIC_EPI_IGDN : NIC_EPI_GDN; g.a_square = 1;
  return launch_simt(g, st);
}

// y[pixels][c_out] = epilogue((x or x^2)[pixels][c_in] . w[c_in][c_out] + bias): the channel-mixing contraction the GDN
// backward (backward.cu) reuses for the norm and for gamma^T . t.  NIC_EPI_GDN / IGDN read x back as the multiplicand.
int conv1x1_fp32(const float* x, long pixels, int cin, int cout, const float* w, const float* bias, float* y, int a_square,
                 int epilogue, cudaStream_t st) {
  if (pixels > 0x7fffffffL) return fail(NIC_E_BADSHAPE, "conv1x1: %ld pixels", pixels);
  SimtParams g{};
  nic_conv_desc gd{};
  gd.n = 1; gd.c_in = cin; gd.c_out = cout; gd.h_in = gd.h_out = 1; gd.w_in = gd.w_out = static_cast<int>(pixels);
  gd.kh = gd.kw = 1; gd.stride = 1;
  if (int rc = build_tap_table(&gd, &g.tt)) return rc;
  g.n = 1; g.cin = cin; g.cout = cout; g.hin = g.hout = 1; g.win = g.wout = static_cast<int>(pixels);
  g.x = x; g.w = w; g.bias = bias; g.y = y;
  set_strides(NIC_LAYOUT_NHWC, cin, 1, pixels, &g.xs_n, &g.xs_c, &g.xs_h, &g.xs_w);
  set_strides(NIC_LAYOUT_NHWC, cout, 1, pixels, &g.ys_n, &g.ys_c, &g.ys_h, &g.ys_w);
  g.epilogue = epilogue; g.a_square = a_square;
  return launch_simt(g, st);
}

// ---------------------------------------------------------------------------------------------
// latent hand-off (Models.py:52-66)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
latent_handoff_kernel(const float* __restrict__ v, int n, int c, int h, int w, int qmode, const float* __restrict__ noise,
                      float* __restrict__ v_nchw, float* __restrict__ vin_nchw, void* __restrict__ vin_nhwc, int out_dtype,
                      __nv_bfloat16* __restrict__ v_lowp, int lowp_dtype, int* __restrict__ lo_nonzero) {
  // 32 x 32 (pixel x channel) transpose tiles through shared memory: coalesced on both layouts
  __shared__ float tile[32][33];
  __shared__ float tile_q[32][33];
  const int hw = h * w;
  const int img = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, tyy = threadIdx.x >> 5;   // 8 rows per pass
  for (int r = tyy; r < 32; r += 8) {
    const int pix = p0 + r, ch = c0 + tx;
    float val = 0.f;
    if (pix < hw && ch < c) {
      val = v[(static_cast<long>(img) * hw + pix) * c + ch];
      if (v_lowp) {
        const __nv_bfloat16 hi = __float2bfloat16_rn(val);
        if (lowp_dtype == NIC_DT_BF16X2) {
          v_lowp[(static_cast<long>(img) * hw + pix) * 2 * c + ch] = hi;
          v_lowp[(static_cast<long>(img) * hw + pix) * 2 * c + c + ch] = __float2bfloat16_rn(val - __bfloat162float(hi));
        } else {
          v_lowp[(static_cast<long>(img) * hw + pix) * c + ch] = hi;
        }
      }
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
  if (vin_nhwc) {
    for (int r = tyy; r < 32; r += 8) {
      const int pix = p0 + r, ch = c0 + tx;
      if (pix < hw && ch < c) {
        const long o = (static_cast<long>(img) * hw + pix) * c + ch;
        if (out_dtype == NIC_DT_BF16) static_cast<__nv_bfloat16*>(vin_nhwc)[o] = __float2bfloat16_rn(tile_q[r][tx]);
        else if (out_dtype == NIC_DT_BF16X2) {
          const long o2 = (static_cast<long>(img) * hw + pix) * 2 * c + ch;
          const __nv_bfloat16 hi = __float2bfloat16_rn(tile_q[r][tx]);
          const float lo = tile_q[r][tx] - __bfloat162float(hi);
          static_cast<__nv_bfloat16*>(vin_nhwc)[o2] = hi;
          static_cast<__nv_bfloat16*>(vin_nhwc)[o2 + c] = __float2bfloat16_rn(lo);
          if (lo_nonzero && lo != 0.f) *lo_nonzero = 1;          // integer symbols below 256 split exactly: lo stays all zero
        } else static_cast<float*>(vin_nhwc)[o] = tile_q[r][tx];
      }
    }
  }
}

}  // namespace nic

using namespace nic;

extern "C" {

int nic_gdn_fwd(const float* x, int32_t n, int32_t c, int32_t h, int32_t w, int32_t layout, int32_t inverse,
                const float* gamma_packed, const float* beta_eff, float* y, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || c < 1 || h < 1 || w < 1 || !x || !y || !gamma_packed || !beta_eff) return fail(NIC_E_BADSHAPE, "gdn: bad arguments");
  if (n == 0) return NIC_OK;
  return gdn_fwd_fp32(x, n, c, h, w, layout, inverse, gamma_packed, beta_eff, y, as_stream(stream));
}

int nic_latent_handoff(const float* v_nhwc, int32_t n, int32_t c, int32_t h, int32_t w, int32_t qmode,
                       const float* noise_nchw, float* v_nchw, float* v_in_nchw, void* v_in_nhwc,
                       int32_t out_dtype, void* v_nhwc_lowp, int32_t lowp_dtype, void* stream) {
  return nic_latent_handoff_ex(v_nhwc, n, c, h, w, qmode, noise_nchw, v_nchw, v_in_nchw, v_in_nhwc, out_dtype, v_nhwc_lowp, lowp_dtype, nullptr, stream);
}

int nic_latent_handoff_ex(const float* v_nhwc, int32_t n, int32_t c, int32_t h, int32_t w, int32_t qmode,
                          const float* noise_nchw, float* v_nchw, float* v_in_nchw, void* v_in_nhwc,
                          int32_t out_dtype, void* v_nhwc_lowp, int32_t lowp_dtype, int32_t* in_lo_nonzero, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (n < 0 || c < 1 || h < 1 || w < 1) return fail(NIC_E_BADSHAPE, "latent_handoff: n=%d c=%d h=%d w=%d", n, c, h, w);
  if (qmode == NIC_Q_NOISE && !noise_nchw) return fail(NIC_E_BADSHAPE, "latent_handoff: NIC_Q_NOISE needs noise");
  if (n == 0) return NIC_OK;
  if (n > 65535) return fail(NIC_E_BADSHAPE, "latent_handoff: n=%d > 65535", n);
  dim3 grid((h * w + 31) / 32, (c + 31) / 32, n);
  if (in_lo_nonzero) {
    if (int rc = check_cuda(cudaMemsetAsync(in_lo_nonzero, 0, sizeof(int32_t), as_stream(stream)), "cudaMemsetAsync")) return rc;
  }
  latent_handoff_kernel<<<grid, 256, 0, as_stream(stream)>>>(v_nhwc, n, c, h, w, qmode, noise_nchw, v_nchw, v_in_nchw, v_in_nhwc, out_dtype,
                                                                   static_cast<__nv_bfloat16*>(v_nhwc_lowp), lowp_dtype, in_lo_nonzero);
  return check_launch("latent_handoff_kernel");
}

}  // extern "C"
