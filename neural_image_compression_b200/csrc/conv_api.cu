// C-ABI entry points of the conv engine: dispatch on nic_conv_desc::precision.
#include "conv_common.cuh"

namespace nic {
// conv_simt.cu
int conv_fwd_fp32(const nic_conv_desc*, const void*, const void*, const float*, const void*, const float*, void*, void*, size_t, cudaStream_t);
__global__ void pack_weight_f32_kernel(const float*, float*, int, int, int, int, int, TapTable);
__global__ void pack_gdn_f32_kernel(int, float, float, float, const float*, const float*, float*, float*);
// conv_tc.cu
int conv_fwd_tc(const nic_conv_desc*, const void*, const void*, const float*, const void*, const float*, void*, void*, size_t, cudaStream_t,
                const int* lo_flag);
int pack_weight_tc(const nic_conv_desc*, const TapTable&, const float*, void*, cudaStream_t);
int pack_gdn_tc(int32_t, float, const float*, const float*, float*, void*, int32_t, cudaStream_t);
size_t packed_weight_elems_tc(const nic_conv_desc*, const TapTable&);
size_t conv_workspace_bytes_tc(const nic_conv_desc*);

// Anchor zeroing of the checkerboard context (include/nic.h, NIC_MASK_CHECKERBOARD): one thread per (anchor pixel, channel of the
// window); `elem` = bytes per element (4: f32, 2: bf16), `halves` = 2 for a hi / lo pair (the lo half c_total channels further on).
__global__ void __launch_bounds__(256)
checkerboard_zero_kernel(char* __restrict__ y, int elem, int nchw, int halves, int n, int h, int w, int c, int c_total, int c_offset) {
  const int wa = (w + 1) / 2;                                    // anchors of a row (at most)
  const long total = static_cast<long>(n) * h * wa * c;
  for (long e = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += static_cast<long>(gridDim.x) * blockDim.x) {
    const int ch = static_cast<int>(e % c);
    const long pr = e / c;
    const int k = static_cast<int>(pr % wa), i = static_cast<int>((pr / wa) % h);
    const long img = pr / (static_cast<long>(wa) * h);
    const int j = (i & 1) + 2 * k;
    if (j >= w) continue;
    for (int half = 0; half < halves; ++half) {
      const long cc = c_offset + ch + static_cast<long>(half) * c_total;
      const long idx = nchw ? ((img * c_total + cc) * h + i) * w + j
                            : ((img * h + i) * w + j) * (static_cast<long>(halves) * c_total) + cc;
      if (elem == 4) reinterpret_cast<float*>(y)[idx] = 0.f;
      else reinterpret_cast<unsigned short*>(y)[idx] = 0;
    }
  }
}

}  // namespace nic

using namespace nic;

extern "C" {

size_t nic_packed_weight_elems(const nic_conv_desc* d) {
  TapTable tt;
  if (build_tap_table(d, &tt)) return 0;
  if (d->precision == NIC_PREC_FP32) return static_cast<size_t>(tt.ntaps) * d->c_in * d->c_out;
  return packed_weight_elems_tc(d, tt);
}

int nic_pack_conv_weight(const nic_conv_desc* d, const float* w_ref, void* w_packed, void* stream) {
  if (int rc = nic_check_device()) return rc;
  TapTable tt;
  if (int rc = build_tap_table(d, &tt)) return rc;
  if (!w_ref || !w_packed) return fail(NIC_E_BADSHAPE, "pack_conv_weight: null pointer");
  if (d->precision == NIC_PREC_FP32) {
    const long total = static_cast<long>(tt.ntaps) * d->c_in * d->c_out;
    const int blocks = static_cast<int>((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
    pack_weight_f32_kernel<<<blocks, 256, 0, as_stream(stream)>>>(w_ref, static_cast<float*>(w_packed), d->c_in, d->c_out,
                                                                 d->kh, d->kw, d->transposed, tt);
    return check_launch("pack_weight_f32_kernel");
  }
  return pack_weight_tc(d, tt, w_ref, w_packed, as_stream(stream));
}

int nic_pack_gdn(int32_t c, float beta_min, const float* beta_raw, const float* gamma_raw,
                 float* beta_eff, void* gamma_packed, int32_t precision, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (c < 1 || !beta_raw || !gamma_raw || !beta_eff || !gamma_packed) return fail(NIC_E_BADSHAPE, "pack_gdn: bad arguments");
  if (precision == NIC_PREC_FP32) {
    // constants of compressai's NonNegativeParametrizer (oracle/gdn.py), evaluated as the fp32 tensors torch holds
    const float pedestal = static_cast<float>(3.814697265625e-06 * 3.814697265625e-06);   // (2^-18)^2
    const float beta_bound = static_cast<float>(sqrt(static_cast<double>(beta_min) + static_cast<double>(pedestal)));
    const float gamma_bound = static_cast<float>(sqrt(static_cast<double>(pedestal)));
    pack_gdn_f32_kernel<<<(c * c + 255) / 256, 256, 0, as_stream(stream)>>>(c, beta_bound, gamma_bound, pedestal, beta_raw, gamma_raw,
                                                                          beta_eff, static_cast<float*>(gamma_packed));
    return check_launch("pack_gdn_f32_kernel");
  }
  return pack_gdn_tc(c, beta_min, beta_raw, gamma_raw, beta_eff, gamma_packed, precision, as_stream(stream));
}

size_t nic_conv_workspace_bytes(const nic_conv_desc* d) {
  if (!d || validate_conv_desc(d)) return 0;
  if (d->precision == NIC_PREC_FP32) {
    if (d->epilogue == NIC_EPI_GDN || d->epilogue == NIC_EPI_IGDN)
      return static_cast<size_t>(d->n) * d->h_out * d->w_out * d->c_out * sizeof(float);
    return 0;
  }
  return conv_workspace_bytes_tc(d);
}

int nic_conv_fwd(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias,
                 const void* gdn_gamma, const float* gdn_beta, void* y,
                 void* workspace, size_t workspace_bytes, void* stream) {
  return nic_conv_fwd_ex(d, x, w_packed, bias, gdn_gamma, gdn_beta, y, workspace, workspace_bytes, nullptr, stream);
}

int nic_conv_fwd_ex(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias,
                    const void* gdn_gamma, const float* gdn_beta, void* y,
                    void* workspace, size_t workspace_bytes, const int32_t* in_lo_nonzero, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (int rc = validate_conv_desc(d)) return rc;
  if (d->n == 0) return NIC_OK;
  if (!x || !w_packed || !bias || !y) return fail(NIC_E_BADSHAPE, "conv: null pointer");
  int rc;
  switch (d->precision) {
    case NIC_PREC_FP32:
      rc = conv_fwd_fp32(d, x, w_packed, bias, gdn_gamma, gdn_beta, y, workspace, workspace_bytes, as_stream(stream));
      break;
    case NIC_PREC_BF16:
    case NIC_PREC_BF16X3:
      rc = conv_fwd_tc(d, x, w_packed, bias, gdn_gamma, gdn_beta, y, workspace, workspace_bytes, as_stream(stream), in_lo_nonzero);
      break;
    default:
      return fail(NIC_E_BADSHAPE, "conv: precision %d", d->precision);
  }
  if (rc || d->mask_a != NIC_MASK_CHECKERBOARD) return rc;
  // checkerboard context: phi = 0 at the anchors (bias included), a separate launch after the conv
  return nic_checkerboard_zero(y, d->out_dtype, d->out_layout, d->n, d->h_out, d->w_out, d->c_out, d->out_c_total ? d->out_c_total : d->c_out,
                               d->out_c_offset, stream);
}

int nic_checkerboard_zero(void* y, int32_t dtype, int32_t layout, int32_t n, int32_t h, int32_t w, int32_t c, int32_t c_total,
                          int32_t c_offset, void* stream) {
  if (n < 0 || h < 1 || w < 1 || c < 1 || c_offset < 0 || c_offset + c > c_total)
    return fail(NIC_E_BADSHAPE, "checkerboard_zero: n=%d h=%d w=%d window [%d,+%d) of %d channels", n, h, w, c_offset, c, c_total);
  if (dtype != NIC_DT_F32 && dtype != NIC_DT_BF16 && dtype != NIC_DT_BF16X2) return fail(NIC_E_BADSHAPE, "checkerboard_zero: dtype %d", dtype);
  if (layout != NIC_LAYOUT_NHWC && (layout != NIC_LAYOUT_NCHW || dtype == NIC_DT_BF16X2))
    return fail(NIC_E_BADSHAPE, "checkerboard_zero: layout %d with dtype %d", layout, dtype);
  if (!y) return fail(NIC_E_BADSHAPE, "checkerboard_zero: null pointer");
  if (n == 0) return NIC_OK;
  const long total = static_cast<long>(n) * h * ((w + 1) / 2) * c;
  const long blocks = (total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096;
  checkerboard_zero_kernel<<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(
      static_cast<char*>(y), dtype == NIC_DT_F32 ? 4 : 2, layout == NIC_LAYOUT_NCHW, dtype == NIC_DT_BF16X2 ? 2 : 1, n, h, w, c, c_total,
      c_offset);
  return check_launch("checkerboard_zero_kernel");
}

int nic_ctx_ep_fwd(const nic_ctx_ep_args* a, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (!a || !a->ctx || !a->ep[0] || !a->ep[1] || !a->ep[2]) return fail(NIC_E_BADSHAPE, "ctx_ep: null descriptor");
  if (!a->y_in_engine || !a->combined || !a->e1 || !a->e2 || !a->raw) return fail(NIC_E_BADSHAPE, "ctx_ep: null buffer");
  const nic_conv_desc* ds[4] = {a->ctx, a->ep[0], a->ep[1], a->ep[2]};
  size_t need = 0;
  for (const nic_conv_desc* d : ds) {
    if (int rc = validate_conv_desc(d)) return rc;
    const size_t b = nic_conv_workspace_bytes(d);
    need = b > need ? b : need;
  }
  if (need && (!a->workspace || a->workspace_bytes < need)) return fail(NIC_E_WORKSPACE, "ctx_ep: workspace %zu < %zu bytes", a->workspace_bytes, need);
  if (a->ep[0]->n != a->ctx->n || a->ep[0]->h_in != a->ctx->h_out || a->ep[0]->w_in != a->ctx->w_out ||
      a->ep[0]->c_in != (a->ctx->out_c_total ? a->ctx->out_c_total : a->ctx->c_out) || a->ep[1]->c_in != a->ep[0]->c_out ||
      a->ep[2]->c_in != a->ep[1]->c_out)
    return fail(NIC_E_BADSHAPE, "ctx_ep: the four descriptors do not chain");
  // phi into its window of `combined` (psi is already in the other one), then the 1x1 stack
  if (int rc = nic_conv_fwd_ex(a->ctx, a->y_in_engine, a->w_ctx, a->b_ctx, nullptr, nullptr, a->combined, a->workspace, a->workspace_bytes,
                               a->y_in_lo_nonzero, stream)) return rc;
  if (int rc = nic_conv_fwd(a->ep[0], a->combined, a->w_ep[0], a->b_ep[0], nullptr, nullptr, a->e1, a->workspace, a->workspace_bytes, stream)) return rc;
  if (int rc = nic_conv_fwd(a->ep[1], a->e1, a->w_ep[1], a->b_ep[1], nullptr, nullptr, a->e2, a->workspace, a->workspace_bytes, stream)) return rc;
  if (int rc = nic_conv_fwd(a->ep[2], a->e2, a->w_ep[2], a->b_ep[2], nullptr, nullptr, a->raw, a->workspace, a->workspace_bytes, stream)) return rc;
  if (!a->p) return NIC_OK;
  if (a->ep[2]->out_layout != NIC_LAYOUT_NCHW || a->ep[2]->out_dtype != NIC_DT_F32)
    return fail(NIC_E_BADSHAPE, "ctx_ep: the likelihood kernel reads raw as NCHW f32");
  return nic_gm_likelihood_fwd(a->y_in, a->raw, a->noise, a->ctx->n, a->m, a->ep[2]->h_out * a->ep[2]->w_out, a->k, a->qmode, a->y_in_out,
                               a->p, a->logp, a->weights, a->mus, a->sigmas, a->logp_partials, stream);
}

}  // extern "C"
