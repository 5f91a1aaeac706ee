/*
 * nic.h - C ABI of libnic_b200.so: hand-written sm_100a kernels for the forward pass
 * (+ likelihood / rate-distortion terms) of the hyperprior / autoregressive-context
 * image codec of achraf-15/neural_image_compression, and for its training step
 * (the backward of that forward + Adam; section "training step" below).
 *
 * The reference has no FFI of its own (it is pure PyTorch); each entry below names the
 * reference Python call (file:line under /root/reference) whose arithmetic it replaces.
 * The Python host in neural_image_compression_b200/ binds these with ctypes
 * (see INTEGRATION.md for the stub a maintainer of the reference would add).
 * 61 entries (tests/test_abi.py checks that the library exports every one).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *     the caller owns every buffer, the library allocates and frees nothing
 *     (except small immutable tables created once per process).
 *   - `stream` is a cudaStream_t passed as void*; nothing here synchronises the device.
 *   - every entry returns 0 on success or a negative NIC_E_* code; nic_last_error()
 *     then holds a thread-local description.  Nothing throws or aborts.
 *   - reductions are deterministic (fixed-order trees, no floating-point atomics).
 *   - the library is compiled for sm_100a only; on any other device entries return
 *     NIC_E_UNSUPPORTED_ARCH.  There is no CPU or multi-architecture fallback.
 */
#ifndef NIC_B200_H
#define NIC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NIC_ABI_VERSION 1

enum {
  NIC_OK = 0,
  NIC_E_BADSHAPE = -1,
  NIC_E_BADALIGN = -2,
  NIC_E_UNSUPPORTED_ARCH = -3,
  NIC_E_CUDA = -4,
  NIC_E_UNSUPPORTED = -5,
  NIC_E_WORKSPACE = -6
};

/* tensor layouts / element types understood by the conv engine */
enum { NIC_LAYOUT_NCHW = 0, NIC_LAYOUT_NHWC = 1 };
enum {
  NIC_DT_F32 = 0,
  NIC_DT_BF16 = 1,
  NIC_DT_BF16X2 = 2   /* fp32 value carried as a bf16 pair: an NHWC tensor with 2*c channels, [hi(c) | lo(c)], hi = bf16(v),
                         lo = bf16(v - hi).  Activation format of the NIC_PREC_BF16X3 arm.  With out_c_total = T a conv
                         writes hi to channels [off, off + c_out) and lo to [T + off, T + off + c_out) of a 2T-channel tensor. */
};

/* arithmetic of the contraction */
enum {
  NIC_PREC_FP32 = 0,   /* CUDA-core FFMA, fp32 operands and accumulation (parity grade)           */
  NIC_PREC_BF16 = 1,   /* tcgen05.mma kind::f16, bf16 operands, fp32 accumulation in TMEM          */
  NIC_PREC_BF16X3 = 2  /* tcgen05, both operands split hi + lo in bf16 and contracted as ONE K-concatenated conv
                          [A_hi | A_lo | A_hi] . [W_hi | W_hi | W_lo] in a single fp32 TMEM accumulation (fp32 grade:
                          ~1e-5 relative, 3x the MMA work).  Every layer type of the path is built, including the
                          3-channel first layer; GDN / IGDN run as a second tensor-core kernel with squares and gamma
                          split the same way (c = 128).  Activations between layers are NIC_DT_BF16X2 pairs.        */
};

/* fused epilogues */
enum {
  NIC_EPI_BIAS = 0,    /* y = acc + b                                   Components.py:16,73,103  */
  NIC_EPI_LRELU = 1,   /* y = leaky_relu(acc + b, 0.01)                 Components.py:70,72,100,102; ParametersModels.py:30,32 */
  NIC_EPI_GDN = 2,     /* v = acc + b; y = v * rsqrt(beta + gamma.v^2)  Components.py:11,13,15 (compressai GDN) */
  NIC_EPI_IGDN = 3     /* v = acc + b; y = v *  sqrt(beta + gamma.v^2)  Components.py:40,42,44 */
};

/* quantisation mode of the likelihood kernels, Models.py:55-66 */
enum {
  NIC_Q_ROUND = 0,     /* x_in = rint(x)   (eval, Models.py:63-64; round-half-even, sign kept)   */
  NIC_Q_NOISE = 1,     /* x_in = x + noise (training, Models.py:57-58; noise injected by caller) */
  NIC_Q_PASSTHRU = 2   /* x_in = x         (caller already quantised)                            */
};

/*
 * One 2-D convolution or transposed convolution, PyTorch semantics
 * (torch.nn.Conv2d / ConvTranspose2d with dilation 1, groups 1).
 * Replaces the nn.Conv2d / nn.ConvTranspose2d (+ GDN / LeakyReLU) pairs of
 * Components.py:9-17, 38-46, 68-74, 98-104, ContextModels.py:18-20 and
 * ParametersModels.py:29-35.
 */
typedef struct nic_conv_desc {
  int32_t n, c_in, h_in, w_in;      /* input  [n, c_in, h_in, w_in] (logical NCHW extents)      */
  int32_t c_out, h_out, w_out;      /* output [n, c_out, h_out, w_out]                          */
  int32_t kh, kw, stride, pad;      /* kernel, stride (1|2), padding                            */
  int32_t transposed;               /* 0: Conv2d, 1: ConvTranspose2d                            */
  int32_t output_padding;           /* ConvTranspose2d only                                     */
  int32_t mask_a;                   /* 1: PixelCNN mask 'A', 2: mask 'B' (ContextModels.py:13-16) */
  int32_t epilogue;                 /* NIC_EPI_*                                                */
  int32_t precision;                /* NIC_PREC_*                                               */
  int32_t in_layout, out_layout;    /* NIC_LAYOUT_*                                             */
  int32_t in_dtype, out_dtype;      /* NIC_DT_*                                                 */
  int32_t out_c_total, out_c_offset;/* output tensor has out_c_total channels; this conv writes
                                       channels [out_c_offset, out_c_offset + c_out) (makes the
                                       torch.cat of Models.py:73 free); 0,0 = plain             */
} nic_conv_desc;

int nic_version(void);
const char* nic_last_error(void);
/* 0 when the current device is sm_100 (B200), NIC_E_UNSUPPORTED_ARCH otherwise */
int nic_check_device(void);
/* number of CUDA kernels this library has launched in this process (all threads) */
uint64_t nic_launch_count(void);
/*
 * The tensor-core kernels bound every mbarrier wait; if one ever expires (a pipeline bug, never expected) the kernel
 * gives up instead of hanging the GPU and raises a device flag.  This reads and clears that flag: 0 = every kernel since
 * the last call ran to completion, 1 = at least one aborted (its output is invalid).  Synchronises the device.
 */
int nic_pipeline_status(void);

/* ---- weight preparation (once per load_state_dict; derived caches, never saved) ---------- */

/* elements (of the packed dtype) the packed weight of `d` occupies */
size_t nic_packed_weight_elems(const nic_conv_desc* d);
/*
 * Re-layout a reference-format weight for the engine: Conv2d [c_out, c_in, kh, kw]
 * (Components.py:10-16), ConvTranspose2d [c_in, c_out, kh, kw] (Components.py:39-45),
 * masked taps dropped when d->mask_a (the reference zeroes them in place, ContextModels.py:19).
 * fp32: [tap][c_in][c_out] f32.  bf16: [tap][c_out][c_in] bf16 (K-major B operand);
 * bf16x3: [tap][c_out][3 c_in] bf16 = [W_hi | W_hi | W_lo] (first layer: [128][192] = hi / lo of the 75 taps in three
 * 64-column panels; last 128 -> 3 transposed layer: its sub-pixel form [9][16][3 c_in]).
 * nic_packed_weight_elems counts 2-byte elements for the two tensor-core precisions.
 */
int nic_pack_conv_weight(const nic_conv_desc* d, const float* w_ref, void* w_packed, void* stream);
/*
 * compressai GDN reparametrisation (oracle/gdn.py):
 *   beta_eff = max(beta, sqrt(beta_min + 2^-36))^2 - 2^-36,  gamma_eff = max(gamma, 2^-18)^2 - 2^-36.
 * gamma_packed: fp32 -> [c_in(j)][c_out(i)] f32; bf16 -> [i][j] bf16; bf16x3 -> [2][i][j] bf16 = hi, then lo.
 */
int nic_pack_gdn(int32_t c, float beta_min, const float* beta_raw, const float* gamma_raw,
                 float* beta_eff, void* gamma_packed, int32_t precision, void* stream);

/* ---- transforms ---------------------------------------------------------------------------- */

size_t nic_conv_workspace_bytes(const nic_conv_desc* d);
/*
 * y = epilogue(conv(x, w) + bias).  gdn_gamma / gdn_beta are the nic_pack_gdn outputs and are
 * only read for NIC_EPI_GDN / NIC_EPI_IGDN.
 */
int nic_conv_fwd(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias,
                 const void* gdn_gamma, const float* gdn_beta, void* y,
                 void* workspace, size_t workspace_bytes, void* stream);
/*
 * nic_conv_fwd with a hint about the input of a NIC_PREC_BF16X3 conv: in_lo_nonzero (device int32 written by
 * nic_latent_handoff_ex, or NULL) == 0 says the lo half of the bf16-pair input is all zero - true for the quantised y_in / z_in the
 * context model, g_s and h_s read in eval mode (Models.py:63-71, 90) - and the kernel then runs 2 of its 3 MMA passes
 * (hi.W_hi + hi.W_lo; the skipped lo.W_hi term is exactly 0).  The flag is read on the device: no host synchronisation, and a
 * CUDA-graph replay follows the data.
 */
int nic_conv_fwd_ex(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias,
                    const void* gdn_gamma, const float* gdn_beta, void* y,
                    void* workspace, size_t workspace_bytes, const int32_t* in_lo_nonzero, void* stream);

/*
 * Context model + entropy-parameter stack (+ likelihoods) as ONE call (SURVEY.md section 8b `nic_ctx_ep_fwd`; replaces
 * ContextModels.py:15-20 -> torch.cat (Models.py:73) -> ParametersModels.py:29-35 (-> ParametersModels.py:43-64 +
 * EntropyModels.py:192-233, Models.py:86-87 when p is given)).  It is a host-side composite, NOT one kernel: it enqueues the masked
 * 5x5 context conv (12 live taps), the three 1x1 layers and, optionally, the likelihood kernel on `stream`, with the intermediates
 * in caller-owned buffers (they stay L2-resident between the launches; DESIGN.md section 4 explains why a single fused kernel
 * does not fit at fp32 grade).  Results are bit-identical to the same five nic_* calls made one by one.
 *   ctx:      descriptor of the context conv; writes phi into its channel window of `combined` (out_c_total / out_c_offset);
 *             the caller has put psi (the h_s output) into the other window, so torch.cat never happens
 *   ep[0..2]: descriptors of the 1x1 layers: combined -> e1 -> e2 -> raw (ep[2]: out_layout NCHW, out_dtype F32)
 *   y_in_engine / y_in_lo_nonzero: the context conv's input in the engine layout and its optional nic_latent_handoff_ex flag
 *   raw:      [n, (1 + 2) K M or 2 M, h, w] f32, always written (the likelihood kernel reads it)
 *   p == NULL: stop after raw.  Otherwise y_in (NCHW f32), m, k, qmode and the outputs are nic_gm_likelihood_fwd's.
 *   workspace: >= the largest nic_conv_workspace_bytes of the four descriptors (the launches are sequential).
 */
typedef struct nic_ctx_ep_args {
  const nic_conv_desc* ctx;
  const nic_conv_desc* ep[3];
  const void* w_ctx;
  const float* b_ctx;
  const void* w_ep[3];
  const float* b_ep[3];
  const void* y_in_engine;
  const int32_t* y_in_lo_nonzero;
  void* combined;
  void* e1;
  void* e2;
  float* raw;
  const float* y_in;
  const float* noise;
  int32_t m, k, qmode, reserved;
  float* y_in_out;
  float* p;
  float* logp;
  float* weights;
  float* mus;
  float* sigmas;
  float* logp_partials;
  void* workspace;
  size_t workspace_bytes;
} nic_ctx_ep_args;
int nic_ctx_ep_fwd(const nic_ctx_ep_args* a, void* stream);

/*
 * Stand-alone GDN / IGDN (compressai.layers.gdn.GDN.forward; call sites Components.py:11-15, 40-44) for
 * callers that invoke the layer on its own: y = x * rsqrt(beta + gamma . x^2) (inverse: * sqrt).
 * x, y: f32 in `layout`; gamma_packed / beta_eff from nic_pack_gdn(NIC_PREC_FP32).
 */
int nic_gdn_fwd(const float* x, int32_t n, int32_t c, int32_t h, int32_t w, int32_t layout, int32_t inverse,
                const float* gamma_packed, const float* beta_eff, float* y, void* stream);

/*
 * Latent hand-off after the last g_a / h_a conv (Models.py:52-66): reads v (NHWC f32, the
 * engine's layout), writes the reference-layout copy `v_nchw` (dict entries 'y' / 'z'),
 * the quantised / noised tensor `v_in_nchw` ('y_in' / 'z_in') and the engine-layout copy
 * `v_in_nhwc` (dtype out_dtype) that h_s / the context model / g_s consume.
 * v_nhwc_lowp (optional) receives an NHWC copy of the UNquantised v (h_a reads y, Models.py:53) in lowp_dtype
 * (NIC_DT_BF16, or NIC_DT_BF16X2 = [hi | lo] with 2c channels).
 * noise_nchw is read only for NIC_Q_NOISE.  Any output pointer may be NULL.
 */
int nic_latent_handoff(const float* v_nhwc, int32_t n, int32_t c, int32_t h, int32_t w, int32_t qmode,
                       const float* noise_nchw, float* v_nchw, float* v_in_nchw, void* v_in_nhwc,
                       int32_t out_dtype, void* v_nhwc_lowp, int32_t lowp_dtype, void* stream);

/* The same; in_lo_nonzero (optional device int32, out): set to 0, then to 1 if any element of the NIC_DT_BF16X2 copy v_in_nhwc has a
 * non-zero lo half.  Rounded symbols below 256 split exactly (lo = 0), and nic_conv_fwd_ex skips one of its three passes on 0. */
int nic_latent_handoff_ex(const float* v_nhwc, int32_t n, int32_t c, int32_t h, int32_t w, int32_t qmode,
                          const float* noise_nchw, float* v_nchw, float* v_in_nchw, void* v_in_nhwc,
                          int32_t out_dtype, void* v_nhwc_lowp, int32_t lowp_dtype, int32_t* in_lo_nonzero, void* stream);

/* ---- likelihoods --------------------------------------------------------------------------- */

/* number of float partial sums per image the likelihood / sse kernels write */
int32_t nic_partials_per_image(void);

/*
 * K-component Gaussian-mixture likelihood (K = 1: mean-scale Gaussian), NCHW f32 throughout.
 * Replaces ParametersModels.py:43-64 (chunk / view / softmax / softplus + 1e-6),
 * EntropyModels.py:192-233 (+ utils.py:6-8, clamp at :31) and the torch.log of Models.py:87,
 * and accumulates sum(logp) per image for RateDistortionLoss.py:13.
 *   y          [b, m, hw]          input latent (quantised here according to qmode)
 *   raw        [b, 3*k*m, hw]      (k = 1: [b, 2*m, hw]) entropy-parameter net output
 *   y_in, p, logp  [b, m, hw]      outputs ('y_in', 'p_y', 'logp_y'); y_in may be NULL
 *   weights, mus, sigmas [b, k, m, hw]  outputs, all three NULL for the lean variant
 *                                   (k = 1: weights must be NULL, mus/sigmas are mu/sigma)
 *   logp_partials [b, nic_partials_per_image()]  per-image partial sums of logp (fixed order)
 */
int nic_gm_likelihood_fwd(const float* y, const float* raw, const float* noise,
                          int32_t b, int32_t m, int32_t hw, int32_t k, int32_t qmode,
                          float* y_in, float* p, float* logp,
                          float* weights, float* mus, float* sigmas,
                          float* logp_partials, void* stream);

/*
 * The reference's conditional-model call on ALREADY-activated parameters, for callers that use
 * GaussianConditional / GaussianMixtureConditional on their own (EntropyModels.py:192-233, clamp :31):
 *   p = max(sum_k w_k * (Phi((x+.5-mu_k)/s_k) - Phi((x-.5-mu_k)/s_k)), 1e-9)
 * x, p [b, m, hw]; weights / mus / sigmas [b, k, m, hw] (k = 1: weights NULL).
 */
int nic_gm_pmf_fwd(const float* x, const float* weights, const float* mus, const float* sigmas,
                   int32_t b, int32_t m, int32_t hw, int32_t k, float* p, void* stream);
/* The same WITHOUT the clamp: GaussianConditional.discretized_gaussian_pmf (EntropyModels.py:192-204, k = 1) and
 * GaussianMixtureConditional.discretized_mixture_pmf (:214-230), public methods of the reference that return the raw mass. */
int nic_gm_pmf_mass_fwd(const float* x, const float* weights, const float* mus, const float* sigmas,
                        int32_t b, int32_t m, int32_t hw, int32_t k, float* mass, void* stream);

/*
 * Factorized prior likelihood (per-channel 1-3-3-3-1 MLP), NCHW f32.
 * Replaces EntropyModels.py:88-151 (+ clamp :31) and the torch.log of Models.py:84.
 *   fparams [c, 43]: per channel, the reference parameters after their fixed transforms:
 *     softplus(matrices.0)[3] bias0[3] tanh(factors.0)[3] softplus(matrices.1)[9] bias1[3]
 *     tanh(factors.1)[3] softplus(matrices.2)[9] bias2[3] tanh(factors.2)[3]
 *     softplus(matrices.3)[3] bias3[1]   (see nic_pack_factorized)
 */
int nic_pack_factorized(int32_t c, const float* m0, const float* b0, const float* f0,
                        const float* m1, const float* b1, const float* f1,
                        const float* m2, const float* b2, const float* f2,
                        const float* m3, const float* b3, float* fparams, void* stream);
int nic_factorized_likelihood_fwd(const float* z, const float* fparams, const float* noise,
                                  int32_t b, int32_t c, int32_t hw, int32_t qmode,
                                  float* z_in, float* p, float* logp,
                                  float* logp_partials, void* stream);

/* ---- distortion + rate-distortion terms ----------------------------------------------------- */

/* per-image partial sums of (x_hat - x)^2, NCHW f32, chw = 3*h*w (RateDistortionLoss.py:26) */
int nic_sse_fwd(const float* x_hat, const float* x, int32_t b, int64_t chw,
                float* sse_partials, void* stream);

/* per-image partial sums of v [b, per_image] f32 (the torch.sum of RateDistortionLoss.py:13-14 when a
 * caller hands rd_loss tensors this library did not produce) */
int nic_sum_fwd(const float* v, int32_t b, int64_t per_image, float* partials, void* stream);

/*
 * Folds the three partial-sum arrays into the rd_loss terms (RateDistortionLoss.py:13-34):
 *   per_image [3][b]: bits_y, bits_z, mse_per_image
 *   scalars   [8]   : bpp_y, bpp_z, bpp_total, mse, psnr, loss, bits_y_mean, bits_z_mean
 * (psnr = -10 log10(mean_b mse + 1e-8); loss = bpp_total + lambda * 255^2 * mse).
 * One launch, one block, fixed summation order.
 */
int nic_rd_finalize(const float* logp_y_partials, const float* logp_z_partials,
                    const float* sse_partials, int32_t b, int32_t num_pixels, int64_t chw,
                    float lambda_rd, float* per_image, float* scalars, void* stream);

/*
 * The same terms from already-reduced per-image rows (data-parallel evaluation: every rank all-gathers the
 * [3][b_local] rows of nic_rd_finalize and folds the global [3][b] array here, in the same fixed order on every rank).
 *   per_image [3][b]: bits_y, bits_z, mse_per_image   ->   scalars [8] as in nic_rd_finalize
 */
int nic_rd_reduce(const float* per_image, int32_t b, int32_t num_pixels, float lambda_rd, float* scalars, void* stream);

/* ---- training step: backward kernels (fp32, CUDA cores) -------------------------------------------------------
 * The reference has no backward code: its gradients are what torch autograd derives from Models.py:49-106 +
 * RateDistortionLoss.py:5-49 when Trainer.py:85 calls loss.backward().  These entries are those derivatives written
 * out; all tensors f32.  The DATA gradient of a conv layer is the adjoint conv and goes through nic_conv_fwd with the
 * mirrored descriptor (Conv2d <-> ConvTranspose2d over the same weight tensor, output_padding chosen to restore the
 * forward input size).
 */

/*
 * Weight (+ bias) gradient of one conv layer.  `d` is the FORWARD descriptor (precision / epilogue ignored; mask_a
 * ignored: the reference masks the weight DATA, ContextModels.py:19, so all taps receive gradient).
 *   x  forward input  (d->in_layout)      g  gradient w.r.t. the conv output before its activation (d->out_layout)
 *   dw reference layout [c_out, c_in, kh, kw] (Conv2d) / [c_in, c_out, kh, kw] (ConvTranspose2d);  db [c_out] or NULL
 * The tensor with the SMALLER spatial extent (g for Conv2d, x for ConvTranspose2d) must be NHWC with c % 4 == 0; the
 * other may be NCHW (the 3-channel image side).  Split-K over pixels with a fixed-order fold: deterministic.
 */
size_t nic_conv_wgrad_workspace_bytes(const nic_conv_desc* d);
int nic_conv_wgrad(const nic_conv_desc* d, const float* x, const float* g, float* dw, float* db,
                   void* workspace, size_t workspace_bytes, void* stream);

/*
 * The same weight gradient on the tcgen05 tensor cores (bf16x3: hi/lo-split operands, fp32 accumulation in TMEM; ~1e-5 relative).
 * x_pair / g_pair are the NIC_DT_BF16X2 NHWC forms (nic_to_pair) of the layer input and of the output gradient; g (f32 NHWC) is
 * only read for db.  The contraction index is the pixel and both tensors are channels-contiguous, so TMA boxes of
 * [pixels][64 channels] are fed to the MMA as MN-major operands with no transposition (csrc/wgrad_tc.cu).
 * Built for c_in % 64 == 0, c_out % 64 == 0, square kernels, both tensors NHWC, >= 8 x 8 pixels on the smaller side:
 * nic_conv_wgrad_tc_workspace_bytes returns 0 for any other layer (use nic_conv_wgrad).
 */
size_t nic_conv_wgrad_tc_workspace_bytes(const nic_conv_desc* d);
int nic_conv_wgrad_tc(const nic_conv_desc* d, const void* x_pair, const void* g_pair, const float* g, float* dw, float* db,
                      void* workspace, size_t workspace_bytes, void* stream);

/* LeakyReLU(0.01) backward from the saved activation OUTPUT: g_pre = out > 0 ? g : 0.01 g (may run in place on g) */
int nic_lrelu_bwd(const float* g, const float* out, float* g_pre, int64_t n, void* stream);

/*
 * compressai GDN / IGDN backward (call sites Components.py:11-15, 40-44), NHWC f32.
 *   u  the layer input (the conv output before the GDN), g  gradient w.r.t. the GDN output
 *   du gradient w.r.t. u;  dbeta_raw [c], dgamma_raw [c, c]: gradients w.r.t. the STORED (reparametrised) parameters,
 *   through eff = LowerBound(raw)^2 - 2^-36 with compressai's rule (passes where raw >= bound or the gradient is < 0).
 */
size_t nic_gdn_bwd_workspace_bytes(int32_t n, int32_t c, int32_t h, int32_t w);
int nic_gdn_bwd(const float* u, const float* g, int32_t n, int32_t c, int32_t h, int32_t w, int32_t inverse, float beta_min,
                const float* beta_raw, const float* gamma_raw, float* du, float* dbeta_raw, float* dgamma_raw,
                void* workspace, size_t workspace_bytes, void* stream);

/*
 * The same GDN forward / backward in pieces, for callers that run the two channel-mixing contractions (norm = beta + gamma . u^2
 * and r = gamma^T . t) elsewhere - the training step runs them as 1x1 convs on the tensor cores (nic_conv_fwd, NIC_PREC_BF16X3):
 *   nic_gdn_reparam     beta_eff [c], gamma_eff [c, c] (= the [c_out, c_in] weight of the norm conv), gamma_eff_t (its transpose)
 *   nic_gdn_apply       out = u * rsqrt(norm)   (inverse: u * sqrt(norm))
 *   nic_gdn_bwd_prep    t = d out / d norm * g,  du = g * rsqrt(norm) (inverse: g * sqrt(norm))
 *   nic_gdn_bwd_finish  du += 2 u r;  dgamma_raw, dbeta_raw from (u, t) through the LowerBound rule; dgamma_eff_in [c, c] /
 *                       dbeta_eff_in [c] (both or neither): the gradients w.r.t. the EFFECTIVE parameters when the caller has
 *                       already formed them (sum_pix t_i u_j^2 is the weight gradient of a 1x1 conv: nic_conv_wgrad_tc)
 */
/* the two halves of nic_gdn_bwd_finish on their own (data path: du += 2 u r; parameter path: the LowerBound chain) - the
 * training step runs the parameter path on a side stream */
int nic_gdn_bwd_du(const float* u, const float* r, float* du, int64_t n, void* stream);
int nic_gdn_reparam_bwd(int32_t c, float beta_min, const float* beta_raw, const float* gamma_raw, const float* dbeta_eff,
                        const float* dgamma_eff, float* dbeta_raw, float* dgamma_raw, void* stream);
int nic_gdn_reparam(int32_t c, float beta_min, const float* beta_raw, const float* gamma_raw, float* beta_eff, float* gamma_eff,
                    float* gamma_eff_t, void* stream);
int nic_gdn_apply(const float* u, const float* norm, int64_t n, int32_t inverse, float* out, void* stream);
/* out = nic_gdn_apply(u, norm) + addend in one pass (the residual sum after the GDN / IGDN of ResidualBlockWithStride /
 * ResidualBlockUpsample, Layers.py:58-60, 85-87); bit-identical to nic_gdn_apply followed by nic_add_inplace */
int nic_gdn_apply_add(const float* u, const float* norm, const float* addend, int64_t n, int32_t inverse, float* out, void* stream);
int nic_gdn_bwd_prep(const float* u, const float* g, const float* norm, int64_t n, int32_t inverse, float* t, float* du, void* stream);
size_t nic_gdn_bwd_finish_workspace_bytes(int64_t pixels, int32_t c);
int nic_gdn_bwd_finish(const float* u, const float* t, const float* r, int64_t pixels, int32_t c, float beta_min,
                       const float* beta_raw, const float* gamma_raw, const float* dgamma_eff_in, const float* dbeta_eff_in,
                       float* du, float* dbeta_raw, float* dgamma_raw, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Backward of nic_gm_likelihood_fwd w.r.t. y_in and the raw entropy-parameter tensor (softmax / softplus / erf-form CDF
 * difference / clamp_min(1e-9) / log chain).  g_logp [b, m, hw] = upstream gradient of logp, or NULL: every element's
 * upstream is g_scalar (rd_loss: -1 / (ln2 * num_pixels * B)).  dy_in [b, m, hw], draw like raw.
 */
int nic_gm_likelihood_bwd(const float* y_in, const float* raw, const float* g_logp, float g_scalar,
                          int32_t b, int32_t m, int32_t hw, int32_t k, float* dy_in, float* draw, void* stream);

/*
 * Backward of nic_factorized_likelihood_fwd: dz_in [b, c, hw]; dparams [c, 43] = gradients w.r.t. the RAW reference
 * parameters (matrices / biases / factors) in nic_pack_factorized order (the softplus / tanh chain is applied).
 */
int nic_factorized_likelihood_bwd(const float* z_in, const float* fparams, const float* g_logp, float g_scalar,
                                  int32_t b, int32_t c, int32_t hw, float* dz_in, float* dparams, void* stream);

/* g_x_hat = coef * (x_hat - x): backward of the MSE term (RateDistortionLoss.py:26-34; coef = g_loss * lambda * 255^2 * 2 / (B*C*H*W)) */
int nic_sse_bwd(const float* x_hat, const float* x, int64_t n, float coef, float* g_x_hat, void* stream);

/* dst += src */
int nic_add_inplace(float* dst, const float* src, int64_t n, void* stream);
/* [n, c, hw] -> [n, hw, c] (to_nhwc = 1) or back (0); accumulate = 1: dst += converted src */
int nic_layout_convert(const float* src, float* dst, int32_t n, int32_t c, int32_t hw, int32_t to_nhwc, int32_t accumulate, void* stream);

/* f32 [rows, c] -> NIC_DT_BF16X2 [rows, 2c] = [hi | lo]: hands fp32 activations / gradients to the bf16x3 convs (c % 4 == 0) */
int nic_to_pair(const float* src, void* dst, int64_t rows, int32_t c, int32_t square /* 1: split src^2 */, void* stream);

/* One torch.optim.Adam update (no weight decay / amsgrad; Main.ipynb:133) of a flat parameter; step = t >= 1 after the increment */
int nic_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                  int32_t step, void* stream);

/*
 * The same update for MANY tensors in one launch (64 tensors per launch).  The *_host arguments are HOST arrays of `count` device
 * pointers / element counts; the pointers travel to the kernel as launch arguments, so there is no table upload and no host
 * synchronisation.  A tensor with n = 0 is skipped.  step_dev (device int32, or NULL): when given, the step count t is read from
 * it by the kernel instead of `step` - a CUDA-graph replay of the launch then sees the t that nic_counter_increment advanced.
 */
int nic_adam_multi_step(float* const* p_host, const float* const* g_host, float* const* m_host, float* const* v_host,
                        const int64_t* n_host, int32_t count, float lr, float beta1, float beta2, float eps, int32_t step,
                        const int32_t* step_dev, void* stream);
/* The same with (a) the learning rate read from DEVICE memory when lr_dev != NULL (an lr scheduler's change - Trainer.py:33-36,
 * 103 - then reaches a captured launch without re-capturing; `lr` is ignored) and (b) every gradient multiplied by grad_scale
 * first (1 / world folds the data-parallel averaging of all-reduced SUMS into the update; 1 = plain Adam). */
int nic_adam_multi_step_ex(float* const* p_host, const float* const* g_host, float* const* m_host, float* const* v_host,
                           const int64_t* n_host, int32_t count, float lr, const float* lr_dev, float grad_scale, float beta1, float beta2,
                           float eps, int32_t step, const int32_t* step_dev, void* stream);
/* *counter += 1 on the device (stream-ordered, graph-capturable) */
int nic_counter_increment(int32_t* counter, void* stream);

/* ---- evaluator-side distortion metrics (Evaluator.py:26-53: compute_metrics on imgs and x_hat.clamp(0, 1)) -------------------- */

/* mse_rgb_y [b][2] = per image: mean over (3, h, w) of (orig - recon)^2, and the same over the luma plane
 * Y = 0.299 R + 0.587 G + 0.114 B (Evaluator.py:27-30, 34, 41-43); clamp01 = 1 clamps recon to [0, 1] on the fly (Evaluator.py:73).
 * NCHW f32; partials [b][nic_partials_per_image()][2] scratch. */
int nic_eval_mse(const float* orig, const float* recon, int32_t b, int32_t h, int32_t w, int32_t clamp01, float* mse_rgb_y, float* partials,
                 void* stream);
/* y [b][h][w] = luma of an NCHW RGB batch; clamp01 = 1 clamps the input to [0, 1] first */
int nic_luma(const float* rgb, float* y, int32_t b, int32_t h, int32_t w, int32_t clamp01, void* stream);
/*
 * The five scales of pytorch_msssim.ms_ssim (11-tap Gaussian, sigma 1.5, valid convolution, 2x2 average pooling with padding
 * size % 2 between scales; third-party package, absent here: the published algorithm restated - parity unpinned):
 * level_means [5][planes][2] = (mean ssim, mean cs) of every scale for `planes` = b * c planes of h x w (f32, plane-contiguous).
 * clamp_y = 1 clamps the second tensor to [0, 1] on the fly (x_hat.clamp(0, 1)).  ms_ssim of a plane =
 * prod_{l<4} relu(cs_l)^w_l * relu(ssim_4)^w_4, w = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333); the smaller side must exceed 160.
 */
size_t nic_ms_ssim_workspace_bytes(int32_t planes, int32_t h, int32_t w);
int nic_ms_ssim_levels(const float* x, const float* y, int32_t planes, int32_t h, int32_t w, float data_range, int32_t clamp_y,
                       float* level_means, void* workspace, size_t workspace_bytes, void* stream);
/*
 * Backward of the level means with respect to the FIRST image (the MS-SSIM loss, DESIGN.md section 13):
 * g_x [planes][h][w] = sum over (level, plane) of g_level[level][plane] * d level_mean / d x, where level_mean is the mean cs of
 * levels 0-3 and the mean ssim of level 4.  `workspace` (>= nic_ms_ssim_bwd_workspace_bytes) must hold what
 * nic_ms_ssim_levels(x, y, planes, h, w, data_range, clamp_y = 0, ...) left in it: the pooled pyramids are read back from there.
 * No atomics: every element of g_x is written by one thread in a fixed order (bit-identical across calls and batch sizes).
 * The first call on a device (as the first nic_ms_ssim_levels call) uploads the window and must run outside a stream capture.
 */
size_t nic_ms_ssim_bwd_workspace_bytes(int32_t planes, int32_t h, int32_t w);
int nic_ms_ssim_bwd(const float* x, const float* y, int32_t planes, int32_t h, int32_t w, float data_range, const float* g_level,
                    float* g_x, void* workspace, size_t workspace_bytes, void* stream);

/* ---- entropy coder (DESIGN.md section 9): byte strings for JointAutoregressiveHierarchical ------------------------------------
 * rANS with a 32-bit state in [2^16, 2^32), 16-bit renormalisation words and 16-bit probabilities.  A table row of one element is
 * a window of n <= NIC_CODEC_WINDOW consecutive integers starting at lo plus an escape bin (index n) for any other value; an
 * escaped value v follows the escape bin as two raw 16-bit words of zigzag(v) (low half first).  Row layout: cdf[0] = 0,
 * cdf[i + 1] = cdf[i] + freq_i (freq_i >= 1), cdf[n + 1] = 2^16; NIC_CODEC_WINDOW + 2 uint32 entries per row.
 * y elements are coded in wavefront order: pixel (i, j) belongs to step t = 3 i + j (3 h + w - 3 steps; the masked 5x5 context of
 * a pixel only reads pixels of earlier steps), pixels of a step with i ascending, lane l holds channels c = l (mod lanes)
 * ascending.  z elements: pixels in raster order, the same channel-to-lane rule.
 */
#define NIC_CODEC_PREC_BITS 16
#define NIC_CODEC_WINDOW 128
enum { NIC_CODEC_GM = 0, NIC_CODEC_FACTORIZED = 1 };   /* y: Gaussian mixture (K = 1: Gaussian); z: factorized prior */
enum { NIC_CODEC_TABLES = 0, NIC_CODEC_SYMBOL = 1 };

/*
 * The quantised tables, the one function both coder directions use (a single compiled kernel with a runtime mode, so the
 * float -> integer step is the same instructions for both).
 *   kind GM:         params = raw entropy parameters [b, (3K | 2) m, h, w] (nic_ctx_ep_fwd's raw), k = K
 *   kind FACTORIZED: params = nic_pack_factorized's [m, 43] (k ignored)
 *   mode TABLES:     GM: the elements of wavefront step t, e = (img * cnt + p) * m + c (p-th pixel of the step) -> cdf [e][W + 2],
 *                    lo [e], nbins [e];  FACTORIZED: one row per channel (e = c; b, h, w only checked)
 *   mode SYMBOL:     every element e of the NCHW latent sym [b, m, h, w] -> code [e] = start | freq << 16 | escape << 32 of its symbol
 */
int nic_codec_tables(int32_t kind, int32_t mode, const float* params, const float* sym, int32_t b, int32_t m, int32_t k, int32_t h,
                     int32_t w, int32_t t, uint32_t* cdf, int32_t* lo, int32_t* nbins, uint64_t* code, void* stream);
/*
 * rANS encode, one thread per (image, lane): code / sym as nic_codec_tables(SYMBOL) saw them.  Lane g = img * lanes + l writes its
 * segment - the final state (2 words, low first) followed by the words in decode order - at the END of words[g * cap, (g + 1) * cap)
 * and its length in words (state included) to count[g].  cap >= 3 * ceil(m / lanes) * h * w + 2.
 */
int nic_codec_encode(int32_t kind, const uint64_t* code, const float* sym, int32_t b, int32_t m, int32_t h, int32_t w, int32_t lanes,
                     int64_t cap, uint16_t* words, int32_t* count, void* stream);
/*
 * rANS decode, one thread per (image, lane).  kind GM: wavefront step t with the step's tables; kind FACTORIZED: all of z with the
 * per-channel tables.  blob holds the byte strings; lane g's segment starts at byte lane_off[g] (4 state bytes, then lane_words[g]
 * words; reads past them return 0).  state / pos [b * lanes] carry each lane's cursor from one step to the next (init = 1: start
 * from the segment).  Symbols go to out, NHWC f32 [b, h, w, m].
 */
int nic_codec_decode(int32_t kind, const uint8_t* blob, const int64_t* lane_off, const int32_t* lane_words, uint32_t* state, int32_t* pos,
                     int32_t init, const uint32_t* cdf, const int32_t* lo, const int32_t* nbins, int32_t b, int32_t m, int32_t h, int32_t w,
                     int32_t lanes, int32_t t, float* out, void* stream);
/*
 * One wavefront step t of y in one launch (DESIGN.md section 11): one CTA per (image, lane) builds the lane's table rows of the step
 * in shared memory from params (raw entropy parameters [b, (3K | 2) m, h, w], NCHW f32, k = K; only the step's pixels are read) with
 * the function nic_codec_tables uses, and decodes them as nic_codec_decode(GM) does with the tables of nic_codec_tables(TABLES):
 * the same symbols, states and read positions.  blob, lane_off, lane_words, state, pos, init and out as nic_codec_decode.
 */
int nic_codec_decode_step(const uint8_t* blob, const int64_t* lane_off, const int32_t* lane_words, uint32_t* state, int32_t* pos,
                          int32_t init, const float* params, int32_t b, int32_t m, int32_t k, int32_t h, int32_t w, int32_t lanes, int32_t t,
                          float* out, void* stream);
/* out [b] = per image sum over the symbols (y [b, y_per_image] then z [b, z_per_image], NCHW f32) of a 32-bit mix of (index, value),
 * mod 2^32 */
int nic_codec_checksum(const float* y, int64_t y_per_image, const float* z, int64_t z_per_image, int32_t b, uint32_t* out, void* stream);

/*
 * Step-local entropy parameters (DESIGN.md section 10; ScalableImageCoding's coder): the masked 5x5 context conv 'A' of a head on
 * m channels -> 2m, then the 1x1 stack (2m + 2M) -> 640 -> 640 -> (2m | 3Km) with LeakyReLU(0.01) after the first two, computed
 * only at the pixels of one launch - every pixel (t = -1) or those of wavefront step t.  fp32 CUDA cores: every output element is
 * one thread's fixed-order __fmaf_rn chain (bias first, then the inputs in the order of the packed weights, zeros at the borders),
 * so a pixel's value is the same bits whichever launch, batch or pixel count computed it.
 * Per head (n_heads = 1 or 2, one launch per layer serves both):
 *   sym     the head's symbols, NHWC f32 [b, h, w, m]; psi = NHWC f32 [b, h, w, 2 M] (shared by the heads)
 *   w_ctx   [12 m][2 m]: live tap s (rows i - 2, i - 1 at columns j - 2 .. j + 2, then row i at j - 2, j - 1), channel c -> row
 *           s m + c; w1 [2 m + 2 M][640] (rows: phi, then psi), w2 [640][640], w3 [640][np m]; biases f32; np = 2 (k = 1) or 3 k
 *   raw     NCHW f32 [b, np m, h, w] (nic_codec_tables' GM params), written at the launch's pixels only
 *   work    n (2 m + 1280) floats, n = b h w (t = -1) or b * (pixels of step t)
 */
typedef struct nic_codec_head {
  const float* sym;
  const float* w_ctx;
  const float* b_ctx;
  const float* w1;
  const float* b1;
  const float* w2;
  const float* b2;
  const float* w3;
  const float* b3;
  float* raw;
  float* work;
  int64_t work_floats;
  int32_t m, reserved;
} nic_codec_head;
int nic_codec_params(const nic_codec_head* heads, int32_t n_heads, const float* psi, int32_t b, int32_t M, int32_t k, int32_t h,
                     int32_t w, int32_t t, void* stream);

/*
 * Image window of the any-size coders (DESIGN.md section 12), on contiguous f32 planes (planes = B x 3):
 *   dst[p, i, j] = src[p, min(i, h_src - 1), min(j, w_src - 1)],  p < planes, i < h_dst, j < w_dst
 * A larger dst is the encoder's edge-replicating pad (down and to the right), a smaller one the decoder's crop.  An exact copy;
 * 64-bit offsets.  Any size < 1 or a null pointer: NIC_E_BADSHAPE, nothing launched.
 */
int nic_image_window(const float* src, int32_t planes, int32_t h_src, int32_t w_src, float* dst, int32_t h_dst, int32_t w_dst,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NIC_B200_H */
