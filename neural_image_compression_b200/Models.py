"""``JointAutoregressiveHierarchical`` of /root/reference/Models.py:10-106 on the sm_100a kernels.

Same constructor, attributes, ``state_dict`` keys and output dict.  ``forward`` issues one fused
chain of C-ABI calls on the current CUDA stream (activations NHWC between layers, nothing returns to
the host):

    g_a   4 x nic_conv_fwd (GDN fused)                              Models.py:52  Components.py:9-17
    y     nic_latent_handoff  -> 'y', 'y_in' (round | + noise)      Models.py:57-64
    h_a   3 x nic_conv_fwd (LeakyReLU fused)                        Models.py:53  Components.py:68-74
    z     nic_latent_handoff  -> 'z', 'z_in'
    h_s   3 x nic_conv_fwd, last one writes channels [2M, 4M)       Models.py:69  Components.py:98-104
    ctx   nic_conv_fwd (12 live taps), writes channels [0, 2M)      Models.py:71  ContextModels.py:18-20
          (so torch.cat([phi, psi]) of Models.py:73 never happens)
    ep    3 x nic_conv_fwd (1x1), last one writes NCHW raw params   Models.py:76-80 ParametersModels.py:29-35
    p_y   nic_gm_likelihood_fwd (+ weights/mus/sigmas, log, sums)   Models.py:86-87
    p_z   nic_factorized_likelihood_fwd (+ log, sums)               Models.py:83-84
    g_s   4 x nic_conv_fwd (IGDN fused), last one writes NCHW x_hat Models.py:90  Components.py:38-46
"""
from __future__ import annotations

import contextlib
import math
import os
from typing import Optional, Tuple

import torch
import torch.nn as nn

from . import _lib, engine
from ._lib import LAYOUT_NCHW, LAYOUT_NHWC, MODEL_PRECISIONS, Q_NOISE, Q_PASSTHRU, Q_ROUND
from .Components import Decoder5x5, Encoder5x5, HyperDecoder5x5, HyperEncoder5x5
from .ContextModels import ChannelContextModel, CheckerboardContextModel, ContextModel
from .EntropyModels import FactorizedEntropyBottleneck, GaussianConditional, GaussianMixtureConditional, gm_likelihood
from .ParametersModels import EntropyParameters


def check_channels(latent_channels, K):
    """The constructor arguments every model shares."""
    if not isinstance(latent_channels, int) or latent_channels < 1:
        raise ValueError(f"latent_channels must be int >= 1, got {latent_channels}")
    if not isinstance(K, int) or K < 1:
        raise ValueError(f"K must be int >= 1, got {K}")


def check_input(x: torch.Tensor):
    """x must be a CUDA tensor [B, 3, H, W] with H and W multiples of 64."""
    engine.require_cuda(x, "x")
    if x.dim() != 4 or x.shape[1] != 3:
        raise ValueError(f"expected x of shape [B, 3, H, W], got {tuple(x.shape)}")
    H, W = x.shape[2:]
    if H % 64 or W % 64:
        raise ValueError(f"H and W must be multiples of 64 (four stride-2 stages in g_a, two in h_a); got {H}x{W}")


def draw_noise(M: int, x: torch.Tensor, noise=None):
    """(noise_z, noise_y) of a training forward: `noise` when given, else U(-0.5, 0.5) drawn z first, then y, as the reference
    does (Models.py:57-58), so seeded runs draw the same noise on every path."""
    if noise is not None:
        return noise
    B, _, H, W = x.shape
    return (torch.rand((B, M, H // 64, W // 64), device=x.device) - 0.5, torch.rand((B, M, H // 16, W // 16), device=x.device) - 0.5)


def precision_arms(precision: str) -> Tuple[str, str]:
    """Model precision -> (arm of g_a and h_a, arm of h_s, the context model, the entropy parameters and g_s): "mixed" keeps
    everything that decides the symbols in fp32."""
    return ("fp32" if precision == "mixed" else precision), ("bf16" if precision == "mixed" else precision)


def _param_names(K: int):
    return ("mu", "sigma") if K == 1 else ("weights", "mus", "sigmas")


def mixture_params(ly: dict, K: int, lean: bool = False) -> list:
    """The distribution parameters of a gm_likelihood result in output order: (mu, sigma) for K == 1, else (weights, mus,
    sigmas); none when lean."""
    return [] if lean else [ly[k] for k in _param_names(K)]


def single_head_outputs(x_hat, logp_y, logp_z, y, y_in, z, z_in, p_z, p_y, parts_y, parts_z, *params, K: int, training: bool) -> dict:
    """The output dict of JointAutoregressiveHierarchical and HierarchicalMixtureResidual (Models.py:92-104, same key order)
    from the values in the order training._forward_impl returns them; params = mixture_params(...).  The per-image sums of
    logp ride along on logp_y / logp_z for rd_loss (RateDistortionLoss.py:13-14)."""
    engine.attach_partials(logp_y, parts_y)
    engine.attach_partials(logp_z, parts_z)
    out = {"x_hat": x_hat, "y": y, "y_in": y_in, "z": z, "z_in": z_in, "p_z": p_z, "logp_z": logp_z, "p_y": p_y, "logp_y": logp_y,
           "training": training}
    out.update(zip(_param_names(K), params))
    return out


def two_head_outputs(x_hat, logp_y1, logp_y2, logp_z, y, y_in, z, z_in, p_z, p_y1, p_y2, parts_y1, parts_y2, parts_z, *params,
                     M1: int, K: int, training: bool) -> dict:
    """The output dict of ScalableImageCoding (Models.py:321-338 without 'F_tilde') from the values in the order
    training_scalable's autograd node returns them; params = mixture_params of head 1, then of head 2."""
    for logp, parts in ((logp_y1, parts_y1), (logp_y2, parts_y2), (logp_z, parts_z)):
        engine.attach_partials(logp, parts)
    y1, y2 = torch.split(y_in, [M1, y_in.shape[1] - M1], dim=1)            # Models.py:279 (views, as in the reference)
    out = {"x_hat": x_hat, "y": y, "y_in": y_in, "y1": y1, "y2": y2, "z": z, "z_in": z_in, "p_z": p_z, "logp_z": logp_z,
           "p_y1": p_y1, "logp_y1": logp_y1, "p_y2": p_y2, "logp_y2": logp_y2, "training": training}
    names = _param_names(K)
    out.update(zip([k + "1" for k in names] + [k + "2" for k in names], params))
    return out


# ---- stages of the fused pair-tensor pipeline (JointAutoregressiveHierarchical, ScalableImageCoding's bf16x3 arm, the codec) ----

def _g_a_nhwc(model, x, prec_up):
    """g_a of the fused pipeline: activations NHWC between layers (bf16 hi/lo pairs in the bf16x3 arm) -> y f32 [B, hy, wy, M]."""
    B, _, H, W = x.shape
    a, h, w, layout = x, H, W, LAYOUT_NCHW
    enc = model.encoder.ops
    for i, op in enumerate(enc):
        a = op.run(a, B, h, w, prec_up, in_layout=layout, out_layout=LAYOUT_NHWC,
                   out_dtype=torch.float32 if i == len(enc) - 1 else None)
        h, w = engine.conv_out_hw(op.conv, h, w)
        layout = LAYOUT_NHWC
    return a


def fused_g_a(model, x, training, noise_y, prec_up, prec):
    """g_a -> y hand-off of the fused pipeline (Models.py:52, 57-64).  Returns (y, y_in, y_in_nhwc, y_src) with y_src = the
    unquantised y in the engine's layout for h_a (Models.py:53)."""
    adt = engine.act_dtype(prec)
    pair = prec == "bf16x3"
    y_nhwc = _g_a_nhwc(model, x, prec_up)
    lowp = prec_up != "fp32"
    y, y_in, y_in_nhwc, y_lowp = engine.latent_handoff(y_nhwc, Q_NOISE if training else Q_ROUND, noise_y, "bf16x2" if pair else adt,
                                                       want_lowp=lowp, lowp_pair=prec_up == "bf16x3")
    return y, y_in, y_in_nhwc, (y_lowp if lowp else y_nhwc)


def _h_a_nhwc(model, y_src, B, hy, wy, prec_up):
    a, h, w = y_src, hy, wy
    ha = model.hyper_encoder.ops
    for i, op in enumerate(ha):
        a = op.run(a, B, h, w, prec_up, out_dtype=torch.float32 if i == len(ha) - 1 else None)
        h, w = engine.conv_out_hw(op.conv, h, w)
    return a


def fused_h_a(model, y_src, B, hy, wy, training, noise_z, prec_up, prec):
    """h_a -> z hand-off (Models.py:53, 57-64).  Returns (z, z_in, z_in_nhwc)."""
    adt = engine.act_dtype(prec)
    z, z_in, z_in_nhwc, _ = engine.latent_handoff(_h_a_nhwc(model, y_src, B, hy, wy, prec_up), Q_NOISE if training else Q_ROUND,
                                                  noise_z, "bf16x2" if prec == "bf16x3" else adt)
    return z, z_in, z_in_nhwc


def engine_dtype(prec: str):
    """The hand-off dtype of the activations a transform of arm `prec` reads (latent_handoff's in_dtype)."""
    return "bf16x2" if prec == "bf16x3" else engine.act_dtype(prec)


def fused_g_a_gained(model, x, training, noise_y, prec_up, prec, gains: "Gains"):
    """fused_g_a with gain units: y = g_y (.) g_a(x) is the tensor that is quantised.  Returns (y, y_in, y_in_nhwc, y_src, gs_in):
    the symbols y_in_nhwc (with their lo-half flag) for the context conv, y_src = y for h_a, gs_in = ginv_y (.) y_in for g_s,
    all written by one nic_latent_handoff_gain pass."""
    src = torch.float32 if prec_up == "fp32" else ("bf16x2" if prec_up == "bf16x3" else torch.bfloat16)
    return engine.latent_handoff_gain(_g_a_nhwc(model, x, prec_up), Q_NOISE if training else Q_ROUND, noise_y, gains.g_y, gains.ginv_y,
                                      engine_dtype(prec), src, engine_dtype(prec))


def fused_h_a_gained(model, y_src, B, hy, wy, training, noise_z, prec_up, prec, gains: "Gains"):
    """fused_h_a with gain units: z = g_z (.) h_a(y) is quantised.  Returns (z, z_in, hs_in) with hs_in = ginv_z (.) z_in, h_s's
    input (no lo-half flag: it is not integer)."""
    z, z_in, _, _, hs_in = engine.latent_handoff_gain(_h_a_nhwc(model, y_src, B, hy, wy, prec_up), Q_NOISE if training else Q_ROUND,
                                                      noise_z, gains.g_z, gains.ginv_z, None, None, engine_dtype(prec))
    return z, z_in, hs_in


def fused_h_s_into(model, z_in_nhwc, B, hz, wz, prec, combined, c_total, c_offset, lo_flag):
    """h_s (Models.py:69) with its last conv writing psi into channels [c_offset, c_offset + 2M) of `combined`.  lo_flag: the
    `_nic_lo_flag` of z_in_nhwc (its first conv skips the MMA pass of an all-zero lo half), or None for all three passes."""
    a, h, w = z_in_nhwc, hz, wz
    hs = model.hyper_decoder.ops
    for i, op in enumerate(hs):
        if i == len(hs) - 1:
            op.run(a, B, h, w, prec, out=combined, out_c_total=c_total, out_c_offset=c_offset)
        else:
            a = op.run(a, B, h, w, prec, in_lo_flag=lo_flag if i == 0 else None)
        h, w = engine.conv_out_hw(op.conv, h, w)


_SIDE_STREAMS = {}


def _branch_stream(device, index: int = 0):
    """A second stream for g_s while the forward pass is being CAPTURED in a CUDA graph: g_s (y_in -> x_hat) and the entropy side
    (h_a, h_s, context, entropy parameters, likelihoods) only share y / y_in, so the graph gets two parallel branches and the small
    launches of the entropy side (32-128 CTAs on 148 SMs) and the tails of the big ones overlap the other branch.  Eager launches
    stay on one stream (they are host-bound; forking costs events).  NIC_EVAL_OVERLAP=0 switches it off."""
    if os.environ.get("NIC_EVAL_OVERLAP", "1") == "0" or not torch.cuda.is_current_stream_capturing():
        return None
    key = (str(device), index)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return _SIDE_STREAMS[key]


def fused_g_s(model, y_in_nhwc, B, hy, wy, prec):
    """g_s (Models.py:90): NHWC symbols -> x_hat NCHW f32."""
    y_flag = getattr(y_in_nhwc, "_nic_lo_flag", None)
    a, h, w = y_in_nhwc, hy, wy
    dec = model.decoder.ops
    for i, op in enumerate(dec):
        last = i == len(dec) - 1
        a = op.run(a, B, h, w, prec, out_layout=LAYOUT_NCHW if last else LAYOUT_NHWC,
                   out_dtype=torch.float32 if last else None, in_lo_flag=y_flag if i == 0 else None)
        h, w = engine.conv_out_hw(op.conv, h, w)
    return a


class JointAutoregressiveHierarchical(nn.Module):
    """
    latent_channels : int, default=192, number of channels in the bottleneck y (M).
    K : int, default=1.  K == 1 -> mean-scale Gaussian; K > 1 -> mixture of K Gaussians.
    precision : arithmetic of the transforms (keyword-only extension; the reference has no such switch):
        None / "auto" (default, or $NIC_PRECISION): "bf16x3" when latent_channels == 128, else "fp32" - both parity grade;
        "fp32"  CUDA-core FFMA kernels, fp32 operands and accumulation - parity grade, any channel count;
        "bf16"  tcgen05 tensor-core kernels, bf16 operands, fp32 accumulation - the throughput arm;
        "mixed" g_a and h_a (everything upstream of the rounding, i.e. what decides the symbols) in fp32, the entropy
                path and g_s in bf16: symbols identical to the fp32 arm at ~2.5x its speed;
        "bf16x3" every transform on the tensor cores at fp32 grade: both operands of every contraction (convs and the GDN
                channel mixing) split into bf16 hi + lo and contracted as hi.hi + lo.hi + hi.lo in one fp32 TMEM accumulation
                (~1e-5 relative; 3x the MMA work), activations carried between layers as bf16 hi/lo pairs - the
                parity-grade tensor-core arm.
    """
    context_model_class = ContextModel

    def __init__(self, latent_channels: int = 192, K: int = 1, *, precision: Optional[str] = None):
        super().__init__()
        check_channels(latent_channels, K)
        self.M = latent_channels
        self.K = K
        self.H = latent_channels
        self.distribution = "Mean-Scale Gaussian" if K == 1 else "Mixture of Gaussians"
        self.conditional = GaussianConditional() if K == 1 else GaussianMixtureConditional()
        # construction order follows Models.py:34-46 so a seeded build draws the same initial weights
        self.encoder = Encoder5x5(latent_channels=self.M)
        self.decoder = Decoder5x5(latent_channels=self.M)
        self.hyper_encoder = HyperEncoder5x5(latent_channels=self.M)
        self.hyper_decoder = HyperDecoder5x5(latent_channels=self.M)
        self.factorized_entropy_model = FactorizedEntropyBottleneck(self.M)
        self.context_model = self.context_model_class(latent_channels=self.M)
        self.entropy_parameters = EntropyParameters(latent_channels=self.M, hyper_latent_channels=self.H, K=self.K)
        self.precision = engine.resolve_precision(precision, latent_channels)
        if self.precision not in MODEL_PRECISIONS:
            raise ValueError(f"precision must be one of {MODEL_PRECISIONS}, got {self.precision}")

    def forward(self, x: torch.Tensor, training: bool = True, *,
                noise: Optional[Tuple[torch.Tensor, torch.Tensor]] = None, lean: bool = False):
        """Returns the reference's dict (Models.py:92-104).

        noise : optional (noise_z, noise_y) in U(-0.5, 0.5) to use instead of drawing them
                (training=True only; the reference draws z's noise first, Models.py:57-58).
        lean  : skip materialising weights/mus/sigmas (mu/sigma); those keys are then absent.
        """
        check_input(x)
        return self._forward(x, training, noise, lean, None)

    def _forward(self, x, training, noise, lean, gains: Optional["Gains"]):
        """forward with the gain units' per-image vectors (GainedCheckerboardHierarchical), or None for the model without them."""
        B, _, H, W = x.shape
        if training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            # the reference's training call (Trainer.py:82): autograd is on, so the step must be differentiable.  One autograd
            # node over the fp32 arm with hand-written backward kernels (training.py); under torch.no_grad() the call below
            # runs the forward-only path of self.precision instead.
            from . import training as _training
            return _training.train_forward(self, x, noise=noise, lean=lean, gains=gains)
        if self.precision == "bf16x3" and self.M not in (128, 192):
            # the fused pair-tensor pipeline (GDN kernels, first layer) is built for 128 and 192 channels (the reference's default);
            # other channel counts that are multiples of 64 run layer by layer: every conv and both GDN contractions on the
            # tcgen05 engine, fp32 NHWC tensors in between (training._forward_impl with rounding instead of noise)
            if self.M % 64:
                raise ValueError(f"precision='bf16x3' needs latent_channels % 64 == 0, got {self.M}")
            from . import training as _training
            with torch.no_grad():
                nz, ny = draw_noise(self.M, x, noise) if training else (None, None)
                _training.forget_pairs()
                res, _ = _training._forward_impl(self, x.contiguous().float(), nz, ny, lean, qmode=Q_NOISE if training else Q_ROUND,
                                                 arm="bf16x3", gains=gains)
                _training.forget_pairs()
            return single_head_outputs(*res, K=self.K, training=training)
        prec_up, prec = precision_arms(self.precision)
        adt = engine.act_dtype(prec)
        pair = prec == "bf16x3"                      # activations are bf16 hi/lo pairs: [hi(c) | lo(c)] channels
        cw = 2 if pair else 1
        M, K = self.M, self.K
        x = x.contiguous().float()
        hy, wy, hz, wz = H // 16, W // 16, H // 64, W // 64
        with torch.cuda.device(x.device), torch.no_grad():
            noise_z, noise_y = draw_noise(M, x, noise) if training else (None, None)
            if gains is None:
                y, y_in, y_in_nhwc, y_src = fused_g_a(self, x, training, noise_y, prec_up, prec)
                gs_in = y_in_nhwc
            else:
                y, y_in, y_in_nhwc, y_src, gs_in = fused_g_a_gained(self, x, training, noise_y, prec_up, prec, gains)

            # ---- two parallel branches while the pass is captured in a CUDA graph: g_s (needs y_in only) and the context conv
            # (y_in only) run beside h_a -> h_s; the context conv joins before the 1x1 stack, g_s at the end
            branch, main_stream = _branch_stream(x.device), torch.cuda.current_stream(x.device)
            if branch is not None:
                branch.wait_stream(main_stream)
                with torch.cuda.stream(branch):
                    x_hat = fused_g_s(self, gs_in, B, hy, wy, prec)
            # phi = combined[..., 0:2M] (context), psi = combined[..., 2M:4M] (h_s): torch.cat([phi, psi]) never happens.
            # (the quantised symbols split into bf16 pairs with an all-zero lo half - the hand-off kernel checks and flags it on the
            #  device: their first consumers - h_s layer 1, the context conv, g_s layer 1 - run 2 of the 3 MMA passes)
            combined = torch.empty((B, hy, wy, cw * 4 * M), dtype=adt, device=x.device)
            self.context_model.masked.apply_mask_()
            branch2 = _branch_stream(x.device, 1)
            if branch2 is not None:
                branch2.wait_stream(main_stream)
            # eager launches (no graph branches): context conv + 1x1 stack + likelihood kernel go out through ONE C-ABI call after
            # h_s (nic_ctx_ep_fwd; same kernels, same results).  While a graph is captured the context conv is its own branch instead.
            one_call = branch2 is None and os.environ.get("NIC_CTX_EP_ONE_CALL", "1") != "0"
            y_flag = getattr(y_in_nhwc, "_nic_lo_flag", None)
            if not one_call:
                with (torch.cuda.stream(branch2) if branch2 is not None else contextlib.nullcontext()):
                    self.context_model.masked._op.run(y_in_nhwc, B, hy, wy, prec, out=combined, out_c_total=4 * M, out_c_offset=0,
                                                      in_lo_flag=y_flag)
            if gains is None:
                z, z_in, hs_in = fused_h_a(self, y_src, B, hy, wy, training, noise_z, prec_up, prec)
            else:
                z, z_in, hs_in = fused_h_a_gained(self, y_src, B, hy, wy, training, noise_z, prec_up, prec, gains)
            fused_h_s_into(self, hs_in, B, hz, wz, prec, combined, 4 * M, 2 * M, getattr(hs_in, "_nic_lo_flag", None))
            if branch2 is not None:
                main_stream.wait_stream(branch2)

            ep = self.entropy_parameters.ops
            if one_call:
                key = (B, hy, wy, prec, bool(lean), str(x.device))
                plans = self.__dict__.setdefault("_ctx_ep_plans", {})
                if key not in plans:
                    plans.clear()                                # one shape at a time: the plan owns the two hidden activations
                    plans[key] = engine.CtxEpPlan(self.context_model.masked._op, ep, B, hy, wy, prec, M, K, x.device, full=not lean)
                raw, ly = plans[key].run(y_in_nhwc, combined, y_in=y_in, qmode=Q_PASSTHRU, in_lo_flag=y_flag)
            else:
                # ---- entropy parameters (1x1 stack) ---------------------------------------------------
                a = ep[0].run(combined, B, hy, wy, prec)
                a = ep[1].run(a, B, hy, wy, prec)
                raw = ep[2].run(a, B, hy, wy, prec, out_layout=LAYOUT_NCHW, out_dtype=torch.float32)
                # ---- likelihoods -------------------------------------------------------------------------
                ly = gm_likelihood(y_in, raw, M, K, Q_PASSTHRU, full=not lean, want_y_in=False)
            _, p_z, logp_z, parts_z = self.factorized_entropy_model.likelihood(z_in, Q_PASSTHRU)

            # ---- g_s -----------------------------------------------------------------------------------
            if branch is not None:
                main_stream.wait_stream(branch)                 # join
            else:
                x_hat = fused_g_s(self, gs_in, B, hy, wy, prec)
        return single_head_outputs(x_hat, ly["logp"], logp_z, y, y_in, z, z_in, p_z, ly["p"], ly["partials"], parts_z,
                                   *mixture_params(ly, K, lean), K=K, training=training)

    def compress(self, x: torch.Tensor) -> dict:
        """x [B, 3, H, W] (any H, W >= 1) -> {"strings": [y_strings, z_strings], "shape": (hz, wz)}: one bytes object per
        image in each list, coded with the eval-mode symbols (the forward's y_in / z_in) of x padded by edge replication to
        multiples of 64 (shape is the padded one).  Format: DESIGN.md sections 9 and 12."""
        from . import codec
        return codec.compress(self, x)

    def decompress(self, strings, shape) -> dict:
        """strings / shape as compress returned them (any subset of the images, in any order) -> {"x_hat", "y_hat", "z_hat"}, NCHW f32;
        x_hat = g_s(y_hat) cropped to the image's size, not clamped; y_hat / z_hat at the padded latent shape.  Raises ValueError on a
        string of another precision arm / M / K, on a malformed string or image size, or when an image's symbol checksum does not match
        (corrupted bytes, other weights)."""
        from . import codec
        return codec.decompress(self, strings, shape)


class JointCheckerboardHierarchical(JointAutoregressiveHierarchical):
    """JointAutoregressiveHierarchical with the checkerboard context model (He et al., CVPR 2021; convention in ContextModels.py
    and DESIGN.md section 14): same constructor, attributes, precision arms, output dict and ``state_dict`` keys, modules built in
    the same order (a seeded build draws the same weights); ``context_model`` is a CheckerboardContextModel.  Anchors (i + j even)
    are coded from the hyperprior alone, non-anchors from the hyperprior and the anchors, so ``decompress`` runs two parameter passes
    and two rANS passes at any image size instead of one wavefront step per 3 hy + wy - 3.  Every forward route (eager, graph
    branches, CtxEpPlan, the layer-by-layer and training forms) gets the anchor zeroing from the conv call itself."""
    context_model_class = CheckerboardContextModel

    def compress(self, x: torch.Tensor) -> dict:
        """x [B, 3, H, W] (any H, W >= 1) -> {"strings": [y_strings, z_strings], "shape": (hz, wz)}: one bytes object per
        image in each list, coded with the eval-mode symbols of x padded by edge replication to multiples of 64 (shape is the
        padded one).  Format 4: DESIGN.md sections 12 and 14."""
        from . import checkerboard_codec
        return checkerboard_codec.compress(self, x)

    def decompress(self, strings, shape) -> dict:
        """strings / shape as compress returned them (any subset of the images, in any order) -> {"x_hat", "y_hat", "z_hat"}, NCHW f32;
        x_hat = g_s(y_hat) cropped to the image's size, not clamped; y_hat / z_hat at the padded latent shape.  Raises ValueError on a
        string of another model, precision arm, M or K, on a malformed string or image size, or when an image's symbol checksum does not
        match (corrupted bytes, other weights)."""
        from . import checkerboard_codec
        return checkerboard_codec.decompress(self, strings, shape)


QUALITY_QUANTUM = 1024                               # every route snaps quality q to q_code / 1024, q_code = round(1024 q)


class GainUnits(nn.Module):
    """The gain units of Cui et al. (CVPR 2021): L learned rows of per-channel gains on y and z and of their inverse gains, stored as
    natural logs (initialised to 0, i.e. gains of 1), each parameter [L, M]."""

    def __init__(self, levels: int, channels: int):
        super().__init__()
        for name in ("y_log_gain", "y_log_inv_gain", "z_log_gain", "z_log_inv_gain"):
            setattr(self, name, nn.Parameter(torch.zeros(levels, channels)))

    def tables(self):
        return self.y_log_gain, self.y_log_inv_gain, self.z_log_gain, self.z_log_inv_gain


class Gains:
    """The per-image gain vectors of one call: vec [4, B, M] = (g_y, ginv_y, g_z, ginv_z) from nic_gain_vectors, q_code int32 [B]."""

    def __init__(self, vec: torch.Tensor, q_code: torch.Tensor):
        self.vec, self.q_code = vec, q_code
        self.g_y, self.ginv_y, self.g_z, self.ginv_z = vec.unbind(0)

    @property
    def quality(self) -> torch.Tensor:
        return self.q_code.float() / QUALITY_QUANTUM


def quality_codes(levels: int, quality, B: int, device) -> torch.Tensor:
    """quality (None = levels - 1, a float, a sequence or tensor of 1 or B values in [0, levels - 1]) -> q_code int32 [B] on `device`,
    q_code = floor(1024 q + 0.5).  Host values are checked (ValueError); a CUDA tensor (the trainer's draws) is snapped and clamped
    on the device without a host synchronisation."""
    top = QUALITY_QUANTUM * (levels - 1)
    if isinstance(quality, torch.Tensor) and quality.is_cuda:
        q = quality.detach().reshape(-1).float()
        if q.numel() not in (1, B):
            raise ValueError(f"quality: expected 1 or {B} values, got {q.numel()}")
        return torch.floor(q * QUALITY_QUANTUM + 0.5).clamp_(0, top).to(torch.int32).expand(B).contiguous()
    if quality is None:
        vals = [float(levels - 1)]
    elif isinstance(quality, torch.Tensor):
        vals = [float(v) for v in quality.reshape(-1).tolist()]
    elif isinstance(quality, (int, float)):
        vals = [float(quality)]
    else:
        vals = [float(v) for v in quality]
    if len(vals) not in (1, B):
        raise ValueError(f"quality: expected 1 or {B} values, got {len(vals)}")
    for v in vals:
        if not (0.0 <= v <= levels - 1):
            raise ValueError(f"quality must lie in [0, {levels - 1}], got {v}")
    codes = [min(int(math.floor(v * QUALITY_QUANTUM + 0.5)), top) for v in vals]
    return torch.tensor(codes * (B // len(codes)) if len(codes) == 1 else codes, dtype=torch.int32).to(device)


def gain_vectors(model, q_code: torch.Tensor) -> Gains:
    """nic_gain_vectors: the per-image gains of the quality codes q_code (device int32 [B]) - the one kernel the forward, the encoder
    and the decoder share."""
    gu = model.gain_units
    tabs = [t.detach().float().contiguous() for t in gu.tables()]
    engine.require_cuda(tabs[0], "gain tables")
    B = q_code.numel()
    L, M = tabs[0].shape
    vec = torch.empty((4, B, M), dtype=torch.float32, device=tabs[0].device)
    with torch.cuda.device(vec.device):
        _lib.check(_lib.load().nic_gain_vectors(*[_lib.ptr(t) for t in tabs], L, M, _lib.ptr(q_code), B, _lib.ptr(vec),
                                                _lib.current_stream()), "nic_gain_vectors")
    return Gains(vec, q_code)


class GainedCheckerboardHierarchical(JointCheckerboardHierarchical):
    """JointCheckerboardHierarchical that codes at any quality q in [0, levels - 1] with gain units (Cui et al., CVPR 2021; DESIGN.md
    section 15).  ``gain_units`` holds four [levels, M] log-gain tables; for image b, l = floor(q), t = q - l and each gain is
    expf((1 - t) log[l] + t log[min(l + 1, levels - 1)]).  y = g_y (.) g_a(x) is quantised; the context conv, the 1x1 stack and the
    likelihood read y_in, h_a reads y, g_s reads ginv_y (.) y_in; z = g_z (.) h_a(y) is quantised, the factorized prior reads z_in
    and h_s reads ginv_z (.) z_in.  With every log-gain 0 it computes exactly JointCheckerboardHierarchical.

    The modules are built in the parent's order with ``gain_units`` last: a seeded build draws the parent's weights, and a parent
    checkpoint loads with ``load_state_dict(..., strict=False)`` (the fine-tuning path from a single-rate model)."""

    def __init__(self, latent_channels: int = 192, K: int = 1, levels: int = 6, *, precision: Optional[str] = None):
        if not isinstance(levels, int) or isinstance(levels, bool) or not 2 <= levels <= 64:
            raise ValueError(f"levels must be an int in [2, 64], got {levels!r}")
        super().__init__(latent_channels, K, precision=precision)
        self.levels = levels
        self.gain_units = GainUnits(levels, self.M)

    def gains(self, quality, B: int, device) -> Gains:
        return gain_vectors(self, quality_codes(self.levels, quality, B, device))

    def forward(self, x: torch.Tensor, training: bool = True, *, quality=None,
                noise: Optional[Tuple[torch.Tensor, torch.Tensor]] = None, lean: bool = False):
        """The parent's dict at quality `quality` (None = levels - 1; a float, or one value per image), plus 'quality': the snapped
        per-image values [B] (round(1024 q) / 1024), which every route (forward, training, compress, decompress) uses."""
        check_input(x)
        gains = self.gains(quality, x.shape[0], x.device)
        out = self._forward(x, training, noise, lean, gains)
        out["quality"] = gains.quality
        return out

    def compress(self, x: torch.Tensor, quality=None) -> dict:
        """x [B, 3, H, W] (any H, W >= 1) at quality `quality` (a float or one value per image) -> {"strings": [y_strings, z_strings],
        "shape": (hz, wz)}.  Format 5: DESIGN.md section 15."""
        from . import gained_codec
        return gained_codec.compress(self, x, quality)

    def decompress(self, strings, shape) -> dict:
        """strings / shape as compress returned them (any subset of the images, in any order) -> {"x_hat", "y_hat", "z_hat",
        "quality"}; each image at the quality its string carries.  Raises ValueError on a string of another model, precision arm, M,
        K or number of levels, on a malformed string, quality or image size, or on a checksum mismatch."""
        from . import gained_codec
        return gained_codec.decompress(self, strings, shape)


def default_slices(M: int) -> Tuple[int, ...]:
    """64-channel slices with any remainder as the last one: (64, 64) at M = 128, (64, 64, 64) at 192, (M,) below 64."""
    n, r = divmod(M, 64)
    return (64,) * n + ((r,) if r else ()) if n else (M,)


def check_slices(slices, M: int) -> Tuple[int, ...]:
    """slices (None = default_slices) -> a tuple of positive ints that sum to M; ValueError otherwise."""
    if slices is None:
        return default_slices(M)
    if not isinstance(slices, (tuple, list)) or not slices or \
            any(not isinstance(m, int) or isinstance(m, bool) or m < 1 for m in slices) or sum(slices) != M:
        raise ValueError(f"slices must be a non-empty tuple of positive ints that sum to latent_channels={M}, got {slices!r}")
    return tuple(slices)


def merge_slices(lys: list, K: int, lean: bool):
    """The likelihood dicts of the channel slices -> (logp, p, per-image partial sums of logp, *mixture params) over all M channels
    in channel order.  One slice: its own tensors (so slices=(M,) returns what JointCheckerboardHierarchical returns)."""
    if len(lys) == 1:
        return (lys[0]["logp"], lys[0]["p"], lys[0]["partials"], *mixture_params(lys[0], K, lean))
    logp = torch.cat([ly["logp"] for ly in lys], dim=1)
    p = torch.cat([ly["p"] for ly in lys], dim=1)
    parts = engine.partials(logp.shape[0], logp.device)
    with torch.cuda.device(logp.device):
        _lib.check(_lib.load().nic_sum_fwd(_lib.ptr(logp), logp.shape[0], logp[0].numel(), _lib.ptr(parts), _lib.current_stream()),
                   "nic_sum_fwd")
    params = [] if lean else [torch.cat([ly[k] for ly in lys], dim=1 if K == 1 else 2) for k in _param_names(K)]
    return (logp, p, parts, *params)


def _channel_window(t: torch.Tensor, c0: int, c1: int, M: int, pair: bool) -> torch.Tensor:
    """Channels [c0, c1) of NHWC symbols with M channels (pairs: [hi(M) | lo(M)] -> [hi | lo] of the window), contiguous."""
    if c0 == 0 and c1 == M:
        return t
    if pair:
        return torch.cat([t[..., c0:c1], t[..., M + c0:M + c1]], dim=-1).contiguous()
    return t[..., c0:c1].contiguous()


def slice_buffers(model, B: int, hy: int, wy: int, prec: str, device) -> list:
    """One NHWC concat buffer per slice, [phi_sp (2 m_s) | phi_ch (2 m_s, s >= 1) | psi (2 M)] (bf16x3: [hi | lo] pairs)."""
    pair = prec == "bf16x3"
    return [torch.empty((B, hy, wy, (2 if pair else 1) * ep.net[0].in_channels), dtype=engine.act_dtype(prec), device=device)
            for ep in model.entropy_parameters]


def slice_psi_into(model, z_eng, B: int, hz: int, wz: int, prec: str, combs: list, lo_flag):
    """h_s writes psi into slice 0's buffer; every other slice's buffer gets a copy (both halves of a pair)."""
    M, pair = model.M, prec == "bf16x3"
    c0 = combs[0].shape[-1] // (2 if pair else 1)
    fused_h_s_into(model, z_eng, B, hz, wz, prec, combs[0], c0, c0 - 2 * M, lo_flag)
    for comb in combs[1:]:
        c = comb.shape[-1] // (2 if pair else 1)
        comb[..., c - 2 * M:c] = combs[0][..., c0 - 2 * M:c0]
        if pair:
            comb[..., 2 * c - 2 * M:] = combs[0][..., 2 * c0 - 2 * M:]


def slice_raw(model, s: int, y_eng: torch.Tensor, comb: torch.Tensor, B: int, hy: int, wy: int, prec: str, lo_flag=None) -> torch.Tensor:
    """The raw entropy parameters [B, (3K | 2) m_s, hy, wy] of slice s from the engine-layout symbols y_eng (all M channels) and
    the slice's buffer with psi in place: checkerboard conv over the slice, channel conv over the slices before it, 1x1 stack.  The
    eval forward and both directions of the coder call this."""
    M, pair = model.M, prec == "bf16x3"
    o, m = model.offsets[s], model.slices[s]
    c = comb.shape[-1] // (2 if pair else 1)
    ctx = model.context_models[s].masked
    ctx.apply_mask_()
    ctx._op.run(_channel_window(y_eng, o, o + m, M, pair), B, hy, wy, prec, out=comb, out_c_total=c, out_c_offset=0, in_lo_flag=lo_flag)
    if s > 0:
        model.channel_contexts[s - 1]._op.run(_channel_window(y_eng, 0, o, M, pair), B, hy, wy, prec, out=comb, out_c_total=c,
                                              out_c_offset=2 * m, in_lo_flag=lo_flag)
    ops = model.entropy_parameters[s].ops
    a = ops[0].run(comb, B, hy, wy, prec)
    a = ops[1].run(a, B, hy, wy, prec)
    return ops[2].run(a, B, hy, wy, prec, out_layout=LAYOUT_NCHW, out_dtype=torch.float32)


class ChannelCheckerboardHierarchical(nn.Module):
    """The space-channel context model (ELIC, He et al., CVPR 2022, after the channel-wise autoregression of Minnen & Singh, ICIP
    2020; DESIGN.md section 16): JointCheckerboardHierarchical's trunk (g_a, g_s, h_a, h_s, factorized prior) with y split into the
    channel slices `slices` (default 64-channel slices, any remainder last).  Slice s, channels [o_s, o_s + m_s), is coded from
    [phi_sp | phi_ch | psi]:
      * phi_sp = context_models[s] (CheckerboardContextModel(m_s)) over the slice: 0 at the anchors;
      * phi_ch = channel_contexts[s - 1] (ChannelContextModel(o_s, m_s), s >= 1) over the slices before it: not zeroed, they are
        fully decoded before slice s starts;
      * psi = h_s(z_hat), shared by every slice;
    through entropy_parameters[s] (1x1 stack, cin = 2 m_s (+ 2 m_s) + 2 M -> 640 -> 640 -> (2 | 3K) m_s).  Training reads the noisy
    y_in of the earlier slices (teacher forcing).  decompress runs two parameter and two rANS passes per slice.

    The trunk is built first and in the parent's order (a seeded build draws the parent's trunk; a parent checkpoint loads its trunk
    with ``load_state_dict(..., strict=False)``), then the slice modules slice by slice.  With slices=(M,) and the parent's weights
    under context_models.0 / entropy_parameters.0 the model computes exactly JointCheckerboardHierarchical.

    precision: "bf16x3" (default when M and every slice width are multiples of 64) or "fp32".  The eval forward runs the fused
    pipeline in fp32 and in bf16x3 at M = 128 / 192, else training._forward_impl without tapes."""

    def __init__(self, latent_channels: int = 192, K: int = 1, slices=None, *, precision: Optional[str] = None):
        super().__init__()
        check_channels(latent_channels, K)
        self.M, self.K, self.H = latent_channels, K, latent_channels
        self.slices = check_slices(slices, latent_channels)
        self.offsets = tuple(sum(self.slices[:s]) for s in range(len(self.slices)))
        tc_ok = all(c % 64 == 0 for c in (self.M,) + self.slices)
        precision = precision or engine.DEFAULT_PRECISION
        self.precision = ("bf16x3" if tc_ok else "fp32") if precision == "auto" else precision
        if self.precision not in ("fp32", "bf16x3") or (self.precision == "bf16x3" and not tc_ok):
            raise ValueError("ChannelCheckerboardHierarchical: precision must be 'fp32', or 'bf16x3' with latent_channels and every "
                             f"slice width multiples of 64; got precision={self.precision!r}, slices={self.slices}")
        self.distribution = "Mean-Scale Gaussian" if K == 1 else "Mixture of Gaussians"
        self.conditional = GaussianConditional() if K == 1 else GaussianMixtureConditional()
        # the trunk in JointCheckerboardHierarchical's order, then the slice modules slice by slice
        self.encoder = Encoder5x5(latent_channels=self.M)
        self.decoder = Decoder5x5(latent_channels=self.M)
        self.hyper_encoder = HyperEncoder5x5(latent_channels=self.M)
        self.hyper_decoder = HyperDecoder5x5(latent_channels=self.M)
        self.factorized_entropy_model = FactorizedEntropyBottleneck(self.M)
        self.context_models, self.channel_contexts, self.entropy_parameters = nn.ModuleList(), nn.ModuleList(), nn.ModuleList()
        for s, (o, m) in enumerate(zip(self.offsets, self.slices)):
            self.context_models.append(CheckerboardContextModel(latent_channels=m))
            if s > 0:
                self.channel_contexts.append(ChannelContextModel(o, m))
            self.entropy_parameters.append(EntropyParameters(latent_channels=m, hyper_latent_channels=self.H, K=K,
                                                             context_channels=2 * m if s > 0 else 0))

    @property
    def fused_pipeline(self) -> bool:
        """True when the eval forward runs the fused pipeline (fp32, or bf16x3 at M = 128 / 192), else training._forward_impl."""
        return self.precision == "fp32" or self.M in (128, 192)

    def forward(self, x: torch.Tensor, training: bool = True, *, noise: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
                lean: bool = False):
        """JointCheckerboardHierarchical's dict: p_y / logp_y and mu / sigma (weights / mus / sigmas) over all M channels in channel
        order; logp_y carries the per-image partial sums for rd_loss."""
        check_input(x)
        from . import training as T
        if training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            return T.train_forward(self, x, noise=noise, lean=lean)
        if self.fused_pipeline:
            return self._forward_fused(x, training, noise, lean)
        with torch.no_grad():
            noise_z, noise_y = draw_noise(self.M, x, noise) if training else (None, None)
            T.forget_pairs()
            outs, _ = T._forward_impl(self, x.contiguous().float(), noise_z, noise_y, lean, qmode=Q_NOISE if training else Q_ROUND,
                                      arm=self.precision, record=False)
            T.forget_pairs()
        return single_head_outputs(*outs, K=self.K, training=training)

    def _forward_fused(self, x, training, noise, lean):
        """The trunk on the fused pipeline (g_s a parallel branch of a captured graph), the slices on slice_raw + the likelihood."""
        B, _, H, W = x.shape
        M, K, prec = self.M, self.K, self.precision
        x = x.contiguous().float()
        hy, wy, hz, wz = H // 16, W // 16, H // 64, W // 64
        with torch.cuda.device(x.device), torch.no_grad():
            noise_z, noise_y = draw_noise(M, x, noise) if training else (None, None)
            y, y_in, y_in_nhwc, y_src = fused_g_a(self, x, training, noise_y, prec, prec)
            branch, main_stream = _branch_stream(x.device), torch.cuda.current_stream(x.device)
            if branch is not None:
                branch.wait_stream(main_stream)
                with torch.cuda.stream(branch):
                    x_hat = fused_g_s(self, y_in_nhwc, B, hy, wy, prec)
            z, z_in, z_in_nhwc = fused_h_a(self, y_src, B, hy, wy, training, noise_z, prec, prec)
            combs = slice_buffers(self, B, hy, wy, prec, x.device)
            slice_psi_into(self, z_in_nhwc, B, hz, wz, prec, combs, getattr(z_in_nhwc, "_nic_lo_flag", None))
            y_flag = getattr(y_in_nhwc, "_nic_lo_flag", None)
            lys = []
            for s, (o, m) in enumerate(zip(self.offsets, self.slices)):
                raw = slice_raw(self, s, y_in_nhwc, combs[s], B, hy, wy, prec, y_flag)
                y_s = y_in if m == M else y_in[:, o:o + m].contiguous()
                lys.append(gm_likelihood(y_s, raw, m, K, Q_PASSTHRU, full=not lean, want_y_in=False))
            logp_y, p_y, parts_y, *params = merge_slices(lys, K, lean)
            _, p_z, logp_z, parts_z = self.factorized_entropy_model.likelihood(z_in, Q_PASSTHRU)
            if branch is not None:
                main_stream.wait_stream(branch)
            else:
                x_hat = fused_g_s(self, y_in_nhwc, B, hy, wy, prec)
        return single_head_outputs(x_hat, logp_y, logp_z, y, y_in, z, z_in, p_z, p_y, parts_y, parts_z, *params, K=K, training=training)

    def compress(self, x: torch.Tensor) -> dict:
        """x [B, 3, H, W] (any H, W >= 1) -> {"strings": [y_strings, z_strings], "shape": (hz, wz)}: one bytes object per image in
        each list, coded with the eval-mode symbols of x padded by edge replication to multiples of 64 (shape is the padded one).
        Format 6: DESIGN.md sections 12 and 16."""
        from . import channel_codec
        return channel_codec.compress(self, x)

    def decompress(self, strings, shape) -> dict:
        """strings / shape as compress returned them (any subset of the images, in any order) -> {"x_hat", "y_hat", "z_hat"}, NCHW f32;
        x_hat = g_s(y_hat) cropped to the image's size, not clamped.  Raises ValueError on a string of another model, precision arm,
        M, K or slices, on a malformed string or image size, or when an image's symbol checksum does not match."""
        from . import channel_codec
        return channel_codec.decompress(self, strings, shape)


class HierarchicalMixtureResidual(nn.Module):
    """``HierarchicalMixtureResidual`` of /root/reference/Models.py:109-205: the same entropy side and output dict as
    JointAutoregressiveHierarchical with the 3x3 residual transforms (Encoder3x3 / Decoder3x3 / HyperEncoder3x3 / HyperDecoder3x3,
    Components.py:20-122, blocks of Layers.py).  Same constructor, attributes and ``state_dict`` keys.

    The transforms run layer by layer on the conv engine (f32 NHWC tensors between layers; residual sums by nic_add_inplace),
    the entropy side on the same kernels as the 5x5 model.  With autograd enabled and training=True the call is the training
    step's forward (training.train_forward: one autograd node; backward = training.Tape over the same C-ABI backward kernels
    as the 5x5 model).  precision: "bf16x3" (default when latent_channels is a multiple of 64: tensor cores with hi/lo-
    split operands; the RGB-input convs of the first block on conv_smallcin_kernel in fp32) or "fp32"."""

    def __init__(self, latent_channels: int = 192, K: int = 1, *, precision: Optional[str] = None):
        super().__init__()
        check_channels(latent_channels, K)
        from .Components import Decoder3x3, Encoder3x3, HyperDecoder3x3, HyperEncoder3x3
        self.M = latent_channels
        self.K = K
        self.H = latent_channels
        self.distribution = "Mean-Scale Gaussian" if K == 1 else "Mixture of Gaussians"
        self.conditional = GaussianConditional() if K == 1 else GaussianMixtureConditional()
        # construction order follows Models.py:133-146 so a seeded build draws the reference's initial weights
        self.encoder = Encoder3x3(latent_channels=self.M)
        self.decoder = Decoder3x3(latent_channels=self.M)
        self.hyper_encoder = HyperEncoder3x3(latent_channels=self.M)
        self.hyper_decoder = HyperDecoder3x3(latent_channels=self.M)
        self.factorized_entropy_model = FactorizedEntropyBottleneck(self.M)
        self.context_model = ContextModel(latent_channels=self.M)
        self.entropy_parameters = EntropyParameters(latent_channels=self.M, hyper_latent_channels=self.H, K=self.K)
        precision = precision or engine.DEFAULT_PRECISION
        self.precision = ("bf16x3" if self.M % 64 == 0 else "fp32") if precision == "auto" else precision
        if self.precision not in ("fp32", "bf16x3") or (self.precision == "bf16x3" and self.M % 64):
            raise ValueError("HierarchicalMixtureResidual: precision must be 'fp32', or 'bf16x3' with latent_channels % 64 == 0")

    def forward(self, x: torch.Tensor, training: bool = True, *, noise: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
                lean: bool = False):
        check_input(x)
        from . import training as T
        if training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            # the training step: ONE autograd node over the hand-written backward (training.Tape walks the residual graphs)
            return T.train_forward(self, x, noise=noise, lean=lean)
        # evaluation: the training forward's layer-by-layer form without tapes (training._forward_impl, record=False)
        with torch.no_grad():
            noise_z, noise_y = draw_noise(self.M, x, noise) if training else (None, None)
            outs, _ = T._forward_impl(self, x.contiguous().float(), noise_z, noise_y, lean, qmode=Q_NOISE if training else Q_ROUND,
                                      arm=self.precision, record=False)
        return single_head_outputs(*outs, K=self.K, training=training)

    def compress(self, x: torch.Tensor) -> dict:
        """x [B, 3, H, W] (any H, W >= 1) -> {"strings": [y_strings, z_strings], "shape": (hz, wz)}: one bytes object per
        image in each list, coded with the eval-mode symbols (the forward's y_in / z_in) of x padded by edge replication to
        multiples of 64 (shape is the padded one).  Format: DESIGN.md sections 11 and 12."""
        from . import residual_codec
        return residual_codec.compress(self, x)

    def decompress(self, strings, shape) -> dict:
        """strings / shape as compress returned them (any subset of the images, in any order) -> {"x_hat", "y_hat", "z_hat"}, NCHW f32;
        x_hat = g_s(y_hat) cropped to the image's size, not clamped; y_hat / z_hat at the padded latent shape.  Raises ValueError on a
        string of another model, precision arm, M or K, on a malformed string or image size, or when an image's symbol checksum does not
        match (corrupted bytes, other weights)."""
        from . import residual_codec
        return residual_codec.decompress(self, strings, shape)


class ScalableImageCoding(nn.Module):
    """The scalable-coding variant of /root/reference/Models.py:208-338: the JointAutoregressiveHierarchical trunk at M
    channels with y split into a base part y1 (M1 channels) and an enhancement part y2 (M - M1), each with its own
    (context model, entropy-parameter net, conditional), both heads sharing the hyper features psi.

    The reference's forward raises as committed (SURVEY.md section 2.4); this class implements the evident intent,
    i.e. the reference with these four repairs, and nothing else:
      * ``self.factorized_entropy_model(z_in, debug)`` (Models.py:302)  ->  ``self.factorized_entropy_model(z_in)``
      * K == 1: ``conditional(y1, mu1=, sigma1=)`` (:293-294, :305-306)  ->  ``conditional(y1, mu=mu1, sigma=sigma1)``
      * K > 1: ``params1`` assigned twice (:298-299)                      ->  ``params2`` holds the second head
      * ``LatentSpaceTransform`` (:256, :319; inconsistent channel counts, Components.py:129-132) is NOT built: the output
        dict has no 'F_tilde', and reference checkpoints load with their ``LST.*`` entries ignored.
    Parity for this class is against the reference's own sub-modules called in that repaired order
    (oracle/make_golden.py: scalable cases) - "parity unpinned" by the reference itself, which has no runnable forward.
    Arithmetic: precision="bf16x3" (default for channel counts that are multiples of 64) runs the convolutions and the GDN
    contractions on the tensor cores, "fp32" on the CUDA cores; both meet the parity bar (tests/test_gpu_scalable.py).
    """

    def __init__(self, latent_channels: int = 192, base_channels: int = 128, K: int = 1, *, precision: Optional[str] = None):
        super().__init__()
        check_channels(latent_channels, K)
        if not isinstance(base_channels, int) or not 0 < base_channels < latent_channels:
            raise ValueError(f"base_channels must be an int in (0, latent_channels), got {base_channels}")
        self.M, self.M1, self.M2 = latent_channels, base_channels, latent_channels - base_channels
        self.H, self.K = latent_channels, K
        self.distribution = "Mean-Scale Gaussian" if K == 1 else "Mixture of Gaussians"
        self.conditional = GaussianConditional() if K == 1 else GaussianMixtureConditional()
        # construction order follows Models.py:237-254 so a seeded build draws the reference's initial weights
        self.encoder = Encoder5x5(latent_channels=self.M)
        self.decoder = Decoder5x5(latent_channels=self.M)
        self.hyper_encoder = HyperEncoder5x5(latent_channels=self.M)
        self.hyper_decoder = HyperDecoder5x5(latent_channels=self.M)
        self.factorized_entropy_model = FactorizedEntropyBottleneck(self.M)
        self.context_model_1 = ContextModel(latent_channels=self.M1)
        self.context_model_2 = ContextModel(latent_channels=self.M2)
        self.entropy_parameters_1 = EntropyParameters(latent_channels=self.M1, hyper_latent_channels=self.H, K=self.K)
        self.entropy_parameters_2 = EntropyParameters(latent_channels=self.M2, hyper_latent_channels=self.H, K=self.K)
        # "bf16x3" (default when every channel count is a multiple of 64, e.g. the reference's 192 / 128): every convolution
        # and the GDN channel contractions on the tcgen05 engine with hi/lo-split operands (fp32 grade), fp32 NHWC tensors
        # between layers split on the fly - the layer-by-layer form the training step uses (training.conv_forward / gdn_forward);
        # "fp32": CUDA cores.
        tc_ok = all(c % 64 == 0 for c in (self.M, self.M1, self.M2))
        precision = precision or engine.DEFAULT_PRECISION
        self.precision = ("bf16x3" if tc_ok else "fp32") if precision == "auto" else precision
        if self.precision not in ("fp32", "bf16x3") or (self.precision == "bf16x3" and not tc_ok):
            raise ValueError("ScalableImageCoding: precision must be 'fp32', or 'bf16x3' with channel counts that are multiples of 64")

    def load_state_dict(self, state_dict, strict: bool = True, **kwargs):
        return super().load_state_dict({k: v for k, v in state_dict.items() if not k.startswith("LST.")}, strict=strict, **kwargs)

    def _forward_pairs(self, x, training, noise):
        """The bf16x3 arm on the fused pipeline of JointAutoregressiveHierarchical (conv -> GDN kernel, activations as bf16 hi/lo
        pairs, no fp32 round trips): the shared trunk, then the two (context, entropy-parameter, likelihood) heads over psi."""
        B, _, H, W = x.shape
        M, M1, M2, K = self.M, self.M1, self.M2, self.K
        prec = "bf16x3"
        x = x.contiguous().float()
        hy, wy, hz, wz = H // 16, W // 16, H // 64, W // 64
        with torch.cuda.device(x.device), torch.no_grad():
            noise_z, noise_y = draw_noise(M, x, noise) if training else (None, None)
            y, y_in, y_in_nhwc, y_src = fused_g_a(self, x, training, noise_y, prec, prec)
            branch, main_stream = _branch_stream(x.device), torch.cuda.current_stream(x.device)
            if branch is not None:                                        # g_s as a parallel branch of a captured graph
                branch.wait_stream(main_stream)
                with torch.cuda.stream(branch):
                    x_hat = fused_g_s(self, y_in_nhwc, B, hy, wy, prec)
            z, z_in, z_in_nhwc = fused_h_a(self, y_src, B, hy, wy, training, noise_z, prec, prec)
            y_flag = getattr(y_in_nhwc, "_nic_lo_flag", None)
            c1, c2 = 2 * M1 + 2 * M, 2 * M2 + 2 * M                       # [phi_i (2 M_i) | psi (2 M)] channels of the two heads
            comb1 = torch.empty((B, hy, wy, 2 * c1), dtype=torch.bfloat16, device=x.device)      # pair tensors: [hi(c) | lo(c)]
            comb2 = torch.empty((B, hy, wy, 2 * c2), dtype=torch.bfloat16, device=x.device)
            fused_h_s_into(self, z_in_nhwc, B, hz, wz, prec, comb1, c1, 2 * M1,                  # psi once, into head 1's buffer
                           getattr(z_in_nhwc, "_nic_lo_flag", None))
            comb2[..., 2 * M2:c2] = comb1[..., 2 * M1:c1]                                        # ... head 2 gets a copy: hi half,
            comb2[..., c2 + 2 * M2:] = comb1[..., c1 + 2 * M1:]                                  # lo half
            y1, y2 = torch.split(y_in, [M1, M2], dim=1)                   # Models.py:279 (views, as in the reference)
            heads = []
            for ctx, ep, comb, ct, lo, hi_, yi in ((self.context_model_1, self.entropy_parameters_1, comb1, c1, 0, M1, y1),
                                                   (self.context_model_2, self.entropy_parameters_2, comb2, c2, M1, M, y2)):
                mi = hi_ - lo
                yi_pair = torch.cat([y_in_nhwc[..., lo:hi_], y_in_nhwc[..., M + lo:M + hi_]], dim=-1).contiguous()
                ctx.masked.apply_mask_()
                ctx.masked._op.run(yi_pair, B, hy, wy, prec, out=comb, out_c_total=ct, out_c_offset=0, in_lo_flag=y_flag)
                a = ep.ops[0].run(comb, B, hy, wy, prec)
                a = ep.ops[1].run(a, B, hy, wy, prec)
                raw = ep.ops[2].run(a, B, hy, wy, prec, out_layout=LAYOUT_NCHW, out_dtype=torch.float32)
                heads.append(gm_likelihood(yi.contiguous(), raw, mi, K, Q_PASSTHRU, full=True, want_y_in=False))
            _, p_z, logp_z, parts_z = self.factorized_entropy_model.likelihood(z_in, Q_PASSTHRU)
            if branch is not None:
                main_stream.wait_stream(branch)
            else:
                x_hat = fused_g_s(self, y_in_nhwc, B, hy, wy, prec)
        l1, l2 = heads
        return two_head_outputs(x_hat, l1["logp"], l2["logp"], logp_z, y, y_in, z, z_in, p_z, l1["p"], l2["p"], l1["partials"],
                                l2["partials"], parts_z, *mixture_params(l1, K), *mixture_params(l2, K), M1=M1, K=K, training=training)

    def forward(self, x: torch.Tensor, training: bool = True, debug=False, *,
                noise: Optional[Tuple[torch.Tensor, torch.Tensor]] = None):
        check_input(x)
        if training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            # the training call with autograd on: one autograd node over the layer-by-layer forward (training_scalable.py)
            from . import training_scalable as _ts
            return _ts.train_forward(self, x, noise=noise)
        if self.fused_pipeline:
            return self._forward_pairs(x, training, noise)
        # fp32, and bf16x3 outside the fused pipeline's channel counts: the training forward's layer-by-layer form without tapes
        from . import training as T
        with torch.no_grad():
            noise_z, noise_y = draw_noise(self.M, x, noise) if training else (None, None)
            outs, _ = T._forward_impl(self, x.contiguous().float(), noise_z, noise_y, False, qmode=Q_NOISE if training else Q_ROUND,
                                      arm=self.precision, record=False)
        return two_head_outputs(*outs, M1=self.M1, K=self.K, training=training)

    @property
    def fused_pipeline(self) -> bool:
        """True when the eval forward runs _forward_pairs (bf16x3 at M = 128 / 192), else training._forward_impl (record=False)."""
        return self.precision == "bf16x3" and self.M in (128, 192) and self.M1 % 64 == 0 and self.M2 % 64 == 0

    def compress(self, x: torch.Tensor) -> dict:
        """x [B, 3, H, W] (any H, W >= 1) -> {"strings": [y1_strings, y2_strings, z_strings], "shape": (hz, wz)}: one bytes
        object per image in each list, coded with the eval-mode symbols of x padded by edge replication to multiples of 64 (shape
        is the padded one).  The base layer (y1 + z) decodes without the y2 strings.  Format: DESIGN.md sections 10 and 12."""
        from . import scalable_codec
        return scalable_codec.compress(self, x)

    def decompress(self, strings, shape, base_only: bool = False) -> dict:
        """strings / shape as compress returned them (any subset of the images, in any order) -> {"x_hat", "y_hat", "y1_hat", "y2_hat",
        "z_hat"}, NCHW f32; x_hat = g_s(y_hat) cropped to the image's size, not clamped; the latents at the padded shape.  base_only=True
        decodes z and y1 alone (strings[1] may be None) and returns {"y1_hat", "z_hat"}.  Raises ValueError on a malformed string, a
        string of another model configuration, or a checksum mismatch of a decoded layer (corrupted bytes, other weights)."""
        from . import scalable_codec
        return scalable_codec.decompress(self, strings, shape, base_only=base_only)
