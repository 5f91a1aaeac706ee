"""The training step of the reference (Trainer.py:79-86: ``model(imgs)`` -> ``rd_loss`` -> ``loss.backward()`` -> ``Adam.step()``)
on the sm_100a kernels.

The reference has no backward code of its own: its gradients are what torch autograd derives from Models.py:49-106 and
RateDistortionLoss.py:5-49.  Here the whole model is ONE autograd node (``_TrainForward``): its forward (``_forward_impl``) runs
layer by layer with fp32 NHWC tensors in between, every transform (g_a, g_s, h_a, h_s; the 5x5 chains and the 3x3 residual
graphs alike) recording its ops and their tensors on a ``Tape``; its backward (``_backward_impl``) walks each transform's tape in
reverse (``Tape.backward``) around the hand-written entropy side (``head_forward`` / ``head_backward`` per entropy head of
``heads``: one for JointAutoregressiveHierarchical and HierarchicalMixtureResidual, two for ScalableImageCoding, whose loss and
autograd wrapping live in training_scalable.py), a hand-scheduled chain of C-ABI calls (include/nic.h, "training step" section):

    data gradient of a conv      nic_conv_fwd with the mirrored descriptor (Conv2d <-> ConvTranspose2d, same weight tensor)
    weight / bias gradients      nic_conv_wgrad_tc (tcgen05, MN-major operands) / nic_conv_wgrad (fp32) - all 25 taps of the masked
                                 conv: ContextModels.py:19 masks the data, not the graph
    GDN / IGDN                   nic_gdn_bwd, or nic_gdn_reparam / _apply / _bwd_prep / _bwd_finish around tensor-core contractions
                                 (incl. compressai's LowerBound gradient rule on the stored parameters)
    LeakyReLU                    nic_lrelu_bwd
    likelihoods                  nic_gm_likelihood_bwd, nic_factorized_likelihood_bwd
    distortion                   nic_sse_bwd (``_RDLoss`` below is rd_loss's autograd node); nic_ms_ssim_bwd for the MS-SSIM
                                 loss (``_MSSSIMRDLoss``, ms_ssim_rd_loss's node)
    optimizer                    nic_adam_multi_step (``Adam`` below: torch.optim.Adam semantics, Main.ipynb:133; one launch)

``step_gradients`` runs the same forward + loss + backward WITHOUT the autograd engine (calling thread, current stream): the form
``parallel.ShardedTrainer(graph=True)`` captures in a CUDA graph.

Differentiable outputs: ``x_hat``, ``logp_y``, ``logp_z`` (what rd_loss consumes).  The other dict entries are returned
detached.

Arithmetic arms of the step (``NIC_TRAIN_PRECISION`` or ``model.train_precision``):
  "bf16x3" (default when M % 64 == 0): the convolutions of the forward pass, the data-gradient convolutions, the weight gradients
           of every layer the kernel is built for and the GDN channel contractions run on the tcgen05 tensor cores with hi/lo-split
           bf16 operands (fp32 grade, the arm the evaluation path uses); activations and gradients stay fp32 NHWC between layers and
           are split on the fly (nic_to_pair, one conversion per tensor and step).  LeakyReLU, the remaining weight gradients and
           the likelihood chain run in fp32 on the CUDA cores.
  "fp32":  everything on the CUDA cores; gradients within 5e-6 of the reference's autograd (tests/test_gpu_train.py).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import _lib, engine
from ._lib import (ConvDesc, DT_F32, EPI_BIAS, EPI_LRELU, LAYOUT_NCHW, LAYOUT_NHWC, PREC_FP32, Q_NOISE, Q_PASSTHRU, Q_ROUND, check, current_stream, ptr)
from .EntropyModels import gm_likelihood
from .Models import draw_noise, mixture_params, single_head_outputs

PREC = "fp32"
WGRAD_TC = os.environ.get("NIC_WGRAD_TC", "1") != "0"      # tensor-core weight gradients in the bf16x3 arm (0: fp32 kernel everywhere)
# Branch parallelism of the step: weight gradients (off the critical path of the data-gradient chain) on one side stream, g_s and
# its backward (independent of the entropy path between y_in and the merge of the y gradients) on another.  Most kernels of a step
# at 8 x 256 x 256 fill only part of the GPU; in a CUDA-graph capture the forks / joins become parallel branches of the graph
# (4.98 -> 3.86 ms per step).  Launched eagerly the step is host-bound and the extra event traffic only costs (7.7 -> 14.7 ms), so
# "auto" forks only while a capture is under way; NIC_STEP_OVERLAP = 0 / 1 forces it off / on.
_OVERLAP_ENV = os.environ.get("NIC_STEP_OVERLAP", "auto")


def _overlap() -> bool:
    if _OVERLAP_ENV == "auto":
        return torch.cuda.is_current_stream_capturing()
    return _OVERLAP_ENV != "0"
_SIDE_STREAMS: Dict[tuple, "torch.cuda.Stream"] = {}


def _side_stream(dev, which: int = 0) -> "torch.cuda.Stream":
    """which = 0: the weight-gradient stream; 1: the synthesis-transform branch (g_s and its backward are independent of the
    entropy path between y_in and the merge of the y gradients)."""
    idx = (dev.index if dev.index is not None else torch.cuda.current_device(), which)
    if idx not in _SIDE_STREAMS:
        _SIDE_STREAMS[idx] = torch.cuda.Stream(device=dev)
    return _SIDE_STREAMS[idx]


def train_precision(model) -> str:
    arm = getattr(model, "train_precision", None) or os.environ.get("NIC_TRAIN_PRECISION", "auto")
    if arm == "auto":
        arm = "bf16x3" if model.M % 64 == 0 else "fp32"
    if arm not in ("fp32", "bf16x3"):
        raise ValueError(f"train precision must be fp32 or bf16x3, got {arm}")
    return arm


def _f32(shape, dev):
    return torch.empty(shape, dtype=torch.float32, device=dev)


def _ws(nbytes: int, dev):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=dev)      # torch allocations are >= 256-byte aligned


# ---- single backward ops ------------------------------------------------------------------------------------------

def wgrad_on_tensor_cores(conv: nn.Module, n: int, h: int, w: int, in_layout: int, out_layout: int, arm: str) -> bool:
    """Whether conv_wgrad will take the tensor-core kernel for this layer (then it consumes the pair forms of x and g)."""
    if arm != "bf16x3" or not WGRAD_TC:
        return False
    d = engine.ConvOp(conv).desc(n, h, w, PREC, in_layout, out_layout, DT_F32, DT_F32)
    d.mask_a = 0
    return _lib.load().nic_conv_wgrad_tc_workspace_bytes(C.byref(d)) > 0


def conv_wgrad(conv: nn.Module, x: torch.Tensor, g: torch.Tensor, n: int, h: int, w: int, in_layout: int, out_layout: int,
               arm: str = "fp32", pairs=None):
    """(dW in the reference layout, db) of one layer; x = forward input, g = gradient w.r.t. the conv output.
    bf16x3 arm: the tensor-core kernel (nic_conv_wgrad_tc) for the layer shapes it is built for, else the fp32 kernel."""
    lib = _lib.load()
    op = engine.ConvOp(conv)
    d = op.desc(n, h, w, PREC, in_layout, out_layout, DT_F32, DT_F32)
    d.mask_a = 0
    dw = torch.empty_like(conv.weight, dtype=torch.float32)
    db = torch.empty_like(conv.bias, dtype=torch.float32)
    if arm == "bf16x3" and WGRAD_TC:
        nbytes = lib.nic_conv_wgrad_tc_workspace_bytes(C.byref(d))
        if nbytes:
            ws = _ws(nbytes, x.device)
            xp, gp = pairs if pairs is not None else (to_pair(x), to_pair(g))   # named: a temporary would be freed before the launch
            check(lib.nic_conv_wgrad_tc(C.byref(d), ptr(xp), ptr(gp), ptr(g), ptr(dw), ptr(db), ptr(ws), ws.numel(),
                                        current_stream()), "nic_conv_wgrad_tc")
            return dw, db
    nbytes = lib.nic_conv_wgrad_workspace_bytes(C.byref(d))
    ws = _ws(nbytes, x.device)
    check(lib.nic_conv_wgrad(C.byref(d), ptr(x), ptr(g), ptr(dw), ptr(db), ptr(ws), ws.numel(), current_stream()), "nic_conv_wgrad")
    return dw, db


_PAIRS: Dict[tuple, tuple] = {}        # (data_ptr, version, square) -> (source tensor, its pair form): one conversion per tensor and step


def to_pair(x: torch.Tensor, square: bool = False) -> torch.Tensor:
    """f32 [..., c] -> bf16 [..., 2c] = [hi | lo] (NIC_DT_BF16X2) of x (or of x^2) through nic_to_pair.
    A layer input is consumed in pair form by its forward conv AND by its weight gradient, a gradient by the data-gradient conv
    AND the weight gradient: the conversions are memoised until the step ends (`forget_pairs`); the source tensor is kept alive
    by the entry, so its address cannot be recycled under the key."""
    key = (x.data_ptr(), x._version, tuple(x.shape), bool(square))
    hit = _PAIRS.get(key)
    if hit is not None:
        return hit[1]
    c = x.shape[-1]
    out = torch.empty(tuple(x.shape[:-1]) + (2 * c,), dtype=torch.bfloat16, device=x.device)
    check(_lib.load().nic_to_pair(ptr(x), ptr(out), x.numel() // c, c, int(square), current_stream()), "nic_to_pair")
    _PAIRS[key] = (x, out)
    return out


def forget_pairs():
    _PAIRS.clear()


def _train_op(conv: nn.Module, epilogue: int, mask_a: bool = False) -> engine.ConvOp:
    """ConvOp of a layer WITHOUT its GDN (the training step keeps the pre-GDN tensor), cached on the module."""
    cache = conv.__dict__.setdefault("_nic_train_ops", {})
    key = (epilogue, mask_a)
    if key not in cache:
        cache[key] = engine.ConvOp(conv, epilogue, mask_a=mask_a)
    return cache[key]


def _is_first_layer_shape(conv: nn.Module) -> bool:
    return (isinstance(conv, nn.Conv2d) and not isinstance(conv, nn.ConvTranspose2d) and conv.in_channels == 3 and conv.out_channels in (128, 192)
            and conv.kernel_size == (5, 5) and conv.stride == (2, 2) and conv.padding == (2, 2))


def conv_forward(arm: str, conv: nn.Module, epilogue: int, x: torch.Tensor, n: int, h: int, w: int, in_layout: int = LAYOUT_NHWC,
                 out_layout: int = LAYOUT_NHWC, out: Optional[torch.Tensor] = None, out_c_total: int = 0, out_c_offset: int = 0,
                 mask_a: bool = False, pair_out: bool = False) -> torch.Tensor:
    """One conv (+ bias / LeakyReLU) with f32 tensors at both ends; the contraction on the tensor cores in the bf16x3 arm.
    pair_out (evaluation chains of the residual family): where the tensor-core kernel runs, leave the result as the bf16 hi/lo
    pair the next conv consumes (no f32 round trip, no nic_to_pair launch); x may itself be such a pair."""
    op = _train_op(conv, epilogue, mask_a)
    if arm == "bf16x3" and _is_first_layer_shape(conv) and in_layout == LAYOUT_NCHW and out_layout == LAYOUT_NHWC and out is None \
            and epilogue == EPI_BIAS and w % 4 == 0:
        return op.run(x, n, h, w, "bf16x3", in_layout=LAYOUT_NCHW, out_dtype=torch.float32)       # the dedicated 3 -> 128 kernel
    if arm == "bf16x3" and in_layout == LAYOUT_NHWC and conv.in_channels % 64 == 0 and conv.out_channels <= 1792:
        as_pair = pair_out and out is None and out_layout == LAYOUT_NHWC and conv.out_channels % 64 == 0
        return op.run(x if x.dtype == torch.bfloat16 else to_pair(x), n, h, w, "bf16x3", out_layout=out_layout, out=out,
                      out_c_total=out_c_total, out_c_offset=out_c_offset, out_dtype=None if as_pair else torch.float32)
    if x.dtype == torch.bfloat16:
        raise ValueError("conv_forward: a bf16 pair input needs the tensor-core path of the bf16x3 arm")
    return op.run(x, n, h, w, PREC, in_layout=in_layout, out_layout=out_layout, out=out, out_c_total=out_c_total,
                  out_c_offset=out_c_offset)


def _gdn_tc(gdn: nn.Module):
    """The two channel-mixing contractions of a GDN layer as 1x1 convs of the tensor-core engine: norm = beta + gamma . u^2
    (weight gamma_eff [i, j], bias beta_eff) and r = gamma^T . t (weight gamma_eff^T).  The effective parameters live in
    persistent buffers refreshed by nic_gdn_reparam whenever beta / gamma changed."""
    st = gdn.__dict__.get("_nic_tc")
    c, dev = gdn.in_channels, gdn.gamma.device
    if st is None or st["dev"] != dev:
        beta_eff, gamma_eff, gamma_t = _f32(c, dev), _f32((c, c, 1, 1), dev), _f32((c, c, 1, 1), dev)
        with torch.device(dev):
            norm_conv, rt_conv = nn.Conv2d(c, c, 1), nn.Conv2d(c, c, 1)
        for m in (norm_conv, rt_conv):
            m.requires_grad_(False)
        norm_conv.weight, norm_conv.bias = nn.Parameter(gamma_eff, requires_grad=False), nn.Parameter(beta_eff, requires_grad=False)
        rt_conv.weight = nn.Parameter(gamma_t, requires_grad=False)
        rt_conv.bias.data.zero_()
        st = {"dev": dev, "beta_eff": beta_eff, "gamma_eff": gamma_eff, "gamma_t": gamma_t, "key": None,
              "norm_op": engine.ConvOp(norm_conv, EPI_BIAS), "rt_op": engine.ConvOp(rt_conv, EPI_BIAS)}
        gdn.__dict__["_nic_tc"] = st
    key = (gdn.beta.data_ptr(), gdn.beta._version, gdn.gamma.data_ptr(), gdn.gamma._version)
    if st["key"] != key:
        check(_lib.load().nic_gdn_reparam(c, float(gdn.beta_min), ptr(gdn.beta.detach().float().contiguous()),
                                          ptr(gdn.gamma.detach().float().contiguous()), ptr(st["beta_eff"]), ptr(st["gamma_eff"]),
                                          ptr(st["gamma_t"]), current_stream()), "nic_gdn_reparam")
        st["norm_op"]._cache.clear(); st["rt_op"]._cache.clear()       # the buffers changed behind torch's back
        st["key"] = key
    return st


def gdn_forward(arm: str, gdn: nn.Module, u: torch.Tensor, n: int, h: int, w: int, addend: Optional[torch.Tensor] = None):
    """GDN / IGDN of an NHWC f32 tensor -> (out, norm | None).  bf16x3 arm: the norm is a tensor-core 1x1 conv over the split
    squares and is kept for the backward; fp32 arm: nic_gdn_fwd (the backward recomputes the norm).
    addend (evaluation chains of the residual family): out = gdn(u) + addend - in the bf16x3 arm in the same pass (nic_gdn_apply_add)."""
    lib = _lib.load()
    c = gdn.in_channels
    if arm == "bf16x3" and c % 64 == 0:
        st = _gdn_tc(gdn)
        norm = st["norm_op"].run(to_pair(u, square=True), n, h, w, "bf16x3", out_dtype=torch.float32)
        out = torch.empty_like(u)
        if addend is not None:
            check(lib.nic_gdn_apply_add(ptr(u), ptr(norm), ptr(addend), u.numel(), int(gdn.inverse), ptr(out), current_stream()),
                  "nic_gdn_apply_add")
        else:
            check(lib.nic_gdn_apply(ptr(u), ptr(norm), u.numel(), int(gdn.inverse), ptr(out), current_stream()), "nic_gdn_apply")
        return out, norm
    gamma = _f32(c * c, u.device)
    beta = _f32(c, u.device)
    check(lib.nic_pack_gdn(c, float(gdn.beta_min), ptr(gdn.beta.detach().float().contiguous()), ptr(gdn.gamma.detach().float().contiguous()),
                           ptr(beta), ptr(gamma), PREC_FP32, current_stream()), "nic_pack_gdn")
    y = torch.empty_like(u)
    check(lib.nic_gdn_fwd(ptr(u), n, c, h, w, LAYOUT_NHWC, int(gdn.inverse), ptr(gamma), ptr(beta), ptr(y), current_stream()), "nic_gdn_fwd")
    if addend is not None:
        add_(y, addend)
    return y, None


def _adjoint(conv: nn.Module, weight: Optional[torch.Tensor], c_in: int, h_in: int, w_in: int):
    """(module, ConvOp) of the adjoint conv of `conv` as a regular layer of the engine, cached on the module:
       Conv2d stride 2      -> ConvTranspose2d over the SAME weight tensor (output_padding restores the input size)
       ConvTranspose2d      -> Conv2d over the same weight tensor
       Conv2d stride 1      -> Conv2d with the flipped, channel-transposed kernel (re-derived every call: the weights move)."""
    transposed = isinstance(conv, nn.ConvTranspose2d)
    k, s, p = conv.kernel_size[0], conv.stride[0], conv.padding[0]
    cache = conv.__dict__.setdefault("_nic_adjoint", {})
    key = (c_in, None if weight is None else weight.shape, h_in % s, w_in % s)
    wsrc = (conv.weight if weight is None else weight).detach()
    if key not in cache:
        dev = wsrc.device
        with torch.device(dev):
            if transposed:
                adj = nn.Conv2d(conv.out_channels, c_in, k, stride=s, padding=p)
            elif s == 1:
                adj = nn.Conv2d(conv.out_channels, c_in, k, stride=1, padding=k - 1 - p)
            else:
                h_out, w_out = engine.conv_out_hw(conv, h_in, w_in)
                oph, opw = h_in - ((h_out - 1) * s - 2 * p + k), w_in - ((w_out - 1) * s - 2 * p + k)
                if oph != opw:
                    raise ValueError("conv_dgrad: height and width need the same output padding")
                adj = nn.ConvTranspose2d(conv.out_channels, c_in, k, stride=s, padding=p, output_padding=oph)
        adj.requires_grad_(False)
        adj.bias.data.zero_()
        cache[key] = (adj, engine.ConvOp(adj, EPI_BIAS))
    adj, op = cache[key]
    if not transposed and s == 1:
        adj.weight = nn.Parameter(wsrc.flip(2, 3).transpose(0, 1).contiguous(), requires_grad=False)
        op._cache.clear()          # a fresh tensor every call: its (address, version) key could repeat with different contents
    elif adj.weight.data_ptr() != wsrc.data_ptr():
        adj.weight = nn.Parameter(wsrc, requires_grad=False)              # shares storage and version counter with the layer's weight
    return adj, op


def conv_dgrad(conv: nn.Module, g: torch.Tensor, n: int, h_in: int, w_in: int, g_layout: int = LAYOUT_NHWC,
               weight: Optional[torch.Tensor] = None, c_in: Optional[int] = None, arm: str = "fp32") -> torch.Tensor:
    """Gradient w.r.t. the layer input (NHWC f32): the adjoint conv through nic_conv_fwd.
    (h_in, w_in) = forward input size.  `weight` / `c_in` select a slice of the layer's input channels
    (weight = the matching slice of conv.weight, contiguous)."""
    if (not isinstance(conv, nn.ConvTranspose2d)) and conv.kernel_size == (1, 1) and conv.stride[0] > 1 and weight is None \
            and g_layout == LAYOUT_NHWC:
        # 1x1 strided conv (the skip of ResidualBlockWithStride, Layers.py:47): the input gradient is W^T g at the sampled positions
        # and zero elsewhere - the contraction as a 1x1 stride-1 conv of the engine, the scatter as a strided view copy
        st = conv.stride[0]
        cache = conv.__dict__.setdefault("_nic_adjoint", {})
        if "pointwise" not in cache:
            with torch.device(conv.weight.device):
                adj1 = nn.Conv2d(conv.out_channels, conv.in_channels, 1)
            adj1.requires_grad_(False)
            adj1.bias.data.zero_()
            cache["pointwise"] = adj1
        adj1 = cache["pointwise"]
        adj1.weight = nn.Parameter(conv.weight.detach().transpose(0, 1).contiguous(), requires_grad=False)
        adj1.__dict__.pop("_nic_train_ops", None)      # a fresh weight tensor every call
        h_out, w_out = engine.conv_out_hw(conv, h_in, w_in)
        t = conv_forward(arm, adj1, EPI_BIAS, g, n, h_out, w_out)
        dx = torch.zeros((n, h_in, w_in, conv.in_channels), dtype=torch.float32, device=g.device)
        dx[:, ::st, ::st, :] = t
        return dx
    if arm == "bf16x3" and g_layout == LAYOUT_NCHW and weight is None and isinstance(conv, nn.ConvTranspose2d) and g.shape[-1] % 4 == 0:
        adj, op = _adjoint(conv, None, conv.in_channels, h_in, w_in)          # ConvTranspose2d(128, 3) backward = the 3 -> 128 conv
        if _is_first_layer_shape(adj):
            h_out, w_out = engine.conv_out_hw(conv, h_in, w_in)
            return op.run(g, n, h_out, w_out, "bf16x3", in_layout=LAYOUT_NCHW, out_dtype=torch.float32)
    if arm == "bf16x3" and g_layout == LAYOUT_NHWC and conv.out_channels % 64 == 0:
        cin = conv.in_channels if c_in is None else c_in
        h_out, w_out = engine.conv_out_hw(conv, h_in, w_in)
        adj, op = _adjoint(conv, weight, cin, h_in, w_in)
        return op.run(to_pair(g), n, h_out, w_out, "bf16x3", out_dtype=torch.float32)
    lib = _lib.load()
    transposed = isinstance(conv, nn.ConvTranspose2d)
    k, s, p = conv.kernel_size[0], conv.stride[0], conv.padding[0]
    h_out, w_out = engine.conv_out_hw(conv, h_in, w_in)
    wt = (conv.weight if weight is None else weight).detach().float().contiguous()
    cin = conv.in_channels if c_in is None else c_in
    d = ConvDesc()
    d.n, d.c_in, d.h_in, d.w_in = n, conv.out_channels, h_out, w_out
    d.c_out, d.h_out, d.w_out = cin, h_in, w_in
    d.kh, d.kw, d.stride, d.pad = k, k, s, p
    d.transposed = 0 if transposed else 1
    d.output_padding = 0 if transposed else h_in - ((h_out - 1) * s - 2 * p + k)
    if not transposed and d.output_padding != w_in - ((w_out - 1) * s - 2 * p + k):
        raise ValueError("conv_dgrad: height and width need the same output padding")
    d.mask_a, d.epilogue, d.precision = 0, EPI_BIAS, PREC_FP32
    d.in_layout, d.out_layout, d.in_dtype, d.out_dtype = g_layout, LAYOUT_NHWC, DT_F32, DT_F32
    dev = g.device
    wp = _f32(lib.nic_packed_weight_elems(C.byref(d)), dev)
    check(lib.nic_pack_conv_weight(C.byref(d), ptr(wt), ptr(wp), current_stream()), "nic_pack_conv_weight")
    zero = torch.zeros(cin, dtype=torch.float32, device=dev)
    out = _f32((n, h_in, w_in, cin), dev)
    check(lib.nic_conv_fwd(C.byref(d), ptr(g), ptr(wp), ptr(zero), None, None, ptr(out), None, 0, current_stream()), "nic_conv_fwd")
    return out


def lrelu_bwd_(g: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    check(_lib.load().nic_lrelu_bwd(ptr(g), ptr(out), ptr(g), g.numel(), current_stream()), "nic_lrelu_bwd")
    return g


def gdn_bwd(gdn: nn.Module, u: torch.Tensor, g: torch.Tensor, n: int, h: int, w: int, norm: Optional[torch.Tensor] = None,
            side=None, keep: Optional[list] = None):
    """(du, dbeta, dgamma): u = the conv output before the GDN (NHWC f32), g = gradient w.r.t. the GDN output.
    With the forward's `norm` (bf16x3 arm) the gamma^T . t contraction runs on the tensor cores."""
    lib = _lib.load()
    c = gdn.in_channels
    du = torch.empty_like(u)
    dbeta = torch.empty_like(gdn.beta, dtype=torch.float32)
    dgamma = torch.empty_like(gdn.gamma, dtype=torch.float32)
    if norm is not None:
        st = _gdn_tc(gdn)
        t = torch.empty_like(u)
        check(lib.nic_gdn_bwd_prep(ptr(u), ptr(g), ptr(norm), u.numel(), int(gdn.inverse), ptr(t), ptr(du), current_stream()), "nic_gdn_bwd_prep")
        tp = to_pair(t)
        r = st["rt_op"].run(tp, n, h, w, "bf16x3", out_dtype=torch.float32)
        pixels = n * h * w
        # d gamma_eff[i][j] = sum_pix t_i u_j^2 is the weight gradient of the norm conv (1x1, input u^2, output gradient t)
        dge = dbe = None
        d = st["norm_op"].desc(n, h, w, PREC, LAYOUT_NHWC, LAYOUT_NHWC, DT_F32, DT_F32)
        nb = lib.nic_conv_wgrad_tc_workspace_bytes(C.byref(d)) if WGRAD_TC else 0
        if nb and side is not None:
            # data path on this stream: du += 2 u r.  Parameter path (gamma / beta gradients + LowerBound chain) on the side stream.
            u2p = to_pair(u, square=True)
            check(lib.nic_gdn_bwd_du(ptr(u), ptr(r), ptr(du), u.numel(), current_stream()), "nic_gdn_bwd_du")
            main = torch.cuda.current_stream(u.device)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                dge, dbe = _f32((c, c), u.device), _f32(c, u.device)
                wws = _ws(nb, u.device)
                check(lib.nic_conv_wgrad_tc(C.byref(d), ptr(u2p), ptr(tp), ptr(t), ptr(dge), ptr(dbe), ptr(wws), wws.numel(), current_stream()),
                      "nic_conv_wgrad_tc")
                check(lib.nic_gdn_reparam_bwd(c, float(gdn.beta_min), ptr(gdn.beta.detach().float().contiguous()),
                                              ptr(gdn.gamma.detach().float().contiguous()), ptr(dbe), ptr(dge), ptr(dbeta), ptr(dgamma),
                                              current_stream()), "nic_gdn_reparam_bwd")
            if keep is not None:
                keep.extend((u, t, tp, u2p, dge, dbe))
            return du, dbeta, dgamma
        if nb:
            dge, dbe = _f32((c, c), u.device), _f32(c, u.device)
            wws = _ws(nb, u.device)
            u2p = to_pair(u, square=True)
            check(lib.nic_conv_wgrad_tc(C.byref(d), ptr(u2p), ptr(tp), ptr(t), ptr(dge), ptr(dbe), ptr(wws), wws.numel(), current_stream()),
                  "nic_conv_wgrad_tc")
        ws = _ws(lib.nic_gdn_bwd_finish_workspace_bytes(pixels, c), u.device)
        check(lib.nic_gdn_bwd_finish(ptr(u), ptr(t), ptr(r), pixels, c, float(gdn.beta_min), ptr(gdn.beta.detach().float().contiguous()),
                                     ptr(gdn.gamma.detach().float().contiguous()), ptr(dge), ptr(dbe), ptr(du), ptr(dbeta), ptr(dgamma),
                                     ptr(ws), ws.numel(), current_stream()), "nic_gdn_bwd_finish")
        return du, dbeta, dgamma
    ws = _ws(lib.nic_gdn_bwd_workspace_bytes(n, c, h, w), u.device)
    check(lib.nic_gdn_bwd(ptr(u), ptr(g), n, c, h, w, int(gdn.inverse), float(gdn.beta_min), ptr(gdn.beta.detach().float().contiguous()),
                          ptr(gdn.gamma.detach().float().contiguous()), ptr(du), ptr(dbeta), ptr(dgamma), ptr(ws), ws.numel(),
                          current_stream()), "nic_gdn_bwd")
    return du, dbeta, dgamma


def to_nhwc(t_nchw: torch.Tensor, accumulate_into: Optional[torch.Tensor] = None) -> torch.Tensor:
    n, c = t_nchw.shape[:2]
    hw = t_nchw[0, 0].numel()
    out = accumulate_into if accumulate_into is not None else _f32((n,) + tuple(t_nchw.shape[2:]) + (c,), t_nchw.device)
    check(_lib.load().nic_layout_convert(ptr(t_nchw), ptr(out), n, c, hw, 1, int(accumulate_into is not None), current_stream()),
          "nic_layout_convert")
    return out


def add_(dst: torch.Tensor, src: torch.Tensor) -> torch.Tensor:
    check(_lib.load().nic_add_inplace(ptr(dst), ptr(src), dst.numel(), current_stream()), "nic_add_inplace")
    return dst


class Tape:
    """Record of one transform's training forward (the 5x5 chains and the 3x3 residual graphs alike, `run_nhwc(..., tape=)`):
    every conv (+ bias / LeakyReLU), GDN / IGDN and residual sum is appended with its input and output tensors; `backward` walks
    the record in reverse, keeps one gradient per tensor (summed where a tensor feeds two consumers: the block input of a residual
    block) and returns the gradient of the transform's input.  Kernels: conv_wgrad, conv_dgrad, gdn_bwd, nic_lrelu_bwd,
    nic_add_inplace."""

    def __init__(self, arm: str, n: int):
        self.arm, self.n, self.recs = arm, n, []

    def conv(self, conv, epilogue, x, h, w, in_layout=LAYOUT_NHWC, out_layout=LAYOUT_NHWC, **out_kw):
        y = conv_forward(self.arm, conv, epilogue, x, self.n, h, w, in_layout=in_layout, out_layout=out_layout, **out_kw)
        self.recs.append(("conv", conv, epilogue, x, h, w, in_layout, out_layout, y))
        return y

    def gdn(self, gdn, u, h, w):
        y, nrm = gdn_forward(self.arm, gdn, u, self.n, h, w)
        self.recs.append(("gdn", gdn, u, nrm, h, w, y))
        return y

    def add(self, a, b):
        y = add_(a.clone(), b)                      # out of place: `a` may be a LeakyReLU output whose signs the backward needs
        self.recs.append(("add", a, b, y))
        return y

    @property
    def output(self):
        return self.recs[-1][-1]

    def backward(self, g_out, g_layout, put, wgrad, root=None, side=None, keep=None):
        """g_out: gradient of `output` (in g_layout).  root: the transform's input tensor; its gradient is returned (None when
        root is None: the image needs none).  put(param, grad) collects parameter gradients, wgrad = conv_wgrad or its
        side-stream form; keep holds what the side stream reads until the caller's join."""
        n, arm = self.n, self.arm
        grads = {id(self.output): (g_out, g_layout)}
        internal = {id(r[-1]) for r in self.recs}

        def give(t, g):
            """Add g to the gradient of tensor t (a tensor made inside the transform, or its input when that is wanted)."""
            if id(t) not in internal and (root is None or t is not root):
                return
            if id(t) in grads:
                grads[id(t)] = (add_(grads[id(t)][0], g), LAYOUT_NHWC)
            else:
                grads[id(t)] = (g, LAYOUT_NHWC)

        for rec in reversed(self.recs):
            if id(rec[-1]) not in grads:
                continue
            g, gl = grads.pop(id(rec[-1]))                  # popped: freed as soon as this op's backward has consumed it
            if rec[0] == "conv":
                _, conv, epi, x, h, w, in_layout, out_layout, y = rec
                if epi == EPI_LRELU:
                    g = lrelu_bwd_(g, y)
                dw, db = wgrad(conv, x, g, n, h, w, in_layout, gl, arm=arm)
                put(conv.weight, dw); put(conv.bias, db)
                if keep is not None and side is not None:
                    keep.append(g)
                if id(x) in internal or (root is not None and x is root):
                    give(x, conv_dgrad(conv, g, n, h, w, gl, arm=arm))
            elif rec[0] == "gdn":
                _, gdn, u, nrm, h, w, y = rec
                g, dbeta, dgamma = gdn_bwd(gdn, u, g, n, h, w, norm=nrm, side=side, keep=keep)
                put(gdn.beta, dbeta); put(gdn.gamma, dgamma)
                give(u, g)
            else:
                _, a, b, y = rec
                give(a, g)
                give(b, g.clone())                                  # the two consumers may modify their gradient in place
        return grads.pop(id(root), (None, None))[0] if root is not None else None


_FACT_SLICES = (("matrices", 0, 0, 3), ("biases", 0, 3, 6), ("factors", 0, 6, 9), ("matrices", 1, 9, 18), ("biases", 1, 18, 21),
                ("factors", 1, 21, 24), ("matrices", 2, 24, 33), ("biases", 2, 33, 36), ("factors", 2, 36, 39),
                ("matrices", 3, 39, 42), ("biases", 3, 42, 43))


# ---- the entropy side: one or more (context model, entropy parameters) heads over channel ranges of y, and the factorized prior

def heads(model) -> list:
    """[(context model, entropy parameters, c0, c1)]: the entropy heads of a model, each over the channels [c0, c1) of y and the
    shared hyper features psi.  One head over all of y (JointAutoregressiveHierarchical, HierarchicalMixtureResidual); the base
    [0, M1) and the enhancement [M1, M) head of ScalableImageCoding."""
    if hasattr(model, "M1"):
        return [(model.context_model_1, model.entropy_parameters_1, 0, model.M1),
                (model.context_model_2, model.entropy_parameters_2, model.M1, model.M)]
    return [(model.context_model, model.entropy_parameters, 0, model.M)]


def gm_likelihood_bwd(y: torch.Tensor, raw: torch.Tensor, g_logp: torch.Tensor, m: int, K: int):
    """(d y, d raw), NCHW f32, of logp = log p(y | raw) (nic_gm_likelihood_bwd) for the upstream gradient g_logp."""
    b, _, h, w = y.shape
    dy, draw = torch.empty_like(y), torch.empty_like(raw)
    check(_lib.load().nic_gm_likelihood_bwd(ptr(y), ptr(raw), ptr(g_logp), 0.0, b, m, h * w, K, ptr(dy), ptr(draw), current_stream()),
          "nic_gm_likelihood_bwd")
    return dy, draw


def head_forward(arm: str, head, K: int, y_i: torch.Tensor, y_i_nhwc: torch.Tensor, comb: torch.Tensor, lean: bool):
    """One entropy head on its symbols y_i (NCHW) / y_i_nhwc: the context conv writes phi into channels [0, 2 m) of the concat
    buffer `comb` (NHWC, psi already at [2 m, 2 m + 2 M)), then the 1x1 stack and the likelihood.  -> (likelihood dict, the
    tensors head_backward reads)."""
    ctx, ep, c0, c1 = head
    B, hy, wy, _ = y_i_nhwc.shape
    ctx.masked.apply_mask_()
    conv_forward(arm, ctx.masked, EPI_BIAS, y_i_nhwc, B, hy, wy, out=comb, out_c_total=comb.shape[-1], out_c_offset=0, mask_a=True)
    ops = ep.ops
    e1 = conv_forward(arm, ops[0].conv, ops[0].epilogue, comb, B, hy, wy)
    e2 = conv_forward(arm, ops[1].conv, ops[1].epilogue, e1, B, hy, wy)
    raw = conv_forward(arm, ops[2].conv, ops[2].epilogue, e2, B, hy, wy, out_layout=LAYOUT_NCHW)
    ly = gm_likelihood(y_i, raw, c1 - c0, K, Q_PASSTHRU, full=not lean, want_y_in=False)
    return ly, dict(comb=comb, e1=e1, e2=e2, raw=raw, y_i=y_i, y_i_nhwc=y_i_nhwc)


def head_backward(arm: str, head, K: int, st: dict, g_logp: torch.Tensor, put, wgrad):
    """Backward of head_forward from the gradient of the head's logp: -> (gradient of y_i, NHWC; gradient of psi, NHWC).
    Parameter gradients go to put(param, grad); wgrad = conv_wgrad or its side-stream form (as in Tape.backward)."""
    ctx, ep, c0, c1 = head
    m = c1 - c0
    B, hy, wy, _ = st["y_i_nhwc"].shape
    dy_lik, draw = gm_likelihood_bwd(st["y_i"], st["raw"], g_logp.contiguous().float(), m, K)
    d_y = to_nhwc(dy_lik)
    g = to_nhwc(draw)
    ops = ep.ops
    for i, (op, a) in reversed(list(enumerate(zip(ops, (st["comb"], st["e1"], st["e2"]))))):
        dw, db = wgrad(op.conv, a, g, B, hy, wy, LAYOUT_NHWC, LAYOUT_NHWC, arm=arm)
        put(op.conv.weight, dw); put(op.conv.bias, db)
        if i > 0:
            g = lrelu_bwd_(conv_dgrad(op.conv, g, B, hy, wy, arm=arm), a)
    # the first 1x1 conv reads [phi | psi]: its data gradient splits along its input channels
    w0 = ops[0].conv.weight.detach()
    d_phi = conv_dgrad(ops[0].conv, g, B, hy, wy, weight=w0[:, :2 * m].contiguous(), c_in=2 * m, arm=arm)
    d_psi = conv_dgrad(ops[0].conv, g, B, hy, wy, weight=w0[:, 2 * m:].contiguous(), c_in=w0.shape[1] - 2 * m, arm=arm)
    dw, db = wgrad(ctx.masked, st["y_i_nhwc"], d_phi, B, hy, wy, LAYOUT_NHWC, LAYOUT_NHWC, arm=arm)
    put(ctx.masked.weight, dw); put(ctx.masked.bias, db)
    return add_(d_y, conv_dgrad(ctx.masked, d_phi, B, hy, wy, arm=arm)), d_psi


def factorized_bwd(fe: nn.Module, z_in: torch.Tensor, fparams: torch.Tensor, g_logp: torch.Tensor, put) -> torch.Tensor:
    """Gradient (NCHW) of z_in from the gradient of the factorized prior's logp; the parameter gradients go to put."""
    b, m, h, w = z_in.shape
    dz = torch.empty_like(z_in)
    dpar = _f32((m, 43), z_in.device)
    check(_lib.load().nic_factorized_likelihood_bwd(ptr(z_in), ptr(fparams), ptr(g_logp.contiguous().float()), 0.0, b, m, h * w,
                                                    ptr(dz), ptr(dpar), current_stream()), "nic_factorized_likelihood_bwd")
    for name, idx, lo, hi in _FACT_SLICES:
        prm = getattr(fe, name)[idx]
        put(prm, dpar[:, lo:hi].reshape(prm.shape).contiguous())
    return dz


# ---- the model as one autograd node ------------------------------------------------------------------------------

def _forward_impl(model, x, noise_z, noise_y, lean, qmode: int = Q_NOISE, arm: Optional[str] = None, record: bool = True):
    """The layer-by-layer forward (fp32 NHWC tensors between layers) of a model with any number of entropy heads (`heads`)
    -> (outputs, saved state S).  Outputs in the order single_head_outputs / two_head_outputs take them: x_hat, the heads' logp,
    logp_z, y, y_in, z, z_in, p_z, the heads' p, the heads' partial sums, the partial sums of z, the heads' mixture_params.
    qmode = Q_NOISE is the training forward; Q_ROUND the evaluation forward.
    record=True (training, and JointAutoregressiveHierarchical's evaluation outside the fused pipeline's channel counts): every
    transform records on a Tape and S keeps what _backward_impl reads; under a CUDA-graph capture g_s runs as a parallel branch.
    record=False (evaluation of the residual family and of ScalableImageCoding outside its fused pipeline): no tapes, so the
    transforms hand bf16 pairs between convs and drop their pair forms per layer; everything on the current stream (a per-layer
    forget_pairs on one stream would free pair tensors another stream still reads); S is None."""
    engine.require_cuda(x, "x")
    dev = x.device
    B, _, H, W = x.shape
    M, K = model.M, model.K
    hy, wy, hz, wz = H // 16, W // 16, H // 64, W // 64
    arm = arm or train_precision(model)
    hds = heads(model)
    S = {t: Tape(arm, B) if record else None for t in ("g_a", "g_s", "h_a", "h_s")}    # each transform's ops and tensors
    with torch.cuda.device(dev):
        y_nhwc, _, _ = model.encoder.run_nhwc(x, B, H, W, arm, in_layout=LAYOUT_NCHW, tape=S["g_a"])
        y, y_in, y_in_nhwc, _ = engine.latent_handoff(y_nhwc, qmode, noise_y, torch.float32)

        def synthesis():
            return model.decoder.run_nhwc(y_in_nhwc, B, hy, wy, arm, tape=S["g_s"], final_kw=dict(out_layout=LAYOUT_NCHW))[0]
        # g_s reads only y_in: it runs as its own branch (a second stream; a parallel branch of a captured graph) beside the
        # entropy path h_a -> h_s -> context -> entropy parameters -> likelihoods
        main = torch.cuda.current_stream(dev)
        branch = _side_stream(dev, 1) if (record and _overlap()) else None
        if branch is not None:
            if arm == "bf16x3":
                to_pair(y_in_nhwc)               # both branches consume the pair form: make it before the fork
            branch.wait_stream(main)
            with torch.cuda.stream(branch):
                x_hat = synthesis()
        # h_a (reads the unquantised y)
        z_nhwc, _, _ = model.hyper_encoder.run_nhwc(y_nhwc, B, hy, wy, arm, tape=S["h_a"])
        z, z_in, z_in_nhwc, _ = engine.latent_handoff(z_nhwc, qmode, noise_z, torch.float32)
        # h_s writes psi into head 0's concat buffer [phi_0 (2 m_0) | psi (2 M)]; every other head's buffer gets a copy of it
        combs = [_f32((B, hy, wy, 2 * (c1 - c0) + 2 * M), dev) for _, _, c0, c1 in hds]
        m0 = hds[0][3] - hds[0][2]
        model.hyper_decoder.run_nhwc(z_in_nhwc, B, hz, wz, arm, tape=S["h_s"],
                                     final_kw=dict(out=combs[0], out_c_total=combs[0].shape[-1], out_c_offset=2 * m0))
        for (_, _, c0, c1), comb in zip(hds[1:], combs[1:]):
            comb[..., 2 * (c1 - c0):] = combs[0][..., 2 * m0:]
        lys, states = [], []
        for head, comb in zip(hds, combs):
            c0, c1 = head[2], head[3]
            ly, st = head_forward(arm, head, K, y_in[:, c0:c1].contiguous(), y_in_nhwc[..., c0:c1].contiguous(), comb, lean)
            lys.append(ly)
            states.append(st)
        _, p_z, logp_z, parts_z = model.factorized_entropy_model.likelihood(z_in, Q_PASSTHRU)
        if branch is not None:
            main.wait_stream(branch)
        else:
            x_hat = synthesis()
    outs = (x_hat, *[ly["logp"] for ly in lys], logp_z, y, y_in, z, z_in, p_z, *[ly["p"] for ly in lys],
            *[ly["partials"] for ly in lys], parts_z, *[t for ly in lys for t in mixture_params(ly, K, lean)])
    if not record:
        return outs, None
    S.update(arm=arm, heads=states, y_in_nhwc=y_in_nhwc, z_in=z_in, z_in_nhwc=z_in_nhwc, y_nhwc=y_nhwc,
             fparams=model.factorized_entropy_model.packed(), shape=(B, H, W))
    return outs, S


def _backward_impl(model, S, g_xhat, g_logp_heads, g_logp_z, partial_hook=None) -> Dict[int, torch.Tensor]:
    """The hand-scheduled backward: {id(parameter): gradient} from the gradients of x_hat / of every head's logp (a list in
    `heads` order) / of logp_z (x_hat's and logp_z's may be None; the entropy heads are skipped unless every head has one).
    partial_hook(grads, streams): called once, when every gradient except g_a's has been ENQUEUED (g_s, the entropy path and h_a
    are done, on `streams`) and only g_a's backward remains - the data-parallel trainer starts the all-reduce of those ~24 of the
    29 MB there, so that it overlaps g_a's backward; the hook may replace entries of `grads` (views of its reduced bucket)."""
    dev = S["y_in_nhwc"].device
    arm = S["arm"]
    grads: Dict[int, torch.Tensor] = {}

    def put(param, g):
        grads[id(param)] = g if id(param) not in grads else grads[id(param)] + g

    main = torch.cuda.current_stream(dev)
    side = _side_stream(dev) if _overlap() else None
    keep = []                      # tensors the side stream reads: held until the join so the allocator cannot recycle them early

    def conv_wgrad_async(conv, a, g, n, h, w, in_layout, out_layout, arm="fp32"):
        """conv_wgrad on the side stream.  The pair forms are made on the CURRENT stream first (the data-gradient conv of the same
        layer reuses them from the memo), then the side stream waits for everything that stream has enqueued so far."""
        if side is None:
            return conv_wgrad(conv, a, g, n, h, w, in_layout, out_layout, arm=arm)
        pairs = (to_pair(a), to_pair(g)) if wgrad_on_tensor_cores(conv, n, h, w, in_layout, out_layout, arm) else None
        side.wait_stream(torch.cuda.current_stream(dev))           # the producing stream: main, or the g_s branch
        with torch.cuda.stream(side):
            out = conv_wgrad(conv, a, g, n, h, w, in_layout, out_layout, arm=arm, pairs=pairs)
        keep.extend((a, g, pairs))
        return out

    with torch.cuda.device(dev), torch.no_grad():
        d_yin = None                                             # NHWC gradient w.r.t. y_in from the entropy path (likelihood, context)
        d_yin_gs = None                                          # ... and from g_s, whose backward runs as its own branch
        branch = _side_stream(dev, 1) if (_overlap() and g_xhat is not None) else None
        # ---- g_s ------------------------------------------------------------------------------------------------
        if g_xhat is not None:
            import contextlib
            if branch is not None:
                branch.wait_stream(main)
            with (torch.cuda.stream(branch) if branch is not None else contextlib.nullcontext()):
                d_yin_gs = S["g_s"].backward(g_xhat.contiguous().float(), LAYOUT_NCHW, put, conv_wgrad_async, root=S["y_in_nhwc"],
                                             side=side, keep=keep)
        # ---- p_y: every head's likelihood, entropy parameters and context model; h_s --------------------------------
        # the y gradient of the entropy path is the channel concatenation of the heads', the psi gradient their sum
        d_zin = None
        if all(g is not None for g in g_logp_heads):
            d_ys, d_psi = [], None
            for head, st, gl in zip(heads(model), S["heads"], g_logp_heads):
                d_y, d_psi_i = head_backward(arm, head, model.K, st, gl, put, conv_wgrad_async)
                d_ys.append(d_y)
                d_psi = d_psi_i if d_psi is None else add_(d_psi, d_psi_i)
            d_yin = d_ys[0] if len(d_ys) == 1 else torch.cat(d_ys, dim=-1)
            del d_ys
            d_zin = S["h_s"].backward(d_psi, LAYOUT_NHWC, put, conv_wgrad_async, root=S["z_in_nhwc"], side=side, keep=keep)
        # ---- p_z ----------------------------------------------------------------------------------------------------
        if g_logp_z is not None:
            dz = factorized_bwd(model.factorized_entropy_model, S["z_in"], S["fparams"], g_logp_z, put)
            d_zin = to_nhwc(dz, accumulate_into=d_zin)
        # ---- h_a (z_in = z + noise: the gradient passes unchanged) --------------------------------------------------
        dy = d_yin
        if d_zin is not None:
            g = S["h_a"].backward(d_zin, LAYOUT_NHWC, put, conv_wgrad_async, root=S["y_nhwc"], side=side, keep=keep)
            dy = g if dy is None else add_(dy, g)
            del g                                                # summed into dy: free it before g_a's backward
        # ---- merge the branches: dy = d(entropy path) + d(h_a) + d(g_s) ---------------------------------------------------------
        if branch is not None:
            main.wait_stream(branch)
        if d_yin_gs is not None:
            dy = d_yin_gs if dy is None else add_(dy, d_yin_gs)
        if partial_hook is not None:
            partial_hook(grads, [st for st in (main, side) if st is not None])
        # ---- g_a (y_in = y + noise) ---------------------------------------------------------------------------------
        if dy is not None:
            S["g_a"].backward(dy, LAYOUT_NHWC, put, conv_wgrad_async, root=None, side=side, keep=keep)
    if side is not None:
        main.wait_stream(side)     # join: every weight gradient is complete before the caller (optimizer, all-reduce) reads it
    keep.clear()
    forget_pairs()
    return grads


class _TrainForward(torch.autograd.Function):
    """The whole model as ONE autograd node (what makes the reference trainer's loss.backward() work, Trainer.py:85)."""

    @staticmethod
    def forward(ctx, model, x, noise_z, noise_y, lean, *params):
        outs, S = _forward_impl(model, x, noise_z, noise_y, lean)
        ctx.model, ctx.S = model, S
        ctx.mark_non_differentiable(*outs[3:])
        return outs

    @staticmethod
    def backward(ctx, g_xhat, g_logp_y, g_logp_z, *unused):
        model, S = ctx.model, ctx.S
        if S is None:
            raise RuntimeError("the saved activations of this forward pass were released by its first backward(); run the forward "
                               "again (retain_graph=True is not supported by the hand-written backward)")
        grads = _backward_impl(model, S, g_xhat, [g_logp_y], g_logp_z)
        ctx.S = None
        params = [p for _, p in model.named_parameters()]
        return (None, None, None, None, None, *[grads.get(id(p)) for p in params])


DISTORTIONS = ("mse", "ms-ssim")


@torch.no_grad()
def step_gradients(model, x: torch.Tensor, lambda_rd: float, noise=None, partial_hook=None, distortion: str = "mse"):
    """forward + rd_loss + backward of one step WITHOUT the autograd engine (everything on the calling thread and its current
    stream - what a CUDA-graph capture needs): accumulates into .grad like loss.backward() and returns
    (loss [device scalar], per_image [3, B], scalars [8]).  distortion="ms-ssim": the loss of ms_ssim_rd_loss, whose x_hat
    gradient comes from nic_ms_ssim_bwd; scalars then has a 9th entry, the batch MS-SSIM, and entry 5 is that loss."""
    from .RateDistortionLoss import check_ms_ssim_shape, ms_ssim_terms, rd_terms
    if distortion not in DISTORTIONS:
        raise ValueError(f"distortion must be one of {DISTORTIONS}, got {distortion!r}")
    if distortion == "ms-ssim":
        check_ms_ssim_shape(tuple(x.shape))
    B, _, H, W = x.shape
    noise_z, noise_y = draw_noise(model.M, x, noise)
    forget_pairs()
    x = x.contiguous().float()
    outs, S = _forward_impl(model, x, noise_z, noise_y, True)
    x_hat, logp_y, logp_z = outs[:3]
    engine.attach_partials(logp_y, outs[9])
    engine.attach_partials(logp_z, outs[10])
    if distortion == "ms-ssim":
        per_image, scalars, _, state = ms_ssim_terms({"x_hat": x_hat, "logp_y": logp_y, "logp_z": logp_z}, x, lambda_rd)
        gx = ms_ssim_x_hat_grad(state, lambda_rd)
    else:
        per_image, scalars = rd_terms({"x_hat": x_hat, "logp_y": logp_y, "logp_z": logp_z}, x, lambda_rd)
        # d loss / d x_hat = lambda * 255^2 * 2 (x_hat - x) / numel  (RateDistortionLoss.py:13-34)
        gx = torch.empty_like(x_hat)
        with torch.cuda.device(x.device):
            check(_lib.load().nic_sse_bwd(ptr(x_hat), ptr(x), x.numel(), float(lambda_rd) * 65025.0 * 2.0 / x.numel(), ptr(gx), current_stream()),
                  "nic_sse_bwd")
    gl = torch.full((1,), -1.0 / (math.log(2.0) * H * W * B), dtype=torch.float32, device=x.device)     # d loss / d logp, both losses
    grads = _backward_impl(model, S, gx, [gl.expand(logp_y.shape)], gl.expand(logp_z.shape), partial_hook=partial_hook)
    for p in model.parameters():
        g = grads.get(id(p))
        if g is not None:
            p.grad = g if p.grad is None else p.grad + g
    return scalars[5], per_image, scalars


def train_forward(model, x: torch.Tensor, noise=None, lean: bool = False) -> dict:
    """``model(x, training=True)`` as a differentiable call (used by JointAutoregressiveHierarchical.forward when autograd is on)."""
    noise_z, noise_y = draw_noise(model.M, x, noise)
    forget_pairs()
    params = [p for _, p in model.named_parameters()]
    res = _TrainForward.apply(model, x.contiguous().float(), noise_z, noise_y, lean, *params)
    return single_head_outputs(*res, K=model.K, training=True)


class _RDLoss(torch.autograd.Function):
    """loss = bpp_total + lambda * 255^2 * mse (RateDistortionLoss.py:13-34) as one node: the value comes from nic_rd_finalize,
    the gradients are d loss / d logp = -1 / (ln 2 * H * W * B) and d loss / d x_hat = lambda * 255^2 * 2 (x_hat - x) / (B * C * H * W)."""

    @staticmethod
    def forward(ctx, logp_y, logp_z, x_hat, x, lambda_rd, scalars):
        ctx.save_for_backward(x_hat, x)
        ctx.lambda_rd, ctx.shapes = float(lambda_rd), (logp_y.shape, logp_z.shape)
        return scalars[5].clone()

    @staticmethod
    def backward(ctx, g):
        x_hat, x = ctx.saved_tensors
        B, C_, H, W = x.shape
        gl = g.float() * (-1.0 / (math.log(2.0) * H * W * B))
        gx = torch.empty_like(x_hat)
        coef = ctx.lambda_rd * 65025.0 * 2.0 / x.numel()
        with torch.cuda.device(x_hat.device):
            check(_lib.load().nic_sse_bwd(ptr(x_hat), ptr(x), x.numel(), coef, ptr(gx), current_stream()), "nic_sse_bwd")
        gx.mul_(g.float())
        return gl.expand(ctx.shapes[0]), gl.expand(ctx.shapes[1]), gx, None, None, None


def ms_ssim_x_hat_grad(state, lambda_rd: float, g: Optional[torch.Tensor] = None) -> torch.Tensor:
    """d loss / d x_hat of loss = bpp + lambda * (1 - mean ms_ssim) (times the upstream scalar g) through nic_ms_ssim_bwd, from the
    state ms_ssim_terms returned: the level coefficients are d loss / d term = -lambda / planes * d value / d term."""
    from .Evaluator import term_grads
    x_hat, x, terms, value, ws = state
    b, c, h, w = x.shape
    coef = term_grads(terms, value) * (-float(lambda_rd) / (b * c))
    if g is not None:
        coef = coef * g.float()
    gx = torch.empty_like(x_hat)
    with torch.cuda.device(x_hat.device):
        check(_lib.load().nic_ms_ssim_bwd(ptr(x_hat), ptr(x), b * c, h, w, 1.0, ptr(coef), ptr(gx), ptr(ws), ws.numel(), current_stream()),
              "nic_ms_ssim_bwd")
    return gx


class _MSSSIMRDLoss(torch.autograd.Function):
    """loss = bpp_total + lambda * (1 - mean_b ms_ssim_b) (RateDistortionLoss.ms_ssim_rd_loss) as one node: the value comes from
    ms_ssim_terms, the gradients are d loss / d logp = -1 / (ln 2 * H * W * B) and the x_hat gradient of nic_ms_ssim_bwd."""

    @staticmethod
    def forward(ctx, logp_y, logp_z, x_hat, lambda_rd, scalars, state):
        ctx.state, ctx.lambda_rd, ctx.shapes = state, float(lambda_rd), (logp_y.shape, logp_z.shape)
        return scalars[5].clone()

    @staticmethod
    def backward(ctx, g):
        B, _, H, W = ctx.state[1].shape
        gl = g.float() * (-1.0 / (math.log(2.0) * H * W * B))
        gx = ms_ssim_x_hat_grad(ctx.state, ctx.lambda_rd, g)
        ctx.state = None
        return gl.expand(ctx.shapes[0]), gl.expand(ctx.shapes[1]), gx, None, None, None


class Adam(torch.optim.Optimizer):
    """torch.optim.Adam(params, lr) (Main.ipynb:133; defaults betas (0.9, 0.999), eps 1e-8, no weight decay) on the one-launch
    update kernel (nic_adam_multi_step_ex).

    A torch.optim.Optimizer: ``param_groups`` (so ``ReduceLROnPlateau`` / ``CosineAnnealingLR`` and ``param_groups[0]['lr']`` of
    Trainer.py:33-36, 103 work), and ``state_dict()`` / ``load_state_dict()`` in torch.optim.Adam's own format (per parameter
    ``step``, ``exp_avg``, ``exp_avg_sq``), so the reference's checkpoints (Trainer.py:52-68) round-trip in both directions.
    The learning rate the kernel uses lives in DEVICE memory and is refreshed from ``param_groups`` before every launch / replay
    (``sync_lr``): a scheduler's change reaches a CUDA-graph replay of the update without re-capturing.  One parameter group."""

    def __init__(self, params, lr: float = 1e-4, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0, amsgrad: bool = False):
        if weight_decay != 0.0 or amsgrad:
            raise ValueError("Adam: weight_decay / amsgrad are not built (the reference trains with torch.optim.Adam(lr) defaults)")
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=0.0, amsgrad=False, maximize=False, foreach=None, capturable=False,
                        differentiable=False, fused=None, decoupled_weight_decay=False)
        super().__init__(params, defaults)
        if len(self.param_groups) != 1:
            raise ValueError("Adam: one parameter group")
        self.params: List[torch.Tensor] = list(self.param_groups[0]["params"])
        self.t = 0                                       # steps taken (host mirror of the device counter)
        self._t_dev = None                               # the step count on the device (what the update kernel reads)
        self._lr_dev, self._lr_host = None, None         # the learning rate on the device + the value last written there
        self.grad_scale = 1.0                            # gradients are multiplied by this inside the kernel (1 / world for SUM all-reduces)
        self.m = [torch.zeros_like(p, dtype=torch.float32) for p in self.params]
        self.v = [torch.zeros_like(p, dtype=torch.float32) for p in self.params]

    # ---- torch.optim.Adam-compatible checkpoint format -------------------------------------------------------------------
    @property
    def lr(self) -> float:
        return float(self.param_groups[0]["lr"])

    @lr.setter
    def lr(self, value: float):
        self.param_groups[0]["lr"] = float(value)

    @property
    def betas(self):
        return tuple(self.param_groups[0]["betas"])

    @property
    def eps(self) -> float:
        return float(self.param_groups[0]["eps"])

    def _publish_state(self):
        """self.state in torch.optim.Adam's layout; exp_avg / exp_avg_sq ALIAS the buffers the kernel updates."""
        for p, m, v in zip(self.params, self.m, self.v):
            self.state[p] = {"step": torch.tensor(float(self.t)), "exp_avg": m, "exp_avg_sq": v}

    def state_dict(self):
        self._publish_state()
        return super().state_dict()

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        self.params = list(self.param_groups[0]["params"])
        steps = set()
        for i, p in enumerate(self.params):
            st = self.state.get(p)
            if not st:
                continue
            self.m[i] = st["exp_avg"].to(device=p.device, dtype=torch.float32).contiguous()
            self.v[i] = st["exp_avg_sq"].to(device=p.device, dtype=torch.float32).contiguous()
            steps.add(int(float(st["step"])))
        if len(steps) > 1:
            raise ValueError(f"Adam.load_state_dict: parameters at different step counts {sorted(steps)} (one shared counter is built)")
        self.t = steps.pop() if steps else 0
        if self._t_dev is not None:
            self._t_dev.fill_(self.t)                     # the device counter follows the restored step count
        self._lr_host = None                              # re-upload the restored learning rate

    def zero_grad(self, set_to_none: bool = True):
        for p in self.params:
            if set_to_none:
                p.grad = None
            elif p.grad is not None:
                p.grad.zero_()

    def sync_lr(self, dev=None):
        """Write param_groups[0]['lr'] to the device scalar if it changed (a 4-byte stream-ordered copy; called before every launch
        and before every graph replay - never inside a capture)."""
        if self._lr_dev is None:
            if dev is None:
                return
            self._lr_dev = torch.empty(1, dtype=torch.float32, device=dev)
        if self._lr_host != self.lr and not torch.cuda.is_current_stream_capturing():
            self._lr_dev.fill_(self.lr)
            self._lr_host = self.lr

    @torch.no_grad()
    def launch(self):
        """Advance the device step counter and update every parameter that has a gradient: two stream-ordered launches
        (nic_counter_increment, nic_adam_multi_step_ex with the pointers as launch arguments), no upload, no host
        synchronisation, capturable in a CUDA graph (the bias corrections are formed on the device from the counter, the
        learning rate is read from its device scalar)."""
        lib = _lib.load()
        live = [(p, p.grad.contiguous().float(), m, v) for p, m, v in zip(self.params, self.m, self.v) if p.grad is not None]
        if not live:
            return
        for p, _, _, _ in live:
            engine.require_cuda(p, "parameter")
        dev = live[0][0].device
        self.prepare(dev)
        n = len(live)
        arr = lambda k: (C.c_void_p * n)(*[t[k].data_ptr() for t in live])     # noqa: E731
        counts = (C.c_int64 * n)(*[t[0].numel() for t in live])
        with torch.cuda.device(dev):
            self.sync_lr(dev)
            check(lib.nic_counter_increment(ptr(self._t_dev), current_stream()), "nic_counter_increment")
            check(lib.nic_adam_multi_step_ex(arr(0), arr(1), arr(2), arr(3), counts, n, self.lr, ptr(self._lr_dev), float(self.grad_scale),
                                             self.betas[0], self.betas[1], self.eps, 1, ptr(self._t_dev), current_stream()),
                  "nic_adam_multi_step_ex")
        self._keep = live                                 # the gradients stay alive until the next launch

    def prepare(self, dev):
        """Create the device step counter and learning-rate scalar (outside any CUDA-graph capture: a captured fill would reset
        them on every replay)."""
        if self._t_dev is None or self._t_dev.device != dev:
            self._t_dev = torch.full((1,), self.t, dtype=torch.int32, device=dev)
        if self._lr_dev is None or self._lr_dev.device != dev:
            self._lr_dev, self._lr_host = torch.full((1,), self.lr, dtype=torch.float32, device=dev), self.lr

    def step(self, closure=None):
        loss = closure() if closure is not None else None
        self.launch()
        self.t += 1
        for p in self.params:
            if p.grad is not None:
                torch.autograd.graph.increment_version(p)       # updated behind torch's back: packed-weight caches key on _version
        return loss
