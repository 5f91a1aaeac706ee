"""The 3x3 residual building blocks of /root/reference/Layers.py on the sm_100a conv engine.

Same class names, constructor arguments and parameter names (``conv1 / conv2 / gdn / skip``, ``subpel_conv.deconv / conv / igdn /
upsample.deconv``, ``conv / shuffle``, ``deconv``) so that ``state_dict`` round-trips with the reference.  Each block executes as
a short chain of C-ABI calls - ``nic_conv_fwd`` with the bias / LeakyReLU epilogue fused, the GDN / IGDN contraction, and
``nic_add_inplace`` for the residual sum - on f32 NHWC tensors (``run_nhwc``); ``forward`` wraps that for stand-alone NCHW calls.
With a ``tape`` (training.Tape) the same chain is the TRAINING forward: every op is recorded for the hand-written backward.
Arithmetic: "bf16x3" (tensor cores, hi/lo-split operands; layers whose input channel count is not a multiple of 64, e.g. the
3-channel first block, run on the fp32 CUDA-core kernels) or "fp32".
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from . import engine
from ._lib import EPI_BIAS, EPI_LRELU, LAYOUT_NCHW, LAYOUT_NHWC
from .gdn import GDN


def _T():
    from . import training
    return training


def _arm(precision: Optional[str], channels: int) -> str:
    p = engine.resolve_precision(precision, channels)
    return p if p in ("fp32", "bf16x3") else "bf16x3"


def _conv(arm, conv, epi, x, n, h, w, in_layout=LAYOUT_NHWC, out_layout=LAYOUT_NHWC, tape=None, pair_out=False, **out_kw):
    """One conv (+ bias / LeakyReLU) -> (f32 tensor, h_out, w_out).  tape: the training forward's record (training.Tape); the RGB
    layer then stays NCHW (it is the transform's output and x_hat is NCHW)."""
    T = _T()
    if tape is not None:
        lay = LAYOUT_NCHW if (out_layout == LAYOUT_NHWC and conv.out_channels % 4) else out_layout
        return (tape.conv(conv, epi, x, h, w, in_layout=in_layout, out_layout=lay, **out_kw),) + engine.conv_out_hw(conv, h, w)
    if out_layout == LAYOUT_NHWC and conv.out_channels % 4:
        # NHWC rows of e.g. 3 floats are not 16-byte aligned (the engine's NHWC stores are vectorised): such layers - the RGB
        # output of g_s - write NCHW, and the chain's NHWC convention is restored by a view permutation
        y = T.conv_forward(arm, conv, epi, x, n, h, w, in_layout=in_layout, out_layout=LAYOUT_NCHW).permute(0, 2, 3, 1).contiguous()
    else:
        # pair_out: the only consumer is the next conv - in the bf16x3 arm the result stays a bf16 hi/lo pair (evaluation only:
        # the training forward keeps f32 activations for the backward)
        y = T.conv_forward(arm, conv, epi, x, n, h, w, in_layout=in_layout, out_layout=out_layout, pair_out=pair_out, **out_kw)
    T.forget_pairs()
    return (y,) + engine.conv_out_hw(conv, h, w)


def _gdn(arm, gdn, u, n, h, w, tape=None, addend=None):
    """GDN / IGDN; addend (evaluation only): + the block's skip branch in the same pass."""
    T = _T()
    if tape is not None:
        return tape.gdn(gdn, u, h, w)
    y = T.gdn_forward(arm, gdn, u, n, h, w, addend=addend)[0]
    T.forget_pairs()
    return y


def _add(out, idn, tape=None):
    return tape.add(out, idn) if tape is not None else _T().add_(out, idn)


class _Block(nn.Module):
    precision = None      # None -> bf16x3 where the channel counts allow, else fp32; set by the owning model

    def run_nhwc(self, x, n, h, w, arm, in_layout=LAYOUT_NHWC, tape=None):
        raise NotImplementedError

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """Stand-alone call with the reference's NCHW f32 tensors at both ends (cold path)."""
        engine.require_cuda(x, "x")
        n, c, h, w = x.shape
        arm = _arm(self.precision, c if c >= 64 else 64)
        with torch.cuda.device(x.device), torch.no_grad():
            y, ho, wo = self.run_nhwc(x.contiguous().float(), n, h, w, arm, in_layout=LAYOUT_NCHW)
        return y.permute(0, 3, 1, 2).contiguous()


class SubpelConv3x3(_Block):
    """Conv2d(in, out * r^2, 3) + PixelShuffle(r) (Layers.py:6-16; unused by the reference's own models, which build
    TransposedDeconv3x3 in its place - kept for API parity).  The shuffle is a pure index permutation (torch view ops)."""

    def __init__(self, in_ch, out_ch, upsample=2):
        super().__init__()
        self.conv = nn.Conv2d(in_ch, out_ch * (upsample ** 2), kernel_size=3, stride=1, padding=1)
        self.shuffle = nn.PixelShuffle(upsample)

    def run_nhwc(self, x, n, h, w, arm, in_layout=LAYOUT_NHWC, tape=None):
        y, h, w = _conv(arm, self.conv, EPI_BIAS, x, n, h, w, in_layout=in_layout, tape=tape)
        r = self.shuffle.upscale_factor
        c = y.shape[-1] // (r * r)
        y = y.reshape(n, h, w, c, r, r).permute(0, 1, 4, 2, 5, 3).reshape(n, h * r, w * r, c).contiguous()
        return y, h * r, w * r


class TransposedDeconv3x3(_Block):
    """ConvTranspose2d(in, out, 3, stride r, padding 1, output_padding r - 1) (Layers.py:18-24)."""

    def __init__(self, in_ch, out_ch, upsample=2):
        super().__init__()
        self.deconv = nn.ConvTranspose2d(in_ch, out_ch, kernel_size=3, stride=upsample, padding=1, output_padding=upsample - 1)

    def run_nhwc(self, x, n, h, w, arm, in_layout=LAYOUT_NHWC, epilogue=EPI_BIAS, tape=None, pair_out=False, **out_kw):
        return _conv(arm, self.deconv, epilogue, x, n, h, w, in_layout=in_layout, tape=tape, pair_out=pair_out, **out_kw)


class ResidualBlockWithStride(_Block):
    """conv3x3(stride) -> LeakyReLU -> conv3x3 -> GDN, plus a 1x1 strided skip (Layers.py:27-61)."""

    def __init__(self, in_ch: int, out_ch: int, stride: int = 2):
        super().__init__()
        self.conv1 = nn.Conv2d(in_ch, out_ch, kernel_size=3, stride=stride, padding=1)
        self.leaky_relu = nn.LeakyReLU(inplace=True)
        self.conv2 = nn.Conv2d(out_ch, out_ch, kernel_size=3, stride=1, padding=1)
        self.gdn = GDN(out_ch, beta_min=1e-6, gamma_init=.1)
        self.skip = nn.Conv2d(in_ch, out_ch, kernel_size=1, stride=stride) if (stride != 1 or in_ch != out_ch) else None

    def run_nhwc(self, x, n, h, w, arm, in_layout=LAYOUT_NHWC, tape=None):
        T = _T()
        u, ho, wo = _conv(arm, self.conv1, EPI_LRELU, x, n, h, w, in_layout=in_layout, tape=tape, pair_out=True)
        u, _, _ = _conv(arm, self.conv2, EPI_BIAS, u, n, ho, wo, tape=tape)
        if tape is not None:
            out = _gdn(arm, self.gdn, u, n, ho, wo, tape=tape)
        if self.skip is not None:
            idn, _, _ = _conv(arm, self.skip, EPI_BIAS, x, n, h, w, in_layout=in_layout, tape=tape)
        else:
            idn = x if in_layout == LAYOUT_NHWC else x.permute(0, 2, 3, 1).contiguous()
        if tape is None:
            return _gdn(arm, self.gdn, u, n, ho, wo, addend=idn), ho, wo            # GDN and the residual sum in one pass
        return _add(out, idn, tape), ho, wo


class ResidualBlockUpsample(_Block):
    """deconv3x3(r) -> LeakyReLU -> conv3x3 -> IGDN, plus a deconv3x3(r) skip (Layers.py:64-88)."""

    def __init__(self, in_ch: int, out_ch: int, upsample: int = 2):
        super().__init__()
        self.subpel_conv = TransposedDeconv3x3(in_ch, out_ch, upsample)
        self.leaky_relu = nn.LeakyReLU(inplace=True)
        self.conv = nn.Conv2d(out_ch, out_ch, kernel_size=3, stride=1, padding=1)
        self.igdn = GDN(out_ch, inverse=True, beta_min=1e-6, gamma_init=.1)
        self.upsample = TransposedDeconv3x3(in_ch, out_ch, upsample)

    def run_nhwc(self, x, n, h, w, arm, in_layout=LAYOUT_NHWC, tape=None):
        T = _T()
        u, ho, wo = self.subpel_conv.run_nhwc(x, n, h, w, arm, in_layout=in_layout, epilogue=EPI_LRELU, tape=tape, pair_out=True)
        u, _, _ = _conv(arm, self.conv, EPI_BIAS, u, n, ho, wo, tape=tape)
        if tape is not None:
            out = _gdn(arm, self.igdn, u, n, ho, wo, tape=tape)
        idn, _, _ = self.upsample.run_nhwc(x, n, h, w, arm, in_layout=in_layout, tape=tape)
        if tape is None:
            return _gdn(arm, self.igdn, u, n, ho, wo, addend=idn), ho, wo           # IGDN and the residual sum in one pass
        return _add(out, idn, tape), ho, wo


class ResidualBlock(_Block):
    """conv3x3 -> LeakyReLU -> conv3x3 -> LeakyReLU, plus the identity (or a 1x1 skip) (Layers.py:91-119)."""

    def __init__(self, in_ch: int, out_ch: int):
        super().__init__()
        self.conv1 = nn.Conv2d(in_ch, out_ch, kernel_size=3, stride=1, padding=1)
        self.leaky_relu = nn.LeakyReLU(inplace=True)
        self.conv2 = nn.Conv2d(out_ch, out_ch, kernel_size=3, stride=1, padding=1)
        self.skip = nn.Conv2d(in_ch, out_ch, kernel_size=1, stride=1) if in_ch != out_ch else None

    def run_nhwc(self, x, n, h, w, arm, in_layout=LAYOUT_NHWC, tape=None):
        T = _T()
        u, _, _ = _conv(arm, self.conv1, EPI_LRELU, x, n, h, w, in_layout=in_layout, tape=tape, pair_out=True)
        out, _, _ = _conv(arm, self.conv2, EPI_LRELU, u, n, h, w, tape=tape)
        if self.skip is not None:
            idn, _, _ = _conv(arm, self.skip, EPI_BIAS, x, n, h, w, in_layout=in_layout, tape=tape)
        else:
            idn = x if in_layout == LAYOUT_NHWC else x.permute(0, 2, 3, 1).contiguous()
        return _add(out, idn, tape), h, w
