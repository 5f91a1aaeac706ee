"""Analysis / synthesis / hyper transforms: the 5x5 family of /root/reference/Components.py.

Same class names, constructor arguments and ``net.<i>`` parameter names as the reference
(Encoder5x5 :6-18, Decoder5x5 :35-47, HyperEncoder5x5 :65-75, HyperDecoder5x5 :94-105), so
``state_dict`` round-trips.  ``forward`` does not execute the ``nn.Sequential``: each
conv (+ the GDN / IGDN / LeakyReLU after it) is one ``nic_conv_fwd`` call with the activation fused
into the epilogue, activations staying NHWC between layers.  ``run_nhwc`` is the layer-by-layer form
the training step records on a ``training.Tape`` (GDN / IGDN as ops of their own).

The 3x3 residual family (Encoder3x3 / Decoder3x3 / HyperEncoder3x3 / HyperDecoder3x3, Components.py:20-32, 49-62, 77-91,
107-122; blocks in Layers.py) runs layer by layer on the same engine (SURVEY.md section 8 row f4).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import Layers as L
from . import engine
from ._lib import EPI_BIAS, EPI_GDN, EPI_IGDN, EPI_LRELU, LAYOUT_NCHW, LAYOUT_NHWC
from .gdn import GDN


def _ops_from_sequential(net: nn.Sequential):
    """Pair every conv with the activation that follows it."""
    ops, mods, i = [], list(net), 0
    while i < len(mods):
        conv = mods[i]
        nxt = mods[i + 1] if i + 1 < len(mods) else None
        if isinstance(nxt, GDN):
            ops.append(engine.ConvOp(conv, EPI_IGDN if nxt.inverse else EPI_GDN, gdn=nxt)); i += 2
        elif isinstance(nxt, nn.LeakyReLU):
            ops.append(engine.ConvOp(conv, EPI_LRELU)); i += 2
        else:
            ops.append(engine.ConvOp(conv, EPI_BIAS)); i += 1
    return ops


class _Transform(nn.Module):
    precision = None   # None -> engine.resolve_precision (fp32 for a stand-alone transform); set by the owning model

    def _build_ops(self):
        self._ops = _ops_from_sequential(self.net)

    @property
    def ops(self):
        return self._ops

    def run_nhwc(self, x, n, h, w, arm, in_layout=None, tape=None, final_kw=None):
        """The chain layer by layer on f32 NHWC tensors (the calls of _Chain.run_nhwc): a conv followed by a GDN / IGDN keeps the
        bias epilogue and the GDN runs as its own op (the training forward keeps the pre-GDN tensor for the GDN backward)."""
        layout = LAYOUT_NHWC if in_layout is None else in_layout
        for i, op in enumerate(self._ops):
            kw = final_kw if (final_kw and i == len(self._ops) - 1) else {}
            x, h, w = L._conv(arm, op.conv, EPI_BIAS if op.gdn is not None else op.epilogue, x, n, h, w, in_layout=layout, tape=tape,
                              **kw)
            if op.gdn is not None:
                x = L._gdn(arm, op.gdn, x, n, h, w, tape=tape)
            layout = LAYOUT_NHWC
        return x, h, w

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        # stand-alone call of one transform: the fp32 arm unless the owner asked for a tensor-core arm explicitly
        return engine.run_sequential_nchw(self._ops, x, engine.resolve_precision(self.precision))


def _conv(cin, cout, k, s):
    return nn.Conv2d(cin, cout, kernel_size=k, stride=s, padding=k // 2)


def _deconv(cin, cout):
    return nn.ConvTranspose2d(cin, cout, kernel_size=5, stride=2, padding=2, output_padding=1)


class Encoder5x5(_Transform):
    """g_a: four 5x5 stride-2 convs, GDN after the first three (Components.py:9-17)."""

    def __init__(self, latent_channels: int = 192):
        super().__init__()
        m, layers, cin = latent_channels, [], 3
        for i in range(4):
            layers.append(_conv(cin, m, 5, 2))
            if i < 3:
                layers.append(GDN(m, beta_min=1e-6, gamma_init=.1))
            cin = m
        self.net = nn.Sequential(*layers)
        self._build_ops()


class Decoder5x5(_Transform):
    """g_s: four 5x5 stride-2 transposed convs, IGDN after the first three (Components.py:38-46)."""

    def __init__(self, latent_channels: int = 192):
        super().__init__()
        m, layers = latent_channels, []
        for i in range(4):
            layers.append(_deconv(m, m if i < 3 else 3))
            if i < 3:
                layers.append(GDN(m, inverse=True, beta_min=1e-6, gamma_init=.1))
        self.net = nn.Sequential(*layers)
        self._build_ops()


class HyperEncoder5x5(_Transform):
    """h_a: 3x3 s1, 5x5 s2, 5x5 s2 with LeakyReLU(0.01) between (Components.py:68-74)."""

    def __init__(self, latent_channels: int = 192):
        super().__init__()
        m = latent_channels
        self.net = nn.Sequential(_conv(m, m, 3, 1), nn.LeakyReLU(inplace=True), _conv(m, m, 5, 2),
                                 nn.LeakyReLU(inplace=True), _conv(m, m, 5, 2))
        self._build_ops()


class HyperDecoder5x5(_Transform):
    """h_s: two 5x5 s2 transposed convs and a 3x3, LeakyReLU(0.01) between (Components.py:98-104)."""

    def __init__(self, latent_channels: int = 192):
        super().__init__()
        m = latent_channels
        self.net = nn.Sequential(_deconv(m, m), nn.LeakyReLU(inplace=True), _deconv(m, int(1.5 * m)),
                                 nn.LeakyReLU(inplace=True), _conv(int(1.5 * m), 2 * m, 3, 1))
        self._build_ops()
        mid = int(1.5 * m)
        if mid % 64 and mid > 64:       # e.g. m = 192: 288 channels travel as 320 on the tensor-core arms (engine.ConvOp)
            pad = (mid + 63) // 64 * 64
            self._ops[1].tc_pad_cout, self._ops[2].tc_pad_cin = pad, pad


# ---- the 3x3 residual family (SURVEY.md section 8 row f4) -----------------------------------------------------------------------

class _Chain(nn.Module):
    """`net` = the reference's nn.Sequential of residual blocks / convs / LeakyReLUs, executed as a chain of engine calls on f32
    NHWC tensors: a conv followed by nn.LeakyReLU runs with the LeakyReLU epilogue fused."""
    precision = None

    def run_nhwc(self, x, n, h, w, arm, in_layout=None, tape=None, final_kw=None):
        """tape: training.Tape that records every op for the backward (training forward); final_kw: output arguments of the LAST
        conv (`out=` window: h_s writes psi straight into the concat buffer of the entropy-parameter stack; out_layout: g_s writes
        x_hat NCHW)."""
        layout = LAYOUT_NHWC if in_layout is None else in_layout
        mods, i = list(self.net), 0
        while i < len(mods):
            m = mods[i]
            nxt = mods[i + 1] if i + 1 < len(mods) else None
            fuse = isinstance(nxt, nn.LeakyReLU)
            kw = final_kw if (final_kw and i == len(mods) - 1) else {}
            after = mods[i + (2 if fuse else 1)] if i + (2 if fuse else 1) < len(mods) else None
            # evaluation: a conv whose only consumer is the next conv hands its result over as a bf16 hi/lo pair (bf16x3 arm)
            pair = tape is None and isinstance(after, (nn.Conv2d, nn.ConvTranspose2d, L.TransposedDeconv3x3))
            if isinstance(m, L.TransposedDeconv3x3):
                x, h, w = m.run_nhwc(x, n, h, w, arm, in_layout=layout, epilogue=EPI_LRELU if fuse else EPI_BIAS, tape=tape, pair_out=pair,
                                    **kw)
            elif isinstance(m, L._Block):
                x, h, w = m.run_nhwc(x, n, h, w, arm, in_layout=layout, tape=tape)
                fuse = False
            elif isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)):
                x, h, w = L._conv(arm, m, EPI_LRELU if fuse else EPI_BIAS, x, n, h, w, in_layout=layout, tape=tape, pair_out=pair, **kw)
            else:
                raise TypeError(f"unexpected module in a transform: {type(m).__name__}")
            layout = LAYOUT_NHWC
            i += 2 if fuse else 1
        return x, h, w

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        engine.require_cuda(x, "x")
        n, c, h, w = x.shape
        arm = L._arm(self.precision, c if c >= 64 else 64)
        with torch.cuda.device(x.device), torch.no_grad():
            y, _, _ = self.run_nhwc(x.contiguous().float(), n, h, w, arm, in_layout=LAYOUT_NCHW)
        return y.permute(0, 3, 1, 2).contiguous()


class Encoder3x3(_Chain):
    """g_a of the residual family: three (strided residual block + GDN, residual block) pairs and a stride-2 3x3 bottleneck
    (Components.py:20-32)."""

    def __init__(self, latent_channels=192):
        super().__init__()
        from .Layers import ResidualBlock, ResidualBlockWithStride
        m, blocks, cin = latent_channels, [], 3
        for _ in range(3):
            blocks += [ResidualBlockWithStride(cin, m, stride=2), ResidualBlock(m, m)]
            cin = m
        self.net = nn.Sequential(*blocks, nn.Conv2d(m, m, kernel_size=3, stride=2, padding=1))


class Decoder3x3(_Chain):
    """g_s: (residual block, upsampling residual block + IGDN) x 3, a residual block and a 3x3 stride-2 transposed conv to RGB
    (Components.py:49-62)."""

    def __init__(self, latent_channels=192):
        super().__init__()
        from .Layers import ResidualBlock, ResidualBlockUpsample, TransposedDeconv3x3
        m, blocks = latent_channels, []
        for _ in range(3):
            blocks += [ResidualBlock(m, m), ResidualBlockUpsample(m, m, 2)]
        self.net = nn.Sequential(*blocks, ResidualBlock(m, m), TransposedDeconv3x3(m, 3, 2))


class HyperEncoder3x3(_Chain):
    """h_a: five 3x3 convs (strides 1, 1, 2, 1, 2) with LeakyReLU between (Components.py:77-91)."""

    def __init__(self, latent_channels=192):
        super().__init__()
        m, layers = latent_channels, []
        for i, s in enumerate((1, 1, 2, 1, 2)):
            layers.append(nn.Conv2d(m, m, kernel_size=3, stride=s, padding=1))
            if i < 4:
                layers.append(nn.LeakyReLU(inplace=True))
        self.net = nn.Sequential(*layers)


class HyperDecoder3x3(_Chain):
    """h_s: conv, deconv x2, conv (-> 1.5 M), deconv x2, conv (-> 2 M), LeakyReLU between (Components.py:107-122)."""

    def __init__(self, latent_channels=192):
        super().__init__()
        from .Layers import TransposedDeconv3x3
        m, mid = latent_channels, int(1.5 * latent_channels)
        act = lambda: nn.LeakyReLU(inplace=True)      # noqa: E731
        self.net = nn.Sequential(nn.Conv2d(m, m, kernel_size=3, stride=1, padding=1), act(), TransposedDeconv3x3(m, m, 2), act(),
                                 nn.Conv2d(m, mid, kernel_size=3, stride=1, padding=1), act(), TransposedDeconv3x3(mid, mid, 2), act(),
                                 nn.Conv2d(mid, 2 * m, kernel_size=3, stride=1, padding=1))
