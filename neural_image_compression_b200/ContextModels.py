"""Masked autoregressive context model (/root/reference/ContextModels.py), the checkerboard context model and the channel context
model of the channel slices.

``MaskedConv2d`` keeps the reference's ``weight`` / ``bias`` parameters and ``mask`` buffer
(:12-16).  The engine packs only the live taps of mask 'A' (12 of 25 for 5x5), so the masked
positions are never multiplied; to stay checkpoint-identical with the reference, whose forward
zeroes them in place (:19), the first forward zeroes them once here too.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import engine
from ._lib import EPI_BIAS, MASK_CHECKERBOARD


class MaskedConv2d(nn.Conv2d):
    def __init__(self, mask_type, *args, **kwargs):
        super().__init__(*args, **kwargs)
        if mask_type not in ("A", "B"):
            raise AssertionError("mask_type must be 'A' or 'B'")
        kh, kw = self.kernel_size
        mask = torch.ones_like(self.weight.data)
        mask[:, :, kh // 2, kw // 2 + (mask_type == "B"):] = 0      # 'B' keeps the centre tap (ContextModels.py:15)
        mask[:, :, kh // 2 + 1:] = 0
        self.register_buffer("mask", mask)
        self.precision = None
        self._op = engine.ConvOp(self, EPI_BIAS, mask_a=1 if mask_type == "A" else 2)
        self._masked_version = None

    def apply_mask_(self):
        """The in-place side effect of ContextModels.py:19, done only when the weight changed."""
        key = (self.weight.data_ptr(), self.weight._version)
        if self._masked_version != key:
            with torch.no_grad():
                self.weight.data *= self.mask
            self._masked_version = (self.weight.data_ptr(), self.weight._version)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        self.apply_mask_()
        return engine.run_sequential_nchw([self._op], x, engine.resolve_precision(self.precision))


class ContextModel(nn.Module):
    def __init__(self, latent_channels: int = 192):
        super().__init__()
        self.masked = MaskedConv2d("A", in_channels=latent_channels, out_channels=2 * latent_channels,
                                   kernel_size=5, stride=1, padding=2)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self.masked(x)



# ---- checkerboard context (He et al., CVPR 2021, "Checkerboard Context Model for Efficient Learned Image Compression") ----------
# The convention, defined here once (DESIGN.md section 14):
#   * anchors are the latent positions (i, j) with i + j even, non-anchors those with i + j odd;
#   * the 5x5 context conv keeps the taps (kh, kw) with kh + kw odd - 12 of 25, no centre tap - so a non-anchor reads anchors only;
#   * its output phi, bias included, is 0 at every anchor before [phi | psi] enters the 1x1 stack, in training (noise) and in
#     evaluation (rounding) alike.  The engine drops the dead taps (nic_conv_desc.mask_a = NIC_MASK_CHECKERBOARD) and zeroes the
#     anchors in the same C-ABI call.
# So an anchor is coded from the hyperprior alone, a non-anchor from the hyperprior and the anchors: two decode passes.

def checkerboard_mask(weight: torch.Tensor) -> torch.Tensor:
    """1 at the taps (kh, kw) with kh + kw odd, else 0, in the shape of `weight`."""
    kh, kw = weight.shape[-2:]
    parity = (torch.arange(kh)[:, None] + torch.arange(kw)[None, :]) % 2
    return parity.to(weight.dtype).expand_as(weight).clone()


def anchor_mask(h: int, w: int, device=None) -> torch.Tensor:
    """bool [h, w]: True at the anchors (i + j even)."""
    return (torch.arange(h, device=device)[:, None] + torch.arange(w, device=device)[None, :]) % 2 == 0


class CheckerboardMaskedConv2d(MaskedConv2d):
    """MaskedConv2d with the checkerboard mask buffer: same parameters, same ``mask`` key.  Loading a ``mask`` other than the
    checkerboard one (a JointAutoregressiveHierarchical checkpoint's mask 'A') raises ValueError: apply_mask_ would otherwise zero
    the live taps of the weights it loads."""

    def __init__(self, *args, **kwargs):
        super().__init__("A", *args, **kwargs)
        self.mask.copy_(checkerboard_mask(self.weight.data))
        self._op = engine.ConvOp(self, EPI_BIAS, mask_a=MASK_CHECKERBOARD)

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        key = prefix + "mask"
        if key in state_dict and not torch.equal(state_dict[key].detach().to("cpu", self.mask.dtype), self.mask.detach().cpu()):
            raise ValueError(f"{key}: not the checkerboard mask (taps with kh + kw odd); a checkpoint of a mask-'A' context model "
                             f"cannot be loaded into a checkerboard context model")
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)


class CheckerboardContextModel(nn.Module):
    """ContextModel with the checkerboard context: ``.masked`` is a CheckerboardMaskedConv2d (5x5, M -> 2M)."""

    def __init__(self, latent_channels: int = 192):
        super().__init__()
        self.masked = CheckerboardMaskedConv2d(in_channels=latent_channels, out_channels=2 * latent_channels, kernel_size=5, stride=1,
                                               padding=2)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self.masked(x)


# ---- channel context (ELIC, He et al., CVPR 2022; Minnen & Singh, ICIP 2020): DESIGN.md section 16 ----------------------------
# Slice s of y (channels [o_s, o_s + m_s)) also reads the slices before it, y[:, :o_s], through one unmasked 5x5 conv.  Those slices
# are fully decoded before slice s starts, so its output phi_ch is NOT zeroed at the anchors.

class ChannelContextModel(nn.Module):
    """``.conv``: an unmasked 5x5 conv with bias, o_s -> 2 m_s, padding 2, over the channels [0, o_s) of y."""

    def __init__(self, in_channels: int, latent_channels: int):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, 2 * latent_channels, kernel_size=5, stride=1, padding=2)
        self._op = engine.ConvOp(self.conv, EPI_BIAS)

    def forward(self, y_prev: torch.Tensor) -> torch.Tensor:
        return engine.run_sequential_nchw([self._op], y_prev, "fp32")
