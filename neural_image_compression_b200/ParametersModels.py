"""Entropy-parameter network (/root/reference/ParametersModels.py:8-64).

Three 1x1 convolutions 2M+2H -> 640 -> 640 -> {2M | 3KM} with LeakyReLU(0.01); the split into
(mu, sigma) or (weights, mus, sigmas) with softmax over K and softplus + 1e-6 is done by the
likelihood kernel (``nic_gm_likelihood_fwd`` also emits these tensors).  Called stand-alone,
``forward`` returns the same tuples as the reference.
"""
from __future__ import annotations

from typing import Tuple

import torch
import torch.nn as nn
from torch import Tensor

from . import engine
from ._lib import EPI_BIAS, EPI_LRELU


class EntropyParameters(nn.Module):
    def __init__(self, latent_channels: int = 192, hyper_latent_channels: int = 192, K: int = 1, *, context_channels: int = 0):
        """context_channels: extra input channels between phi and psi (the channel context of ChannelCheckerboardHierarchical's
        slices: [phi (2M) | phi_ch (context_channels) | psi (2H)]); 0 is the reference's stack."""
        super().__init__()
        if not isinstance(K, int) or K < 1:
            raise ValueError(f"K must be int >= 1, got {K}")
        self.K = K
        self.distribution = "Mean-Scale Gaussian" if K == 1 else "Mixture of Gaussians"
        self.latent_channels = latent_channels
        self.hyper_latent_channels = hyper_latent_channels
        cin = 2 * latent_channels + context_channels + 2 * hyper_latent_channels
        cout = 2 * latent_channels if K == 1 else 3 * K * latent_channels
        self.net = nn.Sequential(nn.Conv2d(cin, 640, kernel_size=1), nn.LeakyReLU(),
                                 nn.Conv2d(640, 640, kernel_size=1), nn.LeakyReLU(),
                                 nn.Conv2d(640, cout, kernel_size=1))
        self.precision = None
        self._ops = [engine.ConvOp(self.net[0], EPI_LRELU), engine.ConvOp(self.net[2], EPI_LRELU),
                     engine.ConvOp(self.net[4], EPI_BIAS)]

    @property
    def ops(self):
        return self._ops

    def raw(self, combined_feat: Tensor) -> Tensor:
        """The [B, 2M | 3KM, H, W] output of the 1x1 stack."""
        return engine.run_sequential_nchw(self._ops, combined_feat, engine.resolve_precision(self.precision))

    def forward(self, combined_feat: Tensor) -> Tuple[Tensor, ...]:
        from .EntropyModels import split_entropy_parameters
        return split_entropy_parameters(self.raw(combined_feat), self.latent_channels, self.K)
