"""CPU oracle of the MS-SSIM training loss (TEST INFRASTRUCTURE, see oracle/__init__.py): torch autograd over the restated forward
(oracle/forward.py), rd_loss's rate and oracle.metrics.ms_ssim, the same construction as oracle/backward.py's MSE oracles."""
from __future__ import annotations

import math

import torch

from . import forward as O
from .backward import parameter_keys
from .metrics import ms_ssim


def loss_and_grads_ms_ssim(sd, x, M: int, K: int, noise_z: torch.Tensor, noise_y: torch.Tensor, lambda_rd: float, residual: bool = False,
                           dtype=torch.float32):
    """The MS-SSIM loss of CompressAI's RateDistortionLoss(metric="ms-ssim"): autograd over forward (or forward_residual) +
    rd_loss's rate + ms_ssim, loss = bpp_total + lambda * (1 - ms_ssim(x_hat, x)) with x_hat unclamped.
    Returns (rd dict with 'loss' and 'ms_ssim' as floats, grads)."""
    keys = set(parameter_keys(sd))
    leaves = {k: (v.detach().to("cpu", dtype).clone().requires_grad_(True) if k in keys else v.detach().clone()) for k, v in sd.items()}
    prev = O.DIFFERENTIABLE
    O.DIFFERENTIABLE = True
    try:
        fwd = O.forward_residual if residual else O.forward
        out = fwd(leaves, x, M, K, training=True, noise_z=noise_z, noise_y=noise_y, dtype=dtype)
        rd = dict(O.rd_loss(out, x, lambda_rd))
        ms = ms_ssim(out["x_hat"], x.to(out["x_hat"].dtype))
        bits = (-torch.sum(out["logp_y"], dim=(1, 2, 3)) - torch.sum(out["logp_z"], dim=(1, 2, 3))) / math.log(2.0)
        loss = (bits / (x.size(2) * x.size(3))).mean() + lambda_rd * (1 - ms)
        loss.backward()
    finally:
        O.DIFFERENTIABLE = prev
    grads = {k: leaves[k].grad.detach() for k in keys if leaves[k].grad is not None}
    rd["loss"], rd["ms_ssim"] = float(loss.detach()), float(ms.detach())
    return rd, grads
