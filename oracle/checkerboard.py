"""CPU oracle of JointCheckerboardHierarchical (TEST INFRASTRUCTURE, see oracle/__init__.py): the forward of oracle/forward.py with
the checkerboard context model, and the training gradients by torch autograd over it, as oracle/backward.py does for the mask-'A'
model.

The checkerboard context (He et al., CVPR 2021) has no reference implementation to pin against, so this restates the convention of
DESIGN.md section 14 ("oracle restatement", unpinned): the 5x5 context conv keeps the taps with kh + kw odd (the weight is masked as
the reference masks mask 'A': in place, so the gradient reaches all 25 taps), and its output phi, bias included, is then set to 0
at the anchors (i + j even), before torch.cat([phi, psi]) enters the entropy-parameter stack."""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from . import forward as O
from .backward import kink_margin as kink_margin_mask_a
from .backward import parameter_keys


def checkerboard_mask(weight):
    """1 at the taps (kh, kw) with kh + kw odd."""
    kh, kw = weight.shape[-2:]
    parity = (torch.arange(kh)[:, None] + torch.arange(kw)[None, :]) % 2
    return parity.to(weight.dtype).expand_as(weight).clone()


def anchors(h, w):
    """bool [h, w]: True at the anchors (i + j even)."""
    return (torch.arange(h)[:, None] + torch.arange(w)[None, :]) % 2 == 0


def context(sd, y_in, dtype=torch.float32, prefix="context_model"):
    """The checkerboard context model: masked 5x5 conv (12 live taps), then phi = 0 at the anchors."""
    w = O._p(sd, f"{prefix}.masked.weight", dtype)
    mask = checkerboard_mask(w)
    w = (w.detach() * mask - w.detach()) + w if O.DIFFERENTIABLE else w * mask
    phi = F.conv2d(y_in, w, O._p(sd, f"{prefix}.masked.bias", dtype), padding=2)
    keep = (~anchors(*y_in.shape[2:])).to(phi.device, phi.dtype)
    return phi * keep


def raw_parameters(sd, y_in, z_in, dtype=torch.float32):
    """The raw entropy parameters [B, (3K | 2) M, hy, wy] of symbols y_in / z_in."""
    psi = O.hyper_synthesis(sd, z_in.to(O.DEVICE, dtype), dtype)
    return O.entropy_parameters_raw(sd, torch.cat([context(sd, y_in.to(O.DEVICE, dtype), dtype), psi], dim=1), dtype)


def forward(sd, x, M: int, K: int, training: bool = False, noise_z=None, noise_y=None, dtype=torch.float32):
    """JointCheckerboardHierarchical.forward: oracle.forward.forward with the checkerboard context."""
    x = x.to(O.DEVICE, dtype)
    y = O.analysis(sd, x, dtype)
    z = O.hyper_analysis(sd, y, dtype)
    if training:
        z_in, y_in = z + noise_z.to(O.DEVICE, dtype), y + noise_y.to(O.DEVICE, dtype)
    else:
        z_in, y_in = torch.round(z), torch.round(y)
    psi = O.hyper_synthesis(sd, z_in, dtype)
    phi = context(sd, y_in, dtype)
    raw = O.entropy_parameters_raw(sd, torch.cat([phi, psi], dim=1), dtype)
    params = O.split_parameters(raw, M, K)
    p_z = O.factorized_likelihood(sd, z_in, dtype)
    p_y = O.conditional_likelihood(y_in, params, K)
    out = {"x_hat": O.synthesis(sd, y_in, dtype), "y": y, "y_in": y_in, "z": z, "z_in": z_in, "p_z": p_z, "logp_z": torch.log(p_z),
           "p_y": p_y, "logp_y": torch.log(p_y), "training": training, "_psi": psi, "_phi": phi, "_raw": raw}
    if K == 1:
        out["mu"], out["sigma"] = params
    else:
        out["weights"], out["mus"], out["sigmas"] = params
    return out


def loss_and_grads(sd, x, M: int, K: int, noise_z, noise_y, lambda_rd: float, distortion: str = "mse", dtype=torch.float32):
    """Autograd over `forward` + rd_loss (distortion "mse") or the MS-SSIM loss of oracle/backward_ms_ssim.py ("ms-ssim").
    Returns (loss as a float, {param key: dLoss/dparam})."""
    from .metrics import ms_ssim
    keys = set(parameter_keys(sd))
    leaves = {k: (v.detach().to("cpu", dtype).clone().requires_grad_(True) if k in keys else v.detach().clone()) for k, v in sd.items()}
    prev = O.DIFFERENTIABLE
    O.DIFFERENTIABLE = True
    try:
        out = forward(leaves, x, M, K, training=True, noise_z=noise_z, noise_y=noise_y, dtype=dtype)
        if distortion == "mse":
            loss = O.rd_loss(out, x, lambda_rd)["loss"]
        else:
            bits = (-torch.sum(out["logp_y"], dim=(1, 2, 3)) - torch.sum(out["logp_z"], dim=(1, 2, 3))) / math.log(2.0)
            loss = (bits / (x.size(2) * x.size(3))).mean() + lambda_rd * (1 - ms_ssim(out["x_hat"], x.to(out["x_hat"].dtype)))
        loss.backward()
    finally:
        O.DIFFERENTIABLE = prev
    return float(loss.detach()), {k: leaves[k].grad.detach() for k in keys if leaves[k].grad is not None}


def kink_margin(sd, x, M: int, K: int, noise_z, noise_y) -> float:
    """oracle/backward.py's kink_margin for this model: the smallest |pre-activation| of the step's LeakyReLU layers, in float64,
    with the entropy-parameter layers evaluated on the checkerboard context (the mask-'A' figure is kept too: it covers h_a and h_s)."""
    dt = torch.float64
    y = O.analysis(sd, x.to("cpu", dt), dt)
    z = O.hyper_analysis(sd, y, dt)
    y_in, z_in = y + noise_y.to(dt), z + noise_z.to(dt)
    h = torch.cat([context(sd, y_in, dt), O.hyper_synthesis(sd, z_in, dt)], dim=1)
    pre0 = F.conv2d(h, O._p(sd, "entropy_parameters.net.0.weight", dt), O._p(sd, "entropy_parameters.net.0.bias", dt))
    pre1 = F.conv2d(F.leaky_relu(pre0, 0.01), O._p(sd, "entropy_parameters.net.2.weight", dt), O._p(sd, "entropy_parameters.net.2.bias", dt))
    return min(kink_margin_mask_a(sd, x, M, K, noise_z, noise_y), float(pre0.abs().min()), float(pre1.abs().min()))


def noise_with_margin(sd, x, M: int, K: int, first_seed: int, margin: float = 1e-6, tries: int = 64):
    """oracle/backward.py's noise_with_margin with this model's kink_margin."""
    B, _, H, W = x.shape
    for seed in range(first_seed, first_seed + tries):
        torch.manual_seed(seed)
        nz = torch.rand(B, M, H // 64, W // 64) - 0.5
        ny = torch.rand(B, M, H // 16, W // 16) - 0.5
        if kink_margin(sd, x, M, K, nz, ny) >= margin:
            return seed, nz, ny
    raise RuntimeError("no noise draw with the requested LeakyReLU margin")
