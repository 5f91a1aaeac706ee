"""CPU oracle of ChannelCheckerboardHierarchical (TEST INFRASTRUCTURE, see oracle/__init__.py): the forward of oracle/forward.py with
y split into channel slices, each coded from the checkerboard context of oracle/checkerboard.py over the slice, a channel context
over the slices before it, and psi; the training gradients by torch autograd over it.

The space-channel context (ELIC, He et al., CVPR 2022) has no reference implementation in this repository to pin against, so this
restates the convention of DESIGN.md section 16 ("oracle restatement", unpinned): slice s covers the channels [o_s, o_s + m_s);
phi_sp = the checkerboard context of the slice (0 at the anchors); phi_ch = an unmasked 5x5 conv (bias, padding 2) over
y_in[:, :o_s] for s >= 1, not zeroed; raw_s = entropy_parameters.{s}(cat[phi_sp, phi_ch, psi])."""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from . import checkerboard as OC
from . import forward as O
from .backward import parameter_keys


def offsets(slices):
    return [sum(slices[:s]) for s in range(len(slices))]


def channel_context(sd, y_prev, s, dtype=torch.float32):
    """phi_ch of slice s >= 1 from the slices before it."""
    return F.conv2d(y_prev, O._p(sd, f"channel_contexts.{s - 1}.conv.weight", dtype), O._p(sd, f"channel_contexts.{s - 1}.conv.bias", dtype),
                    padding=2)


def slice_features(sd, y_in, psi, slices, s, dtype=torch.float32):
    """The input of slice s's 1x1 stack: [phi_sp | phi_ch | psi]."""
    o, m = offsets(slices)[s], slices[s]
    feats = [OC.context(sd, y_in[:, o:o + m], dtype, prefix=f"context_models.{s}")]
    if s > 0:
        feats.append(channel_context(sd, y_in[:, :o], s, dtype))
    return torch.cat(feats + [psi], dim=1)


def raw_parameters(sd, y_in, z_in, slices, dtype=torch.float32):
    """[raw_s]: the raw entropy parameters [B, (3K | 2) m_s, hy, wy] of every slice, from symbols y_in / z_in."""
    psi = O.hyper_synthesis(sd, z_in.to(O.DEVICE, dtype), dtype)
    y_in = y_in.to(O.DEVICE, dtype)
    return [O.entropy_parameters_raw(sd, slice_features(sd, y_in, psi, slices, s, dtype), dtype, prefix=f"entropy_parameters.{s}")
            for s in range(len(slices))]


def forward(sd, x, M: int, K: int, slices, training: bool = False, noise_z=None, noise_y=None, dtype=torch.float32):
    """ChannelCheckerboardHierarchical.forward: p_y and the mixture parameters over all M channels in channel order."""
    x = x.to(O.DEVICE, dtype)
    y = O.analysis(sd, x, dtype)
    z = O.hyper_analysis(sd, y, dtype)
    if training:
        z_in, y_in = z + noise_z.to(O.DEVICE, dtype), y + noise_y.to(O.DEVICE, dtype)
    else:
        z_in, y_in = torch.round(z), torch.round(y)
    raws = raw_parameters(sd, y_in, z_in, slices, dtype)
    p_ys, params = [], []
    for o, m, raw in zip(offsets(slices), slices, raws):
        prm = O.split_parameters(raw, m, K)
        p_ys.append(O.conditional_likelihood(y_in[:, o:o + m], prm, K))
        params.append(prm)
    p_y = torch.cat(p_ys, dim=1)
    p_z = O.factorized_likelihood(sd, z_in, dtype)
    out = {"x_hat": O.synthesis(sd, y_in, dtype), "y": y, "y_in": y_in, "z": z, "z_in": z_in, "p_z": p_z, "logp_z": torch.log(p_z),
           "p_y": p_y, "logp_y": torch.log(p_y), "training": training, "_raw": raws}
    names = ("mu", "sigma") if K == 1 else ("weights", "mus", "sigmas")
    for i, name in enumerate(names):
        out[name] = torch.cat([prm[i] for prm in params], dim=1 if K == 1 else 2)
    return out


def loss_and_grads(sd, x, M: int, K: int, slices, noise_z, noise_y, lambda_rd: float, distortion: str = "mse", dtype=torch.float32):
    """Autograd over `forward` + rd_loss (distortion "mse") or the MS-SSIM loss ("ms-ssim").  Returns (loss as a float,
    {param key: dLoss/dparam})."""
    from .metrics import ms_ssim
    keys = set(parameter_keys(sd))
    leaves = {k: (v.detach().to("cpu", dtype).clone().requires_grad_(True) if k in keys else v.detach().clone()) for k, v in sd.items()}
    prev = O.DIFFERENTIABLE
    O.DIFFERENTIABLE = True
    try:
        out = forward(leaves, x, M, K, slices, training=True, noise_z=noise_z, noise_y=noise_y, dtype=dtype)
        if distortion == "mse":
            loss = O.rd_loss(out, x, lambda_rd)["loss"]
        else:
            bits = (-torch.sum(out["logp_y"], dim=(1, 2, 3)) - torch.sum(out["logp_z"], dim=(1, 2, 3))) / math.log(2.0)
            loss = (bits / (x.size(2) * x.size(3))).mean() + lambda_rd * (1 - ms_ssim(out["x_hat"], x.to(out["x_hat"].dtype)))
        loss.backward()
    finally:
        O.DIFFERENTIABLE = prev
    return float(loss.detach()), {k: leaves[k].grad.detach() for k in keys if leaves[k].grad is not None}


def kink_margin(sd, x, M: int, K: int, slices, noise_z, noise_y) -> float:
    """oracle/backward.py's kink_margin for this model: the smallest |pre-activation| of the step's LeakyReLU layers (h_a, h_s and
    every slice's entropy-parameter stack), in float64."""
    dt = torch.float64
    P = lambda k: O._p(sd, k, dt)                  # noqa: E731
    y = O.analysis(sd, x.to("cpu", dt), dt)
    margins = []

    def act(h):
        margins.append(float(h.abs().min()))
        return F.leaky_relu(h, 0.01)
    h = act(F.conv2d(y, P("hyper_encoder.net.0.weight"), P("hyper_encoder.net.0.bias"), padding=1))
    h = act(F.conv2d(h, P("hyper_encoder.net.2.weight"), P("hyper_encoder.net.2.bias"), stride=2, padding=2))
    z = F.conv2d(h, P("hyper_encoder.net.4.weight"), P("hyper_encoder.net.4.bias"), stride=2, padding=2)
    z_in, y_in = z + noise_z.to(dt), y + noise_y.to(dt)
    h = act(F.conv_transpose2d(z_in, P("hyper_decoder.net.0.weight"), P("hyper_decoder.net.0.bias"), stride=2, padding=2, output_padding=1))
    h = act(F.conv_transpose2d(h, P("hyper_decoder.net.2.weight"), P("hyper_decoder.net.2.bias"), stride=2, padding=2, output_padding=1))
    psi = F.conv2d(h, P("hyper_decoder.net.4.weight"), P("hyper_decoder.net.4.bias"), padding=1)
    for s in range(len(slices)):
        h = act(F.conv2d(slice_features(sd, y_in, psi, slices, s, dt), P(f"entropy_parameters.{s}.net.0.weight"),
                         P(f"entropy_parameters.{s}.net.0.bias")))
        act(F.conv2d(h, P(f"entropy_parameters.{s}.net.2.weight"), P(f"entropy_parameters.{s}.net.2.bias")))
    return min(margins)


def noise_with_margin(sd, x, M: int, K: int, slices, first_seed: int, margin: float = 1e-6, tries: int = 64):
    """oracle/backward.py's noise_with_margin with this model's kink_margin."""
    B, _, H, W = x.shape
    for seed in range(first_seed, first_seed + tries):
        torch.manual_seed(seed)
        nz = torch.rand(B, M, H // 64, W // 64) - 0.5
        ny = torch.rand(B, M, H // 16, W // 16) - 0.5
        if kink_margin(sd, x, M, K, slices, nz, ny) >= margin:
            return seed, nz, ny
    raise RuntimeError("no noise draw with the requested LeakyReLU margin")
