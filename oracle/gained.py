"""CPU oracle of GainedCheckerboardHierarchical (TEST INFRASTRUCTURE, see oracle/__init__.py): oracle/checkerboard.py's forward with
the gain units of DESIGN.md section 15, and the training gradients by torch autograd over it.  Unpinned, as section 14's restatement:
gain units have no reference implementation here.

For image b at quality q_b (snapped to round(1024 q) / 1024): l = floor(q), t = q - l, each gain is
exp((1 - t) log[l] + t log[min(l + 1, L - 1)]).  y = g_y * g_a(x) and z = g_z * h_a(y) are quantised (or noised); the context model,
the entropy parameters and the likelihoods read the symbols, g_s reads ginv_y * y_in and h_s reads ginv_z * z_in."""
from __future__ import annotations

import math

import torch

from . import checkerboard as OC
from . import forward as O
from .backward import parameter_keys

TABLES = ("y_log_gain", "y_log_inv_gain", "z_log_gain", "z_log_inv_gain")


def snap(quality, levels: int, B: int):
    """quality (float or B values) -> q_code int64 [B] = floor(1024 q + 0.5)."""
    q = torch.as_tensor(quality, dtype=torch.float64).reshape(-1).expand(B)
    return torch.clamp(torch.floor(q * 1024 + 0.5), 0, 1024 * (levels - 1)).long()


def gains(sd, q_code, dtype=torch.float32):
    """{table name: [B, M] gain vectors} of the quality codes."""
    out = {}
    for name in TABLES:
        tab = O._p(sd, f"gain_units.{name}", dtype)
        L = tab.shape[0]
        l0 = torch.div(q_code, 1024, rounding_mode="floor").clamp(0, L - 1)
        l1 = (l0 + 1).clamp(max=L - 1)
        t = ((q_code - 1024 * l0).to(dtype) / 1024)[:, None]
        out[name] = torch.exp((1 - t) * tab[l0] + t * tab[l1])
    return out


def _bc(v):
    return v[:, :, None, None]


def forward(sd, x, M: int, K: int, quality, training: bool = False, noise_z=None, noise_y=None, dtype=torch.float32):
    """GainedCheckerboardHierarchical.forward at `quality` (a float or one value per image)."""
    x = x.to(O.DEVICE, dtype)
    L = sd["gain_units.y_log_gain"].shape[0]
    q_code = snap(quality, L, x.shape[0])
    g = gains(sd, q_code, dtype)
    y = _bc(g["y_log_gain"]) * O.analysis(sd, x, dtype)
    z = _bc(g["z_log_gain"]) * O.hyper_analysis(sd, y, dtype)
    if training:
        z_in, y_in = z + noise_z.to(O.DEVICE, dtype), y + noise_y.to(O.DEVICE, dtype)
    else:
        z_in, y_in = torch.round(z), torch.round(y)
    psi = O.hyper_synthesis(sd, _bc(g["z_log_inv_gain"]) * z_in, dtype)
    phi = OC.context(sd, y_in, dtype)
    raw = O.entropy_parameters_raw(sd, torch.cat([phi, psi], dim=1), dtype)
    params = O.split_parameters(raw, M, K)
    p_z = O.factorized_likelihood(sd, z_in, dtype)
    p_y = O.conditional_likelihood(y_in, params, K)
    out = {"x_hat": O.synthesis(sd, _bc(g["y_log_inv_gain"]) * y_in, dtype), "y": y, "y_in": y_in, "z": z, "z_in": z_in, "p_z": p_z,
           "logp_z": torch.log(p_z), "p_y": p_y, "logp_y": torch.log(p_y), "training": training, "quality": q_code.to(dtype) / 1024,
           "_psi": psi, "_raw": raw}
    if K == 1:
        out["mu"], out["sigma"] = params
    else:
        out["weights"], out["mus"], out["sigmas"] = params
    return out


def loss_and_grads(sd, x, M: int, K: int, quality, noise_z, noise_y, lambdas, distortion: str = "mse", dtype=torch.float32):
    """Autograd over `forward` + the loss with per-image lambdas (a float or B values): bpp_total + mean_b(lambda_b 255^2 mse_b), or
    for "ms-ssim" bpp_total + mean_b(lambda_b (1 - ms_ssim_b)).  Returns (loss as a float, {param key: dLoss/dparam})."""
    from .metrics import ms_ssim
    B = x.shape[0]
    lam = torch.as_tensor(lambdas, dtype=dtype).reshape(-1).expand(B)
    keys = set(parameter_keys(sd))
    leaves = {k: (v.detach().to("cpu", dtype).clone().requires_grad_(True) if k in keys else v.detach().clone()) for k, v in sd.items()}
    prev = O.DIFFERENTIABLE
    O.DIFFERENTIABLE = True
    try:
        out = forward(leaves, x, M, K, quality, training=True, noise_z=noise_z, noise_y=noise_y, dtype=dtype)
        bits = (-torch.sum(out["logp_y"], dim=(1, 2, 3)) - torch.sum(out["logp_z"], dim=(1, 2, 3))) / math.log(2.0)
        bpp = (bits / (x.size(2) * x.size(3))).mean()
        xd = x.to(out["x_hat"].dtype)
        if distortion == "mse":
            mse = ((out["x_hat"] - xd) ** 2).mean(dim=(1, 2, 3))
            loss = bpp + (lam * 255 ** 2 * mse).mean()
        else:
            ms = torch.stack([ms_ssim(out["x_hat"][b:b + 1], xd[b:b + 1]) for b in range(B)])
            loss = bpp + (lam * (1 - ms)).mean()
        loss.backward()
    finally:
        O.DIFFERENTIABLE = prev
    return float(loss.detach()), {k: leaves[k].grad.detach() for k in keys if leaves[k].grad is not None}


def kink_margin(sd, x, M: int, K: int, quality, noise_z, noise_y) -> float:
    """oracle/backward.py's kink_margin for this model at `quality`: the smallest |pre-activation| of the step's six LeakyReLU layers
    (h_a 0/2, h_s 0/2, entropy parameters 0/2) in float64, with the gains where the forward applies them."""
    import torch.nn.functional as F
    dt = torch.float64
    P = lambda k: sd[k].detach().to("cpu", dt)     # noqa: E731
    g = gains(sd, snap(quality, sd["gain_units.y_log_gain"].shape[0], x.shape[0]), dt)
    y = _bc(g["y_log_gain"]) * O.analysis(sd, x.to("cpu", dt), dt)
    margins = []

    def act(h):
        margins.append(float(h.abs().min()))
        return F.leaky_relu(h, 0.01)
    h = act(F.conv2d(y, P("hyper_encoder.net.0.weight"), P("hyper_encoder.net.0.bias"), padding=1))
    h = act(F.conv2d(h, P("hyper_encoder.net.2.weight"), P("hyper_encoder.net.2.bias"), stride=2, padding=2))
    z = _bc(g["z_log_gain"]) * F.conv2d(h, P("hyper_encoder.net.4.weight"), P("hyper_encoder.net.4.bias"), stride=2, padding=2)
    z_in, y_in = z + noise_z.to(dt), y + noise_y.to(dt)
    h = act(F.conv_transpose2d(_bc(g["z_log_inv_gain"]) * z_in, P("hyper_decoder.net.0.weight"), P("hyper_decoder.net.0.bias"), stride=2,
                               padding=2, output_padding=1))
    h = act(F.conv_transpose2d(h, P("hyper_decoder.net.2.weight"), P("hyper_decoder.net.2.bias"), stride=2, padding=2, output_padding=1))
    psi = F.conv2d(h, P("hyper_decoder.net.4.weight"), P("hyper_decoder.net.4.bias"), padding=1)
    h = act(F.conv2d(torch.cat([OC.context(sd, y_in, dt), psi], dim=1), P("entropy_parameters.net.0.weight"),
                     P("entropy_parameters.net.0.bias")))
    act(F.conv2d(h, P("entropy_parameters.net.2.weight"), P("entropy_parameters.net.2.bias")))
    return min(margins)


def noise_with_margin(sd, x, M: int, K: int, quality, first_seed: int, margin: float = 1e-6, tries: int = 64):
    """oracle/backward.py's noise_with_margin with this model's kink_margin."""
    B, _, H, W = x.shape
    for seed in range(first_seed, first_seed + tries):
        torch.manual_seed(seed)
        nz = torch.rand(B, M, H // 64, W // 64) - 0.5
        ny = torch.rand(B, M, H // 16, W // 16) - 0.5
        if kink_margin(sd, x, M, K, quality, nz, ny) >= margin:
            return seed, nz, ny
    raise RuntimeError("no noise draw with the requested LeakyReLU margin")
