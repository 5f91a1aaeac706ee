"""``rd_loss`` of /root/reference/RateDistortionLoss.py:5-49 on the device.

Same signature and key set.  The per-image sums of log-likelihoods come from the partial sums the
likelihood kernels already produced (or from ``nic_sum_fwd`` when the dict was not produced by this
package), the squared error from ``nic_sse_fwd``, and ``nic_rd_finalize`` folds them into every term
in one launch; the seven Python floats cost one device-to-host copy instead of the reference's eight
``.item()`` synchronisations (:38-47).
"""
from __future__ import annotations

import torch

from . import _lib, engine
from ._lib import check, current_stream, ptr


def _check_pipeline():
    """The tensor-core kernels bound every barrier wait and raise a device flag instead of hanging; this is the natural place to
    look at it: the loss has just synchronised with the device anyway.  An aborted kernel means the outputs above are garbage."""
    if _lib.load().nic_pipeline_status() != 0:
        raise _lib.NicError("a tensor-core kernel gave up on an expired pipeline wait (nic_pipeline_status): the results of this "
                            "forward pass are invalid")


def _logp_partials(logp: torch.Tensor) -> torch.Tensor:
    parts = getattr(logp, "_nic_partials", None)
    if parts is not None and getattr(logp, "_nic_partials_version", None) == logp._version:
        return parts                                       # the sums the likelihood kernel produced alongside logp (still valid: logp unmodified)
    lib = _lib.load()
    b = logp.shape[0]
    logp = logp.contiguous().float()
    parts = engine.partials(b, logp.device)
    check(lib.nic_sum_fwd(ptr(logp), b, logp[0].numel(), ptr(parts), current_stream()), "nic_sum_fwd")
    return parts


def rd_terms(model_out: dict, x: torch.Tensor, lambda_rd: float):
    """Device-resident terms: (per_image [3, B]: bits_y, bits_z, mse; scalars [8]), no host sync."""
    lib = _lib.load()
    x_hat = model_out["x_hat"]
    engine.require_cuda(x_hat, "x_hat")
    x = x.to(x_hat.device).contiguous().float()
    x_hat = x_hat.contiguous().float()
    b = x.size(0)
    chw = x[0].numel()
    with torch.cuda.device(x_hat.device):
        py = _logp_partials(model_out["logp_y"])
        pz = _logp_partials(model_out["logp_z"])
        se = engine.partials(b, x_hat.device)
        check(lib.nic_sse_fwd(ptr(x_hat), ptr(x), b, chw, ptr(se), current_stream()), "nic_sse_fwd")
        per_image = torch.empty((3, b), dtype=torch.float32, device=x_hat.device)
        scalars = torch.empty(8, dtype=torch.float32, device=x_hat.device)
        check(lib.nic_rd_finalize(ptr(py), ptr(pz), ptr(se), b, x.size(2) * x.size(3), chw, float(lambda_rd),
                                  ptr(per_image), ptr(scalars), current_stream()), "nic_rd_finalize")
    return per_image, scalars


def rd_loss_device(model_out: dict, x: torch.Tensor, lambda_rd: float):
    """(loss, per_image [3, B], scalars [8]) without touching the host: `loss` is differentiable when the model output is
    (Trainer.py:85 calls results['loss'].backward(): one autograd node over logp_y, logp_z, x_hat).  CUDA-graph safe."""
    with torch.no_grad():
        per_image, scalars = rd_terms(model_out, x, lambda_rd)
    loss = scalars[5]
    diff = [model_out[k] for k in ("logp_y", "logp_z", "x_hat")]
    if torch.is_grad_enabled() and any(t.requires_grad for t in diff):
        from .training import _RDLoss
        xd = x.to(diff[2].device).contiguous().float()
        loss = _RDLoss.apply(diff[0], diff[1], diff[2].contiguous().float(), xd, float(lambda_rd), scalars)
    return loss, per_image, scalars


def rd_loss(model_out: dict, x: torch.Tensor, lambda_rd: float):
    loss, per_image, scalars = rd_loss_device(model_out, x, lambda_rd)
    s = scalars.tolist()                                   # the one host synchronisation
    _check_pipeline()
    mse_per_image = per_image[2]
    return {
        "loss": loss,
        "bpp_y": s[0], "bpp_z": s[1], "bpp_total": s[2], "mse": s[3], "psnr": s[4],
        "mse_per_image": mse_per_image,
        "psnr_per_image": -10 * torch.log10(mse_per_image + 1e-8),
        "bits_y": s[6], "bits_z": s[7], "bits_total": s[6] + s[7],
    }


MS_SSIM_MIN_SIDE = (11 - 1) * 2 ** 4        # five scales of an 11-tap VALID window: the smaller side must exceed 160


def check_ms_ssim_shape(shape):
    """ValueError (before any launch) for images whose smaller side is 160 pixels or less."""
    if len(shape) != 4 or min(shape[2], shape[3]) <= MS_SSIM_MIN_SIDE:
        raise ValueError(f"the MS-SSIM loss needs NCHW images whose smaller side exceeds {MS_SSIM_MIN_SIDE} pixels, got {tuple(shape)}")


def ms_ssim_terms(model_out: dict, x: torch.Tensor, lambda_rd: float):
    """Device-resident terms of the MS-SSIM loss, no host sync: (per_image [3, B], scalars [9], ms_ssim_per_image [B], state).
    scalars = nic_rd_finalize's 8 with entry 5 replaced by loss = bpp_total + lambda * (1 - mean_b ms_ssim_b), then the batch
    MS-SSIM.  x_hat is not clamped.  state = (x_hat, x, terms, value, workspace): what ms_ssim_x_hat_grad reads."""
    from .Evaluator import combine_levels, ms_ssim_levels
    check_ms_ssim_shape(tuple(model_out["x_hat"].shape))
    per_image, scalars = rd_terms(model_out, x, lambda_rd)
    x_hat = model_out["x_hat"].detach().contiguous().float()
    x = x.to(x_hat.device).contiguous().float()
    b, c, h, w = x.shape
    ws = torch.empty(_lib.load().nic_ms_ssim_bwd_workspace_bytes(b * c, h, w), dtype=torch.uint8, device=x.device)
    terms, value = combine_levels(ms_ssim_levels(x_hat, x, 1.0, False, workspace=ws))
    per_img = value.view(b, c).mean(1)
    ms = per_img.mean()
    loss = scalars[2] + float(lambda_rd) * (1.0 - ms)
    scalars = torch.cat([scalars[:5], loss.view(1), scalars[6:], ms.view(1)])
    return per_image, scalars, per_img, (x_hat, x, terms, value, ws)


def ms_ssim_rd_loss(model_out: dict, x: torch.Tensor, lambda_rd: float):
    """CompressAI's RateDistortionLoss(metric="ms-ssim"): loss = bpp_total + lambda * (1 - ms_ssim(x_hat, x, data_range=1)), the
    MS-SSIM of pytorch_msssim averaged over the batch, x_hat unclamped.  rd_loss's keys ('mse' / 'psnr' still reported) plus
    'ms_ssim' (float) and 'ms_ssim_per_image' (device tensor [B]); one host synchronisation.  'loss' is differentiable when the
    model output is (training._MSSSIMRDLoss: nic_ms_ssim_bwd for x_hat, the rate gradient for logp_y / logp_z)."""
    with torch.no_grad():
        per_image, scalars, per_img, state = ms_ssim_terms(model_out, x, lambda_rd)
    loss = scalars[5]
    diff = [model_out[k] for k in ("logp_y", "logp_z", "x_hat")]
    if torch.is_grad_enabled() and any(t.requires_grad for t in diff):
        from .training import _MSSSIMRDLoss
        loss = _MSSSIMRDLoss.apply(diff[0], diff[1], diff[2], float(lambda_rd), scalars, state)
    s = scalars.tolist()                                   # the one host synchronisation
    _check_pipeline()
    mse_per_image = per_image[2]
    return {
        "loss": loss,
        "bpp_y": s[0], "bpp_z": s[1], "bpp_total": s[2], "mse": s[3], "psnr": s[4],
        "mse_per_image": mse_per_image,
        "psnr_per_image": -10 * torch.log10(mse_per_image + 1e-8),
        "bits_y": s[6], "bits_z": s[7], "bits_total": s[6] + s[7],
        "ms_ssim": s[8], "ms_ssim_per_image": per_img,
    }


def vision_rd_loss(model_out: dict, x: torch.Tensor, lambda_rd: float, gamma: float = 0.0, frozen_activation=None, V=None):
    """``vision_rd_loss`` of /root/reference/RateDistortionLoss.py:52-121 for ScalableImageCoding outputs: rate terms of the
    two latent parts and of z, reconstruction MSE / PSNR, ``loss = bpp_total + lambda_rd * mse`` (:98, no 255^2 here).
    The feature-space term (:89-95) needs a frozen third-party detector and the latent-space transform, neither of which
    is on this path: ``frozen_activation`` / ``V`` must be None and 'vision_mse' is 0.0, as in the reference's own
    ``V is None`` branch."""
    if frozen_activation is not None or V is not None:
        raise NotImplementedError("the feature-space distortion term (frozen detector + LST) is outside the hot path")
    lib = _lib.load()
    x_hat = model_out["x_hat"]
    engine.require_cuda(x_hat, "x_hat")
    x = x.to(x_hat.device).contiguous().float()
    x_hat = x_hat.contiguous().float()
    b, chw, npix = x.size(0), x[0].numel(), x.size(2) * x.size(3)
    with torch.cuda.device(x_hat.device):
        p1, p2, pz = (_logp_partials(model_out[k]) for k in ("logp_y1", "logp_y2", "logp_z"))
        se = engine.partials(b, x_hat.device)
        check(lib.nic_sse_fwd(ptr(x_hat), ptr(x), b, chw, ptr(se), current_stream()), "nic_sse_fwd")
        rows, scal = [], []
        for py in (p1, p2):                      # the same fold as rd_loss, once per latent part (bits_z / mse repeat)
            per_image = torch.empty((3, b), dtype=torch.float32, device=x_hat.device)
            scalars = torch.empty(8, dtype=torch.float32, device=x_hat.device)
            check(lib.nic_rd_finalize(ptr(py), ptr(pz), ptr(se), b, npix, chw, 0.0, ptr(per_image), ptr(scalars),
                                      current_stream()), "nic_rd_finalize")
            rows.append(per_image); scal.append(scalars)
    s1, s2 = scal[0].tolist(), scal[1].tolist()
    _check_pipeline()
    bpp_y1, bpp_y2, bpp_z, mse, psnr = s1[0], s2[0], s1[1], s1[3], s1[4]
    bpp_total = bpp_y1 + bpp_y2 + bpp_z
    mse_per_image = rows[0][2]
    bits_y1, bits_y2, bits_z = s1[6], s2[6], s1[7]
    loss = scal[0][0] + scal[1][0] + scal[0][1] + lambda_rd * scal[0][3]
    diff = [model_out[k] for k in ("logp_y1", "logp_y2", "logp_z", "x_hat")]
    if torch.is_grad_enabled() and any(t.requires_grad for t in diff):
        from .training_scalable import _VisionRDLoss          # the loss as one autograd node (the trainer calls loss.backward())
        loss = _VisionRDLoss.apply(diff[0], diff[1], diff[2], diff[3].contiguous().float(), x, float(lambda_rd), loss)
    return {
        "loss": loss,
        "bpp_y1": bpp_y1, "bpp_y2": bpp_y2, "bpp_y": bpp_y1 + bpp_y2, "bpp_z": bpp_z, "bpp_total": bpp_total,
        "mse": mse, "reconstruction_mse": mse, "psnr": psnr, "vision_mse": 0.0,
        "mse_per_image": mse_per_image, "reconstruction_mse_per_image": mse_per_image,
        "psnr_per_image": -10 * torch.log10(mse_per_image + 1e-8), "vision_mse_per_image": 0.0,
        "bits_y1": bits_y1, "bits_y2": bits_y2, "bits_y": bits_y1 + bits_y2, "bits_z": bits_z,
        "bits_total": bits_y1 + bits_y2 + bits_z,
    }
