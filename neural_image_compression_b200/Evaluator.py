"""``CompressionEvaluator`` of /root/reference/Evaluator.py:17-92 with the metrics computed on the device.

Same constructor, ``rgb_to_luma``, ``compute_metrics(orig, recon)`` key set and ``evaluate(rd_loss_fn)`` return value; the
plotting / report helpers of the reference (matplotlib, Evaluator.py:94-243) are outside the hot path.  ``compute_metrics``
takes the UNclamped reconstruction too (``clamp=True``: the kernels clamp on the fly, so ``x_hat.clamp(0, 1)`` is never
materialised); MS-SSIM restates ``pytorch_msssim.ms_ssim`` (absent third-party package: parity unpinned, see csrc/metrics.cu).

``evaluate`` keeps the reference's reporting quirk by default: its 'BPP' entry is the mean of bpp_y, not of bpp_total
(Evaluator.py:81); ``fix_bpp=True`` reports bpp_total there.
"""
from __future__ import annotations

import math
import os

import numpy as np
import torch

from . import _lib, engine
from ._lib import check, current_stream, ptr

MS_SSIM_WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)


def ms_ssim_levels(x: torch.Tensor, y: torch.Tensor, data_range: float = 1.0, clamp_y: bool = False,
                   workspace: torch.Tensor = None) -> torch.Tensor:
    """[5, planes, 2] = (mean ssim, mean cs) of every scale of the NCHW f32 planes of x and y (nic_ms_ssim_levels).  `workspace`
    (uint8, default: a fresh one) keeps the pooled pyramids, which nic_ms_ssim_bwd reads back."""
    lib = _lib.load()
    b, c, h, w = x.shape
    planes = b * c
    lev = torch.empty((5, planes, 2), dtype=torch.float32, device=x.device)
    ws = workspace if workspace is not None else torch.empty(lib.nic_ms_ssim_workspace_bytes(planes, h, w), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        check(lib.nic_ms_ssim_levels(ptr(x), ptr(y), planes, h, w, float(data_range), int(clamp_y), ptr(lev), ptr(ws), ws.numel(),
                                     current_stream()), "nic_ms_ssim_levels")
    return lev


_WEIGHTS = {}


def _weights(device) -> torch.Tensor:
    """The MS-SSIM weights on `device`, uploaded once: the training step's first (warm-up) call makes them, so a CUDA-graph
    capture of the step never copies from the host."""
    if device not in _WEIGHTS:
        _WEIGHTS[device] = torch.tensor(MS_SSIM_WEIGHTS, dtype=torch.float32, device=device)
    return _WEIGHTS[device]


def combine_levels(lev: torch.Tensor):
    """(terms [5, planes], value [planes]): the terms are the cs of scales 0-3 and the ssim of scale 4; the value of a plane is
    prod relu(term)^w (pytorch_msssim's per-channel MS-SSIM)."""
    wts = _weights(lev.device)
    terms = torch.cat([lev[:4, :, 1], lev[4:, :, 0]], dim=0)
    return terms, torch.prod(torch.relu(terms) ** wts.view(-1, 1), dim=0)


def term_grads(terms: torch.Tensor, value: torch.Tensor) -> torch.Tensor:
    """d value / d term [5, planes]: w_l value / term_l where term_l > 0, else 0 - the relu rule autograd applies to
    combine_levels (a channel with any term <= 0 has value 0 and no gradient at all)."""
    wts = _weights(terms.device).view(-1, 1)
    pos = terms > 0
    return torch.where(pos, wts * value / torch.where(pos, terms, torch.ones_like(terms)), torch.zeros_like(terms))


def ms_ssim(x: torch.Tensor, y: torch.Tensor, data_range: float = 1.0, size_average: bool = True, clamp_y: bool = False) -> torch.Tensor:
    """pytorch_msssim.ms_ssim(x, y, data_range, size_average) for NCHW f32 batches on the device (Evaluator.py:38, 45)."""
    engine.require_cuda(x, "x")
    x, y = x.contiguous().float(), y.contiguous().float()
    if x.shape != y.shape or x.dim() != 4:
        raise ValueError(f"Input images should have the same 4-d shape, got {tuple(x.shape)} and {tuple(y.shape)}")
    b, c, h, w = x.shape
    if min(h, w) <= (11 - 1) * 2 ** 4:
        raise AssertionError("Image size should be larger than 160 due to the 4 downsamplings in ms-ssim")
    _, val = combine_levels(ms_ssim_levels(x, y, data_range, clamp_y))
    val = val.view(b, c)
    return val.mean() if size_average else val.mean(1)


class CompressionEvaluator:
    def __init__(self, model, dataloader, device, lambda_val, save_dir="./eval_results"):
        self.model, self.dataloader, self.device, self.lambda_val = model, dataloader, device, lambda_val
        os.makedirs(save_dir, exist_ok=True)
        self.save_dir = save_dir

    @staticmethod
    def rgb_to_luma(x, clamp: bool = False):
        """[B, 3, H, W] in [0, 1] -> [B, H, W] (Evaluator.py:26-30)."""
        engine.require_cuda(x, "x")
        x = x.contiguous().float()
        b, _, h, w = x.shape
        y = torch.empty((b, h, w), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            check(_lib.load().nic_luma(ptr(x), ptr(y), b, h, w, int(clamp), current_stream()), "nic_luma")
        return y

    def compute_metrics(self, orig, recon, clamp: bool = False):
        """Evaluator.py:32-53.  orig, recon: [B, 3, H, W]; with clamp=True `recon` is clamped to [0, 1] inside the kernels."""
        lib = _lib.load()
        engine.require_cuda(orig, "orig")
        orig, recon = orig.contiguous().float(), recon.contiguous().float()
        b, _, h, w = orig.shape
        mse = torch.empty((b, 2), dtype=torch.float32, device=orig.device)
        parts = torch.empty((b, lib.nic_partials_per_image(), 2), dtype=torch.float32, device=orig.device)
        with torch.cuda.device(orig.device):
            check(lib.nic_eval_mse(ptr(orig), ptr(recon), b, h, w, int(clamp), ptr(mse), ptr(parts), current_stream()), "nic_eval_mse")
        msssim_rgb = ms_ssim(orig, recon, data_range=1.0, size_average=True, clamp_y=clamp)     # symmetric in its two images
        y_o = self.rgb_to_luma(orig).unsqueeze(1)
        y_r = self.rgb_to_luma(recon, clamp=clamp).unsqueeze(1)
        msssim_y = ms_ssim(y_r, y_o, data_range=1.0, size_average=True)
        m = mse.double().mean(0).tolist()                  # torch.mean over the whole batch (the reference evaluates one image at a time)
        mse_rgb, mse_y = m[0], m[1]
        return {
            "MSE(255)": mse_rgb * (255 ** 2),
            "PSNR(RGB)": 10 * np.log10(1.0 / mse_rgb) if mse_rgb > 0 else float("inf"),
            "MS-SSIM(RGB)": float(msssim_rgb),
            "PSNR(Y)": 10 * np.log10(1.0 / mse_y) if mse_y > 0 else float("inf"),
            "MS-SSIM(Y)": float(msssim_y),
        }

    def evaluate(self, rd_loss_fn, fix_bpp: bool = False):
        """Evaluator.py:55-92: model(imgs, training=False) + rd_loss + compute_metrics over the loader; returns
        (avg_metrics, imgs_list, recon_list).  'BPP' is the mean of bpp_y as in the reference (:81) unless fix_bpp."""
        self.model.eval()
        total_metrics, bpp_t, bpp_y, bpp_z, imgs_list, recon_list = [], [], [], [], [], []
        with torch.no_grad():
            for imgs in self.dataloader:
                imgs = imgs.to(self.device)
                out = self.model(imgs, training=False)
                results = rd_loss_fn(out, imgs, self.lambda_val)
                bpp_t.append(results["bpp_total"]); bpp_y.append(results["bpp_y"]); bpp_z.append(results["bpp_z"])
                total_metrics.append(self.compute_metrics(imgs, out["x_hat"], clamp=True))
                imgs_list.append(imgs[0].cpu())
                recon_list.append(out["x_hat"][0].cpu().clamp(0, 1))
        avg = {k: np.mean([m[k] for m in total_metrics]) for k in total_metrics[0]}
        avg["BPP"] = float(np.mean(bpp_t if fix_bpp else bpp_y))
        avg["BPP(y)"] = float(np.mean(bpp_y))
        avg["BPP(z)"] = float(np.mean(bpp_z))
        return avg, imgs_list, recon_list
