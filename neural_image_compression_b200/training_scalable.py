"""Training step of ``ScalableImageCoding`` (reference Models.py:208-338 with the repairs of SURVEY.md section 2.4, loss
``vision_rd_loss`` of RateDistortionLoss.py:52-121 with V = None): forward with noise, loss, hand-written backward.

The forward and the backward are training.py's (``_forward_impl`` / ``_backward_impl`` over ``training.heads``): the model's base
head (M1 channels of y) and enhancement head (M - M1), each a (context model, entropy-parameter net) over the SHARED hyper features
psi, so the psi gradient is the sum over the two heads and the y gradient of the entropy path the channel concatenation of the
heads'.  What is here is the loss and the autograd wrapping.
``train_forward`` makes ``model(x)`` ONE autograd node (with ``_VisionRDLoss`` for the loss, so the reference-style
``vision_rd_loss(...)['loss'].backward()`` works); ``step_gradients`` runs the same forward + loss + backward on the calling thread
without the autograd engine (what ``parallel.ShardedTrainer`` uses and captures).  Oracle: torch autograd over
``oracle.forward.forward_scalable`` + ``vision_rd_loss`` (``oracle/backward.py: loss_and_grads_scalable``); the reference itself
has no runnable forward for this class, so parity is against that repaired restatement (parity unpinned by the reference).
"""
from __future__ import annotations

import math

import torch

from . import _lib, engine
from . import training as T
from ._lib import check, current_stream, ptr
from .Models import draw_noise, two_head_outputs


@torch.no_grad()
def step_gradients(model, x: torch.Tensor, lambda_rd: float, noise=None):
    """One training step's forward + vision_rd_loss + backward on the calling thread.  Returns (loss [device scalar], terms dict)."""
    engine.require_cuda(x, "x")
    lib = _lib.load()
    dev = x.device
    x = x.contiguous().float()
    B, _, H, W = x.shape
    noise_z, noise_y = draw_noise(model.M, x, noise)
    T.forget_pairs()
    outs, S = T._forward_impl(model, x, noise_z, noise_y, False)
    x_hat, logp_y1, logp_y2, logp_z = outs[:4]
    parts_y, parts_z = outs[11:13], outs[13]                            # two_head_outputs' order
    with torch.cuda.device(dev):
        # ---------------------------------------------------------------- loss -------------------------------------------------
        # vision_rd_loss (RateDistortionLoss.py:52-121, V = None): loss = bpp_y1 + bpp_y2 + bpp_z + lambda * mse  (no 255^2 here)
        chw, npix = x[0].numel(), H * W
        se = engine.partials(B, dev)
        check(lib.nic_sse_fwd(ptr(x_hat), ptr(x), B, chw, ptr(se), current_stream()), "nic_sse_fwd")
        scal = []
        for parts in parts_y:
            per_image = T._f32((3, B), dev)
            scalars = T._f32(8, dev)
            check(lib.nic_rd_finalize(ptr(parts), ptr(parts_z), ptr(se), B, npix, chw, 0.0, ptr(per_image), ptr(scalars), current_stream()),
                  "nic_rd_finalize")
            scal.append(scalars)
        loss = scal[0][0] + scal[1][0] + scal[0][1] + float(lambda_rd) * scal[0][3]
        terms = {"bpp_y1": scal[0][0], "bpp_y2": scal[1][0], "bpp_z": scal[0][1], "mse": scal[0][3], "psnr": scal[0][4], "loss": loss}
        gl = torch.full((1,), -1.0 / (math.log(2.0) * npix * B), dtype=torch.float32, device=dev)
        g = torch.empty_like(x_hat)
        check(lib.nic_sse_bwd(ptr(x_hat), ptr(x), x.numel(), float(lambda_rd) * 2.0 / x.numel(), ptr(g), current_stream()), "nic_sse_bwd")
    grads = T._backward_impl(model, S, g, [gl.expand(logp_y1.shape), gl.expand(logp_y2.shape)], gl.expand(logp_z.shape))
    for p in model.parameters():
        gp = grads.get(id(p))
        if gp is not None:
            p.grad = gp if p.grad is None else p.grad + gp
    return loss, terms


class _ScalableTrainForward(torch.autograd.Function):
    """ScalableImageCoding as ONE autograd node: differentiable outputs x_hat, logp_y1, logp_y2, logp_z."""

    @staticmethod
    def forward(ctx, model, x, noise_z, noise_y, *params):
        outs, S = T._forward_impl(model, x, noise_z, noise_y, False)
        ctx.model, ctx.S = model, S
        ctx.mark_non_differentiable(*outs[4:])
        return outs

    @staticmethod
    def backward(ctx, g_xhat, g1, g2, gz, *unused):
        model, S = ctx.model, ctx.S
        if g_xhat is None or g1 is None or g2 is None or gz is None:
            raise NotImplementedError("ScalableImageCoding backward needs gradients for x_hat, logp_y1, logp_y2 and logp_z (vision_rd_loss)")
        grads = T._backward_impl(model, S, g_xhat, [g1, g2], gz)
        ctx.S = None
        return (None, None, None, None, *[grads.get(id(p)) for _, p in model.named_parameters()])


def train_forward(model, x: torch.Tensor, noise=None) -> dict:
    """``model(x, training=True)`` of ScalableImageCoding as a differentiable call (reference dict keys, Models.py:321-338 minus F_tilde)."""
    noise_z, noise_y = draw_noise(model.M, x, noise)
    T.forget_pairs()
    params = [p for _, p in model.named_parameters()]
    res = _ScalableTrainForward.apply(model, x.contiguous().float(), noise_z, noise_y, *params)
    return two_head_outputs(*res, M1=model.M1, K=model.K, training=True)


class _VisionRDLoss(torch.autograd.Function):
    """loss = bpp_y1 + bpp_y2 + bpp_z + lambda * mse (RateDistortionLoss.py:98, V = None) as one node."""

    @staticmethod
    def forward(ctx, logp_y1, logp_y2, logp_z, x_hat, x, lambda_rd, loss_value):
        ctx.save_for_backward(x_hat, x)
        ctx.lambda_rd, ctx.shapes = float(lambda_rd), (logp_y1.shape, logp_y2.shape, logp_z.shape)
        return loss_value.clone()

    @staticmethod
    def backward(ctx, g):
        x_hat, x = ctx.saved_tensors
        B, _, H, W = x.shape
        gl = g.float() * (-1.0 / (math.log(2.0) * H * W * B))
        gx = torch.empty_like(x_hat)
        with torch.cuda.device(x_hat.device):
            check(_lib.load().nic_sse_bwd(ptr(x_hat), ptr(x), x.numel(), ctx.lambda_rd * 2.0 / x.numel(), ptr(gx), current_stream()), "nic_sse_bwd")
        gx.mul_(g.float())
        return gl.expand(ctx.shapes[0]), gl.expand(ctx.shapes[1]), gl.expand(ctx.shapes[2]), gx, None, None, None
