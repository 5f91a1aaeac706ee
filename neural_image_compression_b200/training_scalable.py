"""Training step of ``ScalableImageCoding`` (reference Models.py:208-338 with the repairs of SURVEY.md section 2.4, loss
``vision_rd_loss`` of RateDistortionLoss.py:52-121 with V = None): forward with noise, loss, hand-written backward.

Same kernels and helpers as training.py, the transforms recorded on and walked back by the same ``training.Tape``; what differs
from the single-head model is the split of y into a base part (M1 channels) and an enhancement part (M - M1), each with its own
(context model, entropy-parameter net) over the SHARED hyper features psi: the psi gradient is the sum over the two heads, the y
gradient of the entropy path is the channel concatenation of the heads'.
``train_forward`` makes ``model(x)`` ONE autograd node (with ``_VisionRDLoss`` for the loss, so the reference-style
``vision_rd_loss(...)['loss'].backward()`` works); ``step_gradients`` runs the same forward + loss + backward on the calling thread
without the autograd engine (what ``parallel.ShardedTrainer`` uses and captures).  Oracle: torch autograd over
``oracle.forward.forward_scalable`` + ``vision_rd_loss`` (``oracle/backward.py: loss_and_grads_scalable``); the reference itself
has no runnable forward for this class, so parity is against that repaired restatement (parity unpinned by the reference).
"""
from __future__ import annotations

import math
from typing import Dict

import torch

from . import _lib, engine
from . import training as T
from ._lib import EPI_BIAS, LAYOUT_NCHW, LAYOUT_NHWC, Q_NOISE, Q_PASSTHRU, check, current_stream, ptr
from .Models import draw_noise, mixture_params, two_head_outputs


def _heads(model):
    return ((model.context_model_1, model.entropy_parameters_1, 0, model.M1), (model.context_model_2, model.entropy_parameters_2, model.M1, model.M))


def _forward_impl(model, x, noise_z, noise_y):
    """Layer-by-layer training forward of the two-head model -> (x_hat, head likelihood dicts, p_z, logp_z, parts_z, y, y_in, z, z_in), S."""
    from .EntropyModels import gm_likelihood
    dev = x.device
    B, _, H, W = x.shape
    M, M1, M2, K = model.M, model.M1, model.M2, model.K
    hy, wy, hz, wz = H // 16, W // 16, H // 64, W // 64
    arm = T.train_precision(model)
    heads = _heads(model)
    S = {t: T.Tape(arm, B) for t in ("g_a", "g_s", "h_a", "h_s")}
    with torch.cuda.device(dev):
        y_nhwc, _, _ = model.encoder.run_nhwc(x, B, H, W, arm, in_layout=LAYOUT_NCHW, tape=S["g_a"])
        y, y_in, y_in_nhwc, _ = engine.latent_handoff(y_nhwc, Q_NOISE, noise_y, torch.float32)
        z_nhwc, _, _ = model.hyper_encoder.run_nhwc(y_nhwc, B, hy, wy, arm, tape=S["h_a"])
        z, z_in, z_in_nhwc, _ = engine.latent_handoff(z_nhwc, Q_NOISE, noise_z, torch.float32)
        combs = [T._f32((B, hy, wy, 2 * (c1 - c0) + 2 * M), dev) for _, _, c0, c1 in heads]
        model.hyper_decoder.run_nhwc(z_in_nhwc, B, hz, wz, arm, tape=S["h_s"],
                                     final_kw=dict(out=combs[0], out_c_total=combs[0].shape[-1], out_c_offset=2 * M1))
        combs[1][..., 2 * M2:] = combs[0][..., 2 * M1:]                       # the second head reads the same psi
        head_state = []
        for (ctx, ep, c0, c1), comb in zip(heads, combs):
            mi = c1 - c0
            yi_nhwc = y_in_nhwc[..., c0:c1].contiguous()
            yi = y_in[:, c0:c1].contiguous()
            ctx.masked.apply_mask_()
            T.conv_forward(arm, ctx.masked, EPI_BIAS, yi_nhwc, B, hy, wy, out=comb, out_c_total=comb.shape[-1], out_c_offset=0, mask_a=True)
            e1 = T.conv_forward(arm, ep.ops[0].conv, ep.ops[0].epilogue, comb, B, hy, wy)
            e2 = T.conv_forward(arm, ep.ops[1].conv, ep.ops[1].epilogue, e1, B, hy, wy)
            raw = T.conv_forward(arm, ep.ops[2].conv, ep.ops[2].epilogue, e2, B, hy, wy, out_layout=LAYOUT_NCHW)
            ly = gm_likelihood(yi, raw, mi, K, Q_PASSTHRU, full=True, want_y_in=False)
            head_state.append(dict(yi=yi, yi_nhwc=yi_nhwc, comb=comb, e1=e1, e2=e2, raw=raw, parts=ly["partials"], ly=ly))
        fe = model.factorized_entropy_model
        _, p_z, logp_z, parts_z = fe.likelihood(z_in, Q_PASSTHRU)
        x_hat, _, _ = model.decoder.run_nhwc(y_in_nhwc, B, hy, wy, arm, tape=S["g_s"])         # the RGB layer writes NCHW
    S.update(arm=arm, shape=(B, H, W), head_state=head_state, y_nhwc=y_nhwc, y_in_nhwc=y_in_nhwc, z_in=z_in, z_in_nhwc=z_in_nhwc,
             fparams=fe.packed())
    return (x_hat, head_state, p_z, logp_z, parts_z, y, y_in, z, z_in), S


def _backward_impl(model, S, g, g_logp_heads, g_logp_z) -> Dict[int, torch.Tensor]:
    """{id(parameter): gradient} from the gradients of x_hat (g, NCHW), of logp_y1 / logp_y2 and of logp_z."""
    lib = _lib.load()
    dev = g.device
    B, H, W = S["shape"]
    M, K = model.M, model.K
    hy, wy, hz, wz = H // 16, W // 16, H // 64, W // 64
    arm, heads, head_state, z_in = S["arm"], _heads(model), S["head_state"], S["z_in"]
    fe = model.factorized_entropy_model
    grads: Dict[int, torch.Tensor] = {}

    def put(param, gr):
        grads[id(param)] = gr if id(param) not in grads else grads[id(param)] + gr

    with torch.cuda.device(dev):
        d_yin_gs = S["g_s"].backward(g, LAYOUT_NCHW, put, T.conv_wgrad, root=S["y_in_nhwc"])
        d_psi, d_yin_parts = None, []
        for (ctx, ep, c0, c1), hsd in zip(heads, head_state):                  # the two entropy heads
            mi = c1 - c0
            glh = g_logp_heads[len(d_yin_parts)].contiguous().float()
            dy_lik = torch.empty_like(hsd["yi"])
            draw = torch.empty_like(hsd["raw"])
            check(lib.nic_gm_likelihood_bwd(ptr(hsd["yi"]), ptr(hsd["raw"]), ptr(glh), 0.0, B, mi, hy * wy, K, ptr(dy_lik), ptr(draw),
                                            current_stream()), "nic_gm_likelihood_bwd")
            d_yi = T.to_nhwc(dy_lik)
            g = T.to_nhwc(draw)
            for j, (op, a) in reversed(list(enumerate(zip(ep.ops, (hsd["comb"], hsd["e1"], hsd["e2"]))))):
                dw, db = T.conv_wgrad(op.conv, a, g, B, hy, wy, LAYOUT_NHWC, LAYOUT_NHWC, arm=arm)
                put(op.conv.weight, dw); put(op.conv.bias, db)
                if j > 0:
                    g = T.lrelu_bwd_(T.conv_dgrad(op.conv, g, B, hy, wy, arm=arm), a)
            w0 = ep.ops[0].conv.weight.detach()
            d_phi = T.conv_dgrad(ep.ops[0].conv, g, B, hy, wy, weight=w0[:, :2 * mi].contiguous(), c_in=2 * mi, arm=arm)
            d_psi_i = T.conv_dgrad(ep.ops[0].conv, g, B, hy, wy, weight=w0[:, 2 * mi:].contiguous(), c_in=2 * M, arm=arm)
            d_psi = d_psi_i if d_psi is None else T.add_(d_psi, d_psi_i)
            dw, db = T.conv_wgrad(ctx.masked, hsd["yi_nhwc"], d_phi, B, hy, wy, LAYOUT_NHWC, LAYOUT_NHWC, arm=arm)
            put(ctx.masked.weight, dw); put(ctx.masked.bias, db)
            d_yin_parts.append(T.add_(d_yi, T.conv_dgrad(ctx.masked, d_phi, B, hy, wy, arm=arm)))
        del g                                                                  # the last head's concat gradient: free it before h_s
        d_zin = S["h_s"].backward(d_psi, LAYOUT_NHWC, put, T.conv_wgrad, root=S["z_in_nhwc"])
        glz = g_logp_z.contiguous().float()                                    # factorized prior
        dz_fac = torch.empty_like(z_in)
        dpar = T._f32((M, 43), dev)
        check(lib.nic_factorized_likelihood_bwd(ptr(z_in), ptr(S["fparams"]), ptr(glz), 0.0, B, M, hz * wz, ptr(dz_fac), ptr(dpar),
                                                current_stream()), "nic_factorized_likelihood_bwd")
        for name, idx, lo, hi in T._FACT_SLICES:
            prm = getattr(fe, name)[idx]
            put(prm, dpar[:, lo:hi].reshape(prm.shape).contiguous())
        d_zin = T.to_nhwc(dz_fac, accumulate_into=d_zin)
        g = S["h_a"].backward(d_zin, LAYOUT_NHWC, put, T.conv_wgrad, root=S["y_nhwc"])
        dy = T.add_(T.add_(g, torch.cat(d_yin_parts, dim=-1).contiguous()), d_yin_gs)
        S["g_a"].backward(dy, LAYOUT_NHWC, put, T.conv_wgrad, root=None)
    T.forget_pairs()
    return grads


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
    (x_hat, head_state, p_z, logp_z, parts_z, y, y_in, z, z_in), S = _forward_impl(model, x, noise_z, noise_y)
    with torch.cuda.device(dev):
        # ---------------------------------------------------------------- loss -------------------------------------------------
        # vision_rd_loss (RateDistortionLoss.py:52-121, V = None): loss = bpp_y1 + bpp_y2 + bpp_z + lambda * mse  (no 255^2 here)
        chw, npix = x[0].numel(), H * W
        se = engine.partials(B, dev)
        check(lib.nic_sse_fwd(ptr(x_hat), ptr(x), B, chw, ptr(se), current_stream()), "nic_sse_fwd")
        scal = []
        for hsd in head_state:
            per_image = T._f32((3, B), dev)
            scalars = T._f32(8, dev)
            check(lib.nic_rd_finalize(ptr(hsd["parts"]), ptr(parts_z), ptr(se), B, npix, chw, 0.0, ptr(per_image), ptr(scalars), current_stream()),
                  "nic_rd_finalize")
            scal.append(scalars)
        loss = scal[0][0] + scal[1][0] + scal[0][1] + float(lambda_rd) * scal[0][3]
        terms = {"bpp_y1": scal[0][0], "bpp_y2": scal[1][0], "bpp_z": scal[0][1], "mse": scal[0][3], "psnr": scal[0][4], "loss": loss}
        gl = torch.full((1,), -1.0 / (math.log(2.0) * npix * B), dtype=torch.float32, device=dev)
        g = torch.empty_like(x_hat)
        check(lib.nic_sse_bwd(ptr(x_hat), ptr(x), x.numel(), float(lambda_rd) * 2.0 / x.numel(), ptr(g), current_stream()), "nic_sse_bwd")
    grads = _backward_impl(model, S, g, [gl.expand(h["yi"].shape) for h in head_state], gl.expand(z_in.shape))
    for p in model.parameters():
        gp = grads.get(id(p))
        if gp is not None:
            p.grad = gp if p.grad is None else p.grad + gp
    return loss, terms


class _ScalableTrainForward(torch.autograd.Function):
    """ScalableImageCoding as ONE autograd node: differentiable outputs x_hat, logp_y1, logp_y2, logp_z."""

    @staticmethod
    def forward(ctx, model, x, noise_z, noise_y, *params):
        (x_hat, head_state, p_z, logp_z, parts_z, y, y_in, z, z_in), S = _forward_impl(model, x, noise_z, noise_y)
        ctx.model, ctx.S = model, S
        l1, l2 = head_state[0]["ly"], head_state[1]["ly"]
        nd = [y, y_in, z, z_in, p_z, l1["p"], l2["p"], l1["partials"], l2["partials"], parts_z] + mixture_params(l1, model.K) + \
            mixture_params(l2, model.K)
        ctx.mark_non_differentiable(*nd)
        return (x_hat, l1["logp"], l2["logp"], logp_z, *nd)

    @staticmethod
    def backward(ctx, g_xhat, g1, g2, gz, *unused):
        model, S = ctx.model, ctx.S
        if g_xhat is None or g1 is None or g2 is None or gz is None:
            raise NotImplementedError("ScalableImageCoding backward needs gradients for x_hat, logp_y1, logp_y2 and logp_z (vision_rd_loss)")
        with torch.no_grad():
            grads = _backward_impl(model, S, g_xhat.contiguous().float(), [g1, g2], gz)
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
