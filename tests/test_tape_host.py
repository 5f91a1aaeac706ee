"""CPU (no GPU): the host logic of the training step's transforms - ``training.Tape`` and the ``tape=`` plumbing of Layers.py /
Components._Transform (5x5) / Components._Chain (3x3) - and of its entropy heads (``training.head_forward`` / ``head_backward``),
with torch stand-ins for the C-ABI calls (conv forward / weight gradient / adjoint conv, GDN forward / backward, LeakyReLU backward,
add, layout conversion, Gaussian(-mixture) likelihood forward / backward).  What is checked is the BOOKKEEPING: every op of the transforms is
recorded once, gradients of tensors with two consumers (the block input feeding the main path and the skip) are summed, the gradient
of the transform's input comes back, and every parameter gets its gradient - against torch autograd over the oracle's restatement
of the same transforms (oracle/forward.py: analysis / synthesis / hyper_* and their _3x3 forms, pinned to the reference's own
classes by tests/test_oracle.py).  The kernels themselves are checked on the GPU (tests/test_gpu_train.py, test_gpu_residual.py)."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import forward as O
from oracle.gdn import gdn_effective

NCHW, NHWC, EPI_LRELU = 0, 1, 1


def _nchw(t, layout):
    return t if layout == NCHW else t.permute(0, 3, 1, 2)


def _fconv(conv, x, w, b):
    if isinstance(conv, nn.ConvTranspose2d):
        return F.conv_transpose2d(x, w, b, stride=conv.stride, padding=conv.padding, output_padding=conv.output_padding)
    return F.conv2d(x, w, b, stride=conv.stride, padding=conv.padding)


def _gdn_fn(gdn, x, beta, gamma):
    be, ga = gdn_effective(beta, gamma, gdn.beta_min)
    c = be.numel()
    norm = F.conv2d(x * x, ga.reshape(c, c, 1, 1), be)
    return x * (torch.sqrt(norm) if gdn.inverse else torch.rsqrt(norm))


@pytest.fixture
def torch_backend(monkeypatch):
    from neural_image_compression_b200 import training as T

    def conv_forward(arm, conv, epi, x, n, h, w, in_layout=NHWC, out_layout=NHWC, out=None, out_c_total=0, out_c_offset=0, mask_a=False,
                     pair_out=False):
        with torch.no_grad():
            y = _fconv(conv, _nchw(x, in_layout).double(), conv.weight.double(), conv.bias.double())
            if epi == EPI_LRELU:
                y = F.leaky_relu(y, 0.01)
            y = y if out_layout == NCHW else y.permute(0, 2, 3, 1)
            if out is not None:
                out[..., out_c_offset:out_c_offset + y.shape[-1]] = y
                return out
            return y.contiguous()

    def conv_wgrad(conv, x, g, n, h, w, in_layout, out_layout, arm="fp32", pairs=None):
        wt, b = conv.weight.detach().double().requires_grad_(), conv.bias.detach().double().requires_grad_()
        with torch.enable_grad():
            y = _fconv(conv, _nchw(x, in_layout).double(), wt, b)
            go = _nchw(g, out_layout).double()
            if go.shape[1] != y.shape[1]:                      # a channel window of a wider buffer (psi inside `combined`)
                go = go[:, -y.shape[1]:]
            return torch.autograd.grad(y, (wt, b), go)

    def conv_dgrad(conv, g, n, h_in, w_in, g_layout=NHWC, weight=None, c_in=None, arm="fp32"):
        # weight / c_in: a slice of the layer's input channels (the [phi | psi] split of the first entropy-parameter conv)
        x = torch.zeros(n, c_in or conv.in_channels, h_in, w_in, dtype=torch.float64, requires_grad=True)
        with torch.enable_grad():
            y = _fconv(conv, x, (conv.weight if weight is None else weight).detach().double(), None)
            return torch.autograd.grad(y, x, _nchw(g, g_layout).double())[0].permute(0, 2, 3, 1).contiguous()

    def gdn_forward(arm, gdn, u, n, h, w):
        with torch.no_grad():
            return _gdn_fn(gdn, u.permute(0, 3, 1, 2), gdn.beta.double(), gdn.gamma.double()).permute(0, 2, 3, 1).contiguous(), None

    def gdn_bwd(gdn, u, g, n, h, w, norm=None, side=None, keep=None):
        x = u.permute(0, 3, 1, 2).detach().requires_grad_()
        beta, gamma = gdn.beta.detach().double().requires_grad_(), gdn.gamma.detach().double().requires_grad_()
        with torch.enable_grad():
            y = _gdn_fn(gdn, x, beta, gamma)
            dx, db, dg = torch.autograd.grad(y, (x, beta, gamma), g.permute(0, 3, 1, 2))
        return dx.permute(0, 2, 3, 1).contiguous(), db, dg

    def lrelu_bwd_(g, out):
        return g.mul_(torch.where(out > 0, torch.ones_like(g), torch.full_like(g, 0.01)))

    def add_(dst, src):
        return dst.add_(src)

    def to_nhwc(t, accumulate_into=None):
        t = t.permute(0, 2, 3, 1)
        return t.contiguous() if accumulate_into is None else accumulate_into.add_(t)
    for name, fn in dict(conv_forward=conv_forward, conv_wgrad=conv_wgrad, conv_dgrad=conv_dgrad, gdn_forward=gdn_forward, gdn_bwd=gdn_bwd,
                         lrelu_bwd_=lrelu_bwd_, add_=add_, to_nhwc=to_nhwc).items():
        monkeypatch.setattr(T, name, fn)
    return T


def _perturb(mod, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in mod.modules():
            if type(m).__name__ == "GDN":
                m.gamma.add_(0.02 * torch.rand(m.gamma.shape, generator=g))
    return mod


_CLASSES = {"encoder": "Encoder", "decoder": "Decoder", "hyper_encoder": "HyperEncoder", "hyper_decoder": "HyperDecoder"}
_ORACLE = {"encoder": "analysis", "decoder": "synthesis", "hyper_encoder": "hyper_analysis", "hyper_decoder": "hyper_synthesis"}


@pytest.mark.parametrize("which", ["encoder", "decoder", "hyper_encoder", "hyper_decoder"])
@pytest.mark.parametrize("family", ["3x3", "5x5"])
def test_tape_routes_gradients_through_the_transforms(torch_backend, family, which):
    from neural_image_compression_b200 import Components as Cm
    T = torch_backend
    M = 8
    torch.manual_seed(3)
    mod = _perturb(getattr(Cm, _CLASSES[which] + family)(latent_channels=M), 4)
    n, h, w = 2, (32 if which == "encoder" else 4), (48 if which == "encoder" else 6)
    x_nchw = (torch.rand(n, 3, h, w) if which == "encoder" else torch.randn(n, M, h, w)).double()
    # oracle: autograd over the restated transform
    sd = {f"{which}.{k}": v.detach().double().clone().requires_grad_(v.dtype.is_floating_point and not k.endswith(("pedestal", "bound")))
          for k, v in mod.state_dict().items()}
    xr = x_nchw.clone().requires_grad_()
    prev, O.DIFFERENTIABLE = O.DIFFERENTIABLE, True
    try:
        fn = getattr(O, _ORACLE[which] + ("_3x3" if family == "3x3" else ""))
        y_ref = fn(sd, xr, torch.float64)
        g_out = torch.randn(y_ref.shape, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
        y_ref.backward(g_out)
    finally:
        O.DIFFERENTIABLE = prev
    # the package's chain with a tape
    tape = T.Tape("fp32", n)
    if which == "encoder":
        x_in, in_layout = x_nchw, NCHW                                     # the image arrives NCHW and needs no gradient
    else:
        x_in, in_layout = x_nchw.permute(0, 2, 3, 1).contiguous(), NHWC
    y, ho, wo = mod.run_nhwc(x_in, n, h, w, "fp32", in_layout=in_layout, tape=tape)
    rgb = which == "decoder"                                               # the RGB layer stays NCHW (x_hat)
    y_nchw = y if rgb else y.permute(0, 3, 1, 2)
    assert torch.allclose(y_nchw, y_ref.detach(), rtol=1e-10, atol=1e-12)
    n_convs = sum(isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)) for m in mod.modules())
    assert sum(r[0] == "conv" for r in tape.recs) == n_convs and tape.output is y
    grads = {}

    def put(p, g):
        grads[id(p)] = g if id(p) not in grads else grads[id(p)] + g
    g_in = tape.backward(g_out if rgb else g_out.permute(0, 2, 3, 1).contiguous(), NCHW if rgb else NHWC, put, T.conv_wgrad,
                         root=None if which == "encoder" else x_in)
    for k, p in mod.named_parameters():
        ref = sd[f"{which}.{k}"].grad
        assert id(p) in grads, k
        assert torch.allclose(grads[id(p)], ref, rtol=1e-8, atol=1e-10 * float(ref.abs().max() + 1)), k
    if which == "encoder":
        assert g_in is None
    else:
        assert torch.allclose(g_in.permute(0, 3, 1, 2), xr.grad, rtol=1e-8, atol=1e-12)


def test_chain_writes_its_last_conv_into_a_channel_window(torch_backend):
    """h_s of the training forward (the 3x3 and the 5x5 family) writes psi straight into its window of the entropy-parameter
    stack's concat buffer (`final_kw`): same values as the plain call, the other window untouched, and the backward starts from the
    window's gradient."""
    from neural_image_compression_b200 import Components as Cm
    T = torch_backend
    M, n, h, w = 8, 1, 2, 3
    for cls in (Cm.HyperDecoder3x3, Cm.HyperDecoder5x5):
        torch.manual_seed(7)
        mod = cls(latent_channels=M)
        x = torch.randn(n, h, w, M).double()
        plain, ho, wo = mod.run_nhwc(x, n, h, w, "fp32", tape=T.Tape("fp32", n))
        combined = torch.full((n, ho, wo, 4 * M), 7.0, dtype=torch.float64)
        tape = T.Tape("fp32", n)
        mod.run_nhwc(x, n, h, w, "fp32", tape=tape, final_kw=dict(out=combined, out_c_total=4 * M, out_c_offset=2 * M))
        assert tape.output is combined and torch.equal(combined[..., 2 * M:], plain) and bool((combined[..., :2 * M] == 7.0).all())
        grads = {}
        g = torch.randn(n, ho, wo, 2 * M, dtype=torch.float64)
        gx = tape.backward(g, NHWC, lambda p, v: grads.__setitem__(id(p), v), T.conv_wgrad, root=x)
        assert gx.shape == x.shape and len(grads) == len(list(mod.parameters())), cls.__name__


@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("scalable", [False, True])
def test_entropy_heads_route_gradients(torch_backend, monkeypatch, scalable, K):
    """training.head_forward / head_backward over training.heads: one head over all of y (JointAutoregressiveHierarchical) or the
    base + enhancement heads of ScalableImageCoding (M1 < M) over the shared psi.  Every context / entropy-parameter gradient, the
    y gradient (the heads' channel concatenation) and the psi gradient (the heads' sum) against autograd over oracle.forward.context
    -> entropy_parameters_raw -> conditional_likelihood."""
    from neural_image_compression_b200 import Models
    T = torch_backend

    def lik(y, raw, m, K_):
        return O.conditional_likelihood(y, O.split_parameters(raw, m, K_), K_)

    def gm_likelihood(y, raw, m, K_, qmode, full=True, want_y_in=True):
        with torch.no_grad():
            p = lik(y, raw, m, K_)
        return {"p": p, "logp": torch.log(p), "partials": None}

    def gm_likelihood_bwd(y, raw, g_logp, m, K_):
        y, raw = y.detach().requires_grad_(), raw.detach().requires_grad_()
        with torch.enable_grad():
            return torch.autograd.grad(torch.log(lik(y, raw, m, K_)), (y, raw), g_logp)
    monkeypatch.setattr(T, "gm_likelihood", gm_likelihood)
    monkeypatch.setattr(T, "gm_likelihood_bwd", gm_likelihood_bwd)
    M, n, h, w = 8, 2, 5, 6
    torch.manual_seed(11)
    model = Models.ScalableImageCoding(M, 3, K, precision="fp32") if scalable else Models.JointAutoregressiveHierarchical(M, K, precision="fp32")
    heads = T.heads(model)
    assert [(c0, c1) for _, _, c0, c1 in heads] == ([(0, 3), (3, M)] if scalable else [(0, M)])
    prefixes = [("context_model_1", "entropy_parameters_1"), ("context_model_2", "entropy_parameters_2")] if scalable else \
        [("context_model", "entropy_parameters")]
    gen = torch.Generator().manual_seed(12)
    y = torch.randint(-3, 4, (n, M, h, w), generator=gen).double()
    psi = torch.randn(n, 2 * M, h, w, generator=gen, dtype=torch.float64)
    g_logp = [torch.randn(n, c1 - c0, h, w, generator=gen).double() for _, _, c0, c1 in heads]       # exact in f32 (head_backward's cast)
    # oracle: autograd over the restated heads
    sd = {k: v.detach().double().clone().requires_grad_() for k, v in model.state_dict().items() if not k.endswith("mask")}
    yr, psir = y.clone().requires_grad_(), psi.clone().requires_grad_()
    prev, O.DIFFERENTIABLE = O.DIFFERENTIABLE, True
    try:
        total = 0
        for (_, _, c0, c1), (cm, ep), g in zip(heads, prefixes, g_logp):
            yi = yr[:, c0:c1]
            raw = O.entropy_parameters_raw(sd, torch.cat([O.context(sd, yi, torch.float64, cm), psir], dim=1), torch.float64, ep)
            total = total + (g * torch.log(lik(yi, raw, c1 - c0, K))).sum()
        total.backward()
    finally:
        O.DIFFERENTIABLE = prev
    # the package's heads
    grads = {}

    def put(p, g):
        grads[id(p)] = g if id(p) not in grads else grads[id(p)] + g
    y_nhwc, psi_nhwc = y.permute(0, 2, 3, 1).contiguous(), psi.permute(0, 2, 3, 1)
    d_y, d_psi = [], None
    for head, g in zip(heads, g_logp):
        c0, c1 = head[2], head[3]
        comb = torch.full((n, h, w, 2 * (c1 - c0) + 2 * M), float("nan"), dtype=torch.float64)
        comb[..., 2 * (c1 - c0):] = psi_nhwc
        ly, st = T.head_forward("fp32", head, K, y[:, c0:c1].contiguous(), y_nhwc[..., c0:c1].contiguous(), comb, False)
        assert torch.allclose(ly["logp"], torch.log(lik(y[:, c0:c1], st["raw"], c1 - c0, K)))
        dy_i, dpsi_i = T.head_backward("fp32", head, K, st, g, put, T.conv_wgrad)
        d_y.append(dy_i)
        d_psi = dpsi_i if d_psi is None else d_psi + dpsi_i
    names = {id(p): k for k, p in model.named_parameters()}
    want = [k for k in sd if k.startswith(tuple(cm + "." for pre in prefixes for cm in pre))]
    assert sorted(names[i] for i in grads) == sorted(want)
    for i, g in grads.items():
        ref = sd[names[i]].grad
        assert torch.allclose(g, ref, rtol=1e-8, atol=1e-10 * float(ref.abs().max() + 1)), names[i]
    assert torch.allclose(torch.cat(d_y, dim=-1).permute(0, 3, 1, 2), yr.grad, rtol=1e-8, atol=1e-12)
    assert torch.allclose(d_psi.permute(0, 3, 1, 2), psir.grad, rtol=1e-8, atol=1e-12)
