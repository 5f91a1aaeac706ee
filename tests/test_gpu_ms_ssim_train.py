"""GPU: the MS-SSIM training loss (RateDistortionLoss.ms_ssim_rd_loss, training.step_gradients(distortion="ms-ssim"),
parallel.ShardedTrainer(distortion="ms-ssim")) and its backward kernel nic_ms_ssim_bwd, against float64 autograd over the oracle.

Kernel tolerance: the gradient within 1e-4 of its norm.  x_hat is x + 5 % Gaussian noise (about 26 dB, a low-rate codec); the
error grows as 1 / |x_hat - x| because the pooled pyramids are stored in fp32 (DESIGN.md section 13)."""
import numpy as np
import pytest
import torch

from oracle import backward as OB
from oracle import backward_ms_ssim as OBM
from oracle import metrics as OM
from tests import helpers as H

pytestmark = pytest.mark.gpu

LAMBDA = 8.0


def _pair(shape, kind="noise", seed=7):
    g = torch.Generator().manual_seed(seed)
    y = torch.rand(*shape, generator=g)
    x = y + 0.05 * torch.randn(*shape, generator=g)
    if kind == "relu":                       # image 0: cs < 0 (its channels are zeroed)
        x[0] = 1 - y[0]
    elif kind == "last":                     # image 0, plane 0: only the last level's ssim <= 0
        x[0, 0] = y[0, 0] - 1
    return x, y


def _device_grad(x, y, per_plane_mean=True):
    """d mean(ms_ssim per plane) / d x (or, per_plane_mean=False, the sum over planes) through nic_ms_ssim_levels + nic_ms_ssim_bwd."""
    from neural_image_compression_b200 import _lib
    from neural_image_compression_b200.Evaluator import combine_levels, ms_ssim_levels, term_grads
    lib = _lib.load()
    x, y = x.cuda().contiguous(), y.cuda().contiguous()
    b, c, h, w = x.shape
    ws = torch.empty(lib.nic_ms_ssim_bwd_workspace_bytes(b * c, h, w), dtype=torch.uint8, device="cuda")
    terms, val = combine_levels(ms_ssim_levels(x, y, workspace=ws))
    coef = term_grads(terms, val) / (b * c if per_plane_mean else 1)
    gx = torch.empty_like(x)
    _lib.check(lib.nic_ms_ssim_bwd(_lib.ptr(x), _lib.ptr(y), b * c, h, w, 1.0, _lib.ptr(coef), _lib.ptr(gx), _lib.ptr(ws), ws.numel(),
                                   _lib.current_stream()), "nic_ms_ssim_bwd")
    torch.cuda.synchronize()
    return gx


def _ref_grad(x, y):
    xr = x.double().clone().requires_grad_(True)
    OM.ms_ssim(xr, y.double()).backward()
    return xr.grad


@pytest.mark.parametrize("shape,kind", [((1, 3, 161, 203), "noise"), ((8, 3, 161, 203), "relu"), ((1, 3, 256, 256), "last"),
                                        ((8, 3, 256, 256), "noise"), ((1, 3, 512, 768), "noise"), ((8, 3, 512, 768), "last"),
                                        ((8, 1, 256, 256), "noise"), ((2, 1, 161, 203), "last"), ((2, 1, 512, 768), "relu")])
def test_backward_kernel_against_float64_autograd(shape, kind):
    x, y = _pair(shape, kind)
    ref = _ref_grad(x, y)
    got = _device_grad(x, y).double().cpu()
    err = float((got - ref).norm() / ref.norm())
    rms = float(ref.norm()) / ref.numel() ** 0.5
    print(shape, kind, "relative error", err, "max element error / rms", float((got - ref).abs().max()) / rms)
    assert err <= 1e-4, err
    assert float((got - ref).abs().max()) <= 1e-2 * rms
    if kind != "noise":                                           # the zeroed channels get exactly zero
        zero = ref.abs().flatten(2).amax(-1) == 0
        assert zero.any() and float(got.flatten(2)[zero].abs().max()) == 0.0


def test_backward_kernel_is_bitwise_deterministic_and_batch_invariant():
    x, y = _pair((8, 3, 256, 320))
    g1 = _device_grad(x, y, per_plane_mean=False)
    g2 = _device_grad(x, y, per_plane_mean=False)
    assert torch.equal(g1, g2)
    for i in (0, 5):
        alone = _device_grad(x[i:i + 1], y[i:i + 1], per_plane_mean=False)
        assert torch.equal(alone[0], g1[i]), i


def test_backward_kernel_rejects_bad_arguments_before_any_launch():
    from neural_image_compression_b200 import _lib
    lib = _lib.load()
    buf = torch.zeros(3 * 256 * 256, device="cuda")
    need = lib.nic_ms_ssim_bwd_workspace_bytes(3, 256, 256)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    p = _lib.ptr(buf)
    assert need > lib.nic_ms_ssim_workspace_bytes(3, 256, 256)
    assert lib.nic_ms_ssim_bwd(p, p, 3, 160, 256, 1.0, p, p, _lib.ptr(ws), need, None) != 0
    assert lib.nic_ms_ssim_bwd(p, p, 0, 256, 256, 1.0, p, p, _lib.ptr(ws), need, None) != 0
    assert lib.nic_ms_ssim_bwd(p, None, 3, 256, 256, 1.0, p, p, _lib.ptr(ws), need, None) != 0
    assert lib.nic_ms_ssim_bwd(p, p, 3, 256, 256, 1.0, p, p, _lib.ptr(ws), need - 1, None) != 0
    torch.cuda.synchronize()


def _models():
    return {"jah": lambda: H.seeded_model(128, 3, "calib", precision="fp32"),
            "res": lambda: H.seeded_residual_model(128, 1, 17.853268, 136.1523, precision="fp32")}


@pytest.mark.parametrize("name,arm,shape", [("jah", "fp32", (2, 3, 192, 256)), ("jah", "bf16x3", (2, 3, 192, 256)),
                                            ("res", "fp32", (1, 3, 256, 192))])
def test_every_gradient_tensor_against_the_oracle(name, arm, shape):
    """ms_ssim_rd_loss(model(x), x, lambda)['loss'].backward() against autograd over the oracle's forward + rate + ms_ssim."""
    from neural_image_compression_b200.RateDistortionLoss import ms_ssim_rd_loss
    from tests.test_gpu_train import grad_tol
    model = _models()[name]()
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    x = H.seeded_input(shape)
    if name == "jah":
        _, nz, ny = OB.noise_with_margin(sd, x, 128, 3, 21, margin=5e-7)     # no draw reaches 1e-6 at this size
    else:
        torch.manual_seed(21)
        B, _, Hh, W = shape
        nz, ny = torch.rand(B, 128, Hh // 64, W // 64) - 0.5, torch.rand(B, 128, Hh // 16, W // 16) - 0.5
    ref_rd, ref_g = OBM.loss_and_grads_ms_ssim(sd, x, 128, model.K, nz, ny, LAMBDA, residual=name == "res")
    model = model.cuda()
    model.train_precision = arm
    rd = ms_ssim_rd_loss(model(x.cuda(), training=True, noise=(nz.cuda(), ny.cuda())), x.cuda(), LAMBDA)
    ltol = 1e-5 if arm == "fp32" else 5e-5
    assert abs(float(rd["loss"].detach()) - ref_rd["loss"]) <= ltol * abs(ref_rd["loss"]), (float(rd["loss"]), ref_rd["loss"])
    assert abs(rd["ms_ssim"] - ref_rd["ms_ssim"]) <= 1e-5, (rd["ms_ssim"], ref_rd["ms_ssim"])
    assert abs(float(rd["ms_ssim_per_image"].mean()) - rd["ms_ssim"]) <= 1e-6 and rd["ms_ssim_per_image"].shape == (shape[0],)
    loss = float(rd["loss"].detach())
    assert abs(rd["bpp_total"] + LAMBDA * (1 - rd["ms_ssim"]) - loss) <= 1e-5 * abs(loss)
    rd["loss"].backward()
    torch.cuda.synchronize()
    worst = {k: float((p.grad.double().cpu() - ref_g[k].double()).norm() / max(float(ref_g[k].double().norm()), 1e-30))
             for k, p in model.named_parameters()}
    assert set(worst) == set(ref_g)
    print(name, arm, "worst gradient errors:", sorted(worst.items(), key=lambda kv: -kv[1])[:5])
    tol = (lambda k: 2e-4) if name == "res" else (lambda k: grad_tol(arm, k))
    bad = {k: v for k, v in worst.items() if v > tol(k)}
    assert not bad, bad


@pytest.mark.parametrize("name", ["jah", "res"])
def test_step_gradients_equals_autograd_backward(name):
    """step_gradients(distortion="ms-ssim") (what the graphed trainer captures) deposits exactly the .grad of the autograd route."""
    from neural_image_compression_b200.RateDistortionLoss import ms_ssim_rd_loss
    from neural_image_compression_b200.training import step_gradients
    model = _models()[name]().cuda()
    if name == "jah":
        model.train_precision = "bf16x3"
    x = H.seeded_input((2, 3, 192, 256)).cuda()
    torch.manual_seed(9)
    noise = (torch.rand(2, 128, 3, 4).cuda() - 0.5, torch.rand(2, 128, 12, 16).cuda() - 0.5)
    rd = ms_ssim_rd_loss(model(x, noise=noise), x, LAMBDA)
    rd["loss"].backward()
    ref = {k: p.grad.clone() for k, p in model.named_parameters()}
    model.zero_grad()
    loss, per_image, scalars = step_gradients(model, x, LAMBDA, noise=noise, distortion="ms-ssim")
    torch.cuda.synchronize()
    assert scalars.shape == (9,) and float(loss) == float(rd["loss"].detach()) and float(scalars[8]) == rd["ms_ssim"]
    for k, p in model.named_parameters():
        assert torch.equal(p.grad, ref[k]), k


def test_graphed_trainer_steps_like_the_eager_one():
    """ShardedTrainer(distortion="ms-ssim", graph=True) against the eager trainer over 30 steps: both losses fall and end in the
    same band, and the batch MS-SSIM rises."""
    from neural_image_compression_b200 import parallel
    x = H.seeded_input((2, 3, 192, 192)).cuda()
    losses, ms = {}, {}
    for mode in (False, True):
        model = H.seeded_model(128, 3, "calib", precision="bf16x3").cuda()
        tr = parallel.ShardedTrainer(model, LAMBDA, lr=1e-4, graph=mode, distortion="ms-ssim")
        ls, ss = [], []
        for _ in range(30):
            rd = tr.step(x)
            ls.append(float(rd["loss"].detach()))
            ss.append(rd["ms_ssim"] if not mode else float(rd["scalars"][8]))
        torch.cuda.synchronize()
        losses[mode], ms[mode] = ls, ss
        assert tr.optimizer.t == 30
    print("losses", losses, "ms-ssim", ms)
    assert abs(losses[True][0] - losses[False][0]) < 0.02 * losses[False][0], (losses[True][0], losses[False][0])
    for mode in (False, True):
        assert losses[mode][-1] < losses[mode][0] and np.mean(ms[mode][-5:]) > np.mean(ms[mode][:5]), (mode, losses[mode], ms[mode])
    assert abs(losses[True][-1] - losses[False][-1]) < 0.05 * losses[False][-1], losses
