"""GPU: GainedCheckerboardHierarchical - zero log-gains compute exactly JointCheckerboardHierarchical; the forward against the oracle
(oracle/gained.py) with random gains and mixed per-image qualities; the gained hand-off and the gain backward kernels; every gradient
against the oracle's autograd with per-image levels and lambdas (MSE and MS-SSIM); the graphed trainer with lambdas; and format 5:
lossless round trips at mixed qualities and any size, the bytes against the reference coder, the quality checksum, the coded rate and
a rate that grows with q."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from neural_image_compression_b200 import _lib, codec, engine
from neural_image_compression_b200.Models import GainedCheckerboardHierarchical, JointCheckerboardHierarchical
from neural_image_compression_b200.RateDistortionLoss import rd_terms
from oracle import checkerboard as OC
from oracle import forward as O
from oracle import gained as OG
from oracle import rans_gained as RG
from tests import helpers as H
from tests.test_gpu_checkerboard import _gpu_tables, _pad, _padded, seeded_cb

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LAMBDA = 0.005


def seeded_gained(M, K, init="calib", precision="fp32", levels=6, log_std=0.0, seed=5):
    """The checkerboard model's seeded weights (seeded_cb) with gain units; log-gains ~ N(0, log_std) when log_std > 0."""
    model = GainedCheckerboardHierarchical(M, K=K, levels=levels, precision=precision)
    model.load_state_dict(seeded_cb(M, K, init, precision).state_dict(), strict=False)
    if log_std:
        g = torch.Generator().manual_seed(seed)
        with torch.no_grad():
            for t in model.gain_units.tables():
                t.copy_(torch.randn(t.shape, generator=g) * log_std)
    return model


def _sd(model):
    return {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}


# ---- identity: zero log-gains are the parent model -------------------------------------------------------------------------------

@pytest.mark.parametrize("arm", ["fp32", "bf16x3"])
def test_zero_gains_are_the_parent(arm):
    parent = seeded_cb(128, 3, "calib", arm).to(DEV)
    model = seeded_gained(128, 3, "calib", arm).to(DEV)
    x = H.seeded_input((2, 3, 256, 320)).to(DEV)
    nz, ny = torch.rand(2, 128, 4, 5, device=DEV) - 0.5, torch.rand(2, 128, 16, 20, device=DEV) - 0.5
    with torch.no_grad():
        for training in (False, True):
            a = parent(x, training=training, noise=(nz, ny))
            b = model(x, training=training, quality=[0.3, 4.7], noise=(nz, ny))
            for k in a:
                if isinstance(a[k], torch.Tensor):
                    assert torch.equal(a[k], b[k]), (arm, training, k)
            assert b["quality"].tolist() == [307 / 1024, 4813 / 1024]
    # the training forward with autograd: outputs bitwise, gradients of the shared parameters at the fp32 arm's bar
    from tests.test_gpu_train import grad_tol
    parent.train_precision = model.train_precision = arm
    xs = H.seeded_input((1, 3, 128, 128)).to(DEV)
    nz, ny = torch.rand(1, 128, 2, 2, device=DEV) - 0.5, torch.rand(1, 128, 8, 8, device=DEV) - 0.5
    outs = []
    for m in (parent, model):
        m.zero_grad()
        out = m(xs, noise=(nz, ny))
        loss = out["x_hat"].square().mean() - out["logp_y"].mean() - out["logp_z"].mean()
        loss.backward()
        outs.append(out)
    for k in ("x_hat", "logp_y", "logp_z", "y", "z"):
        assert torch.equal(outs[0][k], outs[1][k]), k
    gp = dict(parent.named_parameters())
    for k, p in model.named_parameters():
        if k in gp:
            err = float((p.grad - gp[k].grad).norm() / max(float(gp[k].grad.norm()), 1e-30))
            assert err <= grad_tol("fp32", k), (k, err)
        else:
            assert p.grad is not None and torch.isfinite(p.grad).all(), k


# ---- forward parity --------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("arm", ["fp32", "bf16x3"])
@pytest.mark.parametrize("M", [128, 192])
def test_forward_matches_oracle(M, arm):
    """Random log-gains (std 0.5), fractional and mixed per-image qualities: symbols against the oracle's (mismatches only at
    rounding ties), p_y / p_z / x_hat against the oracle evaluated on the device's symbols."""
    model = seeded_gained(M, 3, "calib" if M == 128 else "calib192", arm, log_std=0.5)
    sd = _sd(model)
    x = H.seeded_input((2, 3, 256, 384))
    q = [1.37, 4.5]
    ref = OG.forward(sd, x, M, 3, q)
    with torch.no_grad():
        out = model.to(DEV)(x.to(DEV), training=False, quality=q)
    assert torch.equal(out["quality"].cpu(), ref["quality"])
    for name in ("y_in", "z_in"):
        pre = ref[name[0]]
        real, ties = H.symbol_mismatches(out[name].cpu().numpy(), ref[name].numpy(), pre.numpy(), H.TIE_TAU)
        assert real == 0 and ties <= H.tie_flip_bound(out[name[0]].cpu().numpy(), pre.numpy()), (name, real, ties)
    y_in, z_in = out["y_in"].cpu(), out["z_in"].cpu()
    g = OG.gains(sd, OG.snap(q, 6, 2))
    with torch.no_grad():
        psi = O.hyper_synthesis(sd, g["z_log_inv_gain"][:, :, None, None] * z_in)
        raw = O.entropy_parameters_raw(sd, torch.cat([OC.context(sd, y_in), psi], dim=1))
        p_y = O.conditional_likelihood(y_in, O.split_parameters(raw, M, 3), 3)
        p_z = O.factorized_likelihood(sd, z_in)
        x_hat = O.synthesis(sd, g["y_log_inv_gain"][:, :, None, None] * y_in)
    for name, p, p_ref in (("p_y", out["p_y"], p_y), ("p_z", out["p_z"], p_z)):
        bad, worst = H.likelihood_close(p.cpu().numpy(), p_ref.numpy())
        H.record_report(f"gained_forward[{M},{arm},{name}]", {"outliers": bad, "worst": worst})
        assert bad <= 1e-4 * p_ref.numel(), (name, bad, worst)
    err = float((out["x_hat"].cpu() - x_hat).abs().max())
    assert err <= {"fp32": 1e-4, "bf16x3": 3e-4}[arm], err


# ---- kernels ---------------------------------------------------------------------------------------------------------------------

def test_handoff_gain_is_torch_multiply_then_round():
    n, h, w, c = 3, 5, 37, 70
    v = torch.randn(n, h, w, c, device=DEV) * 6
    g, gi = torch.rand(n, c, device=DEV) * 3 + 0.1, torch.rand(n, c, device=DEV) * 3 + 0.1
    noise = torch.rand(n, c, h, w, device=DEV) - 0.5
    for qmode in (_lib.Q_ROUND, _lib.Q_NOISE, _lib.Q_PASSTHRU):
        y, y_in, sym, src, scaled = engine.latent_handoff_gain(v, qmode, noise if qmode == _lib.Q_NOISE else None, g, gi,
                                                               torch.float32, torch.float32, torch.float32)
        yg = v * g[:, None, None, :]
        q = {_lib.Q_ROUND: torch.round(yg), _lib.Q_NOISE: yg + noise.permute(0, 2, 3, 1), _lib.Q_PASSTHRU: yg}[qmode]
        assert torch.equal(y, yg.permute(0, 3, 1, 2)) and torch.equal(src, yg)
        assert torch.equal(y_in, q.permute(0, 3, 1, 2)) and torch.equal(sym, q)
        assert torch.equal(scaled, q * gi[:, None, None, :])
    # pair forms: the symbols keep the lo-half flag, the scaled output is the pair of the product and carries none
    _, _, sym, src, scaled = engine.latent_handoff_gain(v, _lib.Q_ROUND, None, g, gi, "bf16x2", "bf16x2", "bf16x2")
    q = torch.round(v * g[:, None, None, :])
    assert torch.equal(engine.from_pair(sym), q) and int(sym._nic_lo_flag) == 0
    assert torch.equal(sym, engine.to_pair(q)) and torch.equal(scaled, engine.to_pair(q * gi[:, None, None, :]))
    assert torch.equal(src, engine.to_pair(v * g[:, None, None, :])) and not hasattr(scaled, "_nic_lo_flag")


def test_gain_bwd_accuracy_determinism_batch_invariance():
    from neural_image_compression_b200.training import gain_bwd
    n, hw, c = 4, 1536, 192
    grad, other = torch.randn(n, hw, c, device=DEV), torch.randn(n, hw, c, device=DEV) * 3
    f = torch.rand(n, c, device=DEV) + 0.5
    dst, dg = torch.empty_like(grad), torch.empty(n, c, device=DEV)
    gain_bwd(grad, f, other, n, c, hw, dst, False, dg)
    ref = (grad.double() * other.double()).sum(1)
    assert float((dg.double() - ref).norm() / ref.norm()) <= 1e-6
    assert torch.equal(dst, grad * f[:, None, :])
    acc = torch.ones_like(grad)
    gain_bwd(grad, f, None, n, c, hw, acc, True, None)
    assert torch.equal(acc, 1 + grad * f[:, None, :])
    for _ in range(2):
        dg2 = torch.empty_like(dg)
        gain_bwd(grad, f, other, n, c, hw, None, False, dg2)
        assert torch.equal(dg2, dg)
    one = torch.empty(1, c, device=DEV)
    gain_bwd(grad[2:3].contiguous(), f[2:3].contiguous(), other[2:3].contiguous(), 1, c, hw, None, False, one)
    assert torch.equal(one[0], dg[2])


def test_gain_vectors_and_fold():
    model = seeded_gained(64, 1, "plain", "fp32", levels=5, log_std=0.5).to(DEV)
    q = [0.0, 1.5, 3.999, 4.0, 2.25]
    gains = model.gains(q, 5, DEV)
    ref = OG.gains(_sd(model), OG.snap(q, 5, 5))
    for k, name in enumerate(OG.TABLES):
        torch.testing.assert_close(gains.vec[k].cpu(), ref[name], rtol=2e-7, atol=0)
    again = model.gains(torch.tensor(q, device=DEV), 5, DEV)                 # device quality: same codes, same bits
    assert torch.equal(again.q_code, gains.q_code) and torch.equal(again.vec, gains.vec)
    with pytest.raises(ValueError, match="quality"):
        model.gains(4.01, 5, DEV)


# ---- gradients -------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("distortion", ["mse", "ms-ssim"])
@pytest.mark.parametrize("arm", ["fp32", "bf16x3"])
def test_step_gradients_match_oracle(arm, distortion):
    from neural_image_compression_b200.training import step_gradients
    from tests.test_gpu_train import grad_tol
    model = seeded_gained(128, 3, "calib", "fp32", log_std=0.2)
    sd = _sd(model)
    x = H.seeded_input((2, 3, 192, 192))
    q, lam = [0.75, 3.0], [0.004, 0.02]
    # two 192 x 192 images (MS-SSIM needs a smaller side above 160): draws keep the LeakyReLU pre-activations 3e-7 from 0, no more
    _, nz, ny = OG.noise_with_margin(sd, x, 128, 3, q, 21, margin=3e-7)
    ref_loss, ref_g = OG.loss_and_grads(sd, x, 128, 3, q, nz, ny, lam, distortion=distortion)
    model = model.to(DEV)
    model.train_precision = arm
    loss, _, _ = step_gradients(model, x.to(DEV), torch.tensor(lam, device=DEV), noise=(nz.to(DEV), ny.to(DEV)), distortion=distortion,
                                quality=q)
    torch.cuda.synchronize()
    assert abs(float(loss) - ref_loss) <= (1e-5 if arm == "fp32" else 5e-5) * abs(ref_loss), (float(loss), ref_loss)
    worst = {k: float((p.grad.double().cpu() - ref_g[k].double()).norm() / max(float(ref_g[k].double().norm()), 1e-30))
             for k, p in model.named_parameters()}
    assert set(worst) == set(ref_g)
    print(arm, distortion, "worst gradient errors:", sorted(worst.items(), key=lambda kv: -kv[1])[:6])
    H.record_report(f"gained_grads[{arm},{distortion}]", {k: worst[k] for k in sorted(worst, key=lambda k: -worst[k])[:8]})
    # the gain tables sit upstream of h_a's and h_s's LeakyReLUs: the bf16x3 arm's bar for such tensors
    bad = {k: v for k, v in worst.items() if v > (3e-2 if k.startswith("gain_units") and arm == "bf16x3" else grad_tol(arm, k))}
    assert not bad, bad


def test_autograd_route_equals_step_gradients():
    from neural_image_compression_b200.training import step_gradients
    from neural_image_compression_b200.RateDistortionLoss import rd_loss
    model = seeded_gained(128, 3, "calib", "fp32", log_std=0.2).to(DEV)
    x = H.seeded_input((1, 3, 128, 192)).to(DEV)
    nz, ny = torch.rand(1, 128, 2, 3, device=DEV) - 0.5, torch.rand(1, 128, 8, 12, device=DEV) - 0.5
    model.zero_grad()
    rd_loss(model(x, quality=2.3, noise=(nz, ny)), x, LAMBDA)["loss"].backward()
    auto = {k: p.grad.clone() for k, p in model.named_parameters()}
    assert all(auto[f"gain_units.{n}"].abs().sum() > 0 for n in OG.TABLES)
    model.zero_grad()
    step_gradients(model, x, LAMBDA, noise=(nz, ny), quality=2.3)
    for k, p in model.named_parameters():
        assert torch.equal(p.grad, auto[k]), k


def test_graphed_trainer_with_lambdas_steps_like_the_eager_one():
    from neural_image_compression_b200 import parallel
    x = H.seeded_input((4, 3, 192, 192)).to(DEV)
    lambdas = [0.002, 0.004, 0.008, 0.016, 0.032, 0.064]
    with pytest.raises(ValueError, match="levels"):
        parallel.ShardedTrainer(seeded_gained(128, 3), lambdas=lambdas[:5])
    with pytest.raises(ValueError, match="gain units"):
        parallel.ShardedTrainer(seeded_cb(128, 3), lambdas=lambdas)
    losses = {}
    for mode in (False, True):
        torch.manual_seed(11)
        model = seeded_gained(128, 3, "calib", "bf16x3").to(DEV)
        tr = parallel.ShardedTrainer(model, lambdas=lambdas, lr=1e-4, graph=mode)
        losses[mode] = [float(tr.step(x)["loss"].detach()) for _ in range(30)]
        assert any(float(t.detach().abs().sum()) > 0 for t in model.gain_units.tables())
        torch.cuda.synchronize()
    print("losses", losses)
    for mode in (False, True):
        assert all(math.isfinite(v) for v in losses[mode])
        assert np.mean(losses[mode][-5:]) < np.mean(losses[mode][:5]), (mode, losses[mode])
    # each step draws its own levels (lambdas 32x apart), so single losses scatter: compare the means of the last 20 steps
    assert abs(np.mean(losses[True][-20:]) - np.mean(losses[False][-20:])) < 0.25 * np.mean(losses[False][-20:]), losses


# ---- format 5 --------------------------------------------------------------------------------------------------------------------

ROUND_TRIP = [("fp32", 1, (2, 3, 512, 768)), ("bf16x3", 3, (3, 3, 512, 768)), ("bf16x3", 3, (1, 3, 65, 63)),
              ("bf16x3", 3, (1, 3, 1080, 1920))]


@pytest.mark.parametrize("arm,K,shape", ROUND_TRIP)
def test_round_trip(arm, K, shape):
    model = seeded_gained(128, K, "calib", arm, log_std=0.3).to(DEV)
    x = H.seeded_input(shape).to(DEV)
    B, _, h, w = shape
    q = [0.0, 2.5, 5.0][:B] if B > 1 else 3.3
    with torch.no_grad():
        out = model(_pad(x), training=False, quality=q)
    enc = model.compress(x, quality=q)
    assert all(s[0] & 0x7F == 5 for s in enc["strings"][1])
    dec = model.decompress(**enc)
    assert set(dec) == {"x_hat", "y_hat", "z_hat", "quality"}
    assert torch.equal(dec["quality"], out["quality"])
    assert torch.equal(dec["y_hat"], out["y_in"]) and torch.equal(dec["z_hat"], out["z_in"])
    assert torch.equal(dec["x_hat"], out["x_hat"][..., :h, :w])
    if B > 1:                                                   # any subset, any order
        strings = enc["strings"]
        for k in range(B):
            alone = model.decompress([[s[k]] for s in strings], enc["shape"])
            for key in dec:
                assert torch.equal(alone[key], dec[key][k:k + 1]), (key, k)
        rev = model.decompress([s[::-1] for s in strings], enc["shape"])
        for key in dec:
            assert torch.equal(rev[key], dec[key].flip(0)), key
    assert _lib.load().nic_pipeline_status() == 0


@pytest.mark.parametrize("size", [(320, 256), (65, 63)])
def test_format_pinned_by_reference_coder(size):
    model = seeded_gained(128, 3, "calib", "bf16x3", log_std=0.3).to(DEV)
    x = H.seeded_input((1, 3) + size).to(DEV)
    with torch.no_grad():
        out = model(_pad(x), training=False, quality=1.6)
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    enc = model.compress(x, quality=1.6)
    (ys,), (zs,) = enc["strings"]
    # the tables of the gained parameter path (psi from ginv_z (.) z)
    B, M, hy, wy = y.shape
    path = codec.ParamPath(model, 1, hy, wy, y.device)
    gains = model.gains(1.6, 1, DEV)
    _, comb = path.hyper(z.permute(0, 2, 3, 1).contiguous(), gains.ginv_z)
    raw = path.raw(y.permute(0, 2, 3, 1).contiguous(), comb)
    rows = {}
    from oracle import rans
    for t, pixels in enumerate(rans.wavefront(hy, wy)):
        cdf, lo, n = (a.cpu().numpy() for a in codec.step_tables(raw, M, 3, t))
        cdf = cdf.view(np.uint32).astype(np.int64)
        for p, (i, j) in enumerate(pixels):
            for c in range(M):
                rows[c, i, j] = (cdf[p * M + c], int(lo[p * M + c]), int(n[p * M + c]))
    _, zrows = _gpu_tables(model, y, z)
    fy, fz = (lambda c, i, j: rows[c, i, j]), (lambda c: zrows[c])
    yo, zo, hdr = RG.decode_image(ys, zs, fy, fz, 128, *enc["shape"])
    yq, zq = y[0].cpu().numpy().astype(np.int64), z[0].cpu().numpy().astype(np.int64)
    assert np.array_equal(yo, yq) and np.array_equal(zo, zq)
    csum = int(codec.checksums(y, z).cpu().numpy().view(np.uint32)[0])
    sized = size[0] % 64 or size[1] % 64
    assert hdr == ((0x85 if sized else 5), codec.ARMS.index("bf16x3"), 128, 3, 6, 1638, csum) + (size if sized else _padded(*size))
    assert RG.encode_image(yq, zq, fy, fz, hdr[1:7], size if sized else None) == (ys, zs)


def test_corrupted_quality_fails_the_checksum():
    model = seeded_gained(128, 3, "calib", "bf16x3", log_std=0.3).to(DEV)
    x = H.seeded_input((2, 3, 256, 256)).to(DEV)
    enc = model.compress(x, quality=[2.0, 3.0])
    ys, zs = enc["strings"]
    bad = bytearray(zs[1])
    bad[6:8] = (3 * 1024 + 1).to_bytes(2, "little")                # q_code field
    with pytest.raises(ValueError, match=r"checksum mismatch .*image\(s\) \[1\]"):
        model.decompress([ys, [zs[0], bytes(bad)]], enc["shape"])


def test_rate_close_to_model_bits_and_growing_with_quality():
    model = seeded_gained(128, 3, "calib", "bf16x3")
    with torch.no_grad():
        for t in model.gain_units.tables():
            t.copy_(torch.linspace(math.log(0.25), math.log(4.0), model.levels)[:, None].expand_as(t))
        model.gain_units.y_log_inv_gain.neg_()
        model.gain_units.z_log_inv_gain.neg_()
    model = model.to(DEV)
    x = H.seeded_input((2, 3, 512, 768)).to(DEV)
    bits = []
    for q in (0.0, 1.0, 2.5, 4.0, 5.0):
        with torch.no_grad():
            out = model(x, training=False, quality=q)
        per_image, _ = rd_terms(out, x, LAMBDA)
        model_bits = (per_image[0] + per_image[1]).cpu().numpy()
        ys, zs = model.compress(x, quality=q)["strings"]
        coded = np.array([8 * (len(a) + len(b)) for a, b in zip(ys, zs)])
        assert (coded <= 1.03 * model_bits).all(), (q, coded, model_bits)
        bits.append(coded.sum())
    H.record_report("gained_codec_rate_vs_q", {"coded_bits": [int(b) for b in bits]})
    assert all(b1 > b0 for b0, b1 in zip(bits, bits[1:])), bits
