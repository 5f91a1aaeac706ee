"""GPU: JointCheckerboardHierarchical - the forward against the oracle restatement (oracle/checkerboard.py), the bitwise causality of
the device parameter path the two-pass decoder rests on, the training step against the oracle's autograd gradients (MSE and MS-SSIM)
and the graphed trainer, and format 4: lossless round trips at any size, batch invariance, the bytes against the reference coder,
the coded rate and the checksum."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from neural_image_compression_b200 import _lib, checkerboard_codec, codec
from neural_image_compression_b200.ContextModels import anchor_mask
from neural_image_compression_b200.Models import JointCheckerboardHierarchical
from neural_image_compression_b200.RateDistortionLoss import rd_terms
from oracle import checkerboard as OC
from oracle import forward as O
from oracle import rans_checkerboard as RC
from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LAMBDA = 0.005


def seeded_cb(M, K, init="calib", precision="fp32"):
    """The checkerboard model with helpers.seeded_model's weights (the same seeded draw, the same re-scaling per init)."""
    torch.manual_seed(0)
    model = JointCheckerboardHierarchical(M, K=K, precision=precision)
    if init != "plain":
        model.load_state_dict(H.apply_init({k: v.clone() for k, v in model.state_dict().items()}, init))
    return model


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


# ---- forward ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("arm", ["fp32", "bf16x3"])
@pytest.mark.parametrize("M", [128, 192])
def test_forward_matches_oracle(M, arm):
    """Eval forward at 512 x 768: symbols against the oracle's (mismatches only at rounding ties), p_y / p_z / x_hat against the
    oracle evaluated on the device's symbols (so no flipped symbol's 5x5 footprint needs masking), phi exactly 0 at the anchors."""
    model = seeded_cb(M, 3, "calib" if M == 128 else "calib192", precision=arm)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    x = H.seeded_input((1, 3, 512, 768))
    ref = OC.forward(sd, x, M, 3)
    with torch.no_grad():
        out = model.to(DEV)(x.to(DEV), training=False)
    real, ties = H.symbol_mismatches(out["y_in"].cpu().numpy(), ref["y_in"].numpy(), ref["y"].numpy(), H.TIE_TAU)
    assert real == 0 and ties <= H.tie_flip_bound(out["y"].cpu().numpy(), ref["y"].numpy()), (real, ties)
    y_in, z_in = out["y_in"].cpu(), out["z_in"].cpu()
    with torch.no_grad():
        raw = OC.raw_parameters(sd, y_in, z_in)
        p_y = O.conditional_likelihood(y_in, O.split_parameters(raw, M, 3), 3)
        p_z = O.factorized_likelihood(sd, z_in)
        x_hat = O.synthesis(sd, y_in)
    for name, p, p_ref in (("p_y", out["p_y"], p_y), ("p_z", out["p_z"], p_z)):
        bad, worst = H.likelihood_close(p.cpu().numpy(), p_ref.numpy())
        H.record_report(f"checkerboard_forward[{M},{arm},{name}]", {"outliers": bad, "worst": worst})
        assert bad <= 1e-4 * p_ref.numel(), (name, bad, worst)
    err = float((out["x_hat"].cpu() - x_hat).abs().max())
    assert err <= {"fp32": 1e-4, "bf16x3": 3e-4}[arm], err
    # the context output straight from the engine: 0 at the anchors (bias included), the oracle's phi elsewhere
    ctx = model.context_model.masked
    phi = ctx._op.run(_nhwc(out["y_in"]), 1, 32, 48, "fp32", out_dtype=torch.float32)
    anchor = anchor_mask(32, 48, DEV)
    assert torch.count_nonzero(phi[:, anchor]) == 0
    np.testing.assert_allclose(phi.permute(0, 3, 1, 2).cpu().numpy(), OC.context(sd, y_in).numpy(), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_zero_kernel_windows(dtype):
    """nic_checkerboard_zero on a channel window of a wider NHWC tensor (pairs: both halves) and on NCHW: the anchors of the window
    become 0, nothing else changes."""
    lib = _lib.load()
    for pair in ((False, True) if dtype == torch.bfloat16 else (False,)):
        for layout in ((_lib.LAYOUT_NHWC,) if pair else (_lib.LAYOUT_NHWC, _lib.LAYOUT_NCHW)):
            n, h, w, c, ct, co = 2, 5, 7, 6, 16, 4
            shape = (n, h, w, ct * (2 if pair else 1)) if layout == _lib.LAYOUT_NHWC else (n, ct, h, w)
            t = torch.randn(shape, device=DEV).to(dtype) + 3
            ref = t.clone()
            dt = _lib.DT_BF16X2 if pair else (_lib.DT_F32 if dtype == torch.float32 else _lib.DT_BF16)
            _lib.check(lib.nic_checkerboard_zero(t.data_ptr(), dt, layout, n, h, w, c, ct, co, _lib.current_stream()))
            a = anchor_mask(h, w, DEV)
            chans = list(range(co, co + c)) + ([ct + k for k in range(co, co + c)] if pair else [])
            if layout == _lib.LAYOUT_NHWC:
                r = ref.clone()
                for ch in chans:
                    r[:, :, :, ch][:, a] = 0
            else:
                r = ref.clone()
                for ch in chans:
                    r[:, ch][:, a] = 0
            assert torch.equal(t, r), (dtype, pair, layout)


@pytest.mark.parametrize("arm", ["fp32", "bf16x3", "bf16"])
def test_params_causal(arm):
    """The device parameter path (codec.ParamPath): the raw parameters at the anchors are the same bits from the full y and from
    an all-zero y; those at the non-anchors the same bits from the full y and from y with every non-anchor set to 0.  So the decoder
    rebuilds the encoder's tables."""
    model = seeded_cb(128, 3, "calib", arm).to(DEV)
    x = H.seeded_input((2, 3, 256, 320)).to(DEV)
    with torch.no_grad():
        out = model(x, training=False)
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    B, M, hy, wy = y.shape
    path = codec.ParamPath(model, B, hy, wy, x.device)
    _, comb = path.hyper(_nhwc(z))
    full = path.raw(_nhwc(y), comb).clone()
    anchor = anchor_mask(hy, wy, DEV)
    zero = path.raw(_nhwc(torch.zeros_like(y)), comb)
    assert torch.equal(zero[:, :, anchor], full[:, :, anchor]), arm
    anchors_only = path.raw(_nhwc(y * anchor.float()), comb)
    assert torch.equal(anchors_only[:, :, ~anchor], full[:, :, ~anchor]), arm


# ---- training -----------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("distortion", ["mse", "ms-ssim"])
@pytest.mark.parametrize("arm", ["fp32", "bf16x3"])
def test_step_gradients_match_oracle(arm, distortion):
    from neural_image_compression_b200.training import step_gradients
    from tests.test_gpu_train import grad_tol
    model = seeded_cb(128, 3, "calib", "fp32")
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    # one 192 x 192 image: MS-SSIM needs a smaller side above 160, and at 2 x 192 x 256 no draw of 64 keeps every LeakyReLU
    # pre-activation 5e-7 away from 0
    x = H.seeded_input((1, 3, 192, 192))
    _, nz, ny = OC.noise_with_margin(sd, x, 128, 3, 21, margin=5e-7)
    ref_loss, ref_g = OC.loss_and_grads(sd, x, 128, 3, nz, ny, LAMBDA, distortion=distortion)
    model = model.to(DEV)
    model.train_precision = arm
    loss, _, _ = step_gradients(model, x.to(DEV), LAMBDA, noise=(nz.to(DEV), ny.to(DEV)), distortion=distortion)
    torch.cuda.synchronize()
    assert abs(float(loss) - ref_loss) <= (1e-5 if arm == "fp32" else 5e-5) * abs(ref_loss), (float(loss), ref_loss)
    worst = {k: float((p.grad.double().cpu() - ref_g[k].double()).norm() / max(float(ref_g[k].double().norm()), 1e-30))
             for k, p in model.named_parameters()}
    assert set(worst) == set(ref_g)
    print(arm, distortion, "worst gradient errors:", sorted(worst.items(), key=lambda kv: -kv[1])[:5])
    bad = {k: v for k, v in worst.items() if v > grad_tol(arm, k)}
    assert not bad, bad


def test_graphed_trainer_steps_like_the_eager_one():
    from neural_image_compression_b200 import parallel
    x = H.seeded_input((2, 3, 192, 192)).to(DEV)
    losses = {}
    for mode in (False, True):
        model = seeded_cb(128, 3, "calib", "bf16x3").to(DEV)
        tr = parallel.ShardedTrainer(model, LAMBDA, lr=1e-4, graph=mode)
        losses[mode] = [float(tr.step(x)["loss"].detach()) for _ in range(30)]
        torch.cuda.synchronize()
    print("losses", losses)
    assert abs(losses[True][0] - losses[False][0]) < 0.02 * losses[False][0]
    for mode in (False, True):
        assert losses[mode][-1] < losses[mode][0], (mode, losses[mode])
    assert abs(losses[True][-1] - losses[False][-1]) < 0.05 * losses[False][-1], losses


# ---- codec --------------------------------------------------------------------------------------------------------------------

def _padded(h, w):
    return 64 * (-(-h // 64)), 64 * (-(-w // 64))


def _pad(x):
    hp, wp = _padded(*x.shape[2:])
    return F.pad(x, (0, wp - x.shape[3], 0, hp - x.shape[2]), mode="replicate")


def _round_trip(model, x):
    B, _, h, w = x.shape
    with torch.no_grad():
        out = model(_pad(x), training=False)
    enc = model.compress(x)
    assert enc["shape"] == (_padded(h, w)[0] // 64, _padded(h, w)[1] // 64)
    dec = model.decompress(**enc)
    assert set(dec) == {"x_hat", "y_hat", "z_hat"}
    assert torch.equal(dec["y_hat"], out["y_in"]) and torch.equal(dec["z_hat"], out["z_in"])
    assert torch.equal(dec["x_hat"], out["x_hat"][..., :h, :w])
    return enc, dec, out


ROUND_TRIP = [("fp32", 1, (1, 3, 512, 768)), ("bf16x3", 3, (1, 3, 512, 768)), ("bf16x3", 1, (4, 3, 512, 768)), ("fp32", 3, (4, 3, 512, 768)),
              ("bf16x3", 3, (1, 3, 65, 63)), ("fp32", 1, (2, 3, 200, 328)), ("bf16x3", 3, (2, 3, 200, 328)), ("bf16x3", 3, (1, 3, 1080, 1920))]


@pytest.mark.parametrize("arm,K,shape", ROUND_TRIP)
def test_round_trip(arm, K, shape):
    model = seeded_cb(128, K, "calib", arm).to(DEV)
    x = H.seeded_input(shape).to(DEV)
    enc, dec, _ = _round_trip(model, x)
    assert all(s[0] & 0x7F == 4 for s in enc["strings"][1])
    if shape[0] > 1:                                   # batch invariance: alone, and in a reversed batch
        strings = enc["strings"]
        for k in range(shape[0]):
            one = model.compress(x[k:k + 1])
            assert [s[0] for s in one["strings"]] == [s[k] for s in strings], k
            alone = model.decompress([[s[k]] for s in strings], enc["shape"])
            for key in dec:
                assert torch.equal(alone[key], dec[key][k:k + 1]), (key, k)
        rev = model.decompress([s[::-1] for s in strings], enc["shape"])
        for key in dec:
            assert torch.equal(rev[key], dec[key].flip(0)), key
    assert _lib.load().nic_pipeline_status() == 0


def _gpu_tables(model, y, z):
    """The integer tables of the encoder, as functions for oracle/rans_checkerboard.py: y rows from the raw parameters of the full y
    (equal to the decoder's at every pass's pixels, test_params_causal), one row per element through nic_codec_tables' step form."""
    B, M, hy, wy = y.shape
    path = codec.ParamPath(model, 1, hy, wy, y.device)
    _, comb = path.hyper(_nhwc(z))
    raw = path.raw(_nhwc(y), comb)
    rows = {}
    from oracle import rans
    for t, pixels in enumerate(rans.wavefront(hy, wy)):
        cdf, lo, n = (a.cpu().numpy() for a in codec.step_tables(raw, M, model.K, t))
        cdf = cdf.view(np.uint32).astype(np.int64)
        for p, (i, j) in enumerate(pixels):
            for c in range(M):
                e = p * M + c
                rows[c, i, j] = (cdf[e], int(lo[e]), int(n[e]))
    zc, zlo, zn = (a.cpu().numpy() for a in codec.z_tables(model.factorized_entropy_model.packed(), M))
    zc = zc.view(np.uint32).astype(np.int64)
    return rows, {c: (zc[c], int(zlo[c]), int(zn[c])) for c in range(M)}


@pytest.mark.parametrize("size", [(320, 256), (65, 63)])
def test_format_pinned_by_reference_coder(size):
    model = seeded_cb(128, 3, "calib", "bf16x3").to(DEV)
    x = H.seeded_input((1, 3) + size).to(DEV)
    with torch.no_grad():
        out = model(_pad(x), training=False)
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    enc = model.compress(x)
    (ys,), (zs,) = enc["strings"]
    rows, zrows = _gpu_tables(model, y, z)
    fy, fz = (lambda c, i, j: rows[c, i, j]), (lambda c: zrows[c])
    yo, zo, hdr = RC.decode_image(ys, zs, fy, fz, 128, *enc["shape"])
    yq, zq = y[0].cpu().numpy().astype(np.int64), z[0].cpu().numpy().astype(np.int64)
    assert np.array_equal(yo, yq) and np.array_equal(zo, zq)
    csum = int(codec.checksums(y, z).cpu().numpy().view(np.uint32)[0])
    sized = size[0] % 64 or size[1] % 64
    assert hdr == ((0x84 if sized else 4), codec.ARMS.index("bf16x3"), 128, 3, csum) + (size if sized else _padded(*size))
    assert RC.encode_image(yq, zq, fy, fz, hdr[1:5], size if sized else None) == (ys, zs)


@pytest.mark.parametrize("K", [3, 1])
def test_rate_close_to_model_bits(K):
    model = seeded_cb(128, K, "calib", "bf16x3").to(DEV)
    x = H.seeded_input((2, 3, 512, 768)).to(DEV)
    with torch.no_grad():
        out = model(x, training=False)
    per_image, _ = rd_terms(out, x, LAMBDA)
    model_bits = (per_image[0] + per_image[1]).cpu().numpy()
    ys, zs = model.compress(x)["strings"]
    coded = np.array([8 * (len(a) + len(b)) for a, b in zip(ys, zs)])
    H.record_report(f"checkerboard_codec_rate[K={K}]", {"coded_bits": coded.tolist(), "rd_bits": model_bits.tolist(),
                                                         "ratio": (coded / model_bits).tolist()})
    assert (coded <= 1.03 * model_bits).all(), (coded, model_bits)


def test_checksum_catches_a_flipped_byte():
    model = seeded_cb(128, 3, "calib", "bf16x3").to(DEV)
    x = H.seeded_input((2, 3, 256, 256)).to(DEV)
    enc = model.compress(x)
    ys, zs = enc["strings"]
    lc, lr = checkerboard_codec.y_lanes(128, 16)
    _, offs, words = codec.parse_string(ys[1], lc * lr, False)
    lane = int(np.argmax(words))
    bad = bytearray(ys[1])
    bad[offs[lane] + 4 + words[lane]] ^= 0x5A
    with pytest.raises(ValueError, match=r"checksum mismatch .*image\(s\) \[1\]"):
        model.decompress([[ys[0], bytes(bad)], zs], enc["shape"])
    assert _lib.load().nic_pipeline_status() == 0


def test_decode_is_at_least_4x_faster():
    """The decode of tools/checkerboard_codec_bench.py's two models (M = 128, K = 3, bf16x3, calib weights), alternated call by call:
    the checkerboard decode at least 4x faster than the mask-'A' wavefront decode at 768 x 512 with B = 16 and at 3024 x 4032."""
    import os
    import statistics
    import sys
    sys.path.insert(0, os.path.join(H.ROOT, "tools"))
    from checkerboard_codec_bench import models, wall
    ms = {name: make().to(DEV) for name, make in models().items()}
    for B, Hh, W in ((16, 512, 768), (1, 3024, 4032)):
        x = H.seeded_input((B, 3, Hh, W)).to(DEV)
        encs = {name: m.compress(x) for name, m in ms.items()}
        times = {name: [] for name in ms}
        for _ in range(3):                                  # a warm-up call, then two timed ones, alternated
            for name, m in ms.items():
                times[name].append(wall(lambda: m.decompress(**encs[name]))[0])
        med = {name: statistics.median(t[1:]) for name, t in times.items()}
        speedup = med["JointAutoregressiveHierarchical"] / med["JointCheckerboardHierarchical"]
        H.record_report(f"checkerboard_decode_speedup[{B}x{W}x{Hh}]", {"decode_s": med, "speedup": speedup})
        assert speedup >= 4.0, (B, Hh, W, med)
        del x, encs
        torch.cuda.empty_cache()
