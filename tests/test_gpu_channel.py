"""GPU: ChannelCheckerboardHierarchical - one slice computing exactly JointCheckerboardHierarchical, the forward against the oracle
restatement (oracle/channel.py), the bitwise causality of the device parameter path for every slice pass, the training step against
the oracle's autograd gradients (MSE and MS-SSIM), the autograd node and the graphed trainer, and format 6: lossless round trips at any
size, batch invariance, the bytes against the reference coder, the coded rate, the checksum and the decode speed."""
import numpy as np
import pytest
import torch

from neural_image_compression_b200 import _lib, channel_codec, codec
from neural_image_compression_b200.ContextModels import anchor_mask
from neural_image_compression_b200.Models import ChannelCheckerboardHierarchical
from neural_image_compression_b200.RateDistortionLoss import rd_loss, rd_terms
from oracle import channel as OCH
from oracle import checkerboard as OC
from oracle import forward as O
from oracle import rans_channel as RCH
from tests import helpers as H
from tests.test_channel_host import parent_as_one_slice, seeded_channel
from tests.test_gpu_checkerboard import ROUND_TRIP, _pad, _padded, _round_trip, seeded_cb

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LAMBDA = 0.005


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _outputs_equal(a, b):
    assert set(a) == set(b)
    for k in a:
        if torch.is_tensor(a[k]):
            assert torch.equal(a[k].detach(), b[k].detach()), k
        else:
            assert a[k] == b[k], k


# ---- one slice is the parent ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("arm", ["fp32", "bf16x3"])
def test_one_slice_is_the_parent(arm):
    """slices=(M,) with the parent's weights under remapped keys: the eval forward, the training forward under autograd and the
    gradients of one step are the parent's bits."""
    from neural_image_compression_b200.training import step_gradients
    parent = seeded_cb(128, 3, "calib", arm).to(DEV)
    model = ChannelCheckerboardHierarchical(128, K=3, slices=(128,), precision=arm)
    model.load_state_dict(parent_as_one_slice(parent.state_dict()))
    model = model.to(DEV)
    x = H.seeded_input((2, 3, 256, 320)).to(DEV)
    with torch.no_grad():
        _outputs_equal(model(x, training=False), parent(x, training=False))
    torch.manual_seed(4)
    noise = (torch.rand(2, 128, 4, 5, device=DEV) - 0.5, torch.rand(2, 128, 16, 20, device=DEV) - 0.5)
    _outputs_equal(model(x, noise=noise), parent(x, noise=noise))
    for m in (model, parent):
        m.zero_grad()
        step_gradients(m, x, LAMBDA, noise=noise)
    new_key = {old: new for new, old in parent_as_one_slice({k: k for k, _ in parent.named_parameters()}).items()}
    mp = dict(model.named_parameters())
    for k, p in parent.named_parameters():
        assert torch.equal(mp[new_key[k]].grad, p.grad), k


# ---- forward ------------------------------------------------------------------------------------------------------------------

FORWARD = [(128, (64, 64)), (192, (64, 64, 64)), (192, (64, 128))]


@pytest.mark.parametrize("arm", ["fp32", "bf16x3"])
@pytest.mark.parametrize("M,slices", FORWARD)
def test_forward_matches_oracle(M, slices, arm):
    """Eval forward at 512 x 768 at the checkerboard tests' tolerances: symbols against the oracle's (mismatches only at rounding
    ties), p_y / p_z / x_hat against the oracle evaluated on the device's symbols, phi_sp of every slice exactly 0 at the anchors."""
    model = seeded_channel(M, 3, slices, "calib" if M == 128 else "calib192", precision=arm)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    x = H.seeded_input((1, 3, 512, 768))
    ref = OCH.forward(sd, x, M, 3, slices)
    with torch.no_grad():
        out = model.to(DEV)(x.to(DEV), training=False)
    assert out["p_y"].shape == (1, M, 32, 48) and out["mus"].shape == (1, 3, M, 32, 48)
    real, ties = H.symbol_mismatches(out["y_in"].cpu().numpy(), ref["y_in"].numpy(), ref["y"].numpy(), H.TIE_TAU)
    assert real == 0 and ties <= H.tie_flip_bound(out["y"].cpu().numpy(), ref["y"].numpy()), (real, ties)
    y_in, z_in = out["y_in"].cpu(), out["z_in"].cpu()
    with torch.no_grad():
        raws = OCH.raw_parameters(sd, y_in, z_in, slices)
        p_y = torch.cat([O.conditional_likelihood(y_in[:, o:o + m], O.split_parameters(r, m, 3), 3)
                         for o, m, r in zip(OCH.offsets(slices), slices, raws)], dim=1)
        p_z = O.factorized_likelihood(sd, z_in)
        x_hat = O.synthesis(sd, y_in)
    for name, p, p_ref in (("p_y", out["p_y"], p_y), ("p_z", out["p_z"], p_z)):
        bad, worst = H.likelihood_close(p.cpu().numpy(), p_ref.numpy())
        H.record_report(f"channel_forward[{M},{slices},{arm},{name}]", {"outliers": bad, "worst": worst})
        assert bad <= 1e-4 * p_ref.numel(), (name, bad, worst)
    assert torch.allclose(out["logp_y"].sum(), torch.log(out["p_y"]).sum(), rtol=1e-6)
    err = float((out["x_hat"].cpu() - x_hat).abs().max())
    assert err <= {"fp32": 1e-4, "bf16x3": 3e-4}[arm], err
    anchor = anchor_mask(32, 48, DEV)
    for s, (o, m) in enumerate(zip(OCH.offsets(slices), slices)):
        ctx = model.context_models[s].masked
        phi = ctx._op.run(_nhwc(out["y_in"][:, o:o + m]), 1, 32, 48, "fp32", out_dtype=torch.float32)
        assert torch.count_nonzero(phi[:, anchor]) == 0, s
        np.testing.assert_allclose(phi.permute(0, 3, 1, 2).cpu().numpy(),
                                   OC.context(sd, y_in[:, o:o + m], prefix=f"context_models.{s}").numpy(), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("arm", ["fp32", "bf16x3"])
def test_params_causal_per_slice_pass(arm):
    """The device parameter path (channel_codec.SlicePath): for every slice s, the raw parameters at its anchors are the same bits
    from the full y and from y with slices >= s zeroed (pass 0), those at its non-anchors the same bits from the full y and from y
    with slice s's non-anchors and every later slice zeroed (pass 1).  So the decoder rebuilds the encoder's tables."""
    model = seeded_channel(192, 3, (64, 64, 64), "calib192", arm).to(DEV)
    x = H.seeded_input((2, 3, 256, 320)).to(DEV)
    with torch.no_grad():
        out = model(x, training=False)
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    B, M, hy, wy = y.shape
    path = channel_codec.SlicePath(model, B, hy, wy, x.device)
    path.hyper(_nhwc(z))
    anchor = anchor_mask(hy, wy, DEV)
    y_eng = path.symbols(_nhwc(y))
    for s, (o, m) in enumerate(zip(model.offsets, model.slices)):
        full = path.raw(s, y_eng).clone()
        pass0 = y.clone()
        pass0[:, o:] = 0
        got = path.raw(s, path.symbols(_nhwc(pass0)))
        assert torch.equal(got[:, :, anchor], full[:, :, anchor]), (arm, s)
        pass1 = pass0.clone()
        pass1[:, o:o + m] = y[:, o:o + m] * anchor.float()
        got = path.raw(s, path.symbols(_nhwc(pass1)))
        assert torch.equal(got[:, :, ~anchor], full[:, :, ~anchor]), (arm, s)


# ---- training -----------------------------------------------------------------------------------------------------------------

def _grad_tol(arm, key):
    """tests/test_gpu_train.py's grad_tol with this model's keys: the tensors behind a LeakyReLU get 3e-2 in the bf16x3 arm."""
    if arm == "fp32":
        return 2e-4
    exposed = key.startswith(("hyper_encoder.", "hyper_decoder.", "context_models.", "channel_contexts.")) or \
        (key.startswith("entropy_parameters.") and (".net.0." in key or ".net.2." in key))
    return 3e-2 if exposed else 5e-4


@pytest.mark.parametrize("distortion", ["mse", "ms-ssim"])
@pytest.mark.parametrize("arm", ["fp32", "bf16x3"])
def test_step_gradients_match_oracle(arm, distortion):
    from neural_image_compression_b200.training import step_gradients
    slices = (64, 64)
    model = seeded_channel(128, 3, slices, "calib", "fp32")
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    x = H.seeded_input((1, 3, 192, 192))
    _, nz, ny = OCH.noise_with_margin(sd, x, 128, 3, slices, 21, margin=5e-7)
    ref_loss, ref_g = OCH.loss_and_grads(sd, x, 128, 3, slices, nz, ny, LAMBDA, distortion=distortion)
    model = model.to(DEV)
    model.train_precision = arm
    loss, _, _ = step_gradients(model, x.to(DEV), LAMBDA, noise=(nz.to(DEV), ny.to(DEV)), distortion=distortion)
    torch.cuda.synchronize()
    assert abs(float(loss) - ref_loss) <= (1e-5 if arm == "fp32" else 5e-5) * abs(ref_loss), (float(loss), ref_loss)
    worst = {k: float((p.grad.double().cpu() - ref_g[k].double()).norm() / max(float(ref_g[k].double().norm()), 1e-30))
             for k, p in model.named_parameters()}
    assert set(worst) == set(ref_g)
    print(arm, distortion, "worst gradient errors:", sorted(worst.items(), key=lambda kv: -kv[1])[:5])
    bad = {k: v for k, v in worst.items() if v > _grad_tol(arm, k)}
    assert not bad, bad


def test_autograd_matches_step_gradients():
    """model(x) under autograd + rd_loss(...).backward(): the node splits g_logp_y per slice; the gradients are step_gradients'."""
    from neural_image_compression_b200.training import step_gradients
    model = seeded_channel(192, 1, (64, 128), "calib192", "fp32").to(DEV)
    x = H.seeded_input((2, 3, 128, 192)).to(DEV)
    torch.manual_seed(2)
    noise = (torch.rand(2, 192, 2, 3, device=DEV) - 0.5, torch.rand(2, 192, 8, 12, device=DEV) - 0.5)
    model.zero_grad()
    rd_loss(model(x, noise=noise), x, LAMBDA)["loss"].backward()
    auto = {k: p.grad.clone() for k, p in model.named_parameters()}
    model.zero_grad()
    step_gradients(model, x, LAMBDA, noise=noise)
    for k, p in model.named_parameters():
        assert torch.allclose(p.grad, auto[k], rtol=1e-5, atol=1e-8), k


def test_graphed_trainer_steps_like_the_eager_one():
    from neural_image_compression_b200 import parallel
    x = H.seeded_input((2, 3, 192, 192)).to(DEV)
    losses = {}
    for mode in (False, True):
        model = seeded_channel(128, 3, (64, 64), "calib", "bf16x3").to(DEV)
        tr = parallel.ShardedTrainer(model, LAMBDA, lr=1e-4, graph=mode)
        losses[mode] = [float(tr.step(x)["loss"].detach()) for _ in range(30)]
        torch.cuda.synchronize()
    print("losses", losses)
    assert abs(losses[True][0] - losses[False][0]) < 0.02 * losses[False][0]
    for mode in (False, True):
        assert losses[mode][-1] < losses[mode][0], (mode, losses[mode])
    assert abs(losses[True][-1] - losses[False][-1]) < 0.05 * losses[False][-1], losses


# ---- codec --------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("arm,K,shape", ROUND_TRIP)
def test_round_trip(arm, K, shape):
    model = seeded_channel(128, K, (64, 64), "calib", arm).to(DEV)
    x = H.seeded_input(shape).to(DEV)
    enc, dec, _ = _round_trip(model, x)
    assert all(s[0] & 0x7F == 6 for s in enc["strings"][1])
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


def test_round_trip_uneven_slices():
    model = seeded_channel(192, 3, (64, 128), "calib192", "bf16x3").to(DEV)
    _round_trip(model, H.seeded_input((2, 3, 200, 328)).to(DEV))
    assert _lib.load().nic_pipeline_status() == 0


def _gpu_tables(model, y, z):
    """The integer tables of the encoder, as functions for oracle/rans_channel.py: each slice's rows from its raw parameters over the
    full y (equal to the decoder's at every pass's pixels, test_params_causal_per_slice_pass), one row per element through
    nic_codec_tables' step form."""
    from oracle import rans
    B, M, hy, wy = y.shape
    path = channel_codec.SlicePath(model, 1, hy, wy, y.device)
    path.hyper(_nhwc(z))
    y_eng = path.symbols(_nhwc(y))
    rows = {}
    for s, (o, m) in enumerate(zip(model.offsets, model.slices)):
        raw = path.raw(s, y_eng)
        for t, pixels in enumerate(rans.wavefront(hy, wy)):
            cdf, lo, n = (a.cpu().numpy() for a in codec.step_tables(raw, m, model.K, t))
            cdf = cdf.view(np.uint32).astype(np.int64)
            for p, (i, j) in enumerate(pixels):
                for c in range(m):
                    e = p * m + c
                    rows[o + c, i, j] = (cdf[e], int(lo[e]), int(n[e]))
    zc, zlo, zn = (a.cpu().numpy() for a in codec.z_tables(model.factorized_entropy_model.packed(), M))
    zc = zc.view(np.uint32).astype(np.int64)
    return rows, {c: (zc[c], int(zlo[c]), int(zn[c])) for c in range(M)}


@pytest.mark.parametrize("size", [(320, 256), (65, 63)])
def test_format_pinned_by_reference_coder(size):
    model = seeded_channel(128, 3, (64, 64), "calib", "bf16x3").to(DEV)
    x = H.seeded_input((1, 3) + size).to(DEV)
    with torch.no_grad():
        out = model(_pad(x), training=False)
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    enc = model.compress(x)
    (ys,), (zs,) = enc["strings"]
    rows, zrows = _gpu_tables(model, y, z)
    fy, fz = (lambda c, i, j: rows[c, i, j]), (lambda c: zrows[c])
    yo, zo, hdr = RCH.decode_image(ys, zs, fy, fz, *enc["shape"])
    yq, zq = y[0].cpu().numpy().astype(np.int64), z[0].cpu().numpy().astype(np.int64)
    assert np.array_equal(yo, yq) and np.array_equal(zo, zq)
    csum = int(codec.checksums(y, z).cpu().numpy().view(np.uint32)[0])
    sized = size[0] % 64 or size[1] % 64
    assert hdr == ((0x86 if sized else 6), codec.ARMS.index("bf16x3"), 128, 3, (64, 64), csum) + (size if sized else _padded(*size))
    assert RCH.encode_image(yq, zq, fy, fz, (hdr[1], 128, 3, csum), (64, 64), size if sized else None) == (ys, zs)


@pytest.mark.parametrize("K", [3, 1])
def test_rate_close_to_model_bits(K):
    model = seeded_channel(128, K, (64, 64), "calib", "bf16x3").to(DEV)
    x = H.seeded_input((2, 3, 512, 768)).to(DEV)
    with torch.no_grad():
        out = model(x, training=False)
    per_image, _ = rd_terms(out, x, LAMBDA)
    model_bits = (per_image[0] + per_image[1]).cpu().numpy()
    ys, zs = model.compress(x)["strings"]
    coded = np.array([8 * (len(a) + len(b)) for a, b in zip(ys, zs)])
    H.record_report(f"channel_codec_rate[K={K}]", {"coded_bits": coded.tolist(), "rd_bits": model_bits.tolist(),
                                                    "ratio": (coded / model_bits).tolist()})
    assert (coded <= 1.03 * model_bits).all(), (coded, model_bits)


def test_checksum_catches_a_flipped_byte():
    model = seeded_channel(128, 3, (64, 64), "calib", "bf16x3").to(DEV)
    x = H.seeded_input((2, 3, 256, 256)).to(DEV)
    enc = model.compress(x)
    ys, zs = enc["strings"]
    n = sum(ln for _, ln in channel_codec.slice_lanes(model.slices, 16))
    _, offs, words = codec.parse_string(ys[1], n, False)
    lane = int(np.argmax(words))
    bad = bytearray(ys[1])
    bad[offs[lane] + 4 + words[lane]] ^= 0x5A
    with pytest.raises(ValueError, match=r"checksum mismatch .*image\(s\) \[1\]"):
        model.decompress([[ys[0], bytes(bad)], zs], enc["shape"])
    assert _lib.load().nic_pipeline_status() == 0


def test_decode_is_at_least_4x_faster_than_mask_a():
    """The decode of the channel model of tools/channel_codec_bench.py (M = 128, K = 3, bf16x3, calib weights) against the mask-'A'
    wavefront decode of the same trunk, alternated call by call: at least 4x faster at 768 x 512 with B = 16 and at 3024 x 4032."""
    import os
    import statistics
    import sys
    sys.path.insert(0, os.path.join(H.ROOT, "tools"))
    from channel_codec_bench import models
    from checkerboard_codec_bench import wall
    ms = {"JointAutoregressiveHierarchical": H.seeded_model(128, 3, "calib", precision="bf16x3").to(DEV),
          "ChannelCheckerboardHierarchical": models(128)["ChannelCheckerboardHierarchical"]().to(DEV)}
    for B, Hh, W in ((16, 512, 768), (1, 3024, 4032)):
        x = H.seeded_input((B, 3, Hh, W)).to(DEV)
        encs = {name: m.compress(x) for name, m in ms.items()}
        times = {name: [] for name in ms}
        for _ in range(3):                                  # a warm-up call, then two timed ones, alternated
            for name, m in ms.items():
                times[name].append(wall(lambda: m.decompress(**encs[name]))[0])
        med = {name: statistics.median(t[1:]) for name, t in times.items()}
        speedup = med["JointAutoregressiveHierarchical"] / med["ChannelCheckerboardHierarchical"]
        H.record_report(f"channel_decode_speedup[{B}x{W}x{Hh}]", {"decode_s": med, "speedup": speedup})
        print("decode", B, Hh, W, med, speedup)
        assert speedup >= 4.0, (B, Hh, W, med)
        del x, encs
        torch.cuda.empty_cache()
