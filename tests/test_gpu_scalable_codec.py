"""GPU: the layered coder of ScalableImageCoding - the step-local parameter kernel against the oracle and its bitwise invariances
(the decoder's determinism rests on them), lossless round trips of both layers, the byte format against the reference coder of
oracle/rans.py, the coded rate against the model's, and per-layer corruption detection."""
import numpy as np
import pytest
import torch

from neural_image_compression_b200 import _lib, codec, scalable_codec as sc
from neural_image_compression_b200.RateDistortionLoss import rd_terms
from oracle import forward as O
from oracle import rans, rans_scalable
from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _model(M, M1, K, arm, init="calib"):
    return H.seeded_scalable_model(M, M1, K, init, precision=arm).to(DEV)


def _forward(model, x):
    with torch.no_grad():
        return model(x, training=False)


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _params(model, y, z, all_pixels=True, psi=None):
    """(psi, ParamHeads) over the symbols y (NCHW, both heads), z."""
    psi = sc.psi_nhwc(model, _nhwc(z)) if psi is None else psi
    yn = _nhwc(y)
    return psi, sc.ParamHeads(model, [yn[..., :model.M1].contiguous(), yn[..., model.M1:].contiguous()], psi, all_pixels)


@pytest.mark.parametrize("M,M1,K,arm", [(192, 128, 3, "bf16x3"), (128, 64, 1, "fp32")])
def test_params_kernel_matches_oracle(M, M1, K, arm):
    """Raw parameters of both heads over every pixel against the oracle's context conv + 1x1 stack in float64 on the same symbols,
    psi and weights.  Tolerance: fp32 chains of at most 12 * 128 + 640 + 640 terms through 4 layers - 2e-5 of the largest
    magnitude of the head's parameters plus 2e-5 relative (measured errors are a few 1e-7 relative)."""
    model = _model(M, M1, K, arm)
    x = H.seeded_input((2, 3, 128, 192)).to(DEV)
    out = _forward(model, x)
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    psi, heads = _params(model, y, z)
    heads.run(-1)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    psi64 = psi.permute(0, 3, 1, 2).double().cpu()
    for i, (yi, raw) in enumerate(zip(torch.split(y, [M1, M - M1], dim=1), heads.raw), start=1):
        phi = O.context(sd, yi.double().cpu(), dtype=torch.float64, prefix=f"context_model_{i}")
        ref = O.entropy_parameters_raw(sd, torch.cat([phi, psi64], dim=1), dtype=torch.float64, prefix=f"entropy_parameters_{i}")
        got = raw.double().cpu()
        err = (got - ref).abs()
        bound = 2e-5 * ref.abs().max() + 2e-5 * ref.abs()
        H.record_report(f"scalable_params_vs_oracle[{M},{M1},{K},{arm},head{i}]",
                        {"max_abs_err": float(err.max()), "max_ref": float(ref.abs().max())})
        assert bool((err <= bound).all()), (i, float(err.max()), float(ref.abs().max()))


def test_params_kernel_bitwise_invariances():
    """At 768 x 512 (16 pixels per step and image): step launches equal the all-pixels launch at the step's pixels, an image's
    values are the same at B = 1 and inside B = 4, and values at step t do not change when every position of step >= t is zero."""
    model = _model(192, 128, 3, "bf16x3")
    x = H.seeded_input((4, 3, 512, 768)).to(DEV)
    out = _forward(model, x)
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    B, _, hy, wy = y.shape
    psi, full = _params(model, y, z)
    full.run(-1)
    full_raw = [r.clone() for r in full.raw]
    step = 3 * torch.arange(hy, device=DEV)[:, None] + torch.arange(wy, device=DEV)[None, :]
    steps = (0, 1, (3 * hy + wy - 3) // 2, 3 * hy + wy - 4)
    _, part = _params(model, y, z, all_pixels=False, psi=psi)
    for t in steps:
        part.run(t)
        at = step == t
        for i in range(2):
            assert torch.equal(part.raw[i][:, :, at], full_raw[i][:, :, at]), f"step launch, head {i + 1}, step {t}"
    for k in (0, 3):
        _, one = _params(model, y[k:k + 1], z[k:k + 1], psi=psi[k:k + 1].contiguous())
        one.run(-1)
        for i in range(2):
            assert torch.equal(one.raw[i], full_raw[i][k:k + 1]), f"image {k} at B = 1, head {i + 1}"
        assert torch.equal(sc.psi_nhwc(model, _nhwc(z[k:k + 1])), psi[k:k + 1]), f"psi of image {k}"
    for t in steps:
        _, cut = _params(model, y * (step < t).float(), z, all_pixels=False, psi=psi)
        cut.run(t)
        at = step == t
        for i in range(2):
            assert torch.equal(cut.raw[i][:, :, at], full_raw[i][:, :, at]), f"causality, head {i + 1}, step {t}"


def _check_round_trip(model, x):
    out = _forward(model, x)
    B = x.shape[0]
    enc = model.compress(x)
    y1s, y2s, zs = enc["strings"]
    assert len(y1s) == len(y2s) == len(zs) == B and all(isinstance(s, bytes) for s in y1s + y2s + zs)
    dec = model.decompress(**enc)
    for key, ref in (("y1_hat", out["y1"]), ("y2_hat", out["y2"]), ("y_hat", out["y_in"]), ("z_hat", out["z_in"]),
                     ("x_hat", out["x_hat"])):
        assert torch.equal(dec[key], ref), key
    base = model.decompress([y1s, None, zs], enc["shape"], base_only=True)
    assert set(base) == {"y1_hat", "z_hat"}
    assert torch.equal(base["y1_hat"], out["y1"]) and torch.equal(base["z_hat"], out["z_in"])
    return enc, dec


ROUND_TRIP = [(192, 128, 1, "bf16x3"), (192, 128, 3, "bf16x3"), (192, 128, 1, "fp32"), (192, 128, 3, "fp32"), (128, 64, 3, "fp32")]


@pytest.mark.parametrize("M,M1,K,arm", ROUND_TRIP)
def test_round_trip(M, M1, K, arm):
    model = _model(M, M1, K, arm)
    x = H.seeded_input((3, 3, 256, 192)).to(DEV)
    enc, dec = _check_round_trip(model, x)
    y1s, y2s, zs = enc["strings"]
    for k in range(3):
        one = model.decompress([[y1s[k]], [y2s[k]], [zs[k]]], enc["shape"])
        for key in ("y_hat", "z_hat", "x_hat"):
            assert torch.equal(one[key], dec[key][k:k + 1]), (key, k)
    rev = model.decompress([y1s[::-1], y2s[::-1], zs[::-1]], enc["shape"])
    for key in ("y1_hat", "y2_hat", "z_hat", "x_hat"):
        assert torch.equal(rev[key], dec[key].flip(0)), key
    assert _lib.load().nic_pipeline_status() == 0


def test_round_trip_2048x1536():
    _check_round_trip(_model(192, 128, 1, "bf16x3"), H.seeded_input((1, 3, 1536, 2048)).to(DEV))
    assert _lib.load().nic_pipeline_status() == 0


def _gpu_tables(model, y, z):
    """The integer tables the coder used, per head and for z, as functions for oracle/rans.py (step tables from the all-pixels
    parameters: equal at every step's pixels to the decoder's, test_params_kernel_bitwise_invariances)."""
    _, _, hy, wy = y.shape
    _, heads = _params(model, y, z)
    heads.run(-1)
    rows = [{}, {}]
    for t, pixels in enumerate(rans.wavefront(hy, wy)):
        for i, m in enumerate((model.M1, model.M2)):
            cdf, lo, n = (a.cpu().numpy() for a in codec.step_tables(heads.raw[i], m, model.K, t))
            cdf = cdf.view(np.uint32).astype(np.int64)
            for p, (pi, pj) in enumerate(pixels):
                for c in range(m):
                    e = p * m + c
                    rows[i][c, pi, pj] = (cdf[e], int(lo[e]), int(n[e]))
    zc, zlo, zn = (a.cpu().numpy() for a in codec.z_tables(model.factorized_entropy_model.packed(), model.M))
    zc = zc.view(np.uint32).astype(np.int64)
    return rows, {c: (zc[c], int(zlo[c]), int(zn[c])) for c in range(model.M)}


@pytest.mark.parametrize("init,K", [("calib", 3), ("gain", 1)])
def test_format_pinned_by_reference_coder(init, K):
    model = _model(192, 128, K, "bf16x3", init)
    x = H.seeded_input((1, 3, 128, 192)).to(DEV)
    out = _forward(model, x)
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    enc = model.compress(x)
    (s1,), (s2,), (sz,) = enc["strings"]
    rows, zrows = _gpu_tables(model, y, z)
    f1, f2, fz = (lambda c, i, j: rows[0][c, i, j]), (lambda c, i, j: rows[1][c, i, j]), (lambda c: zrows[c])
    y1o, y2o, zo, hdr = rans_scalable.decode_scalable_image(s1, s2, sz, f1, f2, fz, *enc["shape"])
    yq, zq = y[0].cpu().numpy().astype(np.int64), z[0].cpu().numpy().astype(np.int64)
    assert np.array_equal(y1o, yq[:128]) and np.array_equal(y2o, yq[128:]) and np.array_equal(zo, zq)
    assert hdr[:5] == (2, codec.ARMS.index("bf16x3"), 192, 128, K)
    if init == "gain":
        escapes = sum(not (r[1] <= yq[c, i, j] < r[1] + r[2]) for (c, i, j), r in rows[0].items())
        assert escapes > 0, "the gain weights are meant to exercise the escape path"
    assert rans_scalable.encode_scalable_image(yq[:128], yq[128:], zq, f1, f2, fz, hdr[1:]) == (s1, s2, sz)


def test_rate_close_to_model():
    model = _model(192, 128, 3, "bf16x3")
    x = H.seeded_input((2, 3, 512, 768)).to(DEV)
    out = _forward(model, x)
    bits = []
    for key in ("logp_y1", "logp_y2"):
        per_image, _ = rd_terms({"x_hat": out["x_hat"], "logp_y": out[key], "logp_z": out["logp_z"]}, x, 0.005)
        bits.append(per_image[:2].double().cpu().numpy())
    b1, bz, b2 = bits[0][0], bits[0][1], bits[1][0]
    enc = model.compress(x)
    y1s, y2s, zs = enc["strings"]
    base = np.array([8 * (len(a) + len(c)) for a, c in zip(y1s, zs)])
    total = base + np.array([8 * len(s) for s in y2s])
    H.record_report("scalable_codec_rate[192,128,K=3,calib]", {"base_ratio": (base / (b1 + bz)).tolist(),
                                                               "total_ratio": (total / (b1 + b2 + bz)).tolist()})
    assert (base <= 1.03 * (b1 + bz)).all(), (base, b1 + bz)
    assert (total <= 1.03 * (b1 + b2 + bz)).all(), (total, b1 + b2 + bz)


def _flip(s, lanes):
    _, offs, words = codec.parse_string(s, lanes, False)
    lane = int(np.argmax(words))
    bad = bytearray(s)
    bad[offs[lane] + 4 + words[lane]] ^= 0x5A                  # a byte in the middle of the longest lane's words
    return bytes(bad)


def test_corruption_is_caught_per_layer():
    model = _model(192, 128, 1, "bf16x3")
    x = H.seeded_input((2, 3, 256, 256)).to(DEV)
    out = _forward(model, x)
    enc = model.compress(x)
    y1s, y2s, zs = enc["strings"]
    bad_y2 = [y2s[0], _flip(y2s[1], 32)]
    with pytest.raises(ValueError, match=r"enhancement layer \(y2\) in image\(s\) \[1\]"):
        model.decompress([y1s, bad_y2, zs], enc["shape"])
    base = model.decompress([y1s, bad_y2, zs], enc["shape"], base_only=True)
    assert torch.equal(base["y1_hat"], out["y1"]) and torch.equal(base["z_hat"], out["z_in"])
    with pytest.raises(ValueError, match=r"base layer \(y1 and z\) in image\(s\) \[0\]"):
        model.decompress([[_flip(y1s[0], 32), y1s[1]], None, zs], enc["shape"], base_only=True)
    with pytest.raises(ValueError, match="checksum"):
        _model(192, 128, 1, "bf16x3", "plain").decompress(enc["strings"], enc["shape"])
    assert _lib.load().nic_pipeline_status() == 0
