"""GPU: the entropy coder - compress() / decompress() of JointAutoregressiveHierarchical.

The determinism the decoder rests on (causality of the parameter path, batch-size invariance of the engine), lossless round
trips, the byte format against the reference coder of oracle/rans.py, the coded rate against rd_loss, and the checksum."""
import numpy as np
import pytest
import torch

from neural_image_compression_b200 import _lib, codec
from neural_image_compression_b200.RateDistortionLoss import rd_terms
from oracle import rans
from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _model(M, K, init, arm):
    return H.seeded_model(M, K, init, precision=arm).to(DEV)


def _symbols(model, x):
    with torch.no_grad():
        out = model(x, training=False)
    return out, out["y_in"] + 0.0, out["z_in"] + 0.0


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


@pytest.mark.parametrize("arm", ["fp32", "bf16x3", "bf16"])
def test_params_causal(arm):
    """The raw parameters at step t's pixels are the same bits from the full y and from y with every position of step >= t at 0."""
    model = _model(128, 3, "calib", arm)
    x = H.seeded_input((2, 3, 256, 320)).to(DEV)
    _, y, z = _symbols(model, x)
    B, M, hy, wy = y.shape
    path = codec.ParamPath(model, B, hy, wy, x.device)
    _, comb = path.hyper(_nhwc(z))
    full = path.raw(_nhwc(y), comb).clone()
    step = (3 * torch.arange(hy, device=DEV)[:, None] + torch.arange(wy, device=DEV)[None, :])
    for t in (0, 1, 7, 20, 31, 3 * hy + wy - 4):
        part = path.raw(_nhwc(y * (step < t).float()), comb)
        at = step == t
        assert torch.equal(part[:, :, at], full[:, :, at]), f"{arm}: step {t}"


@pytest.mark.parametrize("arm", ["fp32", "bf16x3", "bf16"])
def test_params_batch_invariant(arm):
    """psi and the raw parameters of an image are the same bits at n = 1 and inside a batch of 16 at 768x512 (the sizes where
    the engine switches tile forms): the decoder may see an image in another batch than the encoder did."""
    model = _model(128, 3, "calib", arm)
    x = H.seeded_input((16, 3, 512, 768)).to(DEV)
    _, y, z = _symbols(model, x)
    B, M, hy, wy = y.shape
    path = codec.ParamPath(model, B, hy, wy, x.device)
    _, comb = path.hyper(_nhwc(z))
    raw = path.raw(_nhwc(y), comb)
    one = codec.ParamPath(model, 1, hy, wy, x.device)
    for k in (0, 5, 15):
        _, comb1 = one.hyper(_nhwc(z[k:k + 1]))
        raw1 = one.raw(_nhwc(y[k:k + 1]), comb1)
        psi = torch.cat([torch.arange(2 * M, 4 * M)] + ([torch.arange(6 * M, 8 * M)] if arm == "bf16x3" else [])).to(DEV)
        assert torch.equal(comb[k:k + 1].index_select(3, psi), comb1.index_select(3, psi)), f"{arm}: psi of image {k}"
        assert torch.equal(raw[k:k + 1], raw1), f"{arm}: image {k}"


ROUND_TRIP = [(128, 3, "calib", "bf16x3"), (128, 1, "calib", "fp32"), (128, 3, "plain", "bf16x3"), (128, 3, "gain", "bf16x3"),
              (192, 1, "calib192", "bf16x3"), (128, 3, "calib", "bf16")]


@pytest.mark.parametrize("M,K,init,arm", ROUND_TRIP)
def test_round_trip(M, K, init, arm):
    model = _model(M, K, init, arm)
    x = H.seeded_input((4, 3, 256, 192)).to(DEV)
    out, _, _ = _symbols(model, x)
    enc = model.compress(x)
    ys, zs = enc["strings"]
    assert len(ys) == len(zs) == 4 and all(isinstance(s, bytes) for s in ys + zs)
    dec = model.decompress(**enc)
    assert torch.equal(dec["y_hat"], out["y_in"]) and torch.equal(dec["z_hat"], out["z_in"])
    assert torch.equal(dec["x_hat"], out["x_hat"])
    for k in range(4):
        one = model.decompress([[ys[k]], [zs[k]]], enc["shape"])
        assert torch.equal(one["y_hat"], dec["y_hat"][k:k + 1]) and torch.equal(one["z_hat"], dec["z_hat"][k:k + 1]), k
        assert torch.equal(one["x_hat"], dec["x_hat"][k:k + 1]), k
    rev = model.decompress([ys[::-1], zs[::-1]], enc["shape"])
    for key in ("y_hat", "z_hat", "x_hat"):
        assert torch.equal(rev[key], dec[key].flip(0)), key
    assert _lib.load().nic_pipeline_status() == 0


def _gpu_tables(model, y, z):
    """The integer tables the coder used, as functions for oracle/rans.py: y rows from the raw parameters of the full y (equal at
    every step's pixels to what the decoder computed, test_params_causal), z rows per channel."""
    B, M, hy, wy = y.shape
    assert B == 1
    path = codec.ParamPath(model, 1, hy, wy, y.device)
    _, comb = path.hyper(_nhwc(z))
    raw = path.raw(_nhwc(y), comb)
    rows = {}
    for t, pixels in enumerate(rans.wavefront(hy, wy)):
        cdf, lo, n = (a.cpu().numpy() for a in codec.step_tables(raw, M, model.K, t))
        cdf = cdf.view(np.uint32).astype(np.int64)
        for p, (i, j) in enumerate(pixels):
            for c in range(M):
                e = p * M + c
                rows[c, i, j] = (cdf[e], int(lo[e]), int(n[e]))
    zc, zlo, zn = (a.cpu().numpy() for a in codec.z_tables(model.factorized_entropy_model.packed(), M))
    zc = zc.view(np.uint32).astype(np.int64)
    zrows = {c: (zc[c], int(zlo[c]), int(zn[c])) for c in range(M)}
    return rows, zrows


@pytest.mark.parametrize("init", ["calib", "gain"])
def test_format_pinned_by_reference_coder(init):
    model = _model(128, 3, init, "bf16x3")
    x = H.seeded_input((1, 3, 128, 192)).to(DEV)
    _, y, z = _symbols(model, x)
    enc = model.compress(x)
    (ys,), (zs,) = enc["strings"]
    rows, zrows = _gpu_tables(model, y, z)
    for cdf, lo, n in list(rows.values()) + list(zrows.values()):              # table invariants
        assert 1 <= n <= _lib.CODEC_WINDOW
        d = np.diff(cdf[:n + 2])
        assert cdf[0] == 0 and cdf[n + 1] == 1 << 16 and d.min() >= 1
    yo, zo, hdr = rans.decode_image(ys, zs, lambda c, i, j: rows[c, i, j], lambda c: zrows[c], 128, *enc["shape"])
    yq, zq = y[0].cpu().numpy().astype(np.int64), z[0].cpu().numpy().astype(np.int64)
    assert np.array_equal(yo, yq) and np.array_equal(zo, zq)
    escapes = sum(not (rows[c, i, j][1] <= yq[c, i, j] < rows[c, i, j][1] + rows[c, i, j][2]) for (c, i, j) in rows)
    if init == "gain":
        assert escapes > 0, "the gain weights are meant to exercise the escape path"
    assert hdr[:4] == (1, codec.ARMS.index("bf16x3"), 128, 3)
    again = rans.encode_image(yq, zq, lambda c, i, j: rows[c, i, j], lambda c: zrows[c], hdr[1:])
    assert again == (ys, zs)


@pytest.mark.parametrize("K,init", [(3, "calib"), (1, "calib"), (3, "plain")])
def test_rate_close_to_rd_loss(K, init):
    model = _model(128, K, init, "bf16x3")
    x = H.seeded_input((2, 3, 512, 768)).to(DEV)
    out, _, _ = _symbols(model, x)
    per_image, _ = rd_terms(out, x, 0.005)
    model_bits = (per_image[0] + per_image[1]).cpu().numpy()
    enc = model.compress(x)
    ys, zs = enc["strings"]
    coded = np.array([8 * (len(a) + len(b)) for a, b in zip(ys, zs)])
    H.record_report(f"codec_rate[K={K},{init}]", {"coded_bits": coded.tolist(), "rd_bits": model_bits.tolist(),
                                                   "ratio": (coded / model_bits).tolist()})
    assert (coded <= 1.03 * model_bits).all(), (coded, model_bits)


def test_checksum_catches_corruption_and_other_weights():
    model = _model(128, 3, "calib", "bf16x3")
    x = H.seeded_input((2, 3, 256, 256)).to(DEV)
    enc = model.compress(x)
    ys, zs = enc["strings"]
    _, offs, words = codec.parse_string(ys[1], codec.Y_LANES, False)
    lane = int(np.argmax(words))
    pos = offs[lane] + 4 + words[lane]                         # a byte in the middle of the longest lane's words
    bad = bytearray(ys[1])
    bad[pos] ^= 0x5A
    with pytest.raises(ValueError, match=r"image\(s\) \[1\]"):
        model.decompress([[ys[0], bytes(bad)], zs], enc["shape"])
    other = _model(128, 3, "plain", "bf16x3")
    with pytest.raises(ValueError, match="checksum"):
        other.decompress(enc["strings"], enc["shape"])
    assert _lib.load().nic_pipeline_status() == 0
