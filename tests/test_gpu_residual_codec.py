"""GPU: the coder of HierarchicalMixtureResidual - the one-launch step decode (nic_codec_decode_step) against the table + decode
pair it replaces, model-free and bit for bit; lossless round trips in both arms; the byte format against the reference coder of
oracle/rans_residual.py; the coded rate against the model's; corruption detection."""
import numpy as np
import pytest
import torch

from neural_image_compression_b200 import _lib, codec, scalable_codec as sc
from neural_image_compression_b200._lib import CODEC_GM, check, current_stream, ptr
from neural_image_compression_b200.RateDistortionLoss import rd_terms
from oracle import rans, rans_residual
from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CALIB = (17.98, 141.28)                 # g_a / h_a output gains of the residual parity cases: rates of a trained model


def _model(M, K, arm, gains=CALIB, sigma_bias=3.0):
    return H.seeded_residual_model(M, K, *gains, precision=arm, sigma_bias=sigma_bias).to(DEV)


def _forward(model, x):
    with torch.no_grad():
        return model(x, training=False)


# ---- the step kernel against the pair, model-free -------------------------------------------------------------------------------

def _random_latent(B, M, K, hy, wy, seed):
    """Raw parameters with sigmas from 0.05 to ~30 and means up to +-60 (windows that clip at 128 bins), symbols around the first
    component with 2 % far outliers: both the window and the escape path are exercised."""
    g = torch.Generator().manual_seed(seed)
    np_ = 2 if K == 1 else 3 * K
    raw = torch.empty((B, np_, M, hy, wy))
    mu_at, s_at = (0, 1) if K == 1 else (K, 2 * K)
    if K > 1:
        raw[:, :K] = torch.randn((B, K, M, hy, wy), generator=g)
    raw[:, mu_at:mu_at + K] = torch.randn((B, K, M, hy, wy), generator=g) * 20
    raw[:, s_at:s_at + K] = torch.rand((B, K, M, hy, wy), generator=g) * 33 - 3
    sigma = torch.nn.functional.softplus(raw[:, s_at])
    sym = torch.round(raw[:, mu_at] + sigma * torch.randn((B, M, hy, wy), generator=g) * 2)
    far = torch.rand((B, M, hy, wy), generator=g) < 0.02
    sym[far] = torch.randint(-50000, 50000, (int(far.sum()),), generator=g).float()
    return raw.reshape(B, np_ * M, hy, wy).to(DEV), sym.to(DEV).contiguous()


@pytest.mark.parametrize("B,M,K,hy,wy,cut", [(1, 192, 1, 96, 128, False),     # 258 rows per lane and step: five chunks
                                            (3, 24, 3, 8, 12, False),         # fewer channels than lanes, B > 1
                                            (2, 192, 3, 16, 24, True)])       # lane 5 of image 1 runs out of words
def test_step_kernel_matches_table_decode_pair(B, M, K, hy, wy, cut):
    lib = _lib.load()
    raw, sym = _random_latent(B, M, K, hy, wy, seed=B * 1000 + M)
    lanes = codec.lanes(codec.Y_LANES, M)
    words, count = codec._encode(CODEC_GM, codec._symbol_codes(CODEC_GM, raw, sym, K), sym, lanes)
    cap = words.shape[1]
    g = torch.arange(B * lanes, device=DEV)
    lane_off = ((g * cap + cap - count) * 2).long()                 # byte offsets of the segments inside `words`
    lane_words = (count - 2).int()
    if cut:
        lane_words[lanes + 5] //= 2
    blob = words.view(torch.uint8)
    out = [torch.zeros((B, hy, wy, M), device=DEV) for _ in range(2)]
    state = [torch.zeros(B * lanes, dtype=torch.int32, device=DEV) for _ in range(2)]
    pos = [torch.zeros(B * lanes, dtype=torch.int32, device=DEV) for _ in range(2)]
    tabs, st = None, current_stream()
    escapes = 0
    for t in range(3 * hy + wy - 3):
        check(lib.nic_codec_decode_step(ptr(blob), ptr(lane_off), ptr(lane_words), ptr(state[0]), ptr(pos[0]), int(t == 0), ptr(raw),
                                        B, M, K, hy, wy, lanes, t, ptr(out[0]), st), "nic_codec_decode_step")
        tabs = codec.step_tables(raw, M, K, t, tabs)
        check(lib.nic_codec_decode(CODEC_GM, ptr(blob), ptr(lane_off), ptr(lane_words), ptr(state[1]), ptr(pos[1]), int(t == 0),
                                   ptr(tabs[0]), ptr(tabs[1]), ptr(tabs[2]), B, M, hy, wy, lanes, t, ptr(out[1]), st), "nic_codec_decode")
        assert torch.equal(out[0], out[1]), f"symbols after step {t}"
        assert torch.equal(state[0], state[1]) and torch.equal(pos[0], pos[1]), f"lane cursors after step {t}"
        rows = [(i, t - 3 * i) for i in range(hy) if 0 <= t - 3 * i < wy]
        n = tabs[2][:B * len(rows) * M].view(B, len(rows), M)
        lo = tabs[1][:B * len(rows) * M].view(B, len(rows), M)
        s = torch.stack([sym[:, :, i, j] for i, j in rows], dim=1)
        escapes += int(((s < lo) | (s >= lo + n)).sum())
    got = out[0].permute(0, 3, 1, 2)
    if cut:
        lost = torch.zeros_like(got, dtype=torch.bool)
        lost[1, 5::lanes] = True
        assert not torch.equal(got[lost], sym[lost]), "the cut lane should have decoded zeros past its end"
        assert torch.equal(got[~lost], sym[~lost])
        assert int((pos[0][lanes + 5] > lane_words[lanes + 5]).item()) == 1
    else:
        assert torch.equal(got, sym)
        assert torch.equal(pos[0], lane_words)
    assert escapes > 0
    assert lib.nic_pipeline_status() == 0


# ---- round trips ----------------------------------------------------------------------------------------------------------------

def _check_round_trip(model, x):
    out = _forward(model, x)
    enc = model.compress(x)
    ys, zs = enc["strings"]
    assert len(ys) == len(zs) == x.shape[0] and all(isinstance(s, bytes) for s in ys + zs)
    dec = model.decompress(**enc)
    for key, ref in (("y_hat", out["y_in"]), ("z_hat", out["z_in"]), ("x_hat", out["x_hat"])):
        assert torch.equal(dec[key], ref), key
    return enc, dec


ROUND_TRIP = [(192, 1, "bf16x3"), (192, 3, "bf16x3"), (192, 1, "fp32"), (192, 3, "fp32"), (128, 1, "bf16x3"), (96, 3, "fp32")]


@pytest.mark.parametrize("M,K,arm", ROUND_TRIP)
def test_round_trip(M, K, arm):
    """y_hat / z_hat / x_hat equal the eval forward's at the same batch.  Decoding an image alone or in a reversed list gives the
    same y_hat / z_hat bits, and - at these shapes - the same x_hat bits: the 3x3 g_s on the conv engine computes an image the
    same way at B = 1 and B = 3 (the maximum difference is recorded as well)."""
    model = _model(M, K, arm)
    x = H.seeded_input((3, 3, 256, 192)).to(DEV)
    enc, dec = _check_round_trip(model, x)
    ys, zs = enc["strings"]
    diffs = []
    for k in range(3):
        one = model.decompress([[ys[k]], [zs[k]]], enc["shape"])
        for key in ("y_hat", "z_hat"):
            assert torch.equal(one[key], dec[key][k:k + 1]), (key, k)
        diffs.append(float((one["x_hat"] - dec["x_hat"][k:k + 1]).abs().max()))
    rev = model.decompress([ys[::-1], zs[::-1]], enc["shape"])
    for key in ("y_hat", "z_hat"):
        assert torch.equal(rev[key], dec[key].flip(0)), key
    diffs.append(float((rev["x_hat"] - dec["x_hat"].flip(0)).abs().max()))
    H.record_report(f"residual_codec_x_hat_batch[{M},{K},{arm}]", {"max_abs_diff": diffs})
    assert max(diffs) == 0.0, diffs
    assert _lib.load().nic_pipeline_status() == 0


def test_round_trip_2048x1536():
    _check_round_trip(_model(192, 1, "bf16x3"), H.seeded_input((1, 3, 1536, 2048)).to(DEV))
    assert _lib.load().nic_pipeline_status() == 0


# ---- format, rate, corruption ---------------------------------------------------------------------------------------------------

def _gpu_tables(model, y, z):
    """The integer tables the coder used, as functions for the reference coder (step tables from the all-pixels parameters: equal
    at every step's pixels to the decoder's, test_gpu_scalable_codec.py::test_params_kernel_bitwise_invariances)."""
    _, _, hy, wy = y.shape
    M, K = model.M, model.K
    heads = sc.ParamHeads(model, [y.permute(0, 2, 3, 1).contiguous()], sc.psi_nhwc(model, z.permute(0, 2, 3, 1).contiguous()), True)
    heads.run(-1)
    rows = {}
    for t, pixels in enumerate(rans.wavefront(hy, wy)):
        cdf, lo, n = (a.cpu().numpy() for a in codec.step_tables(heads.raw[0], M, K, t))
        cdf = cdf.view(np.uint32).astype(np.int64)
        for p, (pi, pj) in enumerate(pixels):
            for c in range(M):
                e = p * M + c
                rows[c, pi, pj] = (cdf[e], int(lo[e]), int(n[e]))
    zc, zlo, zn = (a.cpu().numpy() for a in codec.z_tables(model.factorized_entropy_model.packed(), M))
    zc = zc.view(np.uint32).astype(np.int64)
    return rows, {c: (zc[c], int(zlo[c]), int(zn[c])) for c in range(M)}


@pytest.mark.parametrize("gains,K,arm", [(CALIB, 3, "bf16x3"), ((136.2, 141.28), 1, "fp32")])
def test_format_pinned_by_reference_coder(gains, K, arm):
    model = _model(192, K, arm, gains)
    x = H.seeded_input((1, 3, 128, 192)).to(DEV)
    out = _forward(model, x)
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    enc = model.compress(x)
    (ys,), (zs,) = enc["strings"]
    rows, zrows = _gpu_tables(model, y, z)
    fy, fz = (lambda c, i, j: rows[c, i, j]), (lambda c: zrows[c])
    yo, zo, hdr = rans_residual.decode_residual_image(ys, zs, fy, fz, *enc["shape"])
    yq, zq = y[0].cpu().numpy().astype(np.int64), z[0].cpu().numpy().astype(np.int64)
    assert np.array_equal(yo, yq) and np.array_equal(zo, zq)
    assert hdr[:4] == (3, codec.ARMS.index(arm), 192, K)
    if gains != CALIB:
        escapes = sum(not (r[1] <= yq[c, i, j] < r[1] + r[2]) for (c, i, j), r in rows.items())
        assert escapes > 0, "the gain weights are meant to exercise the escape path"
    assert rans_residual.encode_residual_image(yq, zq, fy, fz, hdr[1:]) == (ys, zs)


def test_rate_close_to_model():
    model = _model(192, 3, "bf16x3")
    x = H.seeded_input((2, 3, 512, 768)).to(DEV)
    out = _forward(model, x)
    per_image, _ = rd_terms(out, x, 0.005)
    by, bz = per_image[:2].double().cpu().numpy()
    enc = model.compress(x)
    coded = np.array([8 * (len(a) + len(b)) for a, b in zip(*enc["strings"])])
    H.record_report("residual_codec_rate[192,K=3,calib]", {"ratio": (coded / (by + bz)).tolist()})
    assert (coded <= 1.03 * (by + bz)).all(), (coded, by + bz)


def _flip(s, lanes):
    _, offs, words = codec.parse_string(s, lanes, False)
    lane = int(np.argmax(words))
    bad = bytearray(s)
    bad[offs[lane] + 4 + words[lane]] ^= 0x5A                  # a byte in the middle of the longest lane's words
    return bytes(bad)


def test_corruption_is_caught():
    model = _model(192, 1, "bf16x3")
    x = H.seeded_input((2, 3, 256, 256)).to(DEV)
    enc = model.compress(x)
    ys, zs = enc["strings"]
    with pytest.raises(ValueError, match=r"checksum mismatch in image\(s\) \[1\]"):
        model.decompress([[ys[0], _flip(ys[1], 32)], zs], enc["shape"])
    with pytest.raises(ValueError, match="checksum"):
        _model(192, 1, "bf16x3", sigma_bias=0.0).decompress(enc["strings"], enc["shape"])
    assert _lib.load().nic_pipeline_status() == 0
