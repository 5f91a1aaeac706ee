"""GPU: images of any size through the three coders (DESIGN.md section 12) - the window kernel against F.pad / slicing, round trips
whose symbols are the eval forward's of the edge-padded image and whose x_hat is its crop, batch invariance at the new shapes, the
unchanged path for sides that are multiples of 64, the sized byte format against the reference coders, the coded rate, and a
corrupted size field."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from neural_image_compression_b200 import _lib, codec
from neural_image_compression_b200.RateDistortionLoss import rd_terms
from oracle import rans_sized
from tests import helpers as H
from tests.test_gpu_codec import _gpu_tables as jah_tables
from tests.test_gpu_residual_codec import CALIB
from tests.test_gpu_residual_codec import _gpu_tables as residual_tables
from tests.test_gpu_scalable_codec import _gpu_tables as scalable_tables

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _padded(h, w):
    return 64 * (-(-h // 64)), 64 * (-(-w // 64))


def _pad(x):
    hp, wp = _padded(*x.shape[2:])
    return F.pad(x, (0, wp - x.shape[3], 0, hp - x.shape[2]), mode="replicate")


# ---- the window kernel ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("B,h,w,hp,wp", [(1, 1, 1, 64, 64), (1, 65, 63, 128, 64), (1, 1080, 1920, 1088, 1920), (3, 200, 328, 256, 384),
                                         (1, 3024, 4032, 3072, 4032)])
def test_window_pads_and_crops_exactly(B, h, w, hp, wp):
    torch.manual_seed(h * w)
    x = torch.randn((B, 3, h, w), device=DEV)
    pad = codec.window(x, hp, wp)
    assert torch.equal(pad, F.pad(x, (0, wp - w, 0, hp - h), mode="replicate"))
    assert torch.equal(codec.window(pad, h, w), x)
    y = torch.randn((B, 3, hp, wp), device=DEV)
    assert torch.equal(codec.window(y, h, w), y[..., :h, :w])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs a second device")
def test_window_runs_on_the_tensors_device():
    """The window launches on its input's device and that device's current stream, whatever device is current."""
    x = torch.randn((1, 3, 65, 63), device="cuda:1")
    with torch.cuda.device(0):
        pad = codec.window(x, 128, 64)
    assert pad.device == x.device
    assert torch.equal(pad, F.pad(x, (0, 1, 0, 63), mode="replicate"))


def test_compress_input_checks():
    """An image without pixels, or a side above 65535 that is not a multiple of 64 (the size field is 16-bit): ValueError before
    any launch."""
    lib = _lib.load()
    for name in MODELS:
        model = MODELS[name]()
        for shape in ((1, 3, 0, 64), (1, 3, 1, 65537), (1, 3, 65537, 1)):
            before = lib.nic_launch_count()
            with pytest.raises(ValueError):
                model.compress(torch.zeros(shape, device=DEV))
            assert lib.nic_launch_count() == before, (name, shape)


# ---- round trips ----------------------------------------------------------------------------------------------------------------

def _jah(M=128, K=3, arm="bf16x3"):
    return H.seeded_model(M, K, "calib", precision=arm).to(DEV)


def _scalable(arm="bf16x3"):
    return H.seeded_scalable_model(192, 128, 1, "calib", precision=arm).to(DEV)


def _residual(arm="bf16x3"):
    return H.seeded_residual_model(192, 1, *CALIB, precision=arm).to(DEV)


MODELS = {"jah": _jah, "scalable": _scalable, "residual": _residual}


def _check_round_trip(model, x):
    """compress / decompress of x against the eval forward of its padded image; -> (enc, dec, forward outputs)."""
    B, _, h, w = x.shape
    with torch.no_grad():
        out = model(_pad(x), training=False)
    enc = model.compress(x)
    assert enc["shape"] == (_padded(h, w)[0] // 64, _padded(h, w)[1] // 64)
    z = enc["strings"][-1]
    assert len(z) == B and all(s[0] & codec.SIZED for s in z)
    dec = model.decompress(**enc)
    refs = {"y_hat": out["y_in"], "z_hat": out["z_in"], "x_hat": out["x_hat"][..., :h, :w]}
    if "y1" in out:
        refs.update(y1_hat=out["y1"], y2_hat=out["y2"])
        base = model.decompress([enc["strings"][0], None, z], enc["shape"], base_only=True)
        assert torch.equal(base["y1_hat"], out["y1"]) and torch.equal(base["z_hat"], out["z_in"])
    assert set(dec) == set(refs)
    for key, ref in refs.items():
        assert torch.equal(dec[key], ref), key
    return enc, dec, out


def _check_batch_invariance(model, x, enc, dec):
    """Image k compressed alone gives the batch's bytes; decoded alone or in a reversed batch it gives the batch's tensors."""
    strings = enc["strings"]
    for k in range(x.shape[0]):
        one = model.compress(x[k:k + 1])
        assert [s[0] for s in one["strings"]] == [s[k] for s in strings], k
        alone = model.decompress([[s[k]] for s in strings], enc["shape"])
        for key in dec:
            assert torch.equal(alone[key], dec[key][k:k + 1]), (key, k)
    rev = model.decompress([s[::-1] for s in strings], enc["shape"])
    for key in dec:
        assert torch.equal(rev[key], dec[key].flip(0)), key


ROUND_TRIP = [("jah", dict(arm="bf16x3")), ("jah", dict(M=64, arm="fp32")), ("scalable", dict(arm="bf16x3")),
              ("residual", dict(arm="bf16x3")), ("residual", dict(arm="fp32"))]


@pytest.mark.parametrize("name,kw", ROUND_TRIP, ids=[f"{n}-{'-'.join(map(str, kw.values()))}" for n, kw in ROUND_TRIP])
def test_round_trips(name, kw):
    model = MODELS[name](**kw)
    _check_round_trip(model, H.seeded_input((1, 3, 65, 63)).to(DEV))
    x = H.seeded_input((2, 3, 200, 328)).to(DEV)
    enc, dec, _ = _check_round_trip(model, x)
    _check_batch_invariance(model, x, enc, dec)


def _model_bits(name, out, xp):
    """Per image (coded-bit bound for all strings, for the base layer or None) of the model's rate on the padded image."""
    if name == "scalable":
        bits = []
        for key in ("logp_y1", "logp_y2"):
            per_image, _ = rd_terms({"x_hat": out["x_hat"], "logp_y": out[key], "logp_z": out["logp_z"]}, xp, 0.005)
            bits.append(per_image[:2].double().cpu().numpy())
        return bits[0][0] + bits[1][0] + bits[0][1], bits[0][0] + bits[0][1]
    per_image, _ = rd_terms(out, xp, 0.005)
    return (per_image[0] + per_image[1]).double().cpu().numpy(), None


def _header_size(name):
    from neural_image_compression_b200 import scalable_codec
    return scalable_codec.HEADER.size if name == "scalable" else codec.HEADER.size


@pytest.mark.parametrize("name", list(MODELS))
def test_1080p(name):
    """Round trip of a 1080 x 1920 image (z latent 17 x 30, y latent 68 x 120); the coded bits against the model's rate on the
    padded image at each model's rate-test bound (1.03); W = 1920 rewritten as 1919 in the size field (the same latent shape)
    fails the checksum."""
    model = MODELS[name]()
    x = H.seeded_input((1, 3, 1080, 1920)).to(DEV)
    enc, _, out = _check_round_trip(model, x)
    assert enc["shape"] == (17, 30)
    total, base = _model_bits(name, out, _pad(x))
    coded = np.array([8 * sum(len(s[0]) for s in enc["strings"])])
    ratio = {"ratio": (coded / total).tolist()}
    assert (coded <= 1.03 * total).all(), (coded, total)
    if base is not None:
        coded_base = np.array([8 * (len(enc["strings"][0][0]) + len(enc["strings"][2][0]))])
        ratio["base_ratio"] = (coded_base / base).tolist()
        assert (coded_base <= 1.03 * base).all(), (coded_base, base)
    H.record_report(f"any_size_codec_rate_1080p[{name}]", ratio)
    z = enc["strings"][-1][0]
    at = _header_size(name) + 2
    assert int.from_bytes(z[at:at + 2], "little") == 1920
    bad = enc["strings"][:-1] + [[z[:at] + (1919).to_bytes(2, "little") + z[at + 2:]]]
    with pytest.raises(ValueError, match=r"checksum mismatch .*image\(s\) \[0\]"):
        model.decompress(bad, enc["shape"])


def test_multiples_of_64_stay_unsized():
    x = H.seeded_input((1, 3, 512, 768)).to(DEV)
    xp, size = codec.any_size_input(x)
    assert xp is x and size is None
    for version, name in enumerate(MODELS, start=1):
        model = MODELS[name]()
        enc = model.compress(x)
        z = enc["strings"][-1][0]
        assert z[0] == version, name
        dec = model.decompress(**enc)
        assert dec["x_hat"].shape == x.shape


# ---- the sized byte format against the reference coders -------------------------------------------------------------------------

@pytest.mark.parametrize("name", list(MODELS))
def test_sized_format_pinned_by_reference_coder(name):
    model = MODELS[name]()
    x = H.seeded_input((1, 3, 65, 63)).to(DEV)
    with torch.no_grad():
        out = model(_pad(x), training=False)
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    enc = model.compress(x)
    strings = [s[0] for s in enc["strings"]]
    yq, zq = y[0].cpu().numpy().astype(np.int64), z[0].cpu().numpy().astype(np.int64)
    arm = codec.ARMS.index(model.precision)
    if name == "scalable":
        M1 = model.M1
        rows, zrows = scalable_tables(model, y, z)
        f1, f2, fz = (lambda c, i, j: rows[0][c, i, j]), (lambda c, i, j: rows[1][c, i, j]), (lambda c: zrows[c])
        y1o, y2o, zo, hdr = rans_sized.decode_sized_image(2, *strings, f1, f2, fz, *enc["shape"])
        assert np.array_equal(y1o, yq[:M1]) and np.array_equal(y2o, yq[M1:]) and np.array_equal(zo, zq)
        sums = [int(v) for v in codec.checksums(y[:, :M1].contiguous(), z).cpu().numpy().view(np.uint32)] + \
               [int(v) for v in codec.checksums(y[:, M1:].contiguous(), z).cpu().numpy().view(np.uint32)]
        assert hdr == (0x82, arm, 192, M1, 1, *sums, 65, 63)
        again = rans_sized.encode_sized_image(2, hdr[7:], yq[:M1], yq[M1:], zq, f1, f2, fz, hdr[1:7])
    else:
        rows, zrows = (jah_tables if name == "jah" else residual_tables)(model, y, z)
        fy, fz = (lambda c, i, j: rows[c, i, j]), (lambda c: zrows[c])
        version = 1 if name == "jah" else 3
        yo, zo, hdr = rans_sized.decode_sized_image(version, *strings, fy, fz, *((model.M,) if version == 1 else ()), *enc["shape"])
        assert np.array_equal(yo, yq) and np.array_equal(zo, zq)
        csum = int(codec.checksums(y, z).cpu().numpy().view(np.uint32)[0])
        assert hdr == (0x80 | version, arm, model.M, model.K, csum, 65, 63)
        again = rans_sized.encode_sized_image(version, hdr[5:], yq, zq, fy, fz, hdr[1:5])
    assert list(again) == strings
