"""CPU: GainedCheckerboardHierarchical without a GPU - construction, state_dict keys and seeded weights equal to the parent's, loading
a parent checkpoint with strict=False, the quality snapping and interpolation rule, the oracle at zero gains against the checkerboard
oracle, the format-5 reference coder, and the host-side validation of format-5 strings, which raises before any launch."""
import math

import numpy as np
import pytest
import torch

from neural_image_compression_b200 import checkerboard_codec, codec, gained_codec
from neural_image_compression_b200.Models import GainedCheckerboardHierarchical, JointCheckerboardHierarchical, quality_codes
from oracle import checkerboard as OC
from oracle import gained as OG
from oracle import rans_checkerboard as RC
from oracle import rans_gained as RG
from tests.test_checkerboard_host import _image


def test_construction_matches_the_parent():
    torch.manual_seed(0)
    a = JointCheckerboardHierarchical(64, K=3).state_dict()
    torch.manual_seed(0)
    model = GainedCheckerboardHierarchical(64, K=3, levels=5)
    b = model.state_dict()
    names = ("y_log_gain", "y_log_inv_gain", "z_log_gain", "z_log_inv_gain")
    assert list(b) == list(a) + [f"gain_units.{n}" for n in names]
    for k in a:
        assert torch.equal(a[k], b[k]), k
    for n in names:
        assert b[f"gain_units.{n}"].shape == (5, 64) and torch.count_nonzero(b[f"gain_units.{n}"]) == 0
    assert model.levels == 5 and isinstance(model, JointCheckerboardHierarchical)
    assert GainedCheckerboardHierarchical(16).levels == 6


@pytest.mark.parametrize("levels", [1, 65, 0, 2.0, True])
def test_levels_out_of_range_raise(levels):
    with pytest.raises(ValueError, match="levels"):
        GainedCheckerboardHierarchical(16, levels=levels)


def test_parent_checkpoint_loads_with_strict_false():
    torch.manual_seed(1)
    parent = JointCheckerboardHierarchical(16, K=1)
    model = GainedCheckerboardHierarchical(16, K=1, levels=3)
    res = model.load_state_dict(parent.state_dict(), strict=False)
    assert sorted(res.missing_keys) == sorted(f"gain_units.{n}" for n in OG.TABLES) and not res.unexpected_keys
    for k, v in parent.state_dict().items():
        assert torch.equal(model.state_dict()[k], v)
    with pytest.raises(RuntimeError):
        model.load_state_dict(parent.state_dict())


def test_quality_snapping():
    cpu = torch.device("cpu")
    assert quality_codes(6, None, 2, cpu).tolist() == [5120, 5120]
    assert quality_codes(6, 0.3, 3, cpu).tolist() == [307] * 3                     # 307.2 -> 307
    assert quality_codes(6, [0, 2.5, 5], 3, cpu).tolist() == [0, 2560, 5120]
    assert quality_codes(3, torch.tensor([1 / 2048, 0.75 / 1024]), 2, cpu).tolist() == [1, 1]   # halves round up
    assert quality_codes(6, [0, 2.5, 5], 3, cpu).tolist() == OG.snap([0, 2.5, 5], 6, 3).tolist()
    for bad in (-0.01, 5.001, float("nan"), [1, 2]):
        with pytest.raises(ValueError, match="quality"):
            quality_codes(6, bad, 3, cpu)


def test_interpolation_rule():
    L, M = 4, 3
    torch.manual_seed(2)
    sd = {f"gain_units.{n}": torch.randn(L, M) for n in OG.TABLES}
    q_code = OG.snap([0.0, 1.25, 2.5, 3.0], L, 4)
    g = OG.gains(sd, q_code)
    tab = sd["gain_units.y_log_gain"]
    assert torch.allclose(g["y_log_gain"][0], tab[0].exp())
    assert torch.allclose(g["y_log_gain"][1], (0.75 * tab[1] + 0.25 * tab[2]).exp())
    assert torch.allclose(g["y_log_gain"][2], (0.5 * tab[2] + 0.5 * tab[3]).exp())
    assert torch.allclose(g["y_log_gain"][3], tab[3].exp())                   # l + 1 clamped to L - 1


@pytest.mark.parametrize("training", [False, True])
def test_oracle_at_zero_gains_is_the_checkerboard_oracle(training):
    M, K = 16, 3
    torch.manual_seed(0)
    sd = GainedCheckerboardHierarchical(M, K=K, levels=4).state_dict()
    x = torch.rand(2, 3, 64, 128)
    nz, ny = torch.rand(2, M, 1, 2) - 0.5, torch.rand(2, M, 4, 8) - 0.5
    got = OG.forward(sd, x, M, K, [0.7, 3.0], training=training, noise_z=nz, noise_y=ny)
    ref = OC.forward(sd, x, M, K, training=training, noise_z=nz, noise_y=ny)
    for k in ("x_hat", "y", "y_in", "z", "z_in", "p_y", "p_z", "weights", "mus", "sigmas"):
        assert torch.equal(got[k], ref[k]), k
    assert got["quality"].tolist() == [717 / 1024, 3.0]


def _header_fields(M, L=6, q_code=2560, csum=0x12345678):
    return (codec.ARMS.index("fp32"), M, 1, L, q_code, csum)


@pytest.mark.parametrize("M,hz,wz,size", [(3, 1, 2, None), (40, 5, 1, None), (5, 2, 2, (65, 127))])
def test_reference_coder_round_trips(M, hz, wz, size):
    """Format 5 through the reference coder; the product's host parser reads the quality, size, checksum and lane table it writes,
    and the y string is format 4's."""
    rng = np.random.default_rng(M + hz)
    y, z, ty, tz = _image(rng, M, hz, wz)
    ys, zs = RG.encode_image(y, z, ty, tz, _header_fields(M), size)
    yo, zo, hdr = RG.decode_image(ys, zs, ty, tz, M, hz, wz)
    assert np.array_equal(yo, y) and np.array_equal(zo, z)
    assert hdr == ((5 | (0x80 if size else 0)), 0, M, 1, 6, 2560, 0x12345678) + (size or (64 * hz, 64 * wz))
    assert zs[0] == (0x85 if size else 5) and len(zs) >= gained_codec.HEADER.size
    ys4, zs4 = RC.encode_image(y, z, ty, tz, (0, M, 1, 0x12345678), size)
    assert ys == ys4
    field = gained_codec.HEADER.unpack_from(zs, 0)[6]
    want = (0x12345678 + RG.quality_term(6, 2560)) % (1 << 32)
    if size:
        want = (want + codec.mix32(0xFFFFFFFF, (size[0] << 16) | size[1])) % (1 << 32)
    assert field == want
    model = GainedCheckerboardHierarchical(M, K=1, levels=6, precision="fp32")
    _, _, codes, csum, y_lanes, _, got = gained_codec._parse_sized(model, [[ys], [zs]], (hz, wz))
    assert codes == [2560] and csum == [0x12345678] and got == (size or (64 * hz, 64 * wz))
    assert len(y_lanes[0][0]) == min(32, M) * -(-4 * hz // 16)


def _strings(M=8, L=6, q_code=1234, size=None):
    rng = np.random.default_rng(7)
    y, z, ty, tz = _image(rng, M, 1, 1)
    return RG.encode_image(y, z, ty, tz, _header_fields(M, L, q_code, 5), size)


def test_host_validation():
    """Header, quality, lane table and size errors raise ValueError before any launch, naming the image (or the other model)."""
    model = GainedCheckerboardHierarchical(8, K=1, levels=6, precision="fp32")
    ys, zs = _strings()
    parse = lambda y, z, shape=(1, 1): gained_codec._parse_sized(model, [[ys, y], [zs, z]], shape)   # noqa: E731
    assert parse(ys, zs)[2] == [1234, 1234]
    for v, name in ((1, "JointAutoregressiveHierarchical"), (2, "ScalableImageCoding"), (3, "HierarchicalMixtureResidual"),
                    (4, "JointCheckerboardHierarchical"), (0x84, "JointCheckerboardHierarchical")):
        with pytest.raises(ValueError, match=rf"image 1: a {name} string"):
            parse(ys, bytes([v]) + zs[1:])
    with pytest.raises(ValueError, match="unknown format version 9"):
        parse(ys, bytes([9]) + zs[1:])
    top = gained_codec.HEADER.pack(5, 0, 8, 1, 6, 5121, 0) + zs[gained_codec.HEADER.size:]
    with pytest.raises(ValueError, match="image 1: quality code 5121"):
        parse(ys, top)
    gained_codec._parse_sized(model, [[_strings(q_code=5120)[0]], [_strings(q_code=5120)[1]]], (1, 1))
    for other, what in ((GainedCheckerboardHierarchical(8, K=2, levels=6, precision="fp32"), "K=1"),
                        (GainedCheckerboardHierarchical(16, K=1, levels=6, precision="fp32"), "M=8"),
                        (GainedCheckerboardHierarchical(8, K=1, levels=5, precision="fp32"), "levels=6"),
                        (GainedCheckerboardHierarchical(8, K=1, levels=6, precision="bf16"), "precision='fp32'")):
        with pytest.raises(ValueError, match=what):
            gained_codec._parse_sized(other, [[ys], [zs]], (1, 1))
    with pytest.raises(ValueError, match="truncated"):
        parse(ys, zs[:5])
    with pytest.raises(ValueError, match=r"image 1, y: corrupt string"):
        parse(ys + b"\0", zs)
    with pytest.raises(ValueError, match=r"image 1, z: corrupt string"):
        parse(ys, zs + b"\0\0")
    ys2, zs2 = _strings(size=(65, 63))
    with pytest.raises(ValueError, match=r"image 0: a 65x63 image has a z latent of 2x1"):
        gained_codec._parse_sized(model, [[ys2], [zs2]], (1, 1))
    for bad in ((0, 63), (128, 64)):
        z = bytearray(zs2)
        z[gained_codec.HEADER.size:gained_codec.HEADER.size + 4] = codec.SIZE.pack(*bad)
        with pytest.raises(ValueError, match="image 0"):
            gained_codec._parse_sized(model, [[ys2], [bytes(z)]], (2, 1))
    with pytest.raises(ValueError, match="y strings"):
        gained_codec._parse_sized(model, [[ys], []], (1, 1))


def test_existing_decoders_reject_format_5():
    ys, zs = _strings()
    with pytest.raises(ValueError, match="unknown format version 5"):
        checkerboard_codec._parse_sized(JointCheckerboardHierarchical(8, K=1, precision="fp32"), [[ys], [zs]], (1, 1))
    with pytest.raises(ValueError, match="unknown format version 5"):
        codec._parse_sized(JointCheckerboardHierarchical(8, K=1, precision="fp32"), [[ys], [zs]], (1, 1))


def test_quality_term_is_the_checksum_mix():
    assert RG.quality_term(6, 2560) == gained_codec.quality_term(6, 2560) == codec.mix32(0xFFFFFFFE, (6 << 16) | 2560)
    assert math.isclose(OG.snap(2.5, 6, 1).item() / 1024, 2.5)
