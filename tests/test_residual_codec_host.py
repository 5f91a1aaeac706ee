"""CPU: the byte format of HierarchicalMixtureResidual's coder - the reference coder on random tables, and the validation of
decompress, which must reject every malformed or mismatched input (strings of the other two models included) before anything
reaches a GPU."""
import numpy as np
import pytest
import torch

from neural_image_compression_b200 import _lib, codec, residual_codec, scalable_codec
from neural_image_compression_b200.Models import HierarchicalMixtureResidual, JointAutoregressiveHierarchical, ScalableImageCoding
from oracle import rans, rans_residual
from tests.test_codec_host import random_row


@pytest.mark.parametrize("seed,M", [(0, 6), (1, 40), (2, 3)])
def test_oracle_residual_round_trip(seed, M):
    """Random tables, escapes at +-(2^20 - 1), fewer channels than lanes (M = 6 < 32 y lanes, M = 3 < 4 z lanes)."""
    rng = np.random.default_rng(seed)
    hz, wz = 1, 2
    hy, wy = 4 * hz, 4 * wz
    y = rng.integers(-6, 7, size=(M, hy, wy))
    z = rng.integers(-4, 5, size=(M, hz, wz))
    y[0, 0, 0], y[-1, hy - 1, wy - 1], z[0, 0, 1] = (1 << 20) - 1, -(1 << 20) + 1, (1 << 20) - 1
    ty = {(c, i, j): random_row(rng) for c in range(M) for i in range(hy) for j in range(wy)}
    tz = {c: random_row(rng) for c in range(M)}
    fy, fz = (lambda c, i, j: ty[c, i, j]), (lambda c: tz[c])
    fields = (3, M, 2, 0x12345678)                                              # arm 3: bf16x3
    ys, zs = rans_residual.encode_residual_image(y, z, fy, fz, fields)
    ay, az, hdr = rans_residual.decode_residual_image(ys, zs, fy, fz, hz, wz)
    assert np.array_equal(ay, y) and np.array_equal(az, z)
    assert hdr == (3,) + fields
    # the product parses what the reference writes, with the lane counts of each string
    model = HierarchicalMixtureResidual(M, K=2, precision="bf16x3" if M % 64 == 0 else "fp32")
    if model.precision != "bf16x3":
        ys, zs = rans_residual.encode_residual_image(y, z, fy, fz, (0,) + fields[1:])
    _, _, csum, y_lanes, z_lanes = residual_codec._parse_all(model, [[ys], [zs]], (hz, wz))
    assert csum == [0x12345678] and len(y_lanes[0][0]) == min(32, M) and len(z_lanes[0][0]) == min(4, M)


def _strings(M=192, K=1, arm="bf16x3", version=residual_codec.FORMAT_VERSION):
    rng = np.random.default_rng(9)

    def layer(n):
        return [rans.encode_lane([(0, 100)] * int(rng.integers(0, 5))) for _ in range(n)]
    z = codec.pack_string(codec.HEADER.pack(version, codec.ARMS.index(arm), M, K, 7), layer(min(4, M)))
    return codec.pack_string(b"", layer(min(32, M))), z


def test_malformed_strings_raise_before_any_gpu_call():
    model = HierarchicalMixtureResidual(192, K=1, precision="bf16x3")      # CPU parameters: any launch would raise NicError
    y, z = _strings()
    H = codec.HEADER.size
    bad = {
        "truncated z": [[y], [z[:-1]]],
        "truncated y": [[y[:-3]], [z]],
        "truncated header": [[y], [z[:5]]],
        "empty z": [[y], [b""]],
        "over-long y": [[y + b"\0"], [z]],
        "over-long z": [[y], [z + b"\0"]],
        "bad lane length": [[y], [z[:H] + bytes([0xFF]) + z[H + 1:]]],
        "unknown format": [[y], [bytes([7]) + z[1:]]],
        "other arm": [[y], [_strings(arm="fp32")[1]]],
        "other M": [[y], [_strings(M=256)[1]]],
        "other K": [[y], [_strings(K=3)[1]]],
        "count mismatch": [[y, y], [z]],
        "no images": [[], []],
        "three layers": [[y], [y], [z]],
        "not bytes": [[y], ["abc"]],
        "y not bytes": [[None], [z]],
        "y None": [None, [z]],
    }
    for what, strings in bad.items():
        with pytest.raises(ValueError):
            model.decompress(strings, (2, 3))
            pytest.fail(what)
    for shape in ((0, 3), (2,), (2.5, 3), "ab"):
        with pytest.raises(ValueError):
            model.decompress([[y], [z]], shape)
    with pytest.raises(ValueError, match=r"image 1: the string was written by a model with precision='fp32', M=192, K=1"):
        model.decompress([[y, y], [z, _strings(arm="fp32")[1]]], (2, 3))


def test_strings_of_the_other_models_are_rejected():
    """v1 (JointAutoregressiveHierarchical) and v2 (ScalableImageCoding) strings are named; the other two decoders reject v3 as
    an unknown version."""
    model = HierarchicalMixtureResidual(192, K=1, precision="bf16x3")
    y, z = _strings()
    jah_y, jah_z = _strings(version=codec.FORMAT_VERSION)
    with pytest.raises(ValueError, match="image 0: a JointAutoregressiveHierarchical string"):
        model.decompress([[jah_y], [jah_z]], (2, 3))
    sc_z = codec.pack_string(scalable_codec.HEADER.pack(scalable_codec.FORMAT_VERSION, 3, 192, 128, 1, 7, 8),
                             [rans.encode_lane([])] * 4)
    with pytest.raises(ValueError, match="image 0: a ScalableImageCoding string"):
        model.decompress([[y], [sc_z]], (2, 3))
    with pytest.raises(ValueError, match="unknown format version 3"):
        JointAutoregressiveHierarchical(192, K=1, precision="bf16x3").decompress([[y], [z]], (2, 3))
    y1 = codec.pack_string(b"", [rans.encode_lane([])] * 32)
    with pytest.raises(ValueError, match="unknown format version 3"):
        ScalableImageCoding(192, 128, K=1, precision="bf16x3").decompress([[y1], [y1], [z]], (2, 3))


def test_residual_codec_has_no_cpu_path():
    model = HierarchicalMixtureResidual(192, K=1, precision="bf16x3")
    with pytest.raises(_lib.NicError):
        model.compress(torch.rand(1, 3, 64, 64))
    y, z = _strings()
    with pytest.raises(_lib.NicError):
        model.decompress([[y], [z]], (1, 1))
