"""CPU: the layered byte format of ScalableImageCoding's coder - the reference coder of oracle/rans.py on random tables, and the
validation of decompress, which must reject every malformed or mismatched input before anything reaches a GPU."""
import numpy as np
import pytest
import torch

from neural_image_compression_b200 import _lib, codec, scalable_codec
from neural_image_compression_b200.Models import ScalableImageCoding
from oracle import rans, rans_scalable
from tests.test_codec_host import random_row


@pytest.mark.parametrize("seed,M,M1", [(0, 6, 2), (1, 40, 35), (2, 3, 1)])
def test_oracle_scalable_round_trip(seed, M, M1):
    """Random tables, escapes at +-(2^20 - 1), heads with fewer channels than lanes (M2 = 4 < 32, M = 3 < 4 z lanes)."""
    rng = np.random.default_rng(seed)
    M2, hz, wz = M - M1, 1, 2
    hy, wy = 4 * hz, 4 * wz
    y1 = rng.integers(-6, 7, size=(M1, hy, wy))
    y2 = rng.integers(-6, 7, size=(M2, hy, wy))
    z = rng.integers(-4, 5, size=(M, hz, wz))
    y1[0, 0, 0], y2[-1, hy - 1, wy - 1], z[0, 0, 1] = (1 << 20) - 1, -(1 << 20) + 1, (1 << 20) - 1
    t1 = {(c, i, j): random_row(rng) for c in range(M1) for i in range(hy) for j in range(wy)}
    t2 = {(c, i, j): random_row(rng) for c in range(M2) for i in range(hy) for j in range(wy)}
    tz = {c: random_row(rng) for c in range(M)}
    f1, f2, fz = (lambda c, i, j: t1[c, i, j]), (lambda c, i, j: t2[c, i, j]), (lambda c: tz[c])
    fields = (0, M, M1, 2, 0x12345678, 0x9ABCDEF0)                             # arm 0: fp32
    s1, s2, sz = rans_scalable.encode_scalable_image(y1, y2, z, f1, f2, fz, fields)
    a1, a2, az, hdr = rans_scalable.decode_scalable_image(s1, s2, sz, f1, f2, fz, hz, wz)
    assert np.array_equal(a1, y1) and np.array_equal(a2, y2) and np.array_equal(az, z)
    assert hdr == (2,) + fields
    b1, b2, bz, _ = rans_scalable.decode_scalable_image(s1, None, sz, f1, f2, fz, hz, wz)             # the base layer alone
    assert b2 is None and np.array_equal(b1, y1) and np.array_equal(bz, z)
    # the product parses what the reference writes, with the lane counts of each layer
    model = ScalableImageCoding(M, M1, K=2, precision="fp32")
    strings, lane_tabs, ln, base, enh = scalable_codec._parse_all(model, [[s1], [s2], [sz]], (hz, wz), False)
    assert ln == [min(4, M), min(32, M1), min(32, M2)] and base == [0x12345678] and enh == [0x9ABCDEF0]


def _strings(M=192, M1=128, K=1, arm="bf16x3", version=scalable_codec.FORMAT_VERSION):
    rng = np.random.default_rng(9)

    def layer(n):
        return [rans.encode_lane([(0, 100)] * int(rng.integers(0, 5))) for _ in range(n)]
    z = codec.pack_string(scalable_codec.HEADER.pack(version, codec.ARMS.index(arm), M, M1, K, 7, 8), layer(min(4, M)))
    return codec.pack_string(b"", layer(min(32, M1))), codec.pack_string(b"", layer(min(32, M - M1))), z


def test_malformed_strings_raise_before_any_gpu_call():
    model = ScalableImageCoding(192, 128, K=1, precision="bf16x3")      # CPU parameters: any launch would raise NicError
    y1, y2, z = _strings()
    jah_y, jah_z = codec.pack_string(b"", [rans.encode_lane([])] * 32), codec.pack_string(
        codec.HEADER.pack(codec.FORMAT_VERSION, 3, 192, 1, 7), [rans.encode_lane([])] * 4)
    H = scalable_codec.HEADER.size
    bad = {
        "truncated z": [[y1], [y2], [z[:-1]]],
        "truncated y1": [[y1[:-3]], [y2], [z]],
        "truncated y2": [[y1], [y2[:-1]], [z]],
        "truncated header": [[y1], [y2], [z[:5]]],
        "empty z": [[y1], [y2], [b""]],
        "over-long y1": [[y1 + b"\0"], [y2], [z]],
        "over-long y2": [[y1], [y2 + b"\0"], [z]],
        "bad lane length": [[y1], [y2], [z[:H] + bytes([0xFF]) + z[H + 1:]]],
        "unknown format": [[y1], [y2], [bytes([7]) + z[1:]]],
        "JAH string": [[jah_y], [y2], [jah_z]],
        "other arm": [[y1], [y2], [_strings(arm="fp32")[2]]],
        "other M": [[y1], [y2], [_strings(M=256)[2]]],
        "other M1": [[y1], [y2], [_strings(M1=64)[2]]],
        "other K": [[y1], [y2], [_strings(K=3)[2]]],
        "count mismatch": [[y1, y1], [y2], [z]],
        "count mismatch y2": [[y1], [y2, y2], [z]],
        "no images": [[], [], []],
        "two layers": [[y1], [z]],
        "not bytes": [[y1], [y2], ["abc"]],
        "y2 None": [[y1], None, [z]],
    }
    for what, strings in bad.items():
        with pytest.raises(ValueError):
            model.decompress(strings, (2, 3))
            pytest.fail(what)
    for shape in ((0, 3), (2,), (2.5, 3), "ab"):
        with pytest.raises(ValueError):
            model.decompress([[y1], [y2], [z]], shape)
    with pytest.raises(ValueError):                                     # base_only still checks the base layer
        model.decompress([[y1[:-1]], None, [z]], (2, 3), base_only=True)


def test_jah_decoder_rejects_a_scalable_string():
    from neural_image_compression_b200.Models import JointAutoregressiveHierarchical
    y1, _, z = _strings(M=128, M1=64, K=3)
    with pytest.raises(ValueError, match="unknown format version 2"):
        JointAutoregressiveHierarchical(128, K=3, precision="bf16x3").decompress([[y1], [z]], (2, 3))


def test_scalable_codec_has_no_cpu_path():
    model = ScalableImageCoding(192, 128, K=1, precision="bf16x3")
    with pytest.raises(_lib.NicError):
        model.compress(torch.rand(1, 3, 64, 64))
    y1, y2, z = _strings()
    with pytest.raises(_lib.NicError):
        model.decompress([[y1], [y2], [z]], (1, 1))
    with pytest.raises(_lib.NicError):
        model.decompress([[y1], None, [z]], (1, 1), base_only=True)
