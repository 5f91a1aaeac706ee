"""CPU: the byte format of the entropy coder - the reference rANS coder of oracle/rans.py on random tables, the product's string
layout (header, lane-length table) and its validation, which must reject malformed strings before anything reaches a GPU."""
import numpy as np
import pytest
import torch

from neural_image_compression_b200 import _lib, codec
from neural_image_compression_b200.Models import JointAutoregressiveHierarchical
from oracle import rans


def random_row(rng, n=None):
    n = int(rng.integers(1, 129)) if n is None else n
    f = rng.integers(1, 3000, size=n + 1).astype(np.float64)
    f = np.maximum(1, np.floor(f / f.sum() * (65536 - n - 1))).astype(np.int64) + 0
    f[-1] += 65536 - f.sum()                                   # escape bin takes the rest
    assert f.min() >= 1 and f.sum() == 65536
    cdf = np.concatenate([[0], np.cumsum(f)])
    return cdf, int(rng.integers(-50, 50)), n


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_lane_round_trip(seed):
    rng = np.random.default_rng(seed)
    rows = [random_row(rng, n=1 if k % 7 == 0 else None) for k in range(300)]
    syms = []
    for k, (cdf, lo, n) in enumerate(rows):
        r = rng.random()
        if r < 0.1:                                            # escapes, including the largest magnitudes allowed
            syms.append(int(rng.choice([(1 << 20) - 1, -(1 << 20) + 1, lo - 1, lo + n, 0 if not lo <= 0 < lo + n else lo + n + 3])))
        else:
            syms.append(lo + int(rng.integers(0, n)))
    ops = [op for s, row in zip(syms, rows) for op in rans.symbol_ops(s, *row)]
    seg = rans.encode_lane(ops)
    dec = rans.LaneDecoder(seg)
    assert [dec.symbol(*row) for row in rows] == syms
    assert dec.pos == len(seg[4:]) // 2


def test_oracle_empty_lane_and_image_round_trip():
    assert rans.encode_lane([]) == (1 << 16).to_bytes(4, "little")
    rng = np.random.default_rng(5)
    m, hz, wz = 3, 1, 1                                        # fewer channels than lanes: empty-free lanes = min(lanes, m)
    y = rng.integers(-5, 6, size=(m, 4, 4))
    y[0, 0, 0] = (1 << 20) - 1
    z = rng.integers(-3, 4, size=(m, hz, wz))
    ytab = {(c, i, j): random_row(rng) for c in range(m) for i in range(4) for j in range(4)}
    ztab = {c: random_row(rng) for c in range(m)}
    ys, zs = rans.encode_image(y, z, lambda c, i, j: ytab[c, i, j], lambda c: ztab[c], (3, m, 1, 1234))
    y2, z2, hdr = rans.decode_image(ys, zs, lambda c, i, j: ytab[c, i, j], lambda c: ztab[c], m, hz, wz)
    assert np.array_equal(y, y2) and np.array_equal(z, z2) and hdr == (1, 3, m, 1, 1234)
    # the product parses what the reference writes
    hdr_p, offs, words = codec.parse_string(zs, codec.lanes(codec.Z_LANES, m), True)
    assert hdr_p == hdr and len(offs) == min(4, m)


def test_wavefront_order_is_causal():
    """Every tap of the mask-'A' 5x5 context of pixel (i, j) belongs to an earlier step than the pixel (t = 3 i + j)."""
    taps = [(di, dj) for di in (-2, -1) for dj in range(-2, 3)] + [(0, -2), (0, -1)]
    assert len(taps) == 12
    for i in range(6):
        for j in range(8):
            for di, dj in taps:
                if 0 <= i + di and 0 <= j + dj < 8:
                    assert 3 * (i + di) + (j + dj) < 3 * i + j
    steps = rans.wavefront(32, 48)
    assert len(steps) == 141 and max(len(s) for s in steps) == codec.max_step_pixels(32, 48) == 16
    assert len(rans.wavefront(16, 16)) == 61


def test_string_layout_round_trip():
    rng = np.random.default_rng(3)
    segs = [bytes(rng.integers(0, 256, size=4 + 2 * n, dtype=np.uint8)) for n in (0, 1, 200, 70000, 3)]
    hdr = codec.HEADER.pack(codec.FORMAT_VERSION, 3, 128, 3, 0xDEADBEEF)
    s = codec.pack_string(hdr, segs)
    assert s == rans.pack(hdr, segs)
    h, offs, words = codec.parse_string(s, len(segs), True)
    assert h == (1, 3, 128, 3, 0xDEADBEEF) and words == [0, 1, 200, 70000, 3]
    assert [s[o:o + 4 + 2 * n] for o, n in zip(offs, words)] == segs
    _, offs2, words2 = codec.parse_string(codec.pack_string(b"", segs), len(segs), False)
    assert words2 == words


def _valid_strings(M=128, K=3, arm="bf16x3"):
    rng = np.random.default_rng(9)
    zsegs = [rans.encode_lane([(0, 100)] * int(rng.integers(0, 5))) for _ in range(codec.lanes(codec.Z_LANES, M))]
    ysegs = [rans.encode_lane([(0, 100)] * int(rng.integers(0, 5))) for _ in range(codec.lanes(codec.Y_LANES, M))]
    z = codec.pack_string(codec.HEADER.pack(codec.FORMAT_VERSION, codec.ARMS.index(arm), M, K, 7), zsegs)
    return codec.pack_string(b"", ysegs), z


def test_malformed_strings_raise_before_any_gpu_call():
    model = JointAutoregressiveHierarchical(128, K=3, precision="bf16x3")   # CPU parameters: any launch would raise NicError
    y, z = _valid_strings()
    bad = {
        "truncated z": ([y], [z[:-1]]),
        "truncated y": ([y[:-3]], [z]),
        "truncated header": ([y], [z[:5]]),
        "wrong version": ([y], [bytes([2]) + z[1:]]),
        "extra byte": ([y + b"\0"], [z]),
        "bad length": ([y], [z[:codec.HEADER.size] + bytes([0xFF]) + z[codec.HEADER.size + 1:]]),
        "other arm": ([y], [_valid_strings(arm="fp32")[1]]),
        "other K": ([y], [_valid_strings(K=1)[1]]),
        "count mismatch": ([y, y], [z]),
    }
    for what, strings in bad.items():
        with pytest.raises(ValueError):
            model.decompress(strings, (2, 3))
    with pytest.raises(ValueError):
        model.decompress([[y], [z]], (0, 3))
    with pytest.raises(ValueError):                            # the fused pipeline's channel counts only, outside fp32
        JointAutoregressiveHierarchical(64, K=1, precision="bf16").decompress([[y], [z]], (2, 3))


def test_codec_has_no_cpu_path():
    model = JointAutoregressiveHierarchical(128, K=3, precision="bf16x3")
    with pytest.raises(_lib.NicError):
        model.compress(torch.rand(1, 3, 64, 64))
    y, z = _valid_strings()
    with pytest.raises(_lib.NicError):
        model.decompress([[y], [z]], (1, 1))
