"""CPU: the size extension of the three byte formats (DESIGN.md section 12) - the reference coders on sized strings and the pinned
byte layout (flag bit, size field, checksum term), the product's validation of sizes, which must raise before anything reaches a GPU,
the cross-model messages for flagged versions, and the window entry's shape checks."""
import struct

import numpy as np
import pytest
import torch

from neural_image_compression_b200 import _lib, codec, residual_codec, scalable_codec
from neural_image_compression_b200.Models import HierarchicalMixtureResidual, JointAutoregressiveHierarchical, ScalableImageCoding
from oracle import rans, rans_residual, rans_scalable, rans_sized
from tests.test_codec_host import random_row


def _mix32_np(idx, v):
    """A third statement of csrc/codec.cu's mix32, in uint32 numpy arithmetic."""
    with np.errstate(over="ignore"):
        h = np.uint32(idx) * np.uint32(0x9E3779B1) ^ (np.uint32(v) + np.uint32(0x7F4A7C15))
        h ^= h >> np.uint32(16)
        h *= np.uint32(0x85EBCA6B)
        h ^= h >> np.uint32(13)
        h *= np.uint32(0xC2B2AE35)
        h ^= h >> np.uint32(16)
    return int(h)


def test_mix32_ports_agree():
    rng = np.random.default_rng(4)
    for idx, v in [(0, 0), (0xFFFFFFFF, (1080 << 16) | 1920), (0xFFFFFFFF, (1 << 16) | 1)] + \
            [tuple(int(a) for a in rng.integers(0, 1 << 32, size=2)) for _ in range(50)]:
        assert codec.mix32(idx, v) == rans_sized.mix32(idx, v) == _mix32_np(idx, v), (idx, v)


def _image(rng, M, hz, wz, m1=None):
    hy, wy = 4 * hz, 4 * wz
    y = rng.integers(-6, 7, size=(M, hy, wy))
    z = rng.integers(-4, 5, size=(M, hz, wz))
    y[0, 0, 0], z[0, 0, 0] = (1 << 20) - 1, -(1 << 20) + 1                          # escapes
    ty = {(c, i, j): random_row(rng) for c in range(M) for i in range(hy) for j in range(wy)}
    tz = {c: random_row(rng) for c in range(M)}
    return y, z, (lambda c, i, j: ty[c, i, j]), (lambda c: tz[c])


def _term(h, w):
    return _mix32_np(0xFFFFFFFF, (h << 16) | w)


@pytest.mark.parametrize("size", [(65, 63), (1, 1), (128, 65), (65535, 64)])
def test_sized_strings_round_trip_and_layout(size):
    """All three reference coders: the sized z string is the unsized one with bit 7 of the version byte set, every checksum field
    salted with mix32(0xFFFFFFFF, H << 16 | W) and <HH> = (H, W) between the header and the lane table; the y strings do not change.
    The product parses what the reference writes: the size, the symbol checksums and the lane offsets."""
    H_, W_ = size
    hz, wz = -(-H_ // 64), -(-W_ // 64)
    shape = (hz, wz) if hz * wz <= 4 else None
    rng = np.random.default_rng(H_ + W_)
    if shape is None:
        hz, wz = 1, 1                                          # the reference coders' layout only: one z pixel
    M, K, cs = 6, 2, 0xFFFFFFF0
    y, z, fy, fz = _image(rng, M, hz, wz)
    term = _term(H_, W_)
    # version 1 and version 3
    coders = ((1, lambda ys, zs: (ys, zs, fy, fz, M, hz, wz)), (3, lambda ys, zs: (ys, zs, fy, fz, hz, wz)))
    for version, dec_args in coders:
        ys0, zs0 = (rans.encode_image if version == 1 else rans_residual.encode_residual_image)(y, z, fy, fz, (0, M, K, cs))
        ys, zs = rans_sized.encode_sized_image(version, size, y, z, fy, fz, (0, M, K, cs))
        n = rans.HEADER.size
        assert ys == ys0
        assert zs[0] == 0x80 | version and zs[1:n - 4] == zs0[1:n - 4]
        assert struct.unpack_from("<I", zs, n - 4)[0] == (cs + term) % (1 << 32)
        assert struct.unpack_from("<HH", zs, n) == size and zs[n + 4:] == zs0[n:]
        ay, az, hdr = rans_sized.decode_sized_image(version, *dec_args(ys, zs))
        assert np.array_equal(ay, y) and np.array_equal(az, z) and hdr == (0x80 | version, 0, M, K, cs, H_, W_)
        if shape is not None and version == 3:
            model = HierarchicalMixtureResidual(M, K=K, precision="fp32")
            _, _, csum, y_lanes, z_lanes, got = residual_codec._parse_sized(model, [[ys], [zs]], shape)
            assert csum == [cs] and got == size and len(y_lanes[0][0]) == M and len(z_lanes[0][0]) == 4
        if shape is not None and version == 1:
            model = JointAutoregressiveHierarchical(M, K=K, precision="fp32")
            _, _, csum, _, z_lanes, got = codec._parse_sized(model, [[ys], [zs]], shape)
            assert csum == [cs] and got == size and len(z_lanes[0][0]) == 4
    # version 2: both checksum fields carry the term
    m1 = 2
    y1s, y2s, zs = rans_sized.encode_sized_image(2, size, y[:m1], y[m1:], z, fy, fy, fz, (0, M, m1, K, cs, 7))
    _, _, zs0 = rans_scalable.encode_scalable_image(y[:m1], y[m1:], z, fy, fy, fz, (0, M, m1, K, cs, 7))
    n = rans_scalable.SCALABLE_HEADER.size
    assert zs[0] == 0x82 and zs[1:n - 8] == zs0[1:n - 8]
    assert struct.unpack_from("<II", zs, n - 8) == ((cs + term) % (1 << 32), (7 + term) % (1 << 32))
    assert struct.unpack_from("<HH", zs, n) == size and zs[n + 4:] == zs0[n:]
    a1, a2, az, hdr = rans_sized.decode_sized_image(2, y1s, y2s, zs, fy, fy, fz, hz, wz)
    assert np.array_equal(a1, y[:m1]) and np.array_equal(a2, y[m1:]) and np.array_equal(az, z)
    assert hdr == (0x82, 0, M, m1, K, cs, 7, H_, W_)
    if shape is not None:
        model = ScalableImageCoding(M, m1, K=K, precision="fp32")
        _, _, _, base, enh, got = scalable_codec._parse_sized(model, [[y1s], [y2s], [zs]], shape, False)
        assert base == [cs] and enh == [7] and got == size
        assert scalable_codec._parse_all(model, [[y1s], None, [zs]], shape, True)[3] == [cs]


def test_product_header_is_the_reference_header():
    fields, size = (3, 192, 1, 0x89ABCDEF), (1080, 1920)
    hdr = codec.sized_header(codec.HEADER.pack(residual_codec.FORMAT_VERSION, *fields[:3], codec.salted(fields[3], size)), size)
    assert hdr == rans_sized.to_sized(rans.HEADER.pack(3, *fields), size)
    assert rans_sized.from_sized(hdr) == (rans.HEADER.pack(3, *fields), size)
    fields = (3, 192, 128, 1, 0x89ABCDEF, 17)
    hdr = codec.sized_header(scalable_codec.HEADER.pack(2, *fields[:4], *(codec.salted(c, size) for c in fields[4:])), size)
    assert hdr == rans_sized.to_sized(rans_scalable.SCALABLE_HEADER.pack(2, *fields), size)
    assert codec.salted(codec.salted(5, size), size, -1) == 5


# ---- validation before any launch ----------------------------------------------------------------------------------------------

def _lanes(n, rng):
    return [rans.encode_lane([(0, 100)] * int(rng.integers(0, 5))) for _ in range(n)]


def _strings(name, size, M=192, version=None):
    """Valid strings of one image of `size` ((H, W); None: unsized) for a CPU model of `name`, whose decoder must reject them
    before any launch when they are malformed."""
    rng = np.random.default_rng(3)
    if name == "scalable":
        v = version or scalable_codec.FORMAT_VERSION
        hdr = codec.sized_header(scalable_codec.HEADER.pack(v, 3, M, 128, 1, 7, 8), size)
        return [codec.pack_string(b"", _lanes(32, rng)), codec.pack_string(b"", _lanes(32, rng)), codec.pack_string(hdr, _lanes(4, rng))]
    v = version or (1 if name == "jah" else 3)
    hdr = codec.sized_header(codec.HEADER.pack(v, 3, M, 1, 7), size)
    return [codec.pack_string(b"", _lanes(32, rng)), codec.pack_string(hdr, _lanes(4, rng))]


def _model(name):
    return {"jah": lambda: JointAutoregressiveHierarchical(192, K=1, precision="bf16x3"),
            "scalable": lambda: ScalableImageCoding(192, 128, K=1, precision="bf16x3"),
            "residual": lambda: HierarchicalMixtureResidual(192, K=1, precision="bf16x3")}[name]()


def _batch(*images):
    return [list(layer) for layer in zip(*images)]


@pytest.mark.parametrize("name", ["jah", "scalable", "residual"])
def test_size_validation_raises_before_any_gpu_call(name):
    model = _model(name)                                       # CPU parameters: any launch would raise NicError
    good = _strings(name, (65, 63))
    n = len(codec.HEADER.pack(1, 0, 0, 0, 0)) if name != "scalable" else scalable_codec.HEADER.size
    z = good[-1]
    bad = {
        "sized, both sides multiples of 64": (_batch(_strings(name, (128, 64))), (2, 1), "written unsized"),
        "H = 0": (_batch(_strings(name, (0, 63))), (2, 1), "0x63"),
        "W = 0": (_batch(_strings(name, (65, 0))), (2, 1), "65x0"),
        "H rounds up to another hz": (_batch(good), (1, 1), "not shape"),
        "W rounds up to another wz": (_batch(good), (2, 2), "not shape"),
        "size field cut short": (_batch(good[:-1] + [z[:n + 3]]), (2, 1), "size field is cut short"),
        "two sizes": (_batch(good, _strings(name, (66, 63))), (2, 1), "image 1: a 66x63 image"),
        "sized and unsized": (_batch(good, _strings(name, None)), (2, 1), "image 1: a 128x64 image"),
    }
    for what, (strings, shape, msg) in bad.items():
        with pytest.raises(ValueError, match=msg):
            model.decompress(strings, shape)
            pytest.fail(what)


def test_flagged_versions_of_other_models_are_named():
    y, z = _strings("jah", (65, 63))
    y1, y2, sz = _strings("scalable", (65, 63))
    for strings in ([[y], [z]], [[y1], [sz]]):
        name = "JointAutoregressiveHierarchical" if strings[1][0][0] == 0x81 else "ScalableImageCoding"
        with pytest.raises(ValueError, match=f"image 0: a {name} string"):
            _model("residual").decompress(strings, (2, 1))
    with pytest.raises(ValueError, match="image 0: a JointAutoregressiveHierarchical string"):
        _model("scalable").decompress([[y1], [y2], [z]], (2, 1))
    ry, rz = _strings("residual", (65, 63))
    for strings, model in (([[y1], [sz]], "jah"), ([[ry], [rz]], "jah"), ([[y1], [y2], [rz]], "scalable")):
        with pytest.raises(ValueError, match=r"unknown format version \d \(sized\)"):
            _model(model).decompress(strings, (2, 1))
    with pytest.raises(ValueError, match="unknown format version 7 \\(sized\\)"):
        _model("residual").decompress([[ry], [bytes([0x87]) + rz[1:]]], (2, 1))


@pytest.mark.parametrize("name", ["jah", "scalable", "residual"])
def test_any_size_compress_has_no_cpu_path(name):
    with pytest.raises(_lib.NicError):
        _model(name).compress(torch.rand(1, 3, 65, 63))
    with pytest.raises(_lib.NicError):
        _model(name).decompress(_batch(_strings(name, (65, 63))), (2, 1))


def test_window_rejects_empty_sizes_without_a_launch():
    lib = _lib.load()
    buf = (np.zeros(16, dtype=np.float32)).ctypes.data
    for planes, hs, ws, hd, wd in ((3, 4, 4, 0, 4), (3, 0, 4, 4, 4), (0, 4, 4, 4, 4), (3, 4, -1, 4, 4), (3, 4, 4, 4, 0)):
        assert lib.nic_image_window(buf, planes, hs, ws, buf, hd, wd, None) == -1                 # NIC_E_BADSHAPE
        assert b"image_window" in lib.nic_last_error()
