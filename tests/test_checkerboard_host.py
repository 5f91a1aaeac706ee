"""CPU: JointCheckerboardHierarchical without a GPU - the checkerboard mask, the construction shared with
JointAutoregressiveHierarchical, the refusal of a mask-'A' checkpoint, the causality of the oracle's parameters (what the two-pass
decoder rests on), the format-4 reference coder, and the host-side validation of format-4 strings, which raises before any launch."""
import ctypes as C

import numpy as np
import pytest
import torch

from neural_image_compression_b200 import _lib, checkerboard_codec, codec
from neural_image_compression_b200.ContextModels import anchor_mask, checkerboard_mask
from neural_image_compression_b200.Models import JointAutoregressiveHierarchical, JointCheckerboardHierarchical
from oracle import checkerboard as OC
from oracle import rans_checkerboard as RC
from tests.test_codec_host import random_row


def test_mask_keeps_the_12_odd_parity_taps():
    m = JointCheckerboardHierarchical(16, K=1).context_model.masked.mask
    assert m.shape == (32, 16, 5, 5)
    live = [(kh, kw) for kh in range(5) for kw in range(5) if m[0, 0, kh, kw]]
    assert len(live) == 12 and all((kh + kw) % 2 for kh, kw in live) and (2, 2) not in live
    assert torch.equal(m, checkerboard_mask(m)) and torch.equal(m, OC.checkerboard_mask(m))
    assert torch.equal(anchor_mask(3, 4), OC.anchors(3, 4)) and bool(anchor_mask(3, 4)[0, 0]) and not bool(anchor_mask(3, 4)[0, 1])
    d = _lib.ConvDesc()
    for k, v in dict(n=1, c_in=128, h_in=32, w_in=48, c_out=256, h_out=32, w_out=48, kh=5, kw=5, stride=1, pad=2,
                     mask_a=_lib.MASK_CHECKERBOARD).items():
        setattr(d, k, v)
    assert _lib.load().nic_packed_weight_elems(C.byref(d)) == 12 * 128 * 256


def test_construction_matches_the_mask_a_model():
    """Same state_dict keys, and a seeded build draws the same weights; only the mask buffer differs."""
    torch.manual_seed(0)
    a = JointAutoregressiveHierarchical(64, K=3).state_dict()
    torch.manual_seed(0)
    model = JointCheckerboardHierarchical(64, K=3)
    b = model.state_dict()
    assert list(a) == list(b)
    for k in a:
        assert torch.equal(a[k], b[k]) == (k != "context_model.masked.mask"), k
    assert (model.M, model.K, model.H, model.precision) == (64, 3, 64, "bf16x3")
    assert isinstance(model, JointAutoregressiveHierarchical)


def test_mask_a_checkpoint_is_rejected():
    sd = JointAutoregressiveHierarchical(16, K=1).state_dict()
    model = JointCheckerboardHierarchical(16, K=1)
    with pytest.raises(ValueError, match=r"context_model\.masked\.mask"):
        model.load_state_dict(sd)
    sd["context_model.masked.mask"] = model.context_model.masked.mask.clone()
    model.load_state_dict(sd)                                          # the same weights with the checkerboard mask load


def _oracle_sd(M, K, seed=0):
    torch.manual_seed(seed)
    return JointCheckerboardHierarchical(M, K=K).state_dict()


@pytest.mark.parametrize("K", [1, 3])
def test_oracle_parameters_are_causal(K):
    """The raw parameters at the anchors are the same bits for any y; those at the non-anchors do not change when the non-anchor
    symbols change.  So the decoder's pass over an all-zero y gives the anchors' parameters, its pass over the decoded anchors the
    non-anchors'."""
    M, hy, wy = 8, 8, 12
    sd = _oracle_sd(M, K)
    g = torch.Generator().manual_seed(3)
    y = torch.randint(-5, 6, (1, M, hy, wy), generator=g).float()
    z = torch.randint(-3, 4, (1, M, 2, 3), generator=g).float()
    full = OC.raw_parameters(sd, y, z)
    anchor = OC.anchors(hy, wy)
    other = torch.randint(-5, 6, y.shape, generator=g).float()
    assert torch.equal(OC.raw_parameters(sd, other, z)[..., anchor], full[..., anchor])
    assert torch.equal(OC.raw_parameters(sd, torch.zeros_like(y), z)[..., anchor], full[..., anchor])
    flipped = torch.where(anchor, y, other)
    assert not torch.equal(flipped, y)
    assert torch.equal(OC.raw_parameters(sd, flipped, z)[..., ~anchor], full[..., ~anchor])
    assert not torch.equal(OC.raw_parameters(sd, torch.where(anchor, other, y), z)[..., ~anchor], full[..., ~anchor])
    phi = OC.context(sd, y)
    assert torch.count_nonzero(phi[..., anchor]) == 0 and torch.count_nonzero(phi[..., ~anchor]) > 0


def _image(rng, M, hz, wz):
    hy, wy = 4 * hz, 4 * wz
    y = rng.integers(-6, 7, size=(M, hy, wy))
    z = rng.integers(-4, 5, size=(M, hz, wz))
    y[0, 0, 0], y[M - 1, hy - 1, wy - 1], z[0, 0, 0] = (1 << 20) - 1, -77, -(1 << 20) + 1        # escapes
    ty = {(c, i, j): random_row(rng) for c in range(M) for i in range(hy) for j in range(wy)}
    tz = {c: random_row(rng) for c in range(M)}
    return y, z, (lambda c, i, j: ty[c, i, j]), (lambda c: tz[c])


@pytest.mark.parametrize("M,hz,wz,size", [(3, 1, 2, None), (40, 5, 1, None), (5, 2, 2, (65, 127))])
def test_reference_coder_round_trips(M, hz, wz, size):
    """Format 4 through the reference coder: every lane of Lc channel classes x ceil(hy / 16) row bands covers its channels and rows
    in two passes, anchors first; the product's host parser reads the header, size, checksum and lane table it writes."""
    rng = np.random.default_rng(M + hz)
    y, z, ty, tz = _image(rng, M, hz, wz)
    hy, wy = 4 * hz, 4 * wz
    order = [e for lane in range(RC.y_lane_count(M, hy)) for e in RC.y_lane_order(M, hy, wy, lane)]
    assert sorted(order) == [(c, i, j) for c in range(M) for i in range(hy) for j in range(wy)]
    lane0 = RC.y_lane_order(M, hy, wy, 0)
    first = [(i + j) % 2 for _, i, j in lane0]
    assert first == sorted(first)                                  # the anchors, then the non-anchors
    ys, zs = RC.encode_image(y, z, ty, tz, (codec.ARMS.index("fp32"), M, 1, 0x12345678), size)
    yo, zo, hdr = RC.decode_image(ys, zs, ty, tz, M, hz, wz)
    assert np.array_equal(yo, y) and np.array_equal(zo, z)
    assert hdr == ((4 | (0x80 if size else 0)), 0, M, 1, 0x12345678) + (size or (64 * hz, 64 * wz))
    model = JointCheckerboardHierarchical(M, K=1, precision="fp32")
    _, _, csum, y_lanes, _, got = checkerboard_codec._parse_sized(model, [[ys], [zs]], (hz, wz))
    assert csum == [0x12345678] and got == (size or (64 * hz, 64 * wz))
    assert len(y_lanes[0][0]) == min(32, M) * -(-hy // 16)


def _strings(M=8, hz=1, wz=1, size=None):
    rng = np.random.default_rng(7)
    y, z, ty, tz = _image(rng, M, hz, wz)
    return RC.encode_image(y, z, ty, tz, (codec.ARMS.index("fp32"), M, 1, 5), size)


def test_host_validation():
    """Header, lane table and size errors raise ValueError before any launch, naming the image (or the other model)."""
    model = JointCheckerboardHierarchical(8, K=1, precision="fp32")
    ys, zs = _strings()
    parse = lambda y, z, shape=(1, 1): checkerboard_codec._parse_sized(model, [[ys, y], [zs, z]], shape)   # noqa: E731
    parse(ys, zs)
    for v, name in ((1, "JointAutoregressiveHierarchical"), (2, "ScalableImageCoding"), (3, "HierarchicalMixtureResidual"),
                    (0x81, "JointAutoregressiveHierarchical")):
        with pytest.raises(ValueError, match=rf"image 1: a {name} string"):
            parse(ys, bytes([v]) + zs[1:])
    with pytest.raises(ValueError, match="unknown format version 9"):
        parse(ys, bytes([9]) + zs[1:])
    with pytest.raises(ValueError, match="M=8, K=1"):
        checkerboard_codec._parse_sized(JointCheckerboardHierarchical(8, K=2, precision="fp32"), [[ys], [zs]], (1, 1))
    with pytest.raises(ValueError, match="precision='fp32'"):
        checkerboard_codec._parse_sized(JointCheckerboardHierarchical(8, K=1, precision="bf16"), [[ys], [zs]], (1, 1))
    with pytest.raises(ValueError, match="truncated"):
        parse(ys, zs[:5])
    with pytest.raises(ValueError, match=r"image 1, y: corrupt string"):
        parse(ys + b"\0", zs)
    with pytest.raises(ValueError, match=r"image 1, y: corrupt string"):
        parse(ys[:-2], zs)
    with pytest.raises(ValueError, match=r"image 1, z: corrupt string"):
        parse(ys, zs + b"\0\0")
    with pytest.raises(ValueError, match=r"image 0, y"):
        parse(ys, zs, (5, 1))                                      # hy = 20: two row bands, twice the lanes
    ys2, zs2 = _strings(size=(65, 63))
    with pytest.raises(ValueError, match=r"image 0: a 65x63 image has a z latent of 2x1"):
        checkerboard_codec._parse_sized(model, [[ys2], [zs2]], (1, 1))
    for bad in ((0, 63), (128, 64)):
        z = bytearray(zs2)
        z[codec.HEADER.size:codec.HEADER.size + 4] = codec.SIZE.pack(*bad)
        with pytest.raises(ValueError, match="image 0"):
            checkerboard_codec._parse_sized(model, [[ys2], [bytes(z)]], (2, 1))
    with pytest.raises(ValueError, match="y strings"):
        checkerboard_codec._parse_sized(model, [[ys], []], (1, 1))


def test_existing_decoders_reject_format_4():
    ys, zs = _strings()
    with pytest.raises(ValueError, match="unknown format version 4"):
        codec._parse_sized(JointAutoregressiveHierarchical(8, K=1, precision="fp32"), [[ys], [zs]], (1, 1))
