"""CPU: ChannelCheckerboardHierarchical without a GPU - slice validation and the default slices, the state_dict keys, the trunk shared
with JointCheckerboardHierarchical, parent-checkpoint loading, the causality of the oracle's parameters for every slice pass (what the
2S-pass decoder rests on), the format-6 reference coder, and the host-side validation of format-6 strings, which raises before any
launch."""
import numpy as np
import pytest
import torch

from neural_image_compression_b200 import channel_codec, checkerboard_codec, codec, gained_codec
from neural_image_compression_b200.Models import (ChannelCheckerboardHierarchical, GainedCheckerboardHierarchical,
                                                  JointAutoregressiveHierarchical, JointCheckerboardHierarchical)
from oracle import channel as OCH
from oracle import checkerboard as OC
from oracle import rans_channel as RCH
from tests import helpers as H
from tests.test_codec_host import random_row

TRUNK = ("encoder.", "decoder.", "hyper_encoder.", "hyper_decoder.", "factorized_entropy_model.")


def apply_channel_init(sd, init):
    """helpers.apply_init for the slice heads: the trunk re-scaled as there, the sigma biases of every slice's last 1x1 conv raised."""
    gy, gz, sigma_bias = H.INITS[init]
    for k in ("encoder.net.6.weight", "encoder.net.6.bias"):
        sd[k] = sd[k] * gy
    for k in ("hyper_encoder.net.4.weight", "hyper_encoder.net.4.bias"):
        sd[k] = sd[k] * gz
    for k in [k for k in sd if k.startswith("entropy_parameters.") and k.endswith(".net.4.bias")]:
        b = sd[k].clone()
        n = b.numel()
        b[n // 2 if n % 3 else 2 * n // 3:] += sigma_bias
        sd[k] = b
    return sd


def seeded_channel(M, K, slices=None, init="calib", precision="fp32"):
    torch.manual_seed(0)
    model = ChannelCheckerboardHierarchical(M, K=K, slices=slices, precision=precision)
    if init != "plain":
        model.load_state_dict(apply_channel_init({k: v.clone() for k, v in model.state_dict().items()}, init))
    return model


def parent_as_one_slice(parent_sd):
    """A JointCheckerboardHierarchical state_dict under the keys of ChannelCheckerboardHierarchical(slices=(M,))."""
    out = {}
    for k, v in parent_sd.items():
        k = k.replace("context_model.", "context_models.0.", 1) if k.startswith("context_model.") else k
        k = k.replace("entropy_parameters.", "entropy_parameters.0.", 1) if k.startswith("entropy_parameters.") else k
        out[k] = v
    return out


def test_slices_validation_and_defaults():
    assert ChannelCheckerboardHierarchical(128).slices == (64, 64)
    assert ChannelCheckerboardHierarchical(192).slices == (64, 64, 64)
    assert ChannelCheckerboardHierarchical(100).slices == (64, 36)
    assert ChannelCheckerboardHierarchical(24).slices == (24,)
    m = ChannelCheckerboardHierarchical(192, slices=[64, 128])
    assert m.slices == (64, 128) and m.offsets == (0, 64) and m.precision == "bf16x3"
    assert ChannelCheckerboardHierarchical(128, slices=(32, 96)).precision == "fp32"
    assert ChannelCheckerboardHierarchical(100).precision == "fp32"
    for bad in ((64, 63), (0, 128), (128.0,), "128", (), (True, 127), (64, 64, 0), (-64, 192), 128):
        with pytest.raises(ValueError, match="slices"):
            ChannelCheckerboardHierarchical(128, slices=bad)
    for prec in ("bf16", "mixed", "fp16"):
        with pytest.raises(ValueError, match="precision"):
            ChannelCheckerboardHierarchical(128, precision=prec)
    with pytest.raises(ValueError, match="precision"):
        ChannelCheckerboardHierarchical(128, slices=(32, 96), precision="bf16x3")
    with pytest.raises(ValueError):
        ChannelCheckerboardHierarchical(0)


def test_key_names_and_shapes():
    model = ChannelCheckerboardHierarchical(128, K=3, slices=(64, 32, 32), precision="fp32")
    sd = model.state_dict()
    heads = [k for k in sd if not k.startswith(TRUNK)]
    want = []
    for s in range(3):
        want += [f"context_models.{s}.masked.{n}" for n in ("weight", "bias", "mask")]
        if s:
            want += [f"channel_contexts.{s - 1}.conv.{n}" for n in ("weight", "bias")]
        want += [f"entropy_parameters.{s}.net.{i}.{n}" for i in (0, 2, 4) for n in ("weight", "bias")]
    assert sorted(heads) == sorted(want)
    assert sd["context_models.1.masked.weight"].shape == (64, 32, 5, 5)
    assert torch.equal(sd["context_models.1.masked.mask"], OC.checkerboard_mask(sd["context_models.1.masked.mask"]))
    assert sd["channel_contexts.0.conv.weight"].shape == (64, 64, 5, 5)
    assert sd["channel_contexts.1.conv.weight"].shape == (64, 96, 5, 5)
    assert sd["entropy_parameters.0.net.0.weight"].shape == (640, 2 * 64 + 256, 1, 1)
    assert sd["entropy_parameters.1.net.0.weight"].shape == (640, 4 * 32 + 256, 1, 1)
    assert sd["entropy_parameters.2.net.4.weight"].shape == (9 * 32, 640, 1, 1)
    assert model.channel_contexts[1].conv.padding == (2, 2)


def test_trunk_is_the_parents_seeded_draw():
    torch.manual_seed(0)
    parent = JointCheckerboardHierarchical(128, K=3, precision="fp32").state_dict()
    torch.manual_seed(0)
    sd = ChannelCheckerboardHierarchical(128, K=3, precision="fp32").state_dict()
    trunk = [k for k in parent if k.startswith(TRUNK)]
    assert trunk == [k for k in sd if k.startswith(TRUNK)]
    for k in trunk:
        assert torch.equal(parent[k], sd[k]), k
    # one slice: the whole model is the parent's draw under remapped keys
    torch.manual_seed(0)
    one = ChannelCheckerboardHierarchical(128, K=3, slices=(128,), precision="fp32").state_dict()
    remapped = parent_as_one_slice(parent)
    assert list(one) == list(remapped)
    for k in one:
        assert torch.equal(one[k], remapped[k]), k


def test_parent_checkpoint_loads_the_trunk():
    torch.manual_seed(5)
    parent = JointCheckerboardHierarchical(64, K=1, precision="fp32").state_dict()
    model = ChannelCheckerboardHierarchical(64, K=1, slices=(32, 32), precision="fp32")
    res = model.load_state_dict(parent, strict=False)
    assert set(res.unexpected_keys) == {k for k in parent if not k.startswith(TRUNK)}
    assert set(res.missing_keys) == {k for k in model.state_dict() if not k.startswith(TRUNK)}
    for k, v in model.state_dict().items():
        if k.startswith(TRUNK):
            assert torch.equal(v, parent[k]), k
    # a mask-'A' context model cannot be loaded into a slice's checkerboard context model
    mask_a = parent_as_one_slice(JointAutoregressiveHierarchical(64, K=1, precision="fp32").state_dict())
    one = ChannelCheckerboardHierarchical(64, K=1, slices=(64,), precision="fp32")
    with pytest.raises(ValueError, match=r"context_models\.0\.masked\.mask"):
        one.load_state_dict(mask_a)
    one.load_state_dict(parent_as_one_slice(parent))


@pytest.mark.parametrize("K,slices", [(1, (4, 8)), (3, (3, 5, 4))])
def test_oracle_parameters_are_causal_per_slice_pass(K, slices):
    """In float64, for every slice s: the raw parameters at the anchors of slice s are unchanged when slices >= s are zeroed (pass 0
    of the decoder sees exactly that y); those at the non-anchors are unchanged when slice s's non-anchors and every later slice are
    zeroed (pass 1).  The channel context is live: the anchors of slice s >= 1 move with the slices before it."""
    M, hy, wy = sum(slices), 8, 12
    torch.manual_seed(0)
    sd = {k: v.double() for k, v in ChannelCheckerboardHierarchical(M, K=K, slices=slices, precision="fp32").state_dict().items()}
    g = torch.Generator().manual_seed(3)
    y = torch.randint(-5, 6, (1, M, hy, wy), generator=g).double()
    z = torch.randint(-3, 4, (1, M, 2, 3), generator=g).double()
    dt = torch.float64
    full = OCH.raw_parameters(sd, y, z, slices, dt)
    anchor = OC.anchors(hy, wy)
    for s, o in enumerate(OCH.offsets(slices)):
        m = slices[s]
        pass0 = y.clone()
        pass0[:, o:] = 0
        assert torch.equal(OCH.raw_parameters(sd, pass0, z, slices, dt)[s][..., anchor], full[s][..., anchor]), s
        pass1 = pass0.clone()
        pass1[:, o:o + m] = torch.where(anchor, y[:, o:o + m], torch.zeros_like(y[:, o:o + m]))
        assert torch.equal(OCH.raw_parameters(sd, pass1, z, slices, dt)[s][..., ~anchor], full[s][..., ~anchor]), s
        other = pass1.clone()
        other[:, o:o + m] = torch.where(anchor, -y[:, o:o + m] + 1, other[:, o:o + m])
        assert not torch.equal(OCH.raw_parameters(sd, other, z, slices, dt)[s][..., ~anchor], full[s][..., ~anchor]), s
        if s:
            earlier = y.clone()
            earlier[:, :o] = 0
            assert not torch.equal(OCH.raw_parameters(sd, earlier, z, slices, dt)[s][..., anchor], full[s][..., anchor]), s


def _image(rng, M, hz, wz):
    hy, wy = 4 * hz, 4 * wz
    y = rng.integers(-6, 7, size=(M, hy, wy))
    z = rng.integers(-4, 5, size=(M, hz, wz))
    y[0, 0, 0], y[M - 1, hy - 1, wy - 1], z[0, 0, 0] = (1 << 20) - 1, -77, -(1 << 20) + 1        # escapes
    ty = {(c, i, j): random_row(rng) for c in range(M) for i in range(hy) for j in range(wy)}
    tz = {c: random_row(rng) for c in range(M)}
    return y, z, (lambda c, i, j: ty[c, i, j]), (lambda c: tz[c])


@pytest.mark.parametrize("M,slices,hz,wz,size", [(24, (5, 19), 1, 2, None), (24, (7, 9, 8), 2, 1, (65, 63)), (24, (24,), 1, 1, None),
                                                 (40, (33, 7), 5, 1, None), (12, (6, 6), 2, 2, (100, 127))])
def test_reference_coder_round_trips(M, slices, hz, wz, size):
    """Format 6 through the reference coder: slice-major lanes, each slice's lanes covering its channels in format 4's two passes;
    the product's host parser reads the header, slices, size, checksum and lane table it writes."""
    rng = np.random.default_rng(M + hz + len(slices))
    y, z, ty, tz = _image(rng, M, hz, wz)
    hy, wy = 4 * hz, 4 * wz
    order = RCH.y_lanes(slices, hy)
    assert len(order) == sum(min(32, m) * -(-hy // 16) for m in slices)
    assert [s for s, _, _ in order] == sorted(s for s, _, _ in order)
    ys, zs = RCH.encode_image(y, z, ty, tz, (codec.ARMS.index("fp32"), M, 1, 0x12345678), slices, size)
    yo, zo, hdr = RCH.decode_image(ys, zs, ty, tz, hz, wz)
    assert np.array_equal(yo, y) and np.array_equal(zo, z)
    assert hdr == ((6 | (0x80 if size else 0)), 0, M, 1, slices, 0x12345678) + (size or (64 * hz, 64 * wz))
    model = ChannelCheckerboardHierarchical(M, K=1, slices=slices, precision="fp32")
    _, _, csum, y_lanes, _, got = channel_codec._parse_sized(model, [[ys], [zs]], (hz, wz))
    assert csum == [0x12345678] and got == (size or (64 * hz, 64 * wz))
    assert len(y_lanes[0][0]) == len(order)
    assert zs[0] == (0x86 if size else 6)


def _strings(M=8, slices=(3, 5), hz=1, wz=1, size=None, K=1):
    rng = np.random.default_rng(7)
    y, z, ty, tz = _image(rng, M, hz, wz)
    return RCH.encode_image(y, z, ty, tz, (codec.ARMS.index("fp32"), M, K, 5), slices, size)


def test_host_validation():
    """Every malformed header, lane table and size raises ValueError before any launch, naming the image (or the other model)."""
    model = ChannelCheckerboardHierarchical(8, K=1, slices=(3, 5), precision="fp32")
    ys, zs = _strings()
    parse = lambda y, z, shape=(1, 1): channel_codec._parse_sized(model, [[ys, y], [zs, z]], shape)   # noqa: E731
    parse(ys, zs)
    for v, name in ((1, "JointAutoregressiveHierarchical"), (2, "ScalableImageCoding"), (3, "HierarchicalMixtureResidual"),
                    (4, "JointCheckerboardHierarchical"), (5, "GainedCheckerboardHierarchical"), (0x84, "JointCheckerboardHierarchical")):
        with pytest.raises(ValueError, match=rf"image 1: a {name} string"):
            parse(ys, bytes([v]) + zs[1:])
    with pytest.raises(ValueError, match="unknown format version 9"):
        parse(ys, bytes([9]) + zs[1:])
    mismatch = [ChannelCheckerboardHierarchical(8, K=2, slices=(3, 5), precision="fp32"),
                ChannelCheckerboardHierarchical(8, K=1, slices=(5, 3), precision="fp32"),
                ChannelCheckerboardHierarchical(8, K=1, slices=(3, 3, 2), precision="fp32"),
                ChannelCheckerboardHierarchical(8, K=1, slices=(8,), precision="fp32"),
                ChannelCheckerboardHierarchical(9, K=1, slices=(3, 6), precision="fp32")]
    for other in mismatch:
        with pytest.raises(ValueError, match=r"M=8, K=1, slices=\(3, 5\)"):
            channel_codec._parse_sized(other, [[ys], [zs]], (1, 1))
    bad_arm = bytearray(zs)
    bad_arm[1] = codec.ARMS.index("bf16x3")
    with pytest.raises(ValueError, match="precision='bf16x3'"):
        parse(ys, bytes(bad_arm))
    bad_arm[1] = 17
    with pytest.raises(ValueError, match="arm #17"):
        parse(ys, bytes(bad_arm))
    bad_s = bytearray(zs)
    bad_s[5] = 200                                                 # S = 200: the header would need 405 bytes
    with pytest.raises(ValueError, match="truncated"):
        parse(ys, bytes(bad_s))
    bad_w = bytearray(zs)
    bad_w[6] = 4                                                   # widths (4, 5)
    with pytest.raises(ValueError, match=r"slices=\(4, 5\)"):
        parse(ys, bytes(bad_w))
    for cut in (3, 6, 9, 13):                                      # inside the prefix, the widths, the checksum
        with pytest.raises(ValueError, match="truncated"):
            parse(ys, zs[:cut])
    with pytest.raises(ValueError, match=r"image 1, y: corrupt string"):
        parse(ys + b"\0", zs)
    with pytest.raises(ValueError, match=r"image 1, y: corrupt string"):
        parse(ys[:-2], zs)
    with pytest.raises(ValueError, match=r"image 1, y: truncated"):
        parse(ys[:2], zs)
    with pytest.raises(ValueError, match=r"image 1, z: corrupt string"):
        parse(ys, zs + b"\0\0")
    with pytest.raises(ValueError, match=r"image 0, y"):
        parse(ys, zs, (5, 1))                                      # hy = 20: two row bands, twice the lanes
    ys2, zs2 = _strings(size=(65, 63))
    with pytest.raises(ValueError, match=r"image 0: a 65x63 image has a z latent of 2x1"):
        channel_codec._parse_sized(model, [[ys2], [zs2]], (1, 1))
    hsize = channel_codec.header_struct(2).size
    with pytest.raises(ValueError, match="size field is cut short"):
        channel_codec._parse_sized(model, [[ys2], [zs2[:hsize + 2]]], (2, 1))
    for bad in ((0, 63), (128, 64)):
        z = bytearray(zs2)
        z[hsize:hsize + 4] = codec.SIZE.pack(*bad)
        with pytest.raises(ValueError, match="image 0"):
            channel_codec._parse_sized(model, [[ys2], [bytes(z)]], (2, 1))
    with pytest.raises(ValueError, match="different sizes|image 1: a"):
        channel_codec._parse_sized(model, [[ys2, ys], [zs2, zs]], (2, 1))
    with pytest.raises(ValueError, match="y strings"):
        channel_codec._parse_sized(model, [[ys], []], (1, 1))
    with pytest.raises(ValueError, match="strings must be"):
        channel_codec._parse_sized(model, [ys, zs, zs], (1, 1))
    with pytest.raises(ValueError, match="shape"):
        channel_codec._parse_sized(model, [[ys], [zs]], (0, 1))
    with pytest.raises(ValueError, match="bytes"):
        channel_codec._parse_sized(model, [["y"], [zs]], (1, 1))


def test_existing_decoders_reject_format_6():
    ys, zs = _strings()
    with pytest.raises(ValueError, match="unknown format version 6"):
        codec._parse_sized(JointAutoregressiveHierarchical(8, K=1, precision="fp32"), [[ys], [zs]], (1, 1))
    with pytest.raises(ValueError, match="unknown format version 6"):
        checkerboard_codec._parse_sized(JointCheckerboardHierarchical(8, K=1, precision="fp32"), [[ys], [zs]], (1, 1))
    with pytest.raises(ValueError, match="unknown format version 6"):
        gained_codec._parse_sized(GainedCheckerboardHierarchical(8, K=1, precision="fp32"), [[ys], [zs]], (1, 1))
