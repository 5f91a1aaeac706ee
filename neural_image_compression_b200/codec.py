"""Entropy coder of JointAutoregressiveHierarchical: ``compress(x)`` -> byte strings, ``decompress(strings, shape)`` -> tensors
(CompressAI's interface).  Byte format and determinism argument: DESIGN.md section 9; kernels: csrc/codec.cu.

Both directions compute psi (h_s on z_hat) and the raw entropy parameters (context conv + 1x1 stack) through ParamPath: the same
engine calls with the same descriptors, symbols handed over through nic_latent_handoff in Q_PASSTHRU mode and no lo-half hint.
The decoder recomputes the raw parameters over the whole latent once per wavefront step, with every not-yet-decoded position at 0;
the masked context conv only reads positions of earlier steps, so the parameters at the step's pixels are those the encoder saw.
"""
from __future__ import annotations

import struct
from typing import Sequence, Tuple

import numpy as np
import torch

from . import _lib, engine
from ._lib import (CODEC_FACTORIZED, CODEC_GM, CODEC_SYMBOL, CODEC_TABLES, CODEC_WINDOW, Q_PASSTHRU, check, current_stream,
                   ptr)
from .Models import fused_g_a, fused_g_s, fused_h_a, fused_h_s_into, precision_arms

FORMAT_VERSION = 1
ARMS = ("fp32", "bf16", "mixed", "bf16x3")          # header byte 1
HEADER = struct.Struct("<BBHBI")                    # version, arm, M, K, checksum of the image's y and z symbols
Y_LANES, Z_LANES = 32, 4                            # rANS lanes per string (fewer when M is smaller)
ROW = CODEC_WINDOW + 2                              # cdf entries of one table row
SYMBOL_LIMIT = 1 << 20                              # |symbol| must stay below this (escape values are 21-bit zigzag codes)


def lanes(kind_lanes: int, M: int) -> int:
    return min(kind_lanes, M)


# ---- byte strings (host) ---------------------------------------------------------------------------------------------

def _varint(n: int) -> bytes:
    out = bytearray()
    while True:
        b, n = n & 0x7F, n >> 7
        out.append(b | (0x80 if n else 0))
        if not n:
            return bytes(out)


def _read_varint(data: bytes, pos: int) -> Tuple[int, int]:
    n = 0
    for k in range(4):                              # lane lengths < 2^28 words
        if pos >= len(data):
            raise ValueError("truncated string: lane length table cut short")
        b = data[pos]
        pos += 1
        n |= (b & 0x7F) << (7 * k)
        if not b & 0x80:
            return n, pos
    raise ValueError("corrupt string: lane length longer than 4 bytes")


def pack_string(header: bytes, segments: Sequence[bytes]) -> bytes:
    """header + one varint per lane (its words after the 4 state bytes) + the lane segments."""
    return header + b"".join(_varint((len(s) - 4) // 2) for s in segments) + b"".join(segments)


def parse_string(data: bytes, n_lanes: int, with_header: bool):
    """-> (header tuple | None, byte offset of every lane segment, words of every lane).  Raises ValueError unless the lengths
    account for every byte of `data`."""
    if not isinstance(data, (bytes, bytearray)):
        raise ValueError(f"strings must be bytes, got {type(data).__name__}")
    pos, hdr = 0, None
    if with_header:
        if len(data) < HEADER.size:
            raise ValueError(f"truncated string: {len(data)} bytes, the header alone is {HEADER.size}")
        hdr = HEADER.unpack_from(data, 0)
        if hdr[0] != FORMAT_VERSION:
            raise ValueError(f"unknown format version {hdr[0]} (this build reads version {FORMAT_VERSION})")
        pos = HEADER.size
    words = []
    for _ in range(n_lanes):
        n, pos = _read_varint(data, pos)
        words.append(n)
    offs = []
    for n in words:
        offs.append(pos)
        pos += 4 + 2 * n
    if pos != len(data):
        raise ValueError(f"corrupt string: the lane lengths account for {pos} bytes, the string has {len(data)}")
    return hdr, offs, words


# ---- images of any size (DESIGN.md section 12): the size extension the three formats share -------------------------------------

SIZED = 0x80                                        # version-byte flag: the z string carries the image size
SIZE = struct.Struct("<HH")                         # H, W, right after the model's header
MAX_SIDE = 0xFFFF


def mix32(idx: int, v: int) -> int:
    """codec_checksum_kernel's 32-bit mix of (index, value) (csrc/codec.cu)."""
    h = ((idx * 0x9E3779B1) & 0xFFFFFFFF) ^ ((v + 0x7F4A7C15) & 0xFFFFFFFF)
    h ^= h >> 16
    h = (h * 0x85EBCA6B) & 0xFFFFFFFF
    h ^= h >> 13
    h = (h * 0xC2B2AE35) & 0xFFFFFFFF
    return h ^ (h >> 16)


def salted(csum: int, size, sign: int = 1) -> int:
    """A checksum field of a sized header: the symbol checksum plus mix32(0xFFFFFFFF, H << 16 | W), mod 2^32, so that a corrupted
    size fails the decode even when it rounds up to the same latent shape.  size None: the checksum itself; sign -1 undoes it."""
    if size is None:
        return csum
    return (csum + sign * mix32(0xFFFFFFFF, (size[0] << 16) | size[1])) & 0xFFFFFFFF


def sized_header(header: bytes, size) -> bytes:
    """The model's packed header as written for an image of `size` (None: an image whose sides are multiples of 64, today's
    header): version byte | SIZED, then H, W."""
    return header if size is None else bytes([header[0] | SIZED]) + header[1:] + SIZE.pack(*size)


def version_name(v: int) -> str:
    return f"{v & 0x7F}" + (" (sized)" if v & SIZED else "")


def read_z_header(data, header: struct.Struct, version: int, shape, b: int):
    """The header of one z string of any of the three formats -> (header tuple, image size (H, W), byte offset of the lane table).
    An unsized string has size (64 hz, 64 wz).  ValueError, naming the image, on a header cut short, another version or a size that
    is not the one spelling of an image of `shape`."""
    if not isinstance(data, (bytes, bytearray)):
        raise ValueError(f"image {b}: strings must be bytes, got {type(data).__name__}")
    if len(data) < header.size:
        raise ValueError(f"image {b}: truncated string: {len(data)} bytes, the header alone is {header.size}")
    hdr = header.unpack_from(data, 0)
    if hdr[0] & 0x7F != version:
        raise ValueError(f"image {b}: unknown format version {version_name(hdr[0])} (this build reads version {version})")
    hz, wz = int(shape[0]), int(shape[1])
    if not hdr[0] & SIZED:
        return hdr, (64 * hz, 64 * wz), header.size
    if len(data) < header.size + SIZE.size:
        raise ValueError(f"image {b}: truncated string: the size field is cut short ({len(data)} bytes)")
    size = SIZE.unpack_from(data, header.size)
    H, W = size
    if H == 0 or W == 0:
        raise ValueError(f"image {b}: the string gives an image size of {H}x{W}")
    if H % 64 == 0 and W % 64 == 0:
        raise ValueError(f"image {b}: a sized string for a {H}x{W} image (sides that are multiples of 64 are written unsized)")
    if (-(-H // 64), -(-W // 64)) != (hz, wz):
        raise ValueError(f"image {b}: a {H}x{W} image has a z latent of {-(-H // 64)}x{-(-W // 64)}, not shape {(hz, wz)}")
    return hdr, size, header.size + SIZE.size


def common_size(sizes):
    """The image size of every string in one call -> (H, W); ValueError naming the first image whose size differs."""
    for b, s in enumerate(sizes):
        if s != sizes[0]:
            raise ValueError(f"image {b}: a {s[0]}x{s[1]} image in a call that starts with a {sizes[0][0]}x{sizes[0][1]} one "
                             f"(decode images of different sizes in separate calls)")
    return sizes[0]


def window(x: torch.Tensor, h: int, w: int) -> torch.Tensor:
    """nic_image_window: [B, 3, h, w] f32 from the contiguous f32 x [B, 3, H, W] - its edge-replicating pad or its crop, launched on
    x's device and that device's current stream whatever device is current."""
    B, C, H, W = x.shape
    with torch.cuda.device(x.device):
        out = torch.empty((B, C, h, w), dtype=torch.float32, device=x.device)
        check(_lib.load().nic_image_window(ptr(x), B * C, H, W, ptr(out), h, w, current_stream()), "nic_image_window")
    return out


def any_size_input(x: torch.Tensor):
    """compress()'s input check: a CUDA tensor [B, 3, H, W] with H, W >= 1 -> (the image the model codes, (H, W) when the strings
    carry the size, else None).  Sides that are multiples of 64 pass through untouched; others are padded by repeating the last row
    and column up to the next multiples of 64."""
    engine.require_cuda(x, "x")
    if x.dim() != 4 or x.shape[1] != 3:
        raise ValueError(f"expected x of shape [B, 3, H, W], got {tuple(x.shape)}")
    H, W = x.shape[2:]
    if H < 1 or W < 1:
        raise ValueError(f"expected an image of at least 1x1 pixels, got {H}x{W}")
    if H % 64 == 0 and W % 64 == 0:
        return x, None
    if H > MAX_SIDE or W > MAX_SIDE:
        raise ValueError(f"an image whose sides are not multiples of 64 must be at most {MAX_SIDE} pixels high and wide; "
                         f"got {H}x{W}")
    return window(x.contiguous().float(), 64 * (-(-H // 64)), 64 * (-(-W // 64))), (H, W)


def crop(x_hat: torch.Tensor, size) -> torch.Tensor:
    """x_hat at the padded size -> the image's (H, W) (no launch when they are equal)."""
    if tuple(x_hat.shape[2:]) == tuple(size):
        return x_hat
    return window(x_hat.contiguous(), *size)


# ---- the shared parameter path ---------------------------------------------------------------------------------------

def check_supported(model):
    if model.precision != "fp32" and model.M not in (128, 192):
        raise ValueError(f"compress/decompress: precision={model.precision!r} is built for latent_channels 128 and 192 "
                         f"(the fused pipeline); got {model.M} - use precision='fp32'")
    if model.K > 5:
        raise ValueError(f"compress/decompress: the likelihood kernels are built for K <= 5, got K={model.K}")


class ParamPath:
    """psi and the raw entropy parameters of a (batch, size) - the calls the encoder and the decoder share.  The whole batch goes
    through one call: the decoder may see an image in a batch of another size than the encoder did, and the engine's results do
    not depend on the batch (tests/test_gpu_codec.py::test_params_batch_invariant, at the sizes where it switches tile forms)."""

    def __init__(self, model, B: int, hy: int, wy: int, device):
        self.model, self.B, self.hy, self.wy, self.device = model, B, hy, wy, device
        _, self.prec = precision_arms(model.precision)
        self.hdt = "bf16x2" if self.prec == "bf16x3" else engine.act_dtype(self.prec)     # engine-layout symbols, as the forward's
        M, K = model.M, model.K
        model.context_model.masked.apply_mask_()
        self.plan = engine.CtxEpPlan(model.context_model.masked._op, model.entropy_parameters.ops, B, hy, wy, self.prec, M, K, device,
                                     full=False)

    def hyper(self, z_nhwc: torch.Tensor):
        """z symbols NHWC f32 -> (z_hat NCHW f32, combined: psi in its channels [2M, 4M))."""
        M, B, prec = self.model.M, self.B, self.prec
        hz, wz = z_nhwc.shape[1:3]
        _, z_hat, z_eng, _ = engine.latent_handoff(z_nhwc, Q_PASSTHRU, None, self.hdt)
        combined = torch.empty((B, self.hy, self.wy, (2 if prec == "bf16x3" else 1) * 4 * M), dtype=engine.act_dtype(prec),
                               device=self.device)
        fused_h_s_into(self.model, z_eng, B, hz, wz, prec, combined, 4 * M, 2 * M, None)          # no lo-half hint (module docstring)
        return z_hat, combined

    def raw(self, y_nhwc: torch.Tensor, combined: torch.Tensor) -> torch.Tensor:
        """y symbols NHWC f32 -> raw entropy parameters NCHW f32 [B, (3K | 2) M, hy, wy]."""
        _, _, y_eng, _ = engine.latent_handoff(y_nhwc, Q_PASSTHRU, None, self.hdt)
        return self.plan.run(y_eng, combined)[0]


# ---- tables ----------------------------------------------------------------------------------------------------------

def max_step_pixels(hy: int, wy: int) -> int:
    return min(hy, (wy + 2) // 3)


def step_tables(raw: torch.Tensor, M: int, K: int, t: int, out=None):
    """(cdf [B * cnt * M, ROW] as int32 holding uint32, lo, nbins) of wavefront step t's elements, e = (img * cnt + p) * M + c."""
    lib = _lib.load()
    B, _, hy, wy = raw.shape
    if out is None:
        n = B * max_step_pixels(hy, wy) * M
        out = (torch.empty((n, ROW), dtype=torch.int32, device=raw.device), torch.empty(n, dtype=torch.int32, device=raw.device),
               torch.empty(n, dtype=torch.int32, device=raw.device))
    cdf, lo, nb = out
    check(lib.nic_codec_tables(CODEC_GM, CODEC_TABLES, ptr(raw), None, B, M, K, hy, wy, t, ptr(cdf), ptr(lo), ptr(nb), None,
                               current_stream()), "nic_codec_tables")
    return out


def z_tables(fparams: torch.Tensor, M: int):
    """(cdf [M, ROW], lo [M], nbins [M]): one table per channel of the factorized prior."""
    lib = _lib.load()
    dev = fparams.device
    cdf, lo, nb = (torch.empty((M, ROW), dtype=torch.int32, device=dev), torch.empty(M, dtype=torch.int32, device=dev),
                   torch.empty(M, dtype=torch.int32, device=dev))
    check(lib.nic_codec_tables(CODEC_FACTORIZED, CODEC_TABLES, ptr(fparams), None, 1, M, 1, 1, 1, 0, ptr(cdf), ptr(lo), ptr(nb), None,
                               current_stream()), "nic_codec_tables")
    return cdf, lo, nb


def _symbol_codes(kind, params, sym, K):
    lib = _lib.load()
    B, M, h, w = sym.shape
    code = torch.empty(sym.numel(), dtype=torch.int64, device=sym.device)
    check(lib.nic_codec_tables(kind, CODEC_SYMBOL, ptr(params), ptr(sym), B, M, K, h, w, 0, None, None, None, ptr(code),
                               current_stream()), "nic_codec_tables")
    return code


def _encode(kind, code, sym, n_lanes):
    lib = _lib.load()
    B, M, h, w = sym.shape
    cap = 3 * ((M + n_lanes - 1) // n_lanes) * h * w + 2
    words = torch.empty((B * n_lanes, cap), dtype=torch.int16, device=sym.device)
    count = torch.empty(B * n_lanes, dtype=torch.int32, device=sym.device)
    check(lib.nic_codec_encode(kind, ptr(code), ptr(sym), B, M, h, w, n_lanes, cap, ptr(words), ptr(count), current_stream()),
          "nic_codec_encode")
    return words, count


def checksums(y: torch.Tensor, z: torch.Tensor) -> torch.Tensor:
    """int32 [B] holding the per-image uint32 checksum of the y and z symbols (NCHW f32)."""
    lib = _lib.load()
    out = torch.empty(y.shape[0], dtype=torch.int32, device=y.device)
    check(lib.nic_codec_checksum(ptr(y), y[0].numel(), ptr(z), z[0].numel(), y.shape[0], ptr(out), current_stream()),
          "nic_codec_checksum")
    return out


# ---- compress / decompress -------------------------------------------------------------------------------------------

def compress(model, x: torch.Tensor) -> dict:
    x, size = any_size_input(x)
    B, _, H, W = x.shape
    check_supported(model)
    M, K = model.M, model.K
    prec_up, prec = precision_arms(model.precision)
    hy, wy, hz, wz = H // 16, W // 16, H // 64, W // 64
    ly, lz = lanes(Y_LANES, M), lanes(Z_LANES, M)
    with torch.cuda.device(x.device), torch.no_grad():
        x = x.contiguous().float()
        _, y_in, _, y_src = fused_g_a(model, x, False, None, prec_up, prec)
        _, z_in, _ = fused_h_a(model, y_src, B, hy, wy, False, None, prec_up, prec)
        big = torch.maximum(y_in.abs().amax(), z_in.abs().amax())
        if not bool(big < SYMBOL_LIMIT):
            raise ValueError(f"a latent symbol has magnitude {float(big)} >= 2^20: the stream format cannot carry it")
        y_sym, z_sym = y_in + 0.0, z_in + 0.0                      # -0.0 -> +0.0, as the decoder writes them
        path = ParamPath(model, B, hy, wy, x.device)
        _, combined = path.hyper(z_sym.permute(0, 2, 3, 1).contiguous())
        raw = path.raw(y_sym.permute(0, 2, 3, 1).contiguous(), combined)
        y_words, y_count = _encode(CODEC_GM, _symbol_codes(CODEC_GM, raw, y_sym, K), y_sym, ly)
        fp = model.factorized_entropy_model.packed()
        z_words, z_count = _encode(CODEC_FACTORIZED, _symbol_codes(CODEC_FACTORIZED, fp, z_sym, 1), z_sym, lz)
        small = torch.cat([y_count, z_count, checksums(y_sym, z_sym)]).cpu().numpy()
        y_words, z_words = y_words.cpu().numpy().view("<u2"), z_words.cpu().numpy().view("<u2")
    y_count, z_count = small[:B * ly], small[B * ly:B * (ly + lz)]
    csum = small[B * (ly + lz):].view(np.uint32)
    arm = ARMS.index(model.precision)

    def segments(words, count, n, b):
        cap = words.shape[1]
        return [words[g, cap - count[g]:].tobytes() for g in range(b * n, (b + 1) * n)]
    y_strings = [pack_string(b"", segments(y_words, y_count, ly, b)) for b in range(B)]
    z_strings = [pack_string(sized_header(HEADER.pack(FORMAT_VERSION, arm, M, K, salted(int(csum[b]), size)), size),
                             segments(z_words, z_count, lz, b)) for b in range(B)]
    return {"strings": [y_strings, z_strings], "shape": (hz, wz)}


def _parse_sized(model, strings, shape):
    """Host-side validation of everything decompress reads: ValueError before any launch.  -> (y strings, z strings, symbol
    checksums, y lane (offsets, words) per image, z lane (offsets, words) per image, image size (H, W))."""
    if not isinstance(strings, (list, tuple)) or len(strings) != 2:
        raise ValueError("strings must be [y_strings, z_strings]")
    y_strings, z_strings = strings
    if len(y_strings) != len(z_strings) or len(y_strings) == 0:
        raise ValueError(f"need as many y strings as z strings (>= 1); got {len(y_strings)} and {len(z_strings)}")
    if len(shape) != 2 or any(int(v) != v or v < 1 for v in shape):
        raise ValueError(f"shape must be (hz, wz) with positive ints, got {shape!r}")
    M, K = model.M, model.K
    ly, lz = lanes(Y_LANES, M), lanes(Z_LANES, M)
    csum, sizes, y_lanes, z_lanes = [], [], [], []
    for b, (ys, zs) in enumerate(zip(y_strings, z_strings)):
        hdr, size, start = read_z_header(zs, HEADER, FORMAT_VERSION, shape, b)
        v, arm, m, k, cs = hdr
        if arm >= len(ARMS) or ARMS[arm] != model.precision or m != M or k != K:
            got = ARMS[arm] if arm < len(ARMS) else f"arm #{arm}"
            raise ValueError(f"image {b}: the string was written by a model with precision={got!r}, M={m}, K={k}; this model has "
                             f"precision={model.precision!r}, M={M}, K={K}")
        _, zoff, zwords = parse_string(bytes(zs[start:]), lz, False)
        _, yoff, ywords = parse_string(ys, ly, False)
        csum.append(salted(cs, size if v & SIZED else None, -1))
        sizes.append(size)
        y_lanes.append((yoff, ywords))
        z_lanes.append(([start + o for o in zoff], zwords))
    return y_strings, z_strings, csum, y_lanes, z_lanes, common_size(sizes)


def decompress(model, strings, shape) -> dict:
    y_strings, z_strings, csum, y_lanes, z_lanes, size = _parse_sized(model, strings, shape)
    check_supported(model)
    w0 = model.encoder.ops[0].conv.weight
    engine.require_cuda(w0, "model parameters")
    lib = _lib.load()
    M, K = model.M, model.K
    B = len(y_strings)
    hz, wz = int(shape[0]), int(shape[1])
    hy, wy = 4 * hz, 4 * wz
    ly, lz = lanes(Y_LANES, M), lanes(Z_LANES, M)
    dev = w0.device
    # one blob: z strings, then y strings; lane tables as absolute byte offsets into it
    blob = b"".join(z_strings) + b"".join(y_strings)
    base = np.cumsum([0] + [len(s) for s in list(z_strings) + list(y_strings)])
    z_off = np.array([base[b] + o for b in range(B) for o in z_lanes[b][0]], dtype=np.int64)
    y_off = np.array([base[B + b] + o for b in range(B) for o in y_lanes[b][0]], dtype=np.int64)
    z_nw = np.array([n for b in range(B) for n in z_lanes[b][1]], dtype=np.int32)
    y_nw = np.array([n for b in range(B) for n in y_lanes[b][1]], dtype=np.int32)
    with torch.cuda.device(dev), torch.no_grad():
        st = current_stream()
        blob_d = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(dev)
        z_off_d, y_off_d = torch.from_numpy(z_off).to(dev), torch.from_numpy(y_off).to(dev)
        z_nw_d, y_nw_d = torch.from_numpy(z_nw).to(dev), torch.from_numpy(y_nw).to(dev)
        want = torch.tensor(np.array(csum, dtype=np.uint32).view(np.int32), device=dev)
        # z: every symbol at once from the per-channel tables
        zc, zlo, zn = z_tables(model.factorized_entropy_model.packed(), M)
        z_nhwc = torch.zeros((B, hz, wz, M), dtype=torch.float32, device=dev)
        zs_state, zs_pos = torch.empty(B * lz, dtype=torch.int32, device=dev), torch.empty(B * lz, dtype=torch.int32, device=dev)
        check(lib.nic_codec_decode(CODEC_FACTORIZED, ptr(blob_d), ptr(z_off_d), ptr(z_nw_d), ptr(zs_state), ptr(zs_pos), 1, ptr(zc),
                                   ptr(zlo), ptr(zn), B, M, hz, wz, lz, 0, ptr(z_nhwc), st), "nic_codec_decode")
        path = ParamPath(model, B, hy, wy, dev)
        z_hat, combined = path.hyper(z_nhwc)
        # y: one wavefront step at a time; no host synchronisation inside the loop
        y_nhwc = torch.zeros((B, hy, wy, M), dtype=torch.float32, device=dev)
        ys_state, ys_pos = torch.empty(B * ly, dtype=torch.int32, device=dev), torch.empty(B * ly, dtype=torch.int32, device=dev)
        tabs = None
        for t in range(3 * hy + wy - 3):
            raw = path.raw(y_nhwc, combined)
            tabs = step_tables(raw, M, K, t, tabs)
            check(lib.nic_codec_decode(CODEC_GM, ptr(blob_d), ptr(y_off_d), ptr(y_nw_d), ptr(ys_state), ptr(ys_pos), int(t == 0),
                                       ptr(tabs[0]), ptr(tabs[1]), ptr(tabs[2]), B, M, hy, wy, ly, t, ptr(y_nhwc), st), "nic_codec_decode")
        # g_s reads the symbols through the same hand-off as the forward's (same engine copy, same lo-half flag)
        _, y_hat, y_eng, _ = engine.latent_handoff(y_nhwc, Q_PASSTHRU, None, path.hdt)
        x_hat = crop(fused_g_s(model, y_eng, B, hy, wy, path.prec), size)
        bad = (checksums(y_hat, z_hat) != want).cpu().numpy()
    if bad.any():
        raise ValueError(f"checksum mismatch in image(s) {np.flatnonzero(bad).tolist()}: the strings are corrupted or were written "
                         f"by a model with other weights")
    return {"x_hat": x_hat, "y_hat": y_hat, "z_hat": z_hat}
