"""Entropy coder of ChannelCheckerboardHierarchical: ``compress(x)`` -> [y_strings, z_strings], ``decompress(strings, shape)`` -> tensors
(CompressAI's interface).  Byte format 6: DESIGN.md section 16; kernels: csrc/codec.cu.

z string: ``<BBHBB>`` = version 6, arm, M, K, S, then S ``<H>`` slice widths, then the ``<I>`` checksum field (section 9's y-then-z
symbol checksum, salted by the image size when sized: flag 0x86 and ``<HH>`` = H, W after the checksum, section 12), then section
9's z lanes.  y string: one lane table, then the segments, slice-major: slice s has min(32, m_s) channel classes x ceil(hy / 16) row
bands, each lane walking format 4's two passes over the slice's channels (anchors, then non-anchors, one rANS stream).

Both directions compute slice s's raw parameters with Models.slice_raw over the engine copy of the symbols from nic_latent_handoff in
Q_PASSTHRU mode (no lo-half hint), so the decoder rebuilds the encoder's tables bit for bit: at an anchor of slice s phi_sp is 0
whatever y_s holds and phi_ch reads only the slices before s, which are decoded; at a non-anchor the live checkerboard taps read only
anchors of slice s.  The decoder runs two parameter passes and two decode launches per slice, with no host synchronisation before the
checksum copy.
"""
from __future__ import annotations

import struct

import numpy as np
import torch

from . import _lib, engine
from ._lib import CODEC_FACTORIZED, CODEC_GM, Q_PASSTHRU, check, current_stream, ptr
from .checkerboard_codec import BAND_ROWS
from .codec import (ARMS, SIZED, SYMBOL_LIMIT, Z_LANES, _encode, _symbol_codes, any_size_input, check_supported, checksums,
                    common_size, crop, lanes, pack_string, parse_string, read_z_header, salted, sized_header, version_name, z_tables)
from .Models import fused_g_a, fused_g_s, fused_h_a, slice_buffers, slice_psi_into, slice_raw

FORMAT_VERSION = 6
PREFIX = struct.Struct("<BBHBB")                    # version, arm, M, K, S; then S <H> slice widths and the <I> checksum field
OTHER_FORMATS = {1: "JointAutoregressiveHierarchical", 2: "ScalableImageCoding", 3: "HierarchicalMixtureResidual",
                 4: "JointCheckerboardHierarchical", 5: "GainedCheckerboardHierarchical"}


def header_struct(S: int) -> struct.Struct:
    return struct.Struct("<BBHBB" + "H" * S + "I")


def slice_lanes(slices, hy: int):
    """[(channel classes, lanes)] per slice: min(32, m_s) classes x ceil(hy / 16) row bands."""
    return [(lanes(32, m), lanes(32, m) * -(-hy // BAND_ROWS)) for m in slices]


class SlicePath:
    """psi and the raw parameters of every slice of a (batch, size): the calls the encoder and the decoder share."""

    def __init__(self, model, B: int, hy: int, wy: int, device):
        self.model, self.B, self.hy, self.wy = model, B, hy, wy
        self.prec = model.precision
        self.hdt = "bf16x2" if self.prec == "bf16x3" else torch.float32          # engine-layout symbols, as the forward's
        self.combs = slice_buffers(model, B, hy, wy, self.prec, device)

    def hyper(self, z_nhwc: torch.Tensor) -> torch.Tensor:
        """z symbols NHWC f32 -> z_hat NCHW f32; psi goes into every slice's buffer."""
        _, z_hat, z_eng, _ = engine.latent_handoff(z_nhwc, Q_PASSTHRU, None, self.hdt)
        slice_psi_into(self.model, z_eng, self.B, z_nhwc.shape[1], z_nhwc.shape[2], self.prec, self.combs, None)
        return z_hat

    def symbols(self, y_nhwc: torch.Tensor) -> torch.Tensor:
        return engine.latent_handoff(y_nhwc, Q_PASSTHRU, None, self.hdt)[2]

    def raw(self, s: int, y_eng: torch.Tensor) -> torch.Tensor:
        """Slice s's raw entropy parameters NCHW f32 [B, (3K | 2) m_s, hy, wy] from the engine-layout symbols of all of y."""
        return slice_raw(self.model, s, y_eng, self.combs[s], self.B, self.hy, self.wy, self.prec)


def compress(model, x: torch.Tensor) -> dict:
    x, size = any_size_input(x)
    B, _, H, W = x.shape
    check_supported(model)
    M, K, slices = model.M, model.K, model.slices
    prec = model.precision
    hy, wy, hz, wz = H // 16, W // 16, H // 64, W // 64
    sl = slice_lanes(slices, hy)
    lz = lanes(Z_LANES, M)
    with torch.cuda.device(x.device), torch.no_grad():
        x = x.contiguous().float()
        _, y_in, _, y_src = fused_g_a(model, x, False, None, prec, prec)
        _, z_in, _ = fused_h_a(model, y_src, B, hy, wy, False, None, prec, prec)
        big = torch.maximum(y_in.abs().amax(), z_in.abs().amax())
        if not bool(big < SYMBOL_LIMIT):
            raise ValueError(f"a latent symbol has magnitude {float(big)} >= 2^20: the stream format cannot carry it")
        y_sym, z_sym = y_in + 0.0, z_in + 0.0                      # -0.0 -> +0.0, as the decoder writes them
        path = SlicePath(model, B, hy, wy, x.device)
        path.hyper(z_sym.permute(0, 2, 3, 1).contiguous())
        y_eng = path.symbols(y_sym.permute(0, 2, 3, 1).contiguous())
        # every slice's parameters from the full y, their symbol codes into one [B, M, hy * wy] tensor, then one walk per slice
        code = torch.empty((B, M, hy * wy), dtype=torch.int64, device=x.device)
        for s, (o, m) in enumerate(zip(model.offsets, slices)):
            code[:, o:o + m] = _symbol_codes(CODEC_GM, path.raw(s, y_eng), y_sym[:, o:o + m].contiguous(), K).view(B, m, hy * wy)
        lib = _lib.load()
        y_words, y_count = [], []
        for (o, m), (lc, ln) in zip(zip(model.offsets, slices), sl):
            cap = 3 * ((m + lc - 1) // lc) * BAND_ROWS * wy + 2
            words = torch.empty((B * ln, cap), dtype=torch.int16, device=x.device)
            count = torch.empty(B * ln, dtype=torch.int32, device=x.device)
            check(lib.nic_codec_encode_checkerboard_slice(ptr(code), ptr(y_sym), B, M, o, m, hy, wy, lc, BAND_ROWS, cap, ptr(words),
                                                          ptr(count), current_stream()), "nic_codec_encode_checkerboard_slice")
            y_words.append(words)
            y_count.append(count)
        fp = model.factorized_entropy_model.packed()
        z_words, z_count = _encode(CODEC_FACTORIZED, _symbol_codes(CODEC_FACTORIZED, fp, z_sym, 1), z_sym, lz)
        small = torch.cat(y_count + [z_count, checksums(y_sym, z_sym)]).cpu().numpy()
        y_words = [w.cpu().numpy().view("<u2") for w in y_words]
        z_words = z_words.cpu().numpy().view("<u2")
    starts = np.cumsum([0] + [B * ln for _, ln in sl])
    ny = int(starts[-1])
    z_count, csum = small[ny:ny + B * lz], small[ny + B * lz:].view(np.uint32)
    arm = ARMS.index(model.precision)

    def segments(words, count, n, b):
        cap = words.shape[1]
        return [words[g, cap - count[g]:].tobytes() for g in range(b * n, (b + 1) * n)]
    y_strings = [pack_string(b"", [seg for s, (_, ln) in enumerate(sl)
                                   for seg in segments(y_words[s], small[starts[s]:starts[s + 1]], ln, b)]) for b in range(B)]
    hdr = header_struct(len(slices))
    z_strings = [pack_string(sized_header(hdr.pack(FORMAT_VERSION, arm, M, K, len(slices), *slices, salted(int(csum[b]), size)), size),
                             segments(z_words, z_count, lz, b)) for b in range(B)]
    return {"strings": [y_strings, z_strings], "shape": (hz, wz)}


def parse_z(data, model, n_lanes: int, b: int, shape):
    """-> (symbol checksum, image size, lane offsets, lane words) of a z string; ValueError on anything that is not one of this
    model's."""
    if isinstance(data, (bytes, bytearray)) and len(data) and data[0] & 0x7F in OTHER_FORMATS:
        v = data[0] & 0x7F
        raise ValueError(f"image {b}: a {OTHER_FORMATS[v]} string (format {v}), not a ChannelCheckerboardHierarchical one "
                         f"(format {FORMAT_VERSION})")
    if not isinstance(data, (bytes, bytearray)):
        raise ValueError(f"image {b}: strings must be bytes, got {type(data).__name__}")
    if len(data) < PREFIX.size:
        raise ValueError(f"image {b}: truncated string: {len(data)} bytes, the header alone is at least {PREFIX.size + 4}")
    v, arm, m, k, S = PREFIX.unpack_from(data, 0)
    if v & 0x7F != FORMAT_VERSION:
        raise ValueError(f"image {b}: unknown format version {version_name(v)} (this build reads version {FORMAT_VERSION})")
    hdr_t = header_struct(S)
    if len(data) < hdr_t.size:
        raise ValueError(f"image {b}: truncated string: {len(data)} bytes, the header alone is {hdr_t.size}")
    widths = hdr_t.unpack_from(data, 0)[5:5 + S]
    if arm >= len(ARMS) or ARMS[arm] != model.precision or (m, k) != (model.M, model.K) or tuple(widths) != model.slices:
        got = ARMS[arm] if arm < len(ARMS) else f"arm #{arm}"
        raise ValueError(f"image {b}: the string was written by a model with precision={got!r}, M={m}, K={k}, slices={tuple(widths)}; "
                         f"this model has precision={model.precision!r}, M={model.M}, K={model.K}, slices={model.slices}")
    hdr, size, start = read_z_header(data, hdr_t, FORMAT_VERSION, shape, b)
    try:
        _, offs, words = parse_string(bytes(data[start:]), n_lanes, False)
    except ValueError as e:
        raise ValueError(f"image {b}, z: {e}") from None
    return salted(hdr[-1], size if hdr[0] & SIZED else None, -1), size, [start + o for o in offs], words


def _parse_sized(model, strings, shape):
    """Host-side validation of everything decompress reads: ValueError before any launch.  -> (y strings, z strings, symbol
    checksums, y lane (offsets, words) per image, z lane (offsets, words) per image, image size (H, W))."""
    if not isinstance(strings, (list, tuple)) or len(strings) != 2:
        raise ValueError("strings must be [y_strings, z_strings]")
    y_strings, z_strings = strings
    if not isinstance(y_strings, (list, tuple)) or not isinstance(z_strings, (list, tuple)):
        raise ValueError("each entry of strings must be a list of bytes (one per image)")
    if len(y_strings) != len(z_strings) or len(y_strings) == 0:
        raise ValueError(f"need as many y strings as z strings (>= 1); got {len(y_strings)} and {len(z_strings)}")
    if not isinstance(shape, (list, tuple)) or len(shape) != 2 or any(int(v) != v or v < 1 for v in shape):
        raise ValueError(f"shape must be (hz, wz) with positive ints, got {shape!r}")
    ly = sum(ln for _, ln in slice_lanes(model.slices, 4 * int(shape[0])))
    lz = lanes(Z_LANES, model.M)
    csum, sizes, y_lanes_, z_lanes_ = [], [], [], []
    for b, (ys, zs) in enumerate(zip(y_strings, z_strings)):
        cs, size, zoff, zwords = parse_z(zs, model, lz, b, shape)
        if not isinstance(ys, (bytes, bytearray)):
            raise ValueError(f"image {b}: strings must be bytes, got {type(ys).__name__}")
        try:
            _, yoff, ywords = parse_string(bytes(ys), ly, False)
        except ValueError as e:
            raise ValueError(f"image {b}, y: {e}") from None
        csum.append(cs)
        sizes.append(size)
        y_lanes_.append((yoff, ywords))
        z_lanes_.append((zoff, zwords))
    return [bytes(s) for s in y_strings], [bytes(s) for s in z_strings], csum, y_lanes_, z_lanes_, common_size(sizes)


def decompress(model, strings, shape) -> dict:
    y_strings, z_strings, csum, y_lanes_, z_lanes_, size = _parse_sized(model, strings, shape)
    check_supported(model)
    w0 = model.encoder.ops[0].conv.weight
    engine.require_cuda(w0, "model parameters")
    lib = _lib.load()
    M, K, slices = model.M, model.K, model.slices
    B = len(y_strings)
    hz, wz = int(shape[0]), int(shape[1])
    hy, wy = 4 * hz, 4 * wz
    sl = slice_lanes(slices, hy)
    lz = lanes(Z_LANES, M)
    dev = w0.device
    # one blob: z strings, then y strings; lane tables as absolute byte offsets into it, y lanes ordered slice, image, lane
    start = np.cumsum([0] + [len(s) for s in z_strings + y_strings])
    first = np.cumsum([0] + [ln for _, ln in sl])
    z_off = np.array([start[b] + o for b in range(B) for o in z_lanes_[b][0]], dtype=np.int64)
    z_nw = np.array([n for b in range(B) for n in z_lanes_[b][1]], dtype=np.int32)
    order = [(s, b, first[s] + l) for s, (_, ln) in enumerate(sl) for b in range(B) for l in range(ln)]
    y_off = np.array([start[B + b] + y_lanes_[b][0][g] for s, b, g in order], dtype=np.int64)
    y_nw = np.array([y_lanes_[b][1][g] for s, b, g in order], dtype=np.int32)
    with torch.cuda.device(dev), torch.no_grad():
        st = current_stream()
        blob = torch.frombuffer(bytearray(b"".join(z_strings + y_strings)), dtype=torch.uint8).to(dev)
        z_off_d, y_off_d = torch.from_numpy(z_off).to(dev), torch.from_numpy(y_off).to(dev)
        z_nw_d, y_nw_d = torch.from_numpy(z_nw).to(dev), torch.from_numpy(y_nw).to(dev)
        want = torch.tensor(np.array(csum, dtype=np.uint32).view(np.int32), device=dev)
        zc, zlo, zn = z_tables(model.factorized_entropy_model.packed(), M)
        z_nhwc = torch.zeros((B, hz, wz, M), dtype=torch.float32, device=dev)
        zs_state, zs_pos = torch.empty(B * lz, dtype=torch.int32, device=dev), torch.empty(B * lz, dtype=torch.int32, device=dev)
        check(lib.nic_codec_decode(CODEC_FACTORIZED, ptr(blob), ptr(z_off_d), ptr(z_nw_d), ptr(zs_state), ptr(zs_pos), 1, ptr(zc),
                                   ptr(zlo), ptr(zn), B, M, hz, wz, lz, 0, ptr(z_nhwc), st), "nic_codec_decode")
        path = SlicePath(model, B, hy, wy, dev)
        z_hat = path.hyper(z_nhwc)
        # y: slice by slice, pass 0 (anchors) then pass 1 (non-anchors), each from the parameters of the y decoded so far
        y_nhwc = torch.zeros((B, hy, wy, M), dtype=torch.float32, device=dev)
        n = len(order)
        ys_state, ys_pos = torch.empty(n, dtype=torch.int32, device=dev), torch.empty(n, dtype=torch.int32, device=dev)
        for s, ((o, m), (lc, _)) in enumerate(zip(zip(model.offsets, slices), sl)):
            g0 = B * int(first[s])                                  # the slice's first lane entry
            for p in (0, 1):
                raw = path.raw(s, path.symbols(y_nhwc))
                check(lib.nic_codec_decode_pass_slice(ptr(blob), ptr(y_off_d) + 8 * g0, ptr(y_nw_d) + 4 * g0, ptr(ys_state) + 4 * g0,
                                                      ptr(ys_pos) + 4 * g0, ptr(raw), B, M, o, m, K, hy, wy, lc, BAND_ROWS, p,
                                                      ptr(y_nhwc), st), "nic_codec_decode_pass_slice")
        # g_s reads the symbols through the same hand-off as the forward's (same engine copy, same lo-half flag)
        _, y_hat, y_eng, _ = engine.latent_handoff(y_nhwc, Q_PASSTHRU, None, path.hdt)
        x_hat = crop(fused_g_s(model, y_eng, B, hy, wy, path.prec), size)
        bad = (checksums(y_hat, z_hat) != want).cpu().numpy()
    if bad.any():
        raise ValueError(f"checksum mismatch in image(s) {np.flatnonzero(bad).tolist()}: the strings are corrupted or were written "
                         f"by a model with other weights")
    return {"x_hat": x_hat, "y_hat": y_hat, "z_hat": z_hat}
