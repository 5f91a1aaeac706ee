"""Entropy coder of GainedCheckerboardHierarchical: ``compress(x, quality)`` -> [y_strings, z_strings], ``decompress(strings, shape)``
-> tensors (CompressAI's interface).  Byte format 5: DESIGN.md section 15.

Format 5 is format 4 (checkerboard_codec.py) with the quality in the z string's header: ``<BBHBBHI>`` = version 5, arm, M, K, L,
q_code, checksum, where the checksum field is the symbol checksum plus mix32(0xFFFFFFFE, L << 16 | q_code) mod 2^32 (then section 12's
size salt; the sized flag is 0x85).  A corrupted quality field therefore fails the decode even when the symbols happen to decode.  The
y string and its lanes are format 4's.  Both directions take the gains from nic_gain_vectors of the same q_code, and psi from
ginv_z (.) z_hat through the same gained hand-off (codec.ParamPath.hyper), so the decoder's parameters are the encoder's bit for bit.
"""
from __future__ import annotations

import struct

import numpy as np
import torch

from . import _lib, engine
from ._lib import CODEC_FACTORIZED, CODEC_GM, Q_PASSTHRU, check, current_stream, ptr
from .checkerboard_codec import BAND_ROWS, _encode_y, _segments, y_lanes
from .codec import (ARMS, SIZED, SYMBOL_LIMIT, Z_LANES, ParamPath, _encode, _symbol_codes, any_size_input, check_supported,
                    checksums, common_size, crop, lanes, mix32, pack_string, parse_string, read_z_header, salted, sized_header,
                    z_tables)
from .Models import QUALITY_QUANTUM, fused_g_a_gained, fused_g_s, fused_h_a_gained, gain_vectors, precision_arms, quality_codes

FORMAT_VERSION = 5
HEADER = struct.Struct("<BBHBBHI")                  # version, arm, M, K, L, q_code, checksum
OTHER_FORMATS = {1: "JointAutoregressiveHierarchical", 2: "ScalableImageCoding", 3: "HierarchicalMixtureResidual",
                 4: "JointCheckerboardHierarchical"}


def quality_term(levels: int, q_code: int) -> int:
    return mix32(0xFFFFFFFE, (levels << 16) | q_code)


def compress(model, x: torch.Tensor, quality=None) -> dict:
    x, size = any_size_input(x)
    B, _, H, W = x.shape
    check_supported(model)
    q_code = quality_codes(model.levels, quality, B, x.device)
    M, K, L = model.M, model.K, model.levels
    prec_up, prec = precision_arms(model.precision)
    hy, wy, hz, wz = H // 16, W // 16, H // 64, W // 64
    lc, lr = y_lanes(M, hy)
    ly, lz = lc * lr, lanes(Z_LANES, M)
    with torch.cuda.device(x.device), torch.no_grad():
        x = x.contiguous().float()
        gains = gain_vectors(model, q_code)
        _, y_in, _, y_src, _ = fused_g_a_gained(model, x, False, None, prec_up, prec, gains)
        _, z_in, _ = fused_h_a_gained(model, y_src, B, hy, wy, False, None, prec_up, prec, gains)
        big = torch.maximum(y_in.abs().amax(), z_in.abs().amax())
        if not bool(big < SYMBOL_LIMIT):
            raise ValueError(f"a latent symbol has magnitude {float(big)} >= 2^20: the stream format cannot carry it")
        y_sym, z_sym = y_in + 0.0, z_in + 0.0                      # -0.0 -> +0.0, as the decoder writes them
        path = ParamPath(model, B, hy, wy, x.device)
        _, combined = path.hyper(z_sym.permute(0, 2, 3, 1).contiguous(), gains.ginv_z)
        raw = path.raw(y_sym.permute(0, 2, 3, 1).contiguous(), combined)
        y_words, y_count = _encode_y(_symbol_codes(CODEC_GM, raw, y_sym, K), y_sym, lc)
        fp = model.factorized_entropy_model.packed()
        z_words, z_count = _encode(CODEC_FACTORIZED, _symbol_codes(CODEC_FACTORIZED, fp, z_sym, 1), z_sym, lz)
        small = torch.cat([y_count, z_count, checksums(y_sym, z_sym), q_code]).cpu().numpy()
        y_words, z_words = y_words.cpu().numpy().view("<u2"), z_words.cpu().numpy().view("<u2")
    y_count, z_count = small[:B * ly], small[B * ly:B * (ly + lz)]
    csum = small[B * (ly + lz):B * (ly + lz + 1)].view(np.uint32)
    codes = small[B * (ly + lz + 1):]
    arm = ARMS.index(model.precision)
    y_strings = [pack_string(b"", _segments(y_words, y_count, ly, b)) for b in range(B)]
    z_strings = []
    for b in range(B):
        qc = int(codes[b])
        field = salted((int(csum[b]) + quality_term(L, qc)) & 0xFFFFFFFF, size)
        z_strings.append(pack_string(sized_header(HEADER.pack(FORMAT_VERSION, arm, M, K, L, qc, field), size),
                                     _segments(z_words, z_count, lz, b)))
    return {"strings": [y_strings, z_strings], "shape": (hz, wz)}


def parse_z(data, model, n_lanes: int, b: int, shape):
    """-> (q_code, symbol checksum, image size, lane offsets, lane words) of a z string; ValueError on anything that is not one of
    this model's."""
    if isinstance(data, (bytes, bytearray)) and len(data) and data[0] & 0x7F in OTHER_FORMATS:
        v = data[0] & 0x7F
        raise ValueError(f"image {b}: a {OTHER_FORMATS[v]} string (format {v}), not a GainedCheckerboardHierarchical one "
                         f"(format {FORMAT_VERSION})")
    hdr, size, start = read_z_header(data, HEADER, FORMAT_VERSION, shape, b)
    _, arm, m, k, levels, qc, field = hdr
    if arm >= len(ARMS) or ARMS[arm] != model.precision or (m, k, levels) != (model.M, model.K, model.levels):
        got = ARMS[arm] if arm < len(ARMS) else f"arm #{arm}"
        raise ValueError(f"image {b}: the string was written by a model with precision={got!r}, M={m}, K={k}, levels={levels}; this "
                         f"model has precision={model.precision!r}, M={model.M}, K={model.K}, levels={model.levels}")
    if qc > QUALITY_QUANTUM * (levels - 1):
        raise ValueError(f"image {b}: quality code {qc} above {QUALITY_QUANTUM * (levels - 1)} (quality {levels - 1}) for {levels} levels")
    try:
        _, offs, words = parse_string(bytes(data[start:]), n_lanes, False)
    except ValueError as e:
        raise ValueError(f"image {b}, z: {e}") from None
    csum = (salted(field, size if hdr[0] & SIZED else None, -1) - quality_term(levels, qc)) & 0xFFFFFFFF
    return qc, csum, size, [start + o for o in offs], words


def _parse_sized(model, strings, shape):
    """Host-side validation of everything decompress reads: ValueError before any launch.  -> (y strings, z strings, q codes, symbol
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
    lc, lr = y_lanes(model.M, 4 * int(shape[0]))
    ly, lz = lc * lr, lanes(Z_LANES, model.M)
    codes, csum, sizes, y_lanes_, z_lanes_ = [], [], [], [], []
    for b, (ys, zs) in enumerate(zip(y_strings, z_strings)):
        qc, cs, size, zoff, zwords = parse_z(zs, model, lz, b, shape)
        if not isinstance(ys, (bytes, bytearray)):
            raise ValueError(f"image {b}: strings must be bytes, got {type(ys).__name__}")
        try:
            _, yoff, ywords = parse_string(bytes(ys), ly, False)
        except ValueError as e:
            raise ValueError(f"image {b}, y: {e}") from None
        codes.append(qc)
        csum.append(cs)
        sizes.append(size)
        y_lanes_.append((yoff, ywords))
        z_lanes_.append((zoff, zwords))
    return [bytes(s) for s in y_strings], [bytes(s) for s in z_strings], codes, csum, y_lanes_, z_lanes_, common_size(sizes)


def decompress(model, strings, shape) -> dict:
    y_strings, z_strings, codes, csum, y_lanes_, z_lanes_, size = _parse_sized(model, strings, shape)
    check_supported(model)
    w0 = model.encoder.ops[0].conv.weight
    engine.require_cuda(w0, "model parameters")
    lib = _lib.load()
    M, K = model.M, model.K
    B = len(y_strings)
    hz, wz = int(shape[0]), int(shape[1])
    hy, wy = 4 * hz, 4 * wz
    lc, lr = y_lanes(M, hy)
    ly, lz = lc * lr, lanes(Z_LANES, M)
    dev = w0.device
    start = np.cumsum([0] + [len(s) for s in z_strings + y_strings])
    z_off = np.array([start[b] + o for b in range(B) for o in z_lanes_[b][0]], dtype=np.int64)
    y_off = np.array([start[B + b] + o for b in range(B) for o in y_lanes_[b][0]], dtype=np.int64)
    z_nw = np.array([n for b in range(B) for n in z_lanes_[b][1]], dtype=np.int32)
    y_nw = np.array([n for b in range(B) for n in y_lanes_[b][1]], dtype=np.int32)
    with torch.cuda.device(dev), torch.no_grad():
        st = current_stream()
        blob = torch.frombuffer(bytearray(b"".join(z_strings + y_strings)), dtype=torch.uint8).to(dev)
        z_off_d, y_off_d = torch.from_numpy(z_off).to(dev), torch.from_numpy(y_off).to(dev)
        z_nw_d, y_nw_d = torch.from_numpy(z_nw).to(dev), torch.from_numpy(y_nw).to(dev)
        want = torch.tensor(np.array(csum, dtype=np.uint32).view(np.int32), device=dev)
        q_code = torch.tensor(codes, dtype=torch.int32).to(dev)
        gains = gain_vectors(model, q_code)
        zc, zlo, zn = z_tables(model.factorized_entropy_model.packed(), M)
        z_nhwc = torch.zeros((B, hz, wz, M), dtype=torch.float32, device=dev)
        zs_state, zs_pos = torch.empty(B * lz, dtype=torch.int32, device=dev), torch.empty(B * lz, dtype=torch.int32, device=dev)
        check(lib.nic_codec_decode(CODEC_FACTORIZED, ptr(blob), ptr(z_off_d), ptr(z_nw_d), ptr(zs_state), ptr(zs_pos), 1, ptr(zc),
                                   ptr(zlo), ptr(zn), B, M, hz, wz, lz, 0, ptr(z_nhwc), st), "nic_codec_decode")
        path = ParamPath(model, B, hy, wy, dev)
        z_hat, combined = path.hyper(z_nhwc, gains.ginv_z)
        # format 4's two passes on the integer symbols
        y_nhwc = torch.zeros((B, hy, wy, M), dtype=torch.float32, device=dev)
        ys_state, ys_pos = torch.empty(B * ly, dtype=torch.int32, device=dev), torch.empty(B * ly, dtype=torch.int32, device=dev)
        for s in (0, 1):
            raw = path.raw(y_nhwc, combined)
            check(lib.nic_codec_decode_pass(ptr(blob), ptr(y_off_d), ptr(y_nw_d), ptr(ys_state), ptr(ys_pos), ptr(raw), B, M, K, hy, wy, lc,
                                            BAND_ROWS, s, ptr(y_nhwc), st), "nic_codec_decode_pass")
        # g_s reads ginv_y (.) y_hat from the gained hand-off, as the forward's g_s does
        _, y_hat, _, _, gs_in = engine.latent_handoff_gain(y_nhwc, Q_PASSTHRU, None, None, gains.ginv_y, None, None, path.hdt)
        x_hat = crop(fused_g_s(model, gs_in, B, hy, wy, path.prec), size)
        bad = (checksums(y_hat, z_hat) != want).cpu().numpy()
    if bad.any():
        raise ValueError(f"checksum mismatch in image(s) {np.flatnonzero(bad).tolist()}: the strings are corrupted or were written "
                         f"by a model with other weights")
    return {"x_hat": x_hat, "y_hat": y_hat, "z_hat": z_hat, "quality": gains.quality}
