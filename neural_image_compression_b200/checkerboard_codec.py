"""Entropy coder of JointCheckerboardHierarchical: ``compress(x)`` -> [y_strings, z_strings], ``decompress(strings, shape)`` -> tensors
(CompressAI's interface).  Byte format 4 and determinism argument: DESIGN.md section 14; kernels: csrc/codec.cu.

The y latent is coded in two passes of every lane: the anchors (i + j even), then the non-anchors.  Both directions compute the raw
entropy parameters with codec.ParamPath (the same engine calls, symbols handed over through nic_latent_handoff in Q_PASSTHRU mode, no
lo-half hint).  The encoder runs it once over the true symbols.  The decoder runs it over an all-zero y for the anchors (their context
output phi is 0 whatever y holds) and over the decoded anchors for the non-anchors (whose live context taps read anchors only), so
both get the encoder's parameters bit for bit.  Tables, rANS arithmetic, escapes, checksums and the size extension are section 9's
and section 12's.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, engine
from ._lib import CODEC_FACTORIZED, CODEC_GM, Q_PASSTHRU, check, current_stream, ptr
from .codec import (ARMS, HEADER, SIZED, SYMBOL_LIMIT, Y_LANES, Z_LANES, ParamPath, _encode, _symbol_codes, any_size_input,
                    check_supported, checksums, common_size, crop, lanes, pack_string, parse_string, read_z_header, salted,
                    sized_header, z_tables)
from .Models import fused_g_a, fused_g_s, fused_h_a, precision_arms

FORMAT_VERSION = 4
BAND_ROWS = 16                                      # latent rows of one lane's row band
OTHER_FORMATS = {1: "JointAutoregressiveHierarchical", 2: "ScalableImageCoding", 3: "HierarchicalMixtureResidual"}


def y_lanes(M: int, hy: int):
    """(channel classes Lc, row bands Lr): the y string has Lc * Lr lanes; lane r * Lc + l holds the channels c = l (mod Lc) of the
    latent rows [16 r, 16 r + 16)."""
    return lanes(Y_LANES, M), -(-hy // BAND_ROWS)


def _encode_y(code: torch.Tensor, sym: torch.Tensor, lc: int):
    lib = _lib.load()
    B, M, h, w = sym.shape
    cap = 3 * ((M + lc - 1) // lc) * BAND_ROWS * w + 2
    n = B * lc * (-(-h // BAND_ROWS))
    words = torch.empty((n, cap), dtype=torch.int16, device=sym.device)
    count = torch.empty(n, dtype=torch.int32, device=sym.device)
    check(lib.nic_codec_encode_checkerboard(ptr(code), ptr(sym), B, M, h, w, lc, BAND_ROWS, cap, ptr(words), ptr(count), current_stream()),
          "nic_codec_encode_checkerboard")
    return words, count


def _segments(words, count, n, b):
    cap = words.shape[1]
    return [words[g, cap - count[g]:].tobytes() for g in range(b * n, (b + 1) * n)]


def compress(model, x: torch.Tensor) -> dict:
    x, size = any_size_input(x)
    B, _, H, W = x.shape
    check_supported(model)
    M, K = model.M, model.K
    prec_up, prec = precision_arms(model.precision)
    hy, wy, hz, wz = H // 16, W // 16, H // 64, W // 64
    lc, lr = y_lanes(M, hy)
    ly, lz = lc * lr, lanes(Z_LANES, M)
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
        raw = path.raw(y_sym.permute(0, 2, 3, 1).contiguous(), combined)        # both passes' parameters in one pass
        y_words, y_count = _encode_y(_symbol_codes(CODEC_GM, raw, y_sym, K), y_sym, lc)
        fp = model.factorized_entropy_model.packed()
        z_words, z_count = _encode(CODEC_FACTORIZED, _symbol_codes(CODEC_FACTORIZED, fp, z_sym, 1), z_sym, lz)
        small = torch.cat([y_count, z_count, checksums(y_sym, z_sym)]).cpu().numpy()
        y_words, z_words = y_words.cpu().numpy().view("<u2"), z_words.cpu().numpy().view("<u2")
    y_count, z_count = small[:B * ly], small[B * ly:B * (ly + lz)]
    csum = small[B * (ly + lz):].view(np.uint32)
    arm = ARMS.index(model.precision)
    y_strings = [pack_string(b"", _segments(y_words, y_count, ly, b)) for b in range(B)]
    z_strings = [pack_string(sized_header(HEADER.pack(FORMAT_VERSION, arm, M, K, salted(int(csum[b]), size)), size),
                             _segments(z_words, z_count, lz, b)) for b in range(B)]
    return {"strings": [y_strings, z_strings], "shape": (hz, wz)}


def parse_z(data, model, n_lanes: int, b: int, shape):
    """-> (header tuple with the symbol checksum, image size, lane offsets, lane words) of a z string; ValueError on anything that
    is not one of this model's."""
    if isinstance(data, (bytes, bytearray)) and len(data) and data[0] & 0x7F in OTHER_FORMATS:
        v = data[0] & 0x7F
        raise ValueError(f"image {b}: a {OTHER_FORMATS[v]} string (format {v}), not a JointCheckerboardHierarchical one "
                         f"(format {FORMAT_VERSION})")
    hdr, size, start = read_z_header(data, HEADER, FORMAT_VERSION, shape, b)
    _, arm, m, k, csum = hdr
    if arm >= len(ARMS) or ARMS[arm] != model.precision or (m, k) != (model.M, model.K):
        got = ARMS[arm] if arm < len(ARMS) else f"arm #{arm}"
        raise ValueError(f"image {b}: the string was written by a model with precision={got!r}, M={m}, K={k}; this model has "
                         f"precision={model.precision!r}, M={model.M}, K={model.K}")
    try:
        _, offs, words = parse_string(bytes(data[start:]), n_lanes, False)
    except ValueError as e:
        raise ValueError(f"image {b}, z: {e}") from None
    return hdr[:4] + (salted(csum, size if hdr[0] & SIZED else None, -1),), size, [start + o for o in offs], words


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
    lc, lr = y_lanes(model.M, 4 * int(shape[0]))
    ly, lz = lc * lr, lanes(Z_LANES, model.M)
    csum, sizes, y_lanes_, z_lanes_ = [], [], [], []
    for b, (ys, zs) in enumerate(zip(y_strings, z_strings)):
        hdr, size, zoff, zwords = parse_z(zs, model, lz, b, shape)
        sizes.append(size)
        if not isinstance(ys, (bytes, bytearray)):
            raise ValueError(f"image {b}: strings must be bytes, got {type(ys).__name__}")
        try:
            _, yoff, ywords = parse_string(bytes(ys), ly, False)
        except ValueError as e:
            raise ValueError(f"image {b}, y: {e}") from None
        csum.append(hdr[4])
        y_lanes_.append((yoff, ywords))
        z_lanes_.append((zoff, zwords))
    return [bytes(s) for s in y_strings], [bytes(s) for s in z_strings], csum, y_lanes_, z_lanes_, common_size(sizes)


def decompress(model, strings, shape) -> dict:
    y_strings, z_strings, csum, y_lanes_, z_lanes_, size = _parse_sized(model, strings, shape)
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
    # one blob: z strings, then y strings; lane tables as absolute byte offsets into it
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
        # z: every symbol at once from the per-channel tables
        zc, zlo, zn = z_tables(model.factorized_entropy_model.packed(), M)
        z_nhwc = torch.zeros((B, hz, wz, M), dtype=torch.float32, device=dev)
        zs_state, zs_pos = torch.empty(B * lz, dtype=torch.int32, device=dev), torch.empty(B * lz, dtype=torch.int32, device=dev)
        check(lib.nic_codec_decode(CODEC_FACTORIZED, ptr(blob), ptr(z_off_d), ptr(z_nw_d), ptr(zs_state), ptr(zs_pos), 1, ptr(zc),
                                   ptr(zlo), ptr(zn), B, M, hz, wz, lz, 0, ptr(z_nhwc), st), "nic_codec_decode")
        path = ParamPath(model, B, hy, wy, dev)
        z_hat, combined = path.hyper(z_nhwc)
        # y: pass 0 (anchors) from the parameters of an all-zero y, pass 1 (non-anchors) from those of the decoded anchors
        y_nhwc = torch.zeros((B, hy, wy, M), dtype=torch.float32, device=dev)
        ys_state, ys_pos = torch.empty(B * ly, dtype=torch.int32, device=dev), torch.empty(B * ly, dtype=torch.int32, device=dev)
        for s in (0, 1):
            raw = path.raw(y_nhwc, combined)
            check(lib.nic_codec_decode_pass(ptr(blob), ptr(y_off_d), ptr(y_nw_d), ptr(ys_state), ptr(ys_pos), ptr(raw), B, M, K, hy, wy, lc,
                                            BAND_ROWS, s, ptr(y_nhwc), st), "nic_codec_decode_pass")
        # g_s reads the symbols through the same hand-off as the forward's (same engine copy, same lo-half flag)
        _, y_hat, y_eng, _ = engine.latent_handoff(y_nhwc, Q_PASSTHRU, None, path.hdt)
        x_hat = crop(fused_g_s(model, y_eng, B, hy, wy, path.prec), size)
        bad = (checksums(y_hat, z_hat) != want).cpu().numpy()
    if bad.any():
        raise ValueError(f"checksum mismatch in image(s) {np.flatnonzero(bad).tolist()}: the strings are corrupted or were written "
                         f"by a model with other weights")
    return {"x_hat": x_hat, "y_hat": y_hat, "z_hat": z_hat}
