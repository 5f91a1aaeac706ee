"""Entropy coder of HierarchicalMixtureResidual: ``compress(x)`` -> [y_strings, z_strings], ``decompress(strings, shape)`` -> tensors
(CompressAI's interface).  Byte format and determinism argument: DESIGN.md section 11.

The format is JointAutoregressiveHierarchical's (section 9) with version byte 3.  The parameters come from the scalable coder's
machinery (scalable_codec): psi by h_s one image per call, the raw entropy parameters by nic_codec_params, whose value at a pixel
does not depend on which pixels, batch or launch computed it.  The encoder runs it over every pixel; the decoder over the pixels of
one wavefront step, followed by nic_codec_decode_step, which builds the step's tables in shared memory and decodes them in the same
launch.  Tables, rANS encode, checksum and string helpers are codec.py's.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, engine
from ._lib import CODEC_FACTORIZED, CODEC_GM, check, current_stream, ptr
from .codec import (ARMS, HEADER, SIZED, SYMBOL_LIMIT, Y_LANES, Z_LANES, _encode, _symbol_codes, any_size_input, checksums,
                    common_size, crop, lanes, pack_string, parse_string, read_z_header, salted, sized_header, z_tables)
from .codec import FORMAT_VERSION as JAH_FORMAT_VERSION
from .scalable_codec import FORMAT_VERSION as SCALABLE_FORMAT_VERSION
from .scalable_codec import ParamHeads, _analysis, _segments, check_supported, psi_nhwc, synthesis

FORMAT_VERSION = 3
OTHER_FORMATS = {JAH_FORMAT_VERSION: "JointAutoregressiveHierarchical", SCALABLE_FORMAT_VERSION: "ScalableImageCoding"}


def compress(model, x: torch.Tensor) -> dict:
    x, size = any_size_input(x)
    check_supported(model)
    B, _, H, W = x.shape
    M, K = model.M, model.K
    hz, wz = H // 64, W // 64
    ly, lz = lanes(Y_LANES, M), lanes(Z_LANES, M)
    with torch.cuda.device(x.device), torch.no_grad():
        y_in, z_in = _analysis(model, x.contiguous().float())
        big = torch.maximum(y_in.abs().amax(), z_in.abs().amax())
        if not bool(big < SYMBOL_LIMIT):
            raise ValueError(f"a latent symbol has magnitude {float(big)} >= 2^20: the stream format cannot carry it")
        y_sym, z_sym = y_in + 0.0, z_in + 0.0                      # -0.0 -> +0.0, as the decoder writes them
        psi = psi_nhwc(model, z_sym.permute(0, 2, 3, 1).contiguous())
        heads = ParamHeads(model, [y_sym.permute(0, 2, 3, 1).contiguous()], psi, all_pixels=True)
        heads.run(-1)
        y_words, y_count = _encode(CODEC_GM, _symbol_codes(CODEC_GM, heads.raw[0], y_sym, K), y_sym, ly)
        z_words, z_count = _encode(CODEC_FACTORIZED, _symbol_codes(CODEC_FACTORIZED, model.factorized_entropy_model.packed(), z_sym, 1),
                                   z_sym, lz)
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
        raise ValueError(f"image {b}: a {OTHER_FORMATS[v]} string (format {v}), not a HierarchicalMixtureResidual one "
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
    ly, lz = lanes(Y_LANES, model.M), lanes(Z_LANES, model.M)
    csum, sizes, y_lanes, z_lanes = [], [], [], []
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
        y_lanes.append((yoff, ywords))
        z_lanes.append((zoff, zwords))
    return [bytes(s) for s in y_strings], [bytes(s) for s in z_strings], csum, y_lanes, z_lanes, common_size(sizes)


def _parse_all(model, strings, shape):
    """_parse_sized without the image size: the five values the host tests and tools/residual_codec_bench.py read."""
    return _parse_sized(model, strings, shape)[:-1]


def decompress(model, strings, shape) -> dict:
    y_strings, z_strings, csum, y_lanes, z_lanes, size = _parse_sized(model, strings, shape)
    check_supported(model)
    w0 = model.entropy_parameters.net[0].weight
    engine.require_cuda(w0, "model parameters")
    lib = _lib.load()
    M, K = model.M, model.K
    B = len(y_strings)
    hz, wz = int(shape[0]), int(shape[1])
    hy, wy = 4 * hz, 4 * wz
    ly, lz = lanes(Y_LANES, M), lanes(Z_LANES, M)
    dev = w0.device
    # one blob: z strings, then y strings; lane tables as absolute byte offsets into it
    start = np.cumsum([0] + [len(s) for s in z_strings + y_strings])
    z_off = np.array([start[b] + o for b in range(B) for o in z_lanes[b][0]], dtype=np.int64)
    y_off = np.array([start[B + b] + o for b in range(B) for o in y_lanes[b][0]], dtype=np.int64)
    z_nw = np.array([n for b in range(B) for n in z_lanes[b][1]], dtype=np.int32)
    y_nw = np.array([n for b in range(B) for n in y_lanes[b][1]], dtype=np.int32)
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
        z_hat = z_nhwc.permute(0, 3, 1, 2).contiguous()
        psi = psi_nhwc(model, z_nhwc)
        # y: per wavefront step, the step's parameters (4 launches) and its tables + rANS (1 launch); no host synchronisation
        y_nhwc = torch.zeros((B, hy, wy, M), dtype=torch.float32, device=dev)
        ys_state, ys_pos = torch.empty(B * ly, dtype=torch.int32, device=dev), torch.empty(B * ly, dtype=torch.int32, device=dev)
        heads = ParamHeads(model, [y_nhwc], psi, all_pixels=False)
        for t in range(3 * hy + wy - 3):
            heads.run(t)
            check(lib.nic_codec_decode_step(ptr(blob), ptr(y_off_d), ptr(y_nw_d), ptr(ys_state), ptr(ys_pos), int(t == 0), ptr(heads.raw[0]),
                                            B, M, K, hy, wy, ly, t, ptr(y_nhwc), st), "nic_codec_decode_step")
        y_hat, x_hat = synthesis(model, y_nhwc)
        x_hat = crop(x_hat, size)
        bad = (checksums(y_hat, z_hat) != want).cpu().numpy()
    if bad.any():
        raise ValueError(f"checksum mismatch in image(s) {np.flatnonzero(bad).tolist()}: the strings are corrupted or were written "
                         f"by a model with other weights")
    return {"x_hat": x_hat, "y_hat": y_hat, "z_hat": z_hat}
