"""Layered entropy coder of ScalableImageCoding: ``compress(x)`` -> [y1_strings, y2_strings, z_strings], ``decompress(strings, shape,
base_only)``.  The base layer (z and the M1 channels of y1) decodes without a single byte of y2.  Byte format, decode order and
determinism argument: DESIGN.md section 10; the step-local parameter kernel: csrc/codec_params.cu.  The table, rANS and checksum
kernels and the string helpers are the JointAutoregressiveHierarchical coder's (codec.py).

Both directions compute psi with `psi_nhwc` (h_s, one image per call) and the raw entropy parameters with `nic_codec_params`, whose
value at a pixel does not depend on which pixels, batch or launch computed it: the encoder runs it over every pixel, the decoder
over the pixels of one wavefront step.
"""
from __future__ import annotations

import struct

import numpy as np
import torch

from . import _lib, engine, training
from ._lib import CODEC_FACTORIZED, CODEC_GM, LAYOUT_NCHW, Q_PASSTHRU, Q_ROUND, CodecHead, check, current_stream, ptr
from .codec import (ARMS, SIZED, SYMBOL_LIMIT, Y_LANES, Z_LANES, _encode, _symbol_codes, any_size_input, checksums, common_size,
                    crop, lanes, max_step_pixels, pack_string, parse_string, read_z_header, salted, sized_header, step_tables, z_tables)
from .codec import FORMAT_VERSION as JAH_FORMAT_VERSION
from .Models import fused_g_a, fused_g_s, fused_h_a, fused_h_s_into

FORMAT_VERSION = 2
HEADER = struct.Struct("<BBHHBII")      # version, arm, M, M1, K, base checksum (y1 and z), enhancement checksum (y2 and z)
HIDDEN = 640                            # width of the entropy-parameter stack
LIVE_TAPS = [(a, b) for a in (0, 1) for b in range(5)] + [(2, 0), (2, 1)]       # mask 'A' of the 5x5 context conv, packed order


def check_supported(model):
    if model.K > 5:
        raise ValueError(f"compress/decompress: the likelihood kernels are built for K <= 5, got K={model.K}")


def _heads(model, base_only=False):
    """The entropy heads (training.heads: context model, entropy parameters, c0, c1) a call runs."""
    heads = training.heads(model)
    return heads[:1] if base_only else heads


def packed_head(ctx, ep):
    """[w_ctx, b_ctx, w1, b1, w2, b2, w3, b3] f32 in nic_codec_params' layout (include/nic.h), cached on the context model and
    repacked when a weight's storage or version changes (the key MaskedConv2d.apply_mask_ uses)."""
    masked = ctx.masked
    masked.apply_mask_()
    convs = [masked] + [ep.net[i] for i in (0, 2, 4)]
    key = tuple((t.data_ptr(), t._version, str(t.device)) for c in convs for t in (c.weight, c.bias))
    ent = ctx.__dict__.get("_codec_pack")
    if ent is not None and ent[0] == key:
        return ent[1]
    with torch.no_grad():
        wc = masked.weight.detach().float()                                          # [2m, m, 5, 5]
        w_ctx = torch.stack([wc[:, :, a, b] for a, b in LIVE_TAPS]).transpose(1, 2)  # [12, m, 2m]
        out = [w_ctx.reshape(-1, wc.shape[0]).contiguous(), masked.bias.detach().float().contiguous()]
        for c in convs[1:]:
            out += [c.weight.detach().float()[:, :, 0, 0].t().contiguous(), c.bias.detach().float().contiguous()]
    ctx.__dict__["_codec_pack"] = (key, out)
    return out


class ParamHeads:
    """nic_codec_params for the heads of one call: buffers (raw NCHW [B, np m, hy, wy] per head and the kernel's work) and the
    argument structs are built once; `run(t)` computes the raw parameters at every pixel (t = -1) or at wavefront step t's."""

    def __init__(self, model, sym_nhwc, psi, all_pixels: bool):
        B, hy, wy, _ = psi.shape
        self.model, self.psi, self.B, self.hy, self.wy = model, psi, B, hy, wy
        n = B * (hy * wy if all_pixels else max_step_pixels(hy, wy))
        npar = 2 if model.K == 1 else 3 * model.K
        self.raw, self._keep = [], []
        self.args = (CodecHead * len(sym_nhwc))()
        for a, ((ctx, ep, c0, c1), sym) in zip(self.args, zip(_heads(model), sym_nhwc)):
            m = c1 - c0
            w = packed_head(ctx, ep)
            raw = torch.empty((B, npar * m, hy, wy), dtype=torch.float32, device=psi.device)
            work = torch.empty(n * (2 * m + 2 * HIDDEN), dtype=torch.float32, device=psi.device)
            a.sym, a.w_ctx, a.b_ctx, a.w1, a.b1, a.w2, a.b2, a.w3, a.b3 = (ptr(t) for t in [sym] + w)
            a.raw, a.work, a.work_floats, a.m = ptr(raw), ptr(work), work.numel(), m
            self.raw.append(raw)
            self._keep += [sym, work, w]

    def run(self, t: int):
        m = self.model
        check(_lib.load().nic_codec_params(self.args, len(self.raw), ptr(self.psi), self.B, m.M, m.K, self.hy, self.wy, t,
                                           current_stream()), "nic_codec_params")


def psi_nhwc(model, z_nhwc: torch.Tensor) -> torch.Tensor:
    """psi = h_s(z symbols) as NHWC f32 [B, hy, wy, 2M], one image per call (so an image's psi is the same bits in any batch): the
    z symbols reach h_s through nic_latent_handoff (Q_PASSTHRU) as the forward's do; the fused pipeline's hi/lo pair is folded."""
    B, hz, wz, M = z_nhwc.shape
    hy, wy = 4 * hz, 4 * wz
    psi = torch.empty((B, hy, wy, 2 * M), dtype=torch.float32, device=z_nhwc.device)
    fused = _fused(model)
    pair = torch.empty((1, hy, wy, 4 * M), dtype=torch.bfloat16, device=z_nhwc.device) if fused else None
    for b in range(B):
        _, _, z_eng, _ = engine.latent_handoff(z_nhwc[b:b + 1], Q_PASSTHRU, None, "bf16x2" if fused else torch.float32)
        if fused:
            fused_h_s_into(model, z_eng, 1, hz, wz, "bf16x3", pair, 2 * M, 0, None)
            torch.add(pair[..., :2 * M].float(), pair[..., 2 * M:].float(), out=psi[b:b + 1])
        else:
            model.hyper_decoder.run_nhwc(z_eng, 1, hz, wz, model.precision,
                                         final_kw=dict(out=psi[b:b + 1], out_c_total=2 * M, out_c_offset=0))
    return psi


def _fused(model) -> bool:
    """True when the model's eval forward runs the fused pair-tensor pipeline; a model without one (HierarchicalMixtureResidual)
    takes the transforms' run_nhwc route."""
    return getattr(model, "fused_pipeline", False)


def _analysis(model, x):
    """The eval forward's symbols (y_in, z_in), NCHW f32, through the route the forward takes."""
    B, _, H, W = x.shape
    if _fused(model):
        _, y_in, _, y_src = fused_g_a(model, x, False, None, "bf16x3", "bf16x3")
        _, z_in, _ = fused_h_a(model, y_src, B, H // 16, W // 16, False, None, "bf16x3", "bf16x3")
        return y_in, z_in
    y_nhwc, _, _ = model.encoder.run_nhwc(x, B, H, W, model.precision, in_layout=LAYOUT_NCHW)
    _, y_in, _, _ = engine.latent_handoff(y_nhwc, Q_ROUND, None, torch.float32)
    z_nhwc, _, _ = model.hyper_encoder.run_nhwc(y_nhwc, B, H // 16, W // 16, model.precision)
    _, z_in, _, _ = engine.latent_handoff(z_nhwc, Q_ROUND, None, torch.float32)
    return y_in, z_in


def synthesis(model, y_nhwc):
    """Decoded y symbols NHWC f32 -> (y_hat NCHW, x_hat NCHW): g_s reads them through the same hand-off as the forward's."""
    B, hy, wy, _ = y_nhwc.shape
    fused = _fused(model)
    _, y_hat, y_eng, _ = engine.latent_handoff(y_nhwc, Q_PASSTHRU, None, "bf16x2" if fused else torch.float32)
    x_hat = fused_g_s(model, y_eng, B, hy, wy, "bf16x3") if fused else \
        model.decoder.run_nhwc(y_eng, B, hy, wy, model.precision, final_kw=dict(out_layout=LAYOUT_NCHW))[0]
    return y_hat, x_hat


def _segments(words, count, n, b):
    cap = words.shape[1]
    return [words[g, cap - count[g]:].tobytes() for g in range(b * n, (b + 1) * n)]


def compress(model, x: torch.Tensor) -> dict:
    x, size = any_size_input(x)
    check_supported(model)
    B, _, H, W = x.shape
    M, M1, K = model.M, model.M1, model.K
    hy, wy, hz, wz = H // 16, W // 16, H // 64, W // 64
    ln = [lanes(Y_LANES, c1 - c0) for _, _, c0, c1 in _heads(model)] + [lanes(Z_LANES, M)]
    with torch.cuda.device(x.device), torch.no_grad():
        y_in, z_in = _analysis(model, x.contiguous().float())
        big = torch.maximum(y_in.abs().amax(), z_in.abs().amax())
        if not bool(big < SYMBOL_LIMIT):
            raise ValueError(f"a latent symbol has magnitude {float(big)} >= 2^20: the stream format cannot carry it")
        y_sym, z_sym = y_in + 0.0, z_in + 0.0                      # -0.0 -> +0.0, as the decoder writes them
        psi = psi_nhwc(model, z_sym.permute(0, 2, 3, 1).contiguous())
        y_nhwc = y_sym.permute(0, 2, 3, 1)
        heads = ParamHeads(model, [y_nhwc[..., :M1].contiguous(), y_nhwc[..., M1:].contiguous()], psi, all_pixels=True)
        heads.run(-1)
        parts = [y_sym[:, :M1].contiguous(), y_sym[:, M1:].contiguous()]
        coded = [_encode(CODEC_GM, _symbol_codes(CODEC_GM, raw, sym, K), sym, n) for raw, sym, n in zip(heads.raw, parts, ln)]
        coded.append(_encode(CODEC_FACTORIZED, _symbol_codes(CODEC_FACTORIZED, model.factorized_entropy_model.packed(), z_sym, 1),
                             z_sym, ln[2]))
        small = torch.cat([c for _, c in coded] + [checksums(parts[0], z_sym), checksums(parts[1], z_sym)]).cpu().numpy()
        payload = torch.cat([w.flatten() for w, _ in coded]).cpu().numpy().view("<u2")
        words, pos = [], 0
        for w, _ in coded:
            words.append(payload[pos:pos + w.numel()].reshape(w.shape))
            pos += w.numel()
    counts, pos = [], 0
    for n in ln:
        counts.append(small[pos:pos + B * n])
        pos += B * n
    base, enh = small[pos:pos + B].view(np.uint32), small[pos + B:].view(np.uint32)
    arm = ARMS.index(model.precision)
    y1_strings = [pack_string(b"", _segments(words[0], counts[0], ln[0], b)) for b in range(B)]
    y2_strings = [pack_string(b"", _segments(words[1], counts[1], ln[1], b)) for b in range(B)]
    z_strings = [pack_string(sized_header(HEADER.pack(FORMAT_VERSION, arm, M, M1, K, salted(int(base[b]), size), salted(int(enh[b]), size)),
                                          size), _segments(words[2], counts[2], ln[2], b)) for b in range(B)]
    return {"strings": [y1_strings, y2_strings, z_strings], "shape": (hz, wz)}


def parse_z(data, model, n_lanes: int, b: int, shape):
    """-> (header tuple with the symbol checksums, image size, lane offsets, lane words) of a scalable z string; ValueError on
    anything that is not one of this model's."""
    if isinstance(data, (bytes, bytearray)) and len(data) and data[0] & 0x7F == JAH_FORMAT_VERSION:
        raise ValueError(f"image {b}: a JointAutoregressiveHierarchical string (format {JAH_FORMAT_VERSION}), not a scalable one "
                         f"(format {FORMAT_VERSION})")
    hdr, size, start = read_z_header(data, HEADER, FORMAT_VERSION, shape, b)
    _, arm, m, m1, k, base, enh = hdr
    if arm >= len(ARMS) or ARMS[arm] != model.precision or (m, m1, k) != (model.M, model.M1, model.K):
        got = ARMS[arm] if arm < len(ARMS) else f"arm #{arm}"
        raise ValueError(f"image {b}: the string was written by a model with precision={got!r}, M={m}, M1={m1}, K={k}; this model "
                         f"has precision={model.precision!r}, M={model.M}, M1={model.M1}, K={model.K}")
    _, offs, words = parse_string(bytes(data[start:]), n_lanes, False)
    salt = size if hdr[0] & SIZED else None
    return hdr[:5] + (salted(base, salt, -1), salted(enh, salt, -1)), size, [start + o for o in offs], words


def _parse_sized(model, strings, shape, base_only):
    """Host-side validation of everything decompress reads: ValueError before any launch.  -> (strings of the layers it decodes
    [z, y1(, y2)], their lane (offsets, words) per image, lane counts, base symbol checksums, enhancement symbol checksums, image
    size (H, W))."""
    if not isinstance(strings, (list, tuple)) or len(strings) != 3:
        raise ValueError("strings must be [y1_strings, y2_strings, z_strings]")
    y1s, y2s, zs = strings
    if y2s is None and not base_only:
        raise ValueError("the enhancement strings (strings[1]) are None: pass base_only=True to decode the base layer alone")
    layers = [zs, y1s] + ([] if base_only else [y2s])
    if any(not isinstance(s, (list, tuple)) for s in layers):
        raise ValueError("each entry of strings must be a list of bytes (one per image)")
    if len(zs) == 0 or any(len(s) != len(zs) for s in layers):
        raise ValueError(f"need as many strings per layer as images (>= 1); got {[len(s) for s in layers]}")
    if not isinstance(shape, (list, tuple)) or len(shape) != 2 or any(int(v) != v or v < 1 for v in shape):
        raise ValueError(f"shape must be (hz, wz) with positive ints, got {shape!r}")
    ln = [lanes(Z_LANES, model.M)] + [lanes(Y_LANES, c1 - c0) for _, _, c0, c1 in _heads(model, base_only)]
    lane_tabs, base, enh, sizes = [[] for _ in layers], [], [], []
    for b in range(len(zs)):
        hdr, size, offs, words = parse_z(zs[b], model, ln[0], b, shape)
        sizes.append(size)
        base.append(hdr[5])
        enh.append(hdr[6])
        lane_tabs[0].append((offs, words))
        for li in range(1, len(layers)):
            s = layers[li][b]
            if not isinstance(s, (bytes, bytearray)):
                raise ValueError(f"image {b}: strings must be bytes, got {type(s).__name__}")
            try:
                _, offs, words = parse_string(bytes(s), ln[li], False)
            except ValueError as e:
                raise ValueError(f"image {b}, layer y{li}: {e}") from None
            lane_tabs[li].append((offs, words))
    return [[bytes(s) for s in layer] for layer in layers], lane_tabs, ln, base, enh, common_size(sizes)


def _parse_all(model, strings, shape, base_only):
    """_parse_sized without the image size: the five values the host tests read."""
    return _parse_sized(model, strings, shape, base_only)[:-1]


def decompress(model, strings, shape, base_only: bool = False) -> dict:
    layers, lane_tabs, ln, base, enh, size = _parse_sized(model, strings, shape, base_only)
    check_supported(model)
    w0 = model.encoder.ops[0].conv.weight
    engine.require_cuda(w0, "model parameters")
    lib = _lib.load()
    M, K = model.M, model.K
    B = len(layers[0])
    hz, wz = int(shape[0]), int(shape[1])
    hy, wy = 4 * hz, 4 * wz
    dev = w0.device
    # one blob: the z strings, then the y1 strings (then the y2 strings); lane tables as absolute byte offsets into it
    flat = [s for layer in layers for s in layer]
    start = np.cumsum([0] + [len(s) for s in flat])
    offs = [np.array([start[li * B + b] + o for b in range(B) for o in tabs[b][0]], dtype=np.int64) for li, tabs in enumerate(lane_tabs)]
    nws = [np.array([n for b in range(B) for n in tabs[b][1]], dtype=np.int32) for tabs in lane_tabs]
    with torch.cuda.device(dev), torch.no_grad():
        st = current_stream()
        blob = torch.frombuffer(bytearray(b"".join(flat)), dtype=torch.uint8).to(dev)
        offs = [torch.from_numpy(o).to(dev) for o in offs]
        nws = [torch.from_numpy(n).to(dev) for n in nws]
        state = [torch.empty(B * n, dtype=torch.int32, device=dev) for n in ln]
        pos = [torch.empty(B * n, dtype=torch.int32, device=dev) for n in ln]
        want = torch.tensor(np.array(base + ([] if base_only else enh), dtype=np.uint32).view(np.int32), device=dev)
        # z: every symbol at once from the per-channel tables
        zc, zlo, zn = z_tables(model.factorized_entropy_model.packed(), M)
        z_nhwc = torch.zeros((B, hz, wz, M), dtype=torch.float32, device=dev)
        check(lib.nic_codec_decode(CODEC_FACTORIZED, ptr(blob), ptr(offs[0]), ptr(nws[0]), ptr(state[0]), ptr(pos[0]), 1, ptr(zc),
                                   ptr(zlo), ptr(zn), B, M, hz, wz, ln[0], 0, ptr(z_nhwc), st), "nic_codec_decode")
        z_hat = z_nhwc.permute(0, 3, 1, 2).contiguous()
        psi = psi_nhwc(model, z_nhwc)
        # y1 (and y2): one wavefront step at a time, both heads' parameters in one launch per layer; no host synchronisation
        ms = [c1 - c0 for _, _, c0, c1 in _heads(model, base_only)]
        y_nhwc = [torch.zeros((B, hy, wy, m), dtype=torch.float32, device=dev) for m in ms]
        heads = ParamHeads(model, y_nhwc, psi, all_pixels=False)
        tabs = [None] * len(ms)
        for t in range(3 * hy + wy - 3):
            heads.run(t)
            for i, m in enumerate(ms):
                tabs[i] = step_tables(heads.raw[i], m, K, t, tabs[i])
                check(lib.nic_codec_decode(CODEC_GM, ptr(blob), ptr(offs[i + 1]), ptr(nws[i + 1]), ptr(state[i + 1]), ptr(pos[i + 1]),
                                           int(t == 0), ptr(tabs[i][0]), ptr(tabs[i][1]), ptr(tabs[i][2]), B, m, hy, wy, ln[i + 1], t,
                                           ptr(y_nhwc[i]), st), "nic_codec_decode")
        y_parts = [y.permute(0, 3, 1, 2).contiguous() for y in y_nhwc]
        got = [checksums(y, z_hat) for y in y_parts]
        out = {"y1_hat": y_parts[0], "z_hat": z_hat}
        if not base_only:
            y_hat, x_hat = synthesis(model, torch.cat(y_nhwc, dim=-1).contiguous())
            out = {"x_hat": crop(x_hat, size), "y_hat": y_hat, "y1_hat": y_parts[0], "y2_hat": y_parts[1], "z_hat": z_hat}
        bad = (torch.cat(got) != want).cpu().numpy().reshape(len(got), B)
    for layer, flags in zip(("base layer (y1 and z)", "enhancement layer (y2)"), bad):
        if flags.any():
            raise ValueError(f"checksum mismatch of the {layer} in image(s) {np.flatnonzero(flags).tolist()}: the strings are corrupted "
                             f"or were written by a model with other weights")
    return out
