"""Host-side glue between the nn.Module mirror of the reference and the C ABI (include/nic.h).

Everything here is plumbing: it owns no arithmetic.  Tensors are allocated by PyTorch and passed to
the library as raw device pointers on the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch
import torch.nn as nn

from . import _lib
from ._lib import (ConvDesc, DT_BF16, DT_BF16X2, DT_F32, EPI_BIAS, EPI_GDN, EPI_IGDN, EPI_LRELU, LAYOUT_NCHW, LAYOUT_NHWC,
                   PRECISIONS, PREC_FP32, check, current_stream, ptr)

DEFAULT_PRECISION = os.environ.get("NIC_PRECISION", "auto")


def resolve_precision(precision: Optional[str], latent_channels: Optional[int] = None) -> str:
    """None / "auto" -> the parity-grade tensor-core arm ("bf16x3") where it is built (channel counts that are multiples of 64:
    M = 128 runs the fused pair-tensor pipeline, other M - e.g. the reference's default 192 - the layer-by-layer form with the
    GDN contractions as tensor-core 1x1 convs), else the fp32 CUDA-core arm.  Both meet the reference-parity tolerances."""
    precision = precision or DEFAULT_PRECISION
    if precision == "auto":
        return "bf16x3" if (latent_channels is not None and latent_channels % 64 == 0) else "fp32"
    return precision


def require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise _lib.NicError(f"{what}: expected a CUDA tensor on a B200; this package has no CPU path")


def act_dtype(precision: str):
    return torch.float32 if precision == "fp32" else torch.bfloat16


def conv_out_hw(conv: nn.Module, h: int, w: int):
    k, s, p = conv.kernel_size[0], conv.stride[0], conv.padding[0]
    if isinstance(conv, nn.ConvTranspose2d):
        op = conv.output_padding[0]
        return (h - 1) * s - 2 * p + k + op, (w - 1) * s - 2 * p + k + op
    return (h + 2 * p - k) // s + 1, (w + 2 * p - k) // s + 1


class ConvOp:
    """One reference conv layer (+ the GDN / LeakyReLU that follows it) bound to nic_conv_fwd.

    Holds packed-weight caches keyed by precision; a cache entry is rebuilt when the parameter
    storage or its in-place version counter changes (load_state_dict, optimizer step, .to()).
    """

    def __init__(self, conv: nn.Module, epilogue: int = EPI_BIAS, gdn: Optional[nn.Module] = None, mask_a: bool = False,
                 tc_pad_cin: Optional[int] = None, tc_pad_cout: Optional[int] = None):
        self.conv, self.epilogue, self.gdn, self.mask_a = conv, epilogue, gdn, mask_a
        self.transposed = isinstance(conv, nn.ConvTranspose2d)
        # tensor-core arms only: the layer runs with its input / output channels zero-padded to these counts (the engine walks
        # channels in chunks of 64; h_s of the 192-channel model has a 288-channel tensor between its last two layers, which
        # travels as 320 channels whose last 32 are exactly 0 = LeakyReLU(0 . x + 0))
        self.tc_pad_cin, self.tc_pad_cout = tc_pad_cin, tc_pad_cout
        self._cache = {}

    def channels(self, precision):
        cv, tc = self.conv, precision != "fp32"
        return ((self.tc_pad_cin if tc and self.tc_pad_cin else cv.in_channels),
                (self.tc_pad_cout if tc and self.tc_pad_cout else cv.out_channels))

    def desc(self, n, h, w, precision, in_layout, out_layout, in_dtype, out_dtype, out_c_total=0, out_c_offset=0) -> ConvDesc:
        cv = self.conv
        ho, wo = conv_out_hw(cv, h, w)
        d = ConvDesc()
        cin, cout = self.channels(precision)
        d.n, d.c_in, d.h_in, d.w_in = n, cin, h, w
        d.c_out, d.h_out, d.w_out = cout, ho, wo
        d.kh, d.kw, d.stride, d.pad = cv.kernel_size[0], cv.kernel_size[1], cv.stride[0], cv.padding[0]
        d.transposed = int(self.transposed)
        d.output_padding = cv.output_padding[0] if self.transposed else 0
        d.mask_a = int(self.mask_a)
        d.epilogue, d.precision = self.epilogue, PRECISIONS[precision]
        d.in_layout, d.out_layout, d.in_dtype, d.out_dtype = in_layout, out_layout, in_dtype, out_dtype
        d.out_c_total, d.out_c_offset = out_c_total, out_c_offset
        return d

    def _key(self):
        ts = [self.conv.weight, self.conv.bias]
        if self.gdn is not None:
            ts += [self.gdn.beta, self.gdn.gamma]
        return tuple((t.data_ptr(), t._version, str(t.device)) for t in ts)

    def packed(self, precision: str):
        key = self._key()
        ent = self._cache.get(precision)
        if ent is not None and ent[0] == key:
            return ent[1]
        lib = _lib.load()
        cv = self.conv
        require_cuda(cv.weight, "conv weight")
        dev = cv.weight.device
        d = self.desc(1, 64, 64, precision, LAYOUT_NHWC, LAYOUT_NHWC, DT_F32, DT_F32)
        elems = lib.nic_packed_weight_elems(C.byref(d))
        if elems == 0:
            check(-1, "nic_packed_weight_elems")
        wp = torch.empty(elems, dtype=act_dtype(precision), device=dev)
        with torch.cuda.device(dev):
            w32 = cv.weight.detach().float().contiguous()
            bias = cv.bias.detach().float().contiguous()
            cin, cout = self.channels(precision)
            if (cin, cout) != (cv.in_channels, cv.out_channels):          # zero padding of the channel dimensions (see __init__)
                pi, po = cin - cv.in_channels, cout - cv.out_channels
                w32 = torch.nn.functional.pad(w32, (0, 0, 0, 0, 0, po, 0, pi) if self.transposed else (0, 0, 0, 0, 0, pi, 0, po)).contiguous()
                bias = torch.nn.functional.pad(bias, (0, po)).contiguous()
            check(lib.nic_pack_conv_weight(C.byref(d), ptr(w32), ptr(wp), current_stream()), "nic_pack_conv_weight")
            gamma = beta = None
            if self.gdn is not None:
                c = cv.out_channels
                mult = 2 if precision == "bf16x3" else 1           # bf16x3: gamma as bf16 [hi | lo]
                gamma = torch.empty(c * c * mult, dtype=act_dtype(precision), device=dev)
                beta = torch.empty(c, dtype=torch.float32, device=dev)
                check(lib.nic_pack_gdn(c, float(self.gdn.beta_min), ptr(self.gdn.beta.detach().float().contiguous()),
                                       ptr(self.gdn.gamma.detach().float().contiguous()), ptr(beta), ptr(gamma),
                                       PRECISIONS[precision], current_stream()), "nic_pack_gdn")
        out = (wp, bias, gamma, beta)
        self._cache[precision] = (key, out)
        return out

    def run(self, x: torch.Tensor, n: int, h: int, w: int, precision: str, in_layout=LAYOUT_NHWC, out_layout=LAYOUT_NHWC,
            out: Optional[torch.Tensor] = None, out_c_total: int = 0, out_c_offset: int = 0,
            out_dtype=None, keep_ws: Optional[list] = None, in_lo_flag: Optional[torch.Tensor] = None) -> torch.Tensor:
        """x: contiguous tensor in `in_layout`; returns (or fills) the output in `out_layout`.

        In the "bf16x3" arm bf16 tensors are hi/lo PAIRS (NIC_DT_BF16X2: NHWC with 2*c channels) and the default output
        is a pair too; out_dtype=torch.float32 asks for a plain fp32 result.
        keep_ws: a list that receives the call's workspace tensor (fp32 arm + GDN epilogue: the conv output BEFORE the GDN,
        NHWC f32 - what the training step's backward needs).
        in_lo_flag: device int32 written by latent_handoff (0 = the lo half of the pair input is all zero: quantised symbols) -
        the bf16x3 conv then skips its lo . W_hi pass (nic_conv_fwd_ex)."""
        lib = _lib.load()
        require_cuda(x, "conv input")
        x3 = precision == "bf16x3"
        in_dt = (DT_BF16X2 if x3 else DT_BF16) if x.dtype == torch.bfloat16 else DT_F32
        if out_dtype is None:
            out_dtype = act_dtype(precision)
        pair_out = x3 and out_dtype == torch.bfloat16
        out_dt = DT_BF16X2 if pair_out else (DT_BF16 if out_dtype == torch.bfloat16 else DT_F32)
        d = self.desc(n, h, w, precision, in_layout, out_layout, in_dt, out_dt, out_c_total, out_c_offset)
        ctot = (2 if pair_out else 1) * (out_c_total or d.c_out)       # pair tensors: [hi(c) | lo(c)]
        if out is None:
            shape = (n, d.h_out, d.w_out, ctot) if out_layout == LAYOUT_NHWC else (n, ctot, d.h_out, d.w_out)
            out = torch.empty(shape, dtype=out_dtype, device=x.device)
        wp, bias, gamma, beta = self.packed(precision)
        ws_bytes = lib.nic_conv_workspace_bytes(C.byref(d))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device) if ws_bytes else None
        check(lib.nic_conv_fwd_ex(C.byref(d), ptr(x), ptr(wp), ptr(bias), ptr(gamma), ptr(beta), ptr(out), ptr(ws), ws_bytes,
                                  ptr(in_lo_flag) if x3 else None, current_stream()), "nic_conv_fwd")
        if keep_ws is not None:
            keep_ws.append(ws)
        return out


class CtxEpPlan:
    """The context conv + entropy-parameter stack (+ likelihood kernel) of one (batch, size, precision) as ONE C-ABI call
    (nic_ctx_ep_fwd: ContextModels.py:15-20 -> Models.py:73 -> ParametersModels.py:29-64 -> EntropyModels.py:192-233).
    Descriptors, packed weights and the intermediate buffers are set up once; `run` fills `combined[..., phi window]`, the raw
    parameters and - with y_in - the likelihood outputs.  Results are bit-identical to the four ConvOp.run calls + gm_likelihood."""

    def __init__(self, ctx_op: "ConvOp", ep_ops, n: int, h: int, w: int, precision: str, M: int, K: int, device, full: bool = True):
        lib = _lib.load()
        x3 = precision == "bf16x3"
        adt = act_dtype(precision)
        in_dt = (DT_BF16X2 if x3 else DT_BF16) if adt == torch.bfloat16 else DT_F32
        cw = 2 if (x3 and adt == torch.bfloat16) else 1
        self.n, self.h, self.w, self.M, self.K, self.precision, self.full = n, h, w, M, K, precision, full
        self.descs = [ctx_op.desc(n, h, w, precision, LAYOUT_NHWC, LAYOUT_NHWC, in_dt, in_dt, 4 * M, 0),
                      ep_ops[0].desc(n, h, w, precision, LAYOUT_NHWC, LAYOUT_NHWC, in_dt, in_dt),
                      ep_ops[1].desc(n, h, w, precision, LAYOUT_NHWC, LAYOUT_NHWC, in_dt, in_dt),
                      ep_ops[2].desc(n, h, w, precision, LAYOUT_NHWC, LAYOUT_NCHW, in_dt, DT_F32)]
        self.ops = [ctx_op] + list(ep_ops)
        self.e1 = torch.empty((n, h, w, cw * self.descs[1].c_out), dtype=adt, device=device)
        self.e2 = torch.empty((n, h, w, cw * self.descs[2].c_out), dtype=adt, device=device)
        ws = max(lib.nic_conv_workspace_bytes(C.byref(d)) for d in self.descs)
        self.ws = torch.empty(max(ws, 256), dtype=torch.uint8, device=device)
        self.device = device

    def run(self, y_in_engine: torch.Tensor, combined: torch.Tensor, y_in: Optional[torch.Tensor] = None, qmode: int = 2,
            in_lo_flag: Optional[torch.Tensor] = None):
        """-> (raw [n, C, h, w] f32, likelihood dict | None).  qmode: _lib.Q_* (default Q_PASSTHRU: y_in is already quantised)."""
        lib = _lib.load()
        n, h, w, M, K = self.n, self.h, self.w, self.M, self.K
        packed = [op.packed(self.precision) for op in self.ops]
        raw = torch.empty((n, self.descs[3].c_out, h, w), dtype=torch.float32, device=self.device)
        a = _lib.CtxEpArgs()
        a.ctx = C.pointer(self.descs[0])
        for i in range(3):
            a.ep[i] = C.pointer(self.descs[1 + i])
            a.w_ep[i], a.b_ep[i] = ptr(packed[1 + i][0]), ptr(packed[1 + i][1])
        a.w_ctx, a.b_ctx = ptr(packed[0][0]), ptr(packed[0][1])
        a.y_in_engine, a.y_in_lo_nonzero = ptr(y_in_engine), ptr(in_lo_flag)
        a.combined, a.e1, a.e2, a.raw = ptr(combined), ptr(self.e1), ptr(self.e2), ptr(raw)
        a.workspace, a.workspace_bytes = ptr(self.ws), self.ws.numel()
        out = None
        if y_in is not None:
            p, logp = torch.empty_like(y_in), torch.empty_like(y_in)
            parts = partials(n, self.device)
            out = {"p": p, "logp": logp, "partials": parts}
            a.y_in, a.m, a.k, a.qmode = ptr(y_in), M, K, qmode
            a.p, a.logp, a.logp_partials = ptr(p), ptr(logp), ptr(parts)
            if self.full:
                shape = (n, M, h, w) if K == 1 else (n, K, M, h, w)
                mus, sgs = torch.empty(shape, dtype=torch.float32, device=self.device), torch.empty(shape, dtype=torch.float32, device=self.device)
                a.mus, a.sigmas = ptr(mus), ptr(sgs)
                if K == 1:
                    out["mu"], out["sigma"] = mus, sgs
                else:
                    ws_ = torch.empty(shape, dtype=torch.float32, device=self.device)
                    a.weights = ptr(ws_)
                    out["weights"], out["mus"], out["sigmas"] = ws_, mus, sgs
        with torch.cuda.device(self.device):
            check(lib.nic_ctx_ep_fwd(C.byref(a), current_stream()), "nic_ctx_ep_fwd")
        return raw, out


def to_pair(v: torch.Tensor) -> torch.Tensor:
    """f32 [..., c] -> bf16 [..., 2c] = [hi | lo], hi = bf16(v), lo = bf16(v - hi): the NIC_DT_BF16X2 activation format."""
    hi = v.to(torch.bfloat16)
    lo = (v - hi.float()).to(torch.bfloat16)
    return torch.cat([hi, lo], dim=-1).contiguous()


def from_pair(p: torch.Tensor) -> torch.Tensor:
    c = p.shape[-1] // 2
    return p[..., :c].float() + p[..., c:].float()


def run_sequential_nchw(ops, x: torch.Tensor, precision: str) -> torch.Tensor:
    """A chain of ConvOps with reference (NCHW f32) tensors at both ends; NHWC inside."""
    require_cuda(x, "input")
    x = x.contiguous().float()
    n, cin, h, w = x.shape
    cur, layout = x, LAYOUT_NCHW
    if precision != "fp32" and cin >= 64:
        # stand-alone call of an inner transform in a tensor-core mode: the engine wants NHWC bf16 (cold path)
        cur, layout = x.permute(0, 2, 3, 1).contiguous(), LAYOUT_NHWC
        cur = to_pair(cur) if precision == "bf16x3" else cur.to(torch.bfloat16)
    with torch.cuda.device(x.device):
        for i, op in enumerate(ops):
            last = i == len(ops) - 1
            cur = op.run(cur, n, h, w, precision, in_layout=layout, out_layout=LAYOUT_NCHW if last else LAYOUT_NHWC,
                         out_dtype=torch.float32 if last else None)
            h, w = conv_out_hw(op.conv, h, w)
            layout = LAYOUT_NHWC
    return cur


def latent_handoff(v_nhwc: torch.Tensor, qmode: int, noise: Optional[torch.Tensor], in_dtype: torch.dtype,
                   want_lowp: bool = False, lowp_pair: bool = False):
    """Models.py:52-66.  Returns (v_nchw, v_in_nchw, v_in_nhwc, v_nhwc_lowp | None); lowp_pair -> hi/lo pair (2c channels).
    With a pair-format v_in_nhwc the tensor carries `_nic_lo_flag`: a device int32 that is 0 when its lo half is all zero."""
    lib = _lib.load()
    n, h, w, c = v_nhwc.shape
    v = torch.empty((n, c, h, w), dtype=torch.float32, device=v_nhwc.device)
    v_in = torch.empty_like(v)
    in_pair = in_dtype == "bf16x2"                      # engine-layout copy as a bf16 hi/lo pair (bf16x3 arm)
    if in_pair:
        in_dtype = torch.bfloat16
    v_in_nhwc = torch.empty((n, h, w, 2 * c if in_pair else c), dtype=in_dtype, device=v_nhwc.device)
    v_lowp = torch.empty((n, h, w, 2 * c if lowp_pair else c), dtype=torch.bfloat16, device=v_nhwc.device) if want_lowp else None
    if noise is not None:
        noise = noise.contiguous().float()
    flag = torch.empty(1, dtype=torch.int32, device=v_nhwc.device) if in_pair else None
    check(lib.nic_latent_handoff_ex(ptr(v_nhwc), n, c, h, w, qmode, ptr(noise), ptr(v), ptr(v_in), ptr(v_in_nhwc),
                                    DT_BF16X2 if in_pair else (DT_BF16 if in_dtype == torch.bfloat16 else DT_F32), ptr(v_lowp),
                                    DT_BF16X2 if lowp_pair else DT_BF16, ptr(flag), current_stream()),
          "nic_latent_handoff")
    if flag is not None:
        v_in_nhwc._nic_lo_flag = flag
    return v, v_in, v_in_nhwc, v_lowp


def _nhwc_out(n, h, w, c, dtype, device):
    """(tensor, NIC_DT_*) of an NHWC hand-off output; dtype torch.float32, torch.bfloat16 or "bf16x2" (hi/lo pair, 2c channels)."""
    if dtype == "bf16x2":
        return torch.empty((n, h, w, 2 * c), dtype=torch.bfloat16, device=device), DT_BF16X2
    return torch.empty((n, h, w, c), dtype=dtype, device=device), (DT_BF16 if dtype == torch.bfloat16 else DT_F32)


def latent_handoff_gain(v_nhwc: torch.Tensor, qmode: int, noise: Optional[torch.Tensor], gain: Optional[torch.Tensor],
                        inv_gain: Optional[torch.Tensor], sym_dtype=None, src_dtype=None, scaled_dtype=None):
    """The hand-off with gain units (nic_latent_handoff_gain): v_g = gain (.) v is quantised.  gain / inv_gain: [n, c] f32 per
    image and channel, or None for 1.  Returns (v_g NCHW, v_in NCHW, symbols NHWC in sym_dtype | None, v_g NHWC in src_dtype | None,
    inv_gain (.) v_in NHWC in scaled_dtype | None); dtypes as latent_handoff's in_dtype.  A pair-format symbol tensor carries
    `_nic_lo_flag`; the scaled one never does."""
    lib = _lib.load()
    n, h, w, c = v_nhwc.shape
    dev = v_nhwc.device
    v = torch.empty((n, c, h, w), dtype=torch.float32, device=dev)
    v_in = torch.empty_like(v)
    sym, sym_dt = _nhwc_out(n, h, w, c, sym_dtype, dev) if sym_dtype is not None else (None, DT_F32)
    src, src_dt = _nhwc_out(n, h, w, c, src_dtype, dev) if src_dtype is not None else (None, DT_F32)
    scaled, sc_dt = _nhwc_out(n, h, w, c, scaled_dtype, dev) if scaled_dtype is not None else (None, DT_F32)
    if noise is not None:
        noise = noise.contiguous().float()
    flag = torch.empty(1, dtype=torch.int32, device=dev) if sym_dt == DT_BF16X2 else None
    check(lib.nic_latent_handoff_gain(ptr(v_nhwc), n, c, h, w, qmode, ptr(noise), ptr(gain), ptr(v), ptr(v_in), ptr(sym), sym_dt,
                                      ptr(flag), ptr(src), src_dt, ptr(inv_gain), ptr(scaled), sc_dt, current_stream()),
          "nic_latent_handoff_gain")
    if flag is not None:
        sym._nic_lo_flag = flag
    return v, v_in, sym, src, scaled


def checkerboard_zero_(t: torch.Tensor) -> torch.Tensor:
    """In place: 0 at the anchors (i + j even) of a contiguous NHWC f32 tensor [n, h, w, c] (nic_checkerboard_zero)."""
    n, h, w, c = t.shape
    check(_lib.load().nic_checkerboard_zero(ptr(t), DT_F32, LAYOUT_NHWC, n, h, w, c, c, 0, current_stream()), "nic_checkerboard_zero")
    return t


def attach_partials(logp: torch.Tensor, parts: torch.Tensor) -> None:
    """Let the per-image partial sums the likelihood kernel produced ride along with `logp` for rd_loss (RateDistortionLoss.py:
    13-14), together with logp's version: a caller that modifies logp in place invalidates them (rd_loss then re-sums)."""
    logp._nic_partials = parts
    logp._nic_partials_version = logp._version


def partials(b: int, device) -> torch.Tensor:
    return torch.empty((b, _lib.load().nic_partials_per_image()), dtype=torch.float32, device=device)
