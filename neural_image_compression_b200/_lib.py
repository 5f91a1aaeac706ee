"""ctypes binding of libnic_b200.so - the C ABI declared in include/nic.h.

The product path has no fallback: if the shared object is missing or the device is not a B200
(sm_100), calls raise.  Nothing here imports ``oracle``.
"""
from __future__ import annotations

import ctypes as C
import os
import re

from . import _build

_i32, _i64, _f32, _vp, _sz = C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_size_t

# enums of include/nic.h
LAYOUT_NCHW, LAYOUT_NHWC = 0, 1
DT_F32, DT_BF16, DT_BF16X2 = 0, 1, 2
PREC_FP32, PREC_BF16, PREC_BF16X3 = 0, 1, 2
EPI_BIAS, EPI_LRELU, EPI_GDN, EPI_IGDN = 0, 1, 2, 3
Q_ROUND, Q_NOISE, Q_PASSTHRU = 0, 1, 2
MASK_A, MASK_B, MASK_CHECKERBOARD = 1, 2, 3        # nic_conv_desc.mask_a
PRECISIONS = {"fp32": PREC_FP32, "bf16": PREC_BF16, "bf16x3": PREC_BF16X3}
# model-level modes: "mixed" = g_a and h_a (everything upstream of the rounding) in fp32, the rest in bf16
#                     "bf16x3" = every transform on the tensor cores with hi/lo-split operands (fp32 grade)
MODEL_PRECISIONS = ("fp32", "bf16", "mixed", "bf16x3")


class ConvDesc(C.Structure):
    """struct nic_conv_desc (include/nic.h)."""
    _fields_ = [(n, _i32) for n in (
        "n", "c_in", "h_in", "w_in", "c_out", "h_out", "w_out", "kh", "kw", "stride", "pad",
        "transposed", "output_padding", "mask_a", "epilogue", "precision", "in_layout", "out_layout",
        "in_dtype", "out_dtype", "out_c_total", "out_c_offset")]


class CtxEpArgs(C.Structure):
    """struct nic_ctx_ep_args (include/nic.h): one call for context conv + entropy-parameter stack (+ likelihoods)."""
    _fields_ = [("ctx", C.POINTER(ConvDesc)), ("ep", C.POINTER(ConvDesc) * 3), ("w_ctx", _vp), ("b_ctx", _vp), ("w_ep", _vp * 3),
                ("b_ep", _vp * 3), ("y_in_engine", _vp), ("y_in_lo_nonzero", _vp), ("combined", _vp), ("e1", _vp), ("e2", _vp),
                ("raw", _vp), ("y_in", _vp), ("noise", _vp), ("m", _i32), ("k", _i32), ("qmode", _i32), ("reserved", _i32),
                ("y_in_out", _vp), ("p", _vp), ("logp", _vp), ("weights", _vp), ("mus", _vp), ("sigmas", _vp), ("logp_partials", _vp),
                ("workspace", _vp), ("workspace_bytes", _sz)]


class CodecHead(C.Structure):
    """struct nic_codec_head (include/nic.h): one entropy head of nic_codec_params."""
    _fields_ = [(n, _vp) for n in ("sym", "w_ctx", "b_ctx", "w1", "b1", "w2", "b2", "w3", "b3", "raw", "work")] + \
               [("work_floats", _i64), ("m", _i32), ("reserved", _i32)]


# name -> (restype, argtypes); must list every function include/nic.h declares (tests check this)
SIGNATURES = {
    "nic_version": (C.c_int, []),
    "nic_last_error": (C.c_char_p, []),
    "nic_check_device": (C.c_int, []),
    "nic_launch_count": (C.c_uint64, []),
    "nic_pipeline_status": (C.c_int, []),
    "nic_packed_weight_elems": (_sz, [C.POINTER(ConvDesc)]),
    "nic_pack_conv_weight": (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp]),
    "nic_pack_gdn": (C.c_int, [_i32, _f32, _vp, _vp, _vp, _vp, _i32, _vp]),
    "nic_conv_workspace_bytes": (_sz, [C.POINTER(ConvDesc)]),
    "nic_conv_fwd": (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nic_conv_fwd_ex": (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp]),
    "nic_ctx_ep_fwd": (C.c_int, [C.POINTER(CtxEpArgs), _vp]),
    "nic_gdn_fwd": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "nic_latent_handoff": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _i32, _vp]),
    "nic_latent_handoff_ex": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _i32, _vp, _vp]),
    "nic_partials_per_image": (_i32, []),
    "nic_gm_likelihood_fwd": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nic_gm_pmf_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "nic_gm_pmf_mass_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "nic_pack_factorized": (C.c_int, [_i32] + [_vp] * 11 + [_vp, _vp]),
    "nic_factorized_likelihood_fwd": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "nic_sse_fwd": (C.c_int, [_vp, _vp, _i32, _i64, _vp, _vp]),
    "nic_sum_fwd": (C.c_int, [_vp, _i32, _i64, _vp, _vp]),
    "nic_rd_reduce": (C.c_int, [_vp, _i32, _i32, _f32, _vp, _vp]),
    "nic_rd_finalize": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i64, _f32, _vp, _vp, _vp]),
    # training step (backward)
    "nic_conv_wgrad_workspace_bytes": (_sz, [C.POINTER(ConvDesc)]),
    "nic_conv_wgrad": (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nic_conv_wgrad_tc_workspace_bytes": (_sz, [C.POINTER(ConvDesc)]),
    "nic_conv_wgrad_tc": (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nic_lrelu_bwd": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "nic_gdn_bwd_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32]),
    "nic_gdn_bwd": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nic_gm_likelihood_bwd": (C.c_int, [_vp, _vp, _vp, _f32, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "nic_factorized_likelihood_bwd": (C.c_int, [_vp, _vp, _vp, _f32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "nic_sse_bwd": (C.c_int, [_vp, _vp, _i64, _f32, _vp, _vp]),
    "nic_sse_bwd_per_image": (C.c_int, [_vp, _vp, _i32, _i64, _vp, _vp, _vp]),
    "nic_add_inplace": (C.c_int, [_vp, _vp, _i64, _vp]),
    "nic_layout_convert": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp]),
    "nic_eval_mse": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "nic_luma": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "nic_ms_ssim_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "nic_ms_ssim_levels": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _f32, _i32, _vp, _vp, _sz, _vp]),
    "nic_ms_ssim_bwd_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "nic_ms_ssim_bwd": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _f32, _vp, _vp, _vp, _sz, _vp]),
    "nic_adam_multi_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _f32, _f32, _f32, _f32, _i32, _vp, _vp]),
    "nic_adam_multi_step_ex": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _f32, _vp, _f32, _f32, _f32, _f32, _i32, _vp, _vp]),
    "nic_counter_increment": (C.c_int, [_vp, _vp]),
    "nic_to_pair": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp]),
    "nic_gdn_reparam": (C.c_int, [_i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nic_gdn_apply": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "nic_gdn_apply_add": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _vp]),
    "nic_gdn_bwd_prep": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "nic_gdn_bwd_du": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "nic_gdn_reparam_bwd": (C.c_int, [_i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nic_gdn_bwd_finish_workspace_bytes": (_sz, [_i64, _i32]),
    "nic_gdn_bwd_finish": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nic_adam_step": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _i32, _vp]),
    # entropy coder
    "nic_codec_tables": (C.c_int, [_i32, _i32, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "nic_codec_encode": (C.c_int, [_i32, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i64, _vp, _vp, _vp]),
    "nic_codec_decode": (C.c_int, [_i32, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "nic_codec_decode_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "nic_codec_checksum": (C.c_int, [_vp, _i64, _vp, _i64, _i32, _vp, _vp]),
    "nic_codec_encode_checkerboard": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i64, _vp, _vp, _vp]),
    "nic_codec_decode_pass": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "nic_codec_encode_checkerboard_slice": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i64, _vp, _vp, _vp]),
    "nic_codec_decode_pass_slice": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32,
                                              _vp, _vp]),
    "nic_checkerboard_zero": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "nic_codec_params": (C.c_int, [C.POINTER(CodecHead), _i32, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "nic_image_window": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _i32, _i32, _vp]),
    # gain units
    "nic_gain_vectors": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _i32, _vp, _vp]),
    "nic_latent_handoff_gain": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp,
                                          _i32, _vp]),
    "nic_gain_bwd": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i64, _vp, _i32, _vp, _vp]),
    "nic_gain_fold": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
}

# entropy coder constants of include/nic.h
CODEC_GM, CODEC_FACTORIZED = 0, 1
CODEC_TABLES, CODEC_SYMBOL = 0, 1
CODEC_PREC_BITS, CODEC_WINDOW = 16, 128

_lib = None


class NicError(RuntimeError):
    pass


def header_functions():
    """Function names declared in include/nic.h (used by the ABI test)."""
    hdr = os.path.join(os.path.dirname(_build.PKG_DIR), "include", "nic.h")
    text = re.sub(r"/\*.*?\*/", "", open(hdr).read(), flags=re.S)
    return sorted(set(re.findall(r"\b(nic_[a-z0-9_]+)\s*\(", text)))


def load(build_if_missing: bool = True):
    """Load (building in-tree first if needed) the shared object.  Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if not os.path.exists(path) or (build_if_missing and _build.is_stale() and _has_nvcc()):
        if not build_if_missing:
            raise NicError(f"{path} is missing; run `python __graft_entry__.py` (build) first")
        _build.build()
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def _has_nvcc():
    try:
        _build._nvcc()
        return True
    except RuntimeError:
        return False


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().nic_last_error()
        raise NicError(f"{what or 'libnic_b200'} failed (code {rc}): {msg.decode() if msg else ''}")


def ptr(t):
    """Raw device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def current_stream():
    import torch
    return torch.cuda.current_stream().cuda_stream
