"""ctypes binding of libidf_b200.so (C ABI declared in include/idf_b200.h).

There is deliberately no fallback: if the shared library is missing or the device is not sm_100,
every entry point raises.  The library is built in-tree by ``infodiffusion_b200.build``.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libidf_b200.so"

IDF_CONV_MAX_KB = 160
IDF_CONV_MAX_SRC = 3
EPI_BF16, EPI_F32_NCHW, EPI_SAMPLER = 0, 1, 2


class ConvDesc(C.Structure):
    _fields_ = [
        ("n_src", C.c_int32),
        ("src", C.c_void_p * IDF_CONV_MAX_SRC),
        ("src_rows", C.c_int64 * IDF_CONV_MAX_SRC),
        ("src_ld", C.c_int32 * IDF_CONV_MAX_SRC),
        ("num_kb", C.c_int32),
        ("kb_src", C.c_int32 * IDF_CONV_MAX_KB),
        ("kb_c0", C.c_int32 * IDF_CONV_MAX_KB),
        ("kb_rowoff", C.c_int32 * IDF_CONV_MAX_KB),
        ("weight", C.c_void_p),
        ("cout_pad", C.c_int32),
        ("block_n", C.c_int32),
        ("cout", C.c_int32),
        ("bias", C.c_void_p),
        ("batch", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("epilogue", C.c_int32),
        ("out", C.c_void_p),
        ("out_ld", C.c_int32),
        ("residual", C.c_void_p),
        ("res_ld", C.c_int32),
        ("out_f32", C.c_void_p),
        ("x_io", C.c_void_p),
        ("noise", C.c_void_p),
        ("coef", C.c_void_p),
        ("step_ptr", C.c_void_p),
        ("stats_out", C.c_void_p),
        ("xf_coef", C.c_void_p), ("xf_ctot", C.c_int32), ("xf_silu", C.c_int32), ("kb_xf", C.c_int32 * IDF_CONV_MAX_KB),
        ("up2", C.c_int32),
    ]


class WgradDesc(C.Structure):
    _fields_ = [
        ("dy", C.c_void_p), ("rows", C.c_int64), ("cout", C.c_int32),
        ("x", C.c_void_p), ("x_rows", C.c_int64), ("cin", C.c_int32),
        ("n_taps", C.c_int32), ("tap_off", C.c_int32 * 9),
        ("dw", C.c_void_p),
        ("partials", C.c_void_p),
    ]


class AdaGNArgs(C.Structure):
    _fields_ = [
        ("src0", C.c_void_p), ("c0", C.c_int32),
        ("src1", C.c_void_p), ("c1", C.c_int32),
        ("out", C.c_void_p),
        ("batch", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("gamma", C.c_void_p), ("beta", C.c_void_p),
        ("eps", C.c_float),
        ("mod_t", C.c_void_p), ("mod_t_step_stride", C.c_int64), ("mod_t_batch_stride", C.c_int64),
        ("mod_z", C.c_void_p), ("mod_z_step_stride", C.c_int64), ("mod_z_batch_stride", C.c_int64),
        ("step_ptr", C.c_void_p),
        ("apply_silu", C.c_int32),
        ("stats0", C.c_void_p), ("stats1", C.c_void_p),
        ("dropout_p", C.c_float), ("dropout_seed", C.c_void_p), ("dropout_layer", C.c_uint32),
        ("save_coef", C.c_void_p),
        ("stats_unit0", C.c_int32), ("stats_unit1", C.c_int32),
        ("stats_planes0", C.c_int32), ("stats_planes1", C.c_int32), ("stats_rows0", C.c_int32), ("stats_rows1", C.c_int32),
    ]


class ClipAdamWArgs(C.Structure):
    _fields_ = [
        ("params", C.c_void_p), ("grads", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p),
        ("numel", C.c_void_p), ("chunk_tensor", C.c_void_p), ("chunk_offset", C.c_void_p),
        ("n_chunks", C.c_int32),
        ("bias_corrections", C.c_void_p),
        ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("weight_decay", C.c_float),
        ("max_norm", C.c_float),
        ("partial", C.c_void_p), ("norm_out", C.c_void_p),
    ]


class AdaGNBwdArgs(C.Structure):
    _fields_ = [
        ("f", AdaGNArgs),
        ("dy", C.c_void_p),
        ("dx0", C.c_void_p), ("dx1", C.c_void_p),
        ("acc0", C.c_int32), ("acc1", C.c_int32),
        ("sums", C.c_void_p),
        ("ws", C.c_void_p),
        ("d_mod_t", C.c_void_p), ("d_mod_z", C.c_void_p), ("dgamma", C.c_void_p), ("dbeta", C.c_void_p),
        ("dparam_ws", C.c_void_p), ("dparam_ticket", C.c_void_p),
    ]


# name -> (restype, argtypes); every symbol include/idf_b200.h declares
SIGNATURES = {
    "idf_version": (C.c_int, []),
    "idf_last_error": (C.c_char_p, []),
    "idf_init": (C.c_int, []),
    "idf_set_option": (C.c_int, [C.c_char_p, C.c_int32]),
    "idf_conv_plan_create": (C.c_int, [C.POINTER(ConvDesc), C.POINTER(C.c_void_p)]),
    "idf_conv_plan_destroy": (C.c_int, [C.c_void_p]),
    "idf_conv_run": (C.c_int, [C.c_void_p, C.c_void_p]),
    "idf_conv_plan_tiles": (C.c_int64, [C.c_void_p]),
    "idf_conv_plan_stats_unit": (C.c_int32, [C.c_void_p]),
    "idf_wgrad_plan_create": (C.c_int, [C.POINTER(WgradDesc), C.POINTER(C.c_void_p)]),
    "idf_wgrad_plan_destroy": (C.c_int, [C.c_void_p]),
    "idf_wgrad_run": (C.c_int, [C.c_void_p, C.c_void_p]),
    "idf_wgrad_plan_partials_floats": (C.c_int64, [C.c_void_p]),
    "idf_adagn_coef": (C.c_int, [C.POINTER(AdaGNArgs), C.c_void_p, C.c_void_p]),
    "idf_adagn_silu_fwd": (C.c_int, [C.POINTER(AdaGNArgs), C.c_void_p]),
    "idf_adagn_bwd_ws_floats": (C.c_int64, [C.c_int32, C.c_int32]),
    "idf_adagn_silu_bwd": (C.c_int, [C.POINTER(AdaGNBwdArgs), C.c_void_p]),
    "idf_attn_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                               C.c_void_p]),
    "idf_attn_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                               C.c_float, C.c_void_p]),
    "idf_attn_bwd_ws_bytes": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "idf_linear_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                 C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "idf_gemm_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64,
                               C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "idf_gemm_f32_ordered": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                       C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "idf_gemm_f32_ws_floats": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "idf_scale_layernorm_silu": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_float, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                           C.c_void_p]),
    "idf_clip_adamw": (C.c_int, [C.c_void_p, C.c_void_p]),
    "idf_to_uint8_hwc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "idf_copy2d_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "idf_gather_elems": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "idf_gather_rows_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "idf_im2col_head": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "idf_upsample2x": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "idf_space_to_depth": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_void_p]),
    "idf_nchw_to_padflat": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_void_p]),
    "idf_padflat_to_nchw": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_void_p]),
    "idf_nchw_to_padflat_ld": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_void_p]),
    "idf_upsample2x_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_void_p]),
    "idf_depth_to_space": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_void_p]),
    "idf_colsum_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "idf_colsum_bf16_ordered": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p,
                                          C.c_void_p]),
    "idf_colsum_ws_floats": (C.c_int64, [C.c_int64, C.c_int32]),
    "idf_sampler_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                     C.c_void_p]),
    "idf_mmd_fwd_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                  C.c_void_p]),
    "idf_mmd_fwd_bwd_ordered": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "idf_mmd_ws_floats": (C.c_int64, [C.c_int32]),
}

_lib = None
_launches = 0


class IdfError(RuntimeError):
    pass


def load(build_if_missing: bool = True):
    """dlopen libidf_b200.so and attach the signatures.  Raises if it cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if not build_if_missing:
            raise IdfError(f"{LIB_PATH} is missing; run `python -m infodiffusion_b200.build`")
        from . import build as _build
        _build.build()
    import os
    # kernel development only: A/B an alternative build of the SAME C-ABI (e.g. the previous commit's kernels)
    lib = C.CDLL(os.environ.get("IDF_LIB_AB") or str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().idf_last_error()
        raise IdfError(f"idf_b200 error {rc}: {msg.decode() if msg else '?'}")


_WEIGHT_EPOCH = 0


def bump_weight_epoch() -> None:
    """Called by code that updates parameters behind torch's back (ClipAdamW writes them from a CUDA kernel through
    raw pointers, so tensor._version does not move): cached inference plans hold packed bf16 copies of the weights
    and must be rebuilt."""
    global _WEIGHT_EPOCH
    _WEIGHT_EPOCH += 1


def weight_epoch() -> int:
    return _WEIGHT_EPOCH


def count_launch(n: int = 1) -> None:
    global _launches
    _launches += n


def launches() -> int:
    """Number of idf kernel launches issued through this binding (bench.py's gpu_launches claim)."""
    return _launches
