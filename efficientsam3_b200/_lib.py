"""ctypes binding of libes3.so (the C ABI declared in include/es3.h).

The product path has NO fallback: if the shared library is missing, or the device is not a CC 10.x
GPU, importing/using the ops raises.  Nothing in this package imports `oracle/`.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libes3.so"

_vp, _ll, _i, _f = C.c_void_p, C.c_longlong, C.c_int, C.c_float

# name -> argtypes  (restype is always int unless noted)
SIGNATURES: dict[str, list] = {
    "es3_init": [_i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)],
    "es3_gemm_bf16": [_vp, _ll, _vp, _ll, _vp, _ll, _i, _i, _i, _i, _vp, _vp, _i, _vp, _ll, _i, _vp],
    "es3_gemm_bf16_ex": [_vp, _ll, _vp, _ll, _vp, _ll, _i, _i, _i, _i, _vp, _vp, _i, _vp, _ll, _i, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "es3_win_attn_bias_bf16": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp],
    "es3_layernorm_bf16": [_vp, _vp, _vp, _f, _vp, _ll, _i, _vp],
    "es3_layernorm_f32": [_vp, _vp, _i, _i, _i, _vp, _vp, _f, _vp, _vp, _ll, _i, _vp],
    "es3_im2col_patch": [_vp, _vp, _i, _i, _i, _i, _vp],
    "es3_attention_bf16": [_vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp],
    "es3_attention_tc_bf16": [_vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp],
    "es3_attention_mma_bf16": [_vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp],
    "es3_tokens_f32_to_nchw": [_vp, _vp, _i, _i, _i, _vp],
    "es3_cast_f32_to_f16": [_vp, _vp, _ll, _vp],
    "es3_convt2x2_bf16": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _vp, _i, _i, _vp],
    "es3_dense_pe": [_vp, _i, _i, _i, _vp, _vp],
    "es3_point_embed": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _f, _vp, _vp],
    "es3_mask_downscale_tokens": [_vp] * 12 + [_ll, _vp, _vp, _i, _i, _i, _i, _f, _vp],
    "es3_fill_small_components": [_vp, _vp, _vp, _vp, _i, _i, _i, _f, _f, _f, _vp],
    "es3_add_rows": [_vp, _vp, _ll, _i, _i, _vp, _vp, _vp],
    "es3_nchw_f32_to_tokens": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp],
    "es3_attn_few_queries": [_vp, _ll, _vp, _vp, _ll, _i, _vp, _ll, _i, _i, _i, _i, _i, _f, _vp],
    "es3_attn_few_keys": [_vp, _ll, _vp, _vp, _ll, _vp, _ll, _i, _i, _i, _i, _i, _f, _vp],
    "es3_ln_rows_gelu": [_vp, _vp, _vp, _f, _vp, _ll, _i, _vp],
    "es3_hyper_masks": [_vp, _vp, _vp, _f, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "es3_bilinear_nchw_f32": [_vp, _vp, _vp, _f, _ll, _i, _i, _i, _i, _vp],
    "es3_kd_loss_fwd": [_vp, _vp, _vp, _i, _i, _i, _i, _f, _vp, _vp, _vp, _vp],
    "es3_kd_loss_bwd": [_vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _i, _f, _vp, _vp],
    "es3_grad_norm": [_vp, _ll, _vp, _vp, _vp],
    "es3_adamw_flat": [_vp, _vp, _vp, _vp, _ll, _ll, _f, _f, _f, _f, _f, _f, _f, _vp, _vp, _i, _f, _f, _i, _vp],
    "es3_conv3x3_s2_narrow_bf16": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "es3_channel_mean": [_vp, _vp, _vp, _i, _i, _i, _vp],
    "es3_scale_channels": [_vp, _vp, _vp, _i, _i, _i, _vp],
    "es3_conv3x3_bf16": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp, _i, _vp],
    "es3_gemm_simt": [_vp, _ll, _i, _vp, _ll, _i, _vp, _ll, _i, _i, _i, _i, _vp, _vp, _i, _vp, _ll, _i, _vp],
    "es3_stem_conv3x3_s2": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "es3_dwconv_bf16": [_vp, _ll, _vp, _vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _i, _vp],
    "es3_dwconv_tiled_bf16": [_vp, _ll, _vp, _vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _i, _vp],
    "es3_litemla_aggreg_tiled": [_vp, _ll, _vp, _vp, _i, _i, _i, _i, _vp],
    "es3_mbconv_fused_bf16": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "es3_mbconv_tc_bf16": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "es3_mbconv_tc_s2_bf16": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "es3_dwproj_tc_bf16": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "es3_stem_fused_c16": [_vp] * 10 + [_i, _i, _i, _vp],
    "es3_dsconv_res_bf16": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "es3_bilinear_nhwc_to_nchw": [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "es3_maxpool2x2_bf16": [_vp, _vp, _i, _i, _i, _i, _vp],
    "es3_nhwc_to_nchw_f32": [_vp, _vp, _i, _i, _i, _vp],
    "es3_nchw_f32_to_nhwc": [_vp, _vp, _i, _i, _i, _vp],
    "es3_litemla_aggreg": [_vp, _ll, _vp, _vp, _i, _i, _i, _i, _vp],
    "es3_litemla_aggreg_tc": [_vp, _ll, _vp, _i, _i, _i, _i, _vp],
    "es3_litemla_aggreg_dwpw": [_vp, _ll, _vp, _vp, _i, _i, _i, _i, _vp],
    "es3_litemla_attn_tc": [_vp, _ll, _vp, _vp, _ll, _i, _i, _i, _f, _vp],
    "es3_litemla_attn": [_vp, _ll, _vp, _vp, _ll, _i, _i, _i, _f, _vp],
    "es3_litemla_attn_generic": [_vp, _ll, _vp, _vp, _ll, _i, _i, _i, _i, _f, _vp],
    # student backward (train_bwd.cu)
    "es3_bn_stats": [_vp, _ll, _i, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "es3_affine_act": [_vp, _vp, _vp, _i, _vp, _vp, _ll, _i, _vp],
    "es3_bn_act_bwd_reduce": [_vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _ll, _i, _vp, _vp, _vp, _vp, _vp],
    "es3_bn_act_bwd_apply": [_vp, _vp, _vp, _vp, _i, _vp, _vp, _ll, _i, _vp],
    "es3_add_bf16": [_vp, _ll, _vp, _ll, _vp, _ll, _ll, _i, _vp],
    "es3_wgrad_pw": [_vp, _ll, _vp, _ll, _ll, _i, _i, _i, _i, _i, _i, _vp, _vp, _ll, _ll, _vp],
    "es3_transpose_pad_bf16": [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "es3_accumulate_strided": [_vp, _ll, _i, _ll, _ll, _vp, _vp],
    "es3_dwconv_bwd_data": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "es3_dwconv_wgrad": [_vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    "es3_round_taps_sum_bf16": [_vp, _vp, _i, _i, _vp],
    "es3_dwconv_tc_bf16": [_vp, _ll, _vp, _vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _vp],
    "es3_dwconv_wgrad_win": [_vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    "es3_dwconv_wgrad_tiled": [_vp, _vp, _ll, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    "es3_se_bwd_dgate": [_vp, _vp, _i, _i, _i, _vp, _vp, _vp],
    "es3_se_bwd_apply": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp],
    "es3_layernorm_bwd": [_vp, _vp, _vp, _vp, _f, _vp, _ll, _i, _vp, _vp, _vp, _vp],
    "es3_win_attn_bias_bwd": [_vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _f, _vp],
    "es3_colsum_f32": [_vp, _ll, _ll, _i, _vp, _vp, _vp],
    "es3_pw_small_bf16": [_vp, _ll, _vp, _ll, _vp, _ll, _vp, _ll, _ll, _i, _i, _vp],
    "es3_wgrad_tc": [_vp, _ll, _vp, _ll, _ll, _i, _i, _vp, _vp, _ll, _vp],
    # strict (fp32-class) precision mode (strict_f32.cu)
    "es3_sgemm_f32": [_vp, _ll, _vp, _ll, _vp, _ll, _ll, _i, _i, _vp, _vp, _i, _vp, _ll, _i, _vp],
    "es3_im2col_f32": [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "es3_dwconv_f32": [_vp, _ll, _vp, _vp, _vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _i, _vp],
    "es3_litemla_attn_f32": [_vp, _ll, _vp, _vp, _ll, _i, _i, _i, _i, _f, _vp],
    "es3_bilinear_nhwc_f32_to_nchw": [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "es3_attn_few_keys_f32": [_vp, _ll, _vp, _vp, _ll, _vp, _ll, _i, _i, _i, _i, _i, _f, _vp],
    "es3_ln_rows_gelu_f32": [_vp, _vp, _vp, _f, _vp, _ll, _i, _vp],
    "es3_bias_act_res_f32": [_vp, _vp, _vp, _vp, _ll, _i, _i, _i, _vp],
    "es3_ln_rows_f32": [_vp, _vp, _vp, _f, _vp, _ll, _i, _vp],
    "es3_rope_f32": [_vp, _ll, _ll, _vp, _i, _i, _i, _i, _vp],
    "es3_attention_f32": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp],
    "es3_scale_channels_f32": [_vp, _vp, _vp, _i, _ll, _i, _vp],
    "es3_stem_wgrad": [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp],
    "es3_bilinear_bwd": [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "es3_litemla_attn_bwd_generic": [_vp, _ll, _vp, _ll, _vp, _i, _vp, _vp, _ll, _i, _i, _i, _i, _f, _vp],
    "es3_litemla_attn_bwd": [_vp, _ll, _vp, _ll, _vp, _i, _vp, _vp, _ll, _i, _i, _i, _f, _vp],
    # input preprocessing (preprocess.cu)
    "es3_preprocess_images": [_vp, _vp, _vp, _i, _i, _i, _vp, _vp],
}

# workspace-size helpers: name -> argtypes, restype long long
SIZE_HELPERS: dict[str, list] = {
    "es3_col_reduce_ws_floats": [_ll, _i],
    "es3_wgrad_pw_ws_floats": [_ll, _i, _i],
    "es3_dwconv_wgrad_ws_floats": [_i, _i, _i, _i, _i, _i],
    "es3_dwconv_wgrad_win_ws_floats": [_i, _i, _i, _i, _i, _i],
    "es3_dwconv_wgrad_tiled_ws_floats": [_i, _i, _i, _i, _i],
    "es3_se_bwd_ws_floats": [_i, _i, _i],
    "es3_layernorm_bwd_ws_floats": [_ll, _i],
    "es3_colsum_f32_ws_floats": [_ll, _i],
    "es3_wgrad_tc_ws_floats": [_ll, _i, _i],
    "es3_litemla_attn_f32_ws_floats": [_i, _i, _i, _i],
    "es3_stem_wgrad_ws_floats": [_i, _i, _i, _i],
    "es3_litemla_bwd_ws_floats": [_i, _i, _i],
    "es3_litemla_bwd_generic_ws_floats": [_i, _i, _i, _i],
}

_lib = None


class Es3Error(RuntimeError):
    pass


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load libes3.so, building it in-tree first if it is absent (nvcc needs no GPU)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if not build_if_missing:
            raise Es3Error(f"{LIB_PATH} not built; run `python -m efficientsam3_b200.build`")
        from . import build as _build
        _build.build()
    lib = C.CDLL(str(LIB_PATH))
    lib.es3_last_error.restype = C.c_char_p
    lib.es3_last_error.argtypes = []
    lib.es3_version.restype = _i
    lib.es3_version.argtypes = []
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.restype = _i
        fn.argtypes = argtypes
    for name, argtypes in SIZE_HELPERS.items():
        fn = getattr(lib, name)
        fn.restype = _ll
        fn.argtypes = argtypes
    _lib = lib
    return lib


def last_error() -> str:
    return load().es3_last_error().decode("utf-8", "replace")


def call(name: str, *args) -> None:
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise Es3Error(f"{name} failed ({rc}): {last_error()}")


def size(name: str, *args) -> int:
    """Workspace size (in floats) from one of the *_ws_floats helpers; pure host arithmetic, no GPU needed."""
    return int(getattr(load(), name)(*args))


def call_rc(name: str, *args) -> int:
    """For entry points with a documented negative 'not applicable' return (no error raised for rc < 0)."""
    rc = getattr(load(), name)(*args)
    if rc > 0:
        raise Es3Error(f"{name} failed ({rc}): {last_error()}")
    return rc


_inited: dict[int, tuple[int, int, int]] = {}


def init(device: int = 0) -> tuple[int, int, int]:
    """Validate the device (CC 10.x required).  Returns (sm_count, cc_major, cc_minor)."""
    if device in _inited:
        return _inited[device]
    sm, ma, mi = _i(0), _i(0), _i(0)
    call("es3_init", device, C.byref(sm), C.byref(ma), C.byref(mi))
    _inited[device] = (sm.value, ma.value, mi.value)
    return _inited[device]
