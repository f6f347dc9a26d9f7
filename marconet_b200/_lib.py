"""ctypes binding of libmarconet_b200.so (the C ABI declared in include/marconet_b200.h).

The product path has NO fallback: if the shared library is missing or a symbol cannot be
resolved this module raises at import of the first operator, loudly.
"""
import ctypes
import os
from ctypes import c_longlong, POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmarconet_b200.so")

# enums (mirror include/marconet_b200.h)
ACT_NONE, ACT_RELU, ACT_LRELU02, ACT_TANH, ACT_GELU, ACT_SIGMOID, ACT_RSQRT_EPS = range(7)
PREC_FP32_SIMT, PREC_F16X3_TC, PREC_BF16X3_TC, PREC_F16X1_TC = range(4)


class ConvParams(Structure):
    _fields_ = [
        ("x", c_void_p), ("N", c_int), ("H", c_int), ("W", c_int), ("Cin", c_int), ("x_cs", c_int),
        ("w", c_void_p), ("KH", c_int), ("KW", c_int), ("stride_h", c_int), ("stride_w", c_int),
        ("pad_h", c_int), ("pad_w", c_int), ("Cout", c_int),
        ("y", c_void_p), ("y_cs", c_int),
        ("bias", c_void_p),
        ("out_scale", c_void_p), ("out_scale_stride", c_int),
        ("residual", c_void_p), ("res_cs", c_int),
        ("res_broadcast_n", c_int),
        ("act", c_int), ("act_gain", c_float),
        ("y2", c_void_p), ("y2_cs", c_int), ("y2_scale", c_void_p), ("y2_scale_stride", c_int),
        ("valid_w", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_int64),
        ("split_k", c_int),
        ("precision", c_int),
        ("w_tc_hi", c_void_p), ("w_tc_lo", c_void_p), ("w_tc_scale", c_void_p),
        ("gn_mean_rstd", c_void_p), ("gn_gamma", c_void_p), ("gn_beta", c_void_p), ("gn_swish", c_int),
        ("x_scale", c_float), ("x_absmax", c_void_p), ("range_flag", c_void_p), ("range_tag", c_int32),
        ("y2_ptrs", c_void_p), ("gn_stats_out", c_void_p),
    ]


class DemodDesc(Structure):
    _fields_ = [("wsq", c_void_p), ("s_off", c_int32), ("cin", c_int32), ("cout", c_int32), ("out_off", c_int32)]


class Window(Structure):
    _fields_ = [("line", c_int32), ("x1", c_int32), ("x2", c_int32), ("y1", c_int32)]


# name -> (restype, argtypes); every symbol include/marconet_b200.h declares
SYMBOLS = {
    "mn_last_error": (c_char_p, []),
    "mn_version": (c_int, []),
    "mn_device_is_sm100": (c_int, []),
    "mn_set_max_ctas": (c_int, [c_int]),
    "mn_conv2d_nhwc": (c_int, [POINTER(ConvParams), c_void_p]),
    "mn_conv2d_workspace_bytes": (c_int64, [POINTER(ConvParams)]),
    "mn_conv2d_tc_supported": (c_int, [POINTER(ConvParams)]),
    "mn_groupnorm_stats": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mn_groupnorm_finalize": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "mn_groupnorm_apply": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                   c_void_p, c_void_p]),
    "mn_conv_pack_weights_tc": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mn_pixelnorm": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "mn_select_text": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p]),
    "mn_set_pdl": (c_int, [c_int]),
    "mn_check_labels": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "mn_char_windows": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mn_char_segment_styles": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int,
                                       c_void_p, c_void_p]),
    "mn_demod": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "mn_demod_batched": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "mn_resample_modulate": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mn_torgb": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "mn_groupnorm_swish": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                   c_float, c_int, c_void_p, c_void_p, c_void_p]),
    "mn_adain_concat": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "mn_window_scatter": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                  c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mn_swish": (c_int, [c_void_p, c_void_p, c_longlong, c_void_p]),
    "mn_row_mean_std": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p]),
    "mn_adain_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "mn_layernorm": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p]),
    "mn_linear_small_m": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "mn_linear_small_m_ex": (c_int, [c_void_p, c_longlong, c_longlong, c_int, c_longlong, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p,
                                     c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "mn_linear_small_m_ws": (c_int, [c_void_p, c_longlong, c_longlong, c_int, c_longlong, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p,
                                     c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_longlong, c_void_p]),
    "mn_preprocess_lq_u8": (c_int, [c_void_p, c_int, c_int, c_int, c_double, c_double, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "mn_postprocess_sr_u8": (c_int, [c_void_p, c_longlong, c_longlong, c_longlong, c_longlong, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "mn_token_mix": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "mn_attention": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "mn_nchw_to_nhwc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mn_nhwc_to_nchw": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
}

_lib = None


def load():
    """Load the shared library and bind every declared symbol. Raises RuntimeError when unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"marconet_b200: CUDA library {LIB_PATH} is missing. Build it with "
            f"`python -m marconet_b200.build` (nvcc, sm_100a). There is no CPU/PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise RuntimeError(f"marconet_b200: symbol {name} missing from {LIB_PATH}") from e
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().mn_last_error().decode(errors="replace")
        raise RuntimeError(f"{what} failed (status {rc}): {msg}")
