"""ctypes binding of libfemasr_b200.so (the C ABI declared in include/femasr_b200.h).

There is no CPU fallback: loading fails loudly if the library has not been built, and every
compute entry point returns an error without an sm_100 device.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FEMASR_LIB") or os.path.join(_HERE, "libfemasr_b200.so")

PRO_NONE, PRO_GN_SILU, PRO_LN, PRO_GN_SILU_FAST = 0, 1, 2, 3
ABI_VERSION = 5          # femasr_abi_version() of the library this binding was written against (include/femasr_b200.h)
ACT_NONE, ACT_GELU = 0, 1
TAP_STAGES = ("in_conv", "down", "swin", "up1", "up2", "z", "zq", "after_quant", "dec0", "dec1", "dec2")

c_float_p = C.c_void_p     # raw device/host addresses travel as integers
c_i64_p = C.c_void_p


class FemasrError(RuntimeError):
    pass


_I, _V, _Z, _D, _F = C.c_int, C.c_void_p, C.c_size_t, C.c_double, C.c_float


class NetConfig(C.Structure):
    _fields_ = [("scale_factor", C.c_int), ("n_e", C.c_int), ("e_dim", C.c_int), ("in_channel", C.c_int),
                ("use_quantize", C.c_int), ("use_residual", C.c_int), ("gemm_path", C.c_int),
                ("n_codebooks", C.c_int), ("cb_scale", C.c_int * 3), ("cb_n_e", C.c_int * 3), ("cb_e_dim", C.c_int * 3)]


class IgemmArgs(C.Structure):
    _fields_ = [("x", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p), ("res1", C.c_void_p),
                ("res2", C.c_void_p), ("y", C.c_void_p), ("pro_a", C.c_void_p), ("pro_b", C.c_void_p),
                ("gamma", C.c_void_p), ("beta", C.c_void_p),
                ("B", C.c_int), ("Hin", C.c_int), ("Win", C.c_int), ("Cin", C.c_int), ("Cout", C.c_int),
                ("ksize", C.c_int), ("stride", C.c_int), ("upsample", C.c_int), ("prologue", C.c_int),
                ("act", C.c_int)]


class TcArgs(C.Structure):
    _fields_ = [("a_hi", C.c_void_p), ("a_lo", C.c_void_p), ("w_blob", C.c_void_p), ("bias", C.c_void_p),
                ("res1", C.c_void_p), ("res2", C.c_void_p), ("y", C.c_void_p),
                ("B", C.c_int), ("H", C.c_int), ("W", C.c_int), ("Cin", C.c_int), ("Cout", C.c_int),
                ("ksize", C.c_int), ("act", C.c_int), ("out_hi", C.c_void_p), ("out_lo", C.c_void_p),
                ("stride", C.c_int), ("kb_begin", C.c_int), ("kb_count", C.c_int),
                ("slice_kb", C.c_int), ("pair", C.c_int), ("strip", C.c_int), ("gn_partial", C.c_void_p),
                ("upsample", C.c_int), ("f8", C.c_int)]


# name -> (restype, argtypes); must list every symbol include/femasr_b200.h declares
# (tests/test_abi.py checks the two against each other).
SIGNATURES = {
    "femasr_last_error": (C.c_char_p, []),
    "femasr_abi_version": (_I, []),
    "femasr_device_cc": (_I, []),
    "femasr_net_create": (_I, [C.POINTER(NetConfig), C.POINTER(_V)]),
    "femasr_net_destroy": (None, [_V]),
    "femasr_net_set_param": (_I, [_V, C.c_char_p, _V, _Z, _I, _V]),
    "femasr_net_params_complete": (_I, [_V]),
    "femasr_net_workspace_bytes": (_I, [_V, _I, _I, _I, C.POINTER(_Z)]),
    "femasr_net_forward": (_I, [_V, _V, _V, _V, _V, _I, _I, _I, _V, _Z, _V]),
    "femasr_net_forward_gt": (_I, [_V, _V, _V, _V, _V, _V, _I, _I, _I, _V, _Z, _V]),
    "femasr_net_decode_indices": (_I, [_V, _V, _V, _I, _I, _I, _V, _Z, _V]),
    "femasr_net_decode_workspace_bytes": (_I, [_V, _I, _I, _I, C.POINTER(_Z)]),
    "femasr_net_set_tap": (_I, [_V, C.c_char_p, _V, _Z]),
    "femasr_net_last_launch_count": (_I, [_V]),
    "femasr_net_set_profile": (_I, [_V, _I]),
    "femasr_net_profile_json": (C.c_char_p, [_V]),
    "femasr_net_flops": (_D, [_V, _I, _I, _I]),
    "femasr_flip_pad": (_I, [_V, _V, _I, _I, _I, _I, _I, _I, _V]),
    "femasr_u8_to_input": (_I, [_V, _V, _I, _I, _I, _I, _I, _V]),
    "femasr_output_to_u8": (_I, [_V, _V, _I, _I, _I, _I, _I, _V]),
    "femasr_copy_window": (_I, [_V, _V] + [_I] * 12 + [_V]),
    "femasr_pack_weight": (_I, [_V, _V, _I, _I, _I, _I, _V]),
    "femasr_igemm_simt": (_I, [C.POINTER(IgemmArgs), _V]),
    "femasr_tc_weight_bytes": (_Z, [_I, _I, _I, _I]),
    "femasr_tc_pack_weight": (_I, [_V, _V, _I, _I, _I, _I, _V]),
    "femasr_tc_pack_weight_up2": (_I, [_V, _V, _I, _I, _V]),
    "femasr_tc_prepare": (_I, [_V, _V, _V, _I, _V, _V, _V, _V, _I, _I, _I, _I, _I, _F, _V]),
    "femasr_tc_prepare_f8": (_I, [_V, _V, _V, _I, _V, _V, _I, _I, _I, _I, _V]),
    "femasr_tc_pack_weight_f8": (_I, [_V, _V, _I, _I, _I, _I, _V]),
    "femasr_tc_pack_weight_up2_f8": (_I, [_V, _V, _I, _I, _V]),
    "femasr_tc_igemm": (_I, [C.POINTER(TcArgs), _V]),
    "femasr_tc_gn_partial_rows": (_I, [C.POINTER(TcArgs)]),
    "femasr_gn_finalize_rows": (_I, [_V, _V, _V, _V, _V, _I, _I, _I, _I, _F, _V]),
    "femasr_gn_scratch_floats": (_Z, [_I, _I, _I]),
    "femasr_gn_stats": (_I, [_V, _V, _V, _V, _V, _V, _I, _I, _I, _F, _V]),
    "femasr_ln_stats": (_I, [_V, _V, _V, _I, _I, _F, _V]),
    "femasr_window_attention": (_I, [_V, _V, _V, _I, _I, _I, _I, _I, _I, _V]),
    "femasr_window_attention_mma": (_I, [_V, _V, _V, _V, _V, _I, _I, _I, _I, _I, _I, _V]),
    "femasr_expand_rel_bias": (_I, [_V, _V, _I, _V]),
    "femasr_expand_rel_bias_mma": (_I, [_V, _V, _I, _V]),
    "femasr_row_sumsq": (_I, [_V, _V, _I, _I, _V]),
    "femasr_vq_select": (_I, [_V, _V, _V, _V, _V, _V, _V, _I, _I, _I, _I, _V]),
    "femasr_vq_match_tc": (_I, [_V, _V, _V, _V, _V, _V, _I, _I, _I, _V]),
    "femasr_vq_finish": (_I, [_V, _V, _V, _V, _V, _V, _V, _V, _V, _I, _I, _I, _V]),
    "femasr_packed_code_bytes": (_Z, [_Z, _I]),
    "femasr_pack_codes": (_I, [_V, _V, _Z, _I, _V, _V]),
    "femasr_unpack_codes": (_I, [_V, _V, _Z, _I, _V]),
    "femasr_sum_scaled": (_I, [_V, _V, _Z, _D, _V]),
    "femasr_sum_scaled_add": (_I, [_V, _V, _Z, _D, _V]),
    "femasr_concat_channels": (_I, [_V, _I, _V, _I, _I, _I, _V, _I, _I, _I, _V]),
    "femasr_vq_gt_rows": (_I, [_V, _V, _V, _V, _V, _I, _I, _I, _V]),
    "femasr_gram_diff_tiles": (_I, [_I]),
    "femasr_gram_diff": (_I, [_V, _V, _V, _I, _I, _I, _V]),
    "femasr_codebook_gather": (_I, [_V, _V, _V, _I, _I, _I, _V]),
    "femasr_in_conv4x4": (_I, [_V, _V, _V, _V, _I, _I, _I, _I, _I, _V]),
    "femasr_in_conv_im2col": (_I, [_V, _V, _V, _I, _I, _I, _I, _V]),
    "femasr_in_conv_pad_weight": (_I, [_V, _V, _I, _V]),
    "femasr_out_conv3x3": (_I, [_V, _V, _V, _V, _I, _I, _I, _I, _V]),
    "femasr_out_conv3x3_mma": (_I, [_V, _V, _V, _V, _I, _I, _I, _I, _V]),
    "femasr_nchw_to_nhwc": (_I, [_V, _V, _I, _I, _I, _I, _V]),
    "femasr_nhwc_to_nchw": (_I, [_V, _V, _I, _I, _I, _I, _V]),
}

_lib = None


def load() -> C.CDLL:
    """Load the CUDA library (raises FemasrError if it was never built: no fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FemasrError(
            f"{LIB_PATH} not found. Build it with `python -m femasr_b200.build` "
            "(needs nvcc); femasr_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != 0:
        msg = load().femasr_last_error()
        raise FemasrError(f"femasr_b200 error {status}: {msg.decode() if msg else '?'}")


def require_device() -> int:
    """Compute capability of the current device; raises unless it is sm_100."""
    cc = load().femasr_device_cc()
    if cc < 0:
        check(cc)
    if cc // 10 != 10:
        raise FemasrError(f"femasr_b200 kernels are built for sm_100a only; current device is sm_{cc}")
    return cc
