"""ctypes binding of ``libffsr_b200.so`` (C ABI declared in ``include/ffsr_b200.h``).

Loading never falls back: a missing library raises ``FusionLibraryError`` with the build
command.  ``check(rc)`` turns a non-zero return code into ``RuntimeError`` carrying
``ffsr_last_error()``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libffsr_b200.so")

ACT_NONE, ACT_GELU, ACT_RELU, ACT_SIGMOID = 0, 1, 2, 3
EPI_PLAIN, EPI_RESIDUAL, EPI_LKAGATE, EPI_ACTGRAD = 0, 1, 2, 3
DT_F32, DT_BF16, DT_F16 = 0, 1, 2
CONV_MULTI_ISSUE = 1          # ffsr_conv_params.flags


class FusionLibraryError(RuntimeError):
    pass


class ConvParams(C.Structure):
    _fields_ = [
        ("inp", C.c_void_p),
        ("in_sN", C.c_longlong), ("in_sY", C.c_longlong), ("in_sX", C.c_longlong), ("in_sC", C.c_longlong),
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("Cin", C.c_int), ("Cout", C.c_int), ("ksize", C.c_int),
        ("w", C.c_void_p), ("bias", C.c_void_p), ("groups", C.c_int),
        ("out", C.c_void_p),
        ("out_sN", C.c_longlong), ("out_sY", C.c_longlong), ("out_sX", C.c_longlong),
        ("act", C.c_int), ("epi", C.c_int),
        ("r1", C.c_void_p), ("r1_sN", C.c_longlong), ("r1_sY", C.c_longlong), ("r1_sX", C.c_longlong),
        ("r2", C.c_void_p), ("r2_sN", C.c_longlong), ("r2_sY", C.c_longlong), ("r2_sX", C.c_longlong),
        ("sa", C.c_float), ("sa_ptr", C.c_void_p),
        ("sb", C.c_float), ("sb_ptr", C.c_void_p),
        ("ch_k", C.c_void_p), ("ch_d", C.c_void_p),
        ("in_dtype", C.c_int), ("out_dtype", C.c_int),
        ("w_dtype", C.c_int), ("r1_dtype", C.c_int), ("r2_dtype", C.c_int),
        ("out2", C.c_void_p), ("flags", C.c_int),
    ]


class WgradParams(C.Structure):
    _fields_ = [
        ("x", C.c_void_p),
        ("x_sN", C.c_longlong), ("x_sY", C.c_longlong), ("x_sX", C.c_longlong), ("x_sC", C.c_longlong),
        ("x_dtype", C.c_int),
        ("dy", C.c_void_p),
        ("dy_sN", C.c_longlong), ("dy_sY", C.c_longlong), ("dy_sX", C.c_longlong),
        ("dy_dtype", C.c_int),
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("Cin", C.c_int), ("Cout", C.c_int), ("ksize", C.c_int),
        ("dw", C.c_void_p), ("dbias", C.c_void_p),
    ]


class CacheSegment(C.Structure):
    _fields_ = [
        ("src_offset", C.c_ulonglong), ("dst", C.c_void_p),
        ("C", C.c_int), ("h", C.c_int), ("w", C.c_int),
        ("src_dtype", C.c_int), ("dst_dtype", C.c_int), ("reserved", C.c_int),
    ]


_P, _I, _L, _LL, _SZ = C.c_void_p, C.c_int, C.c_long, C.c_longlong, C.c_size_t
_F, _U64 = C.c_float, C.c_ulonglong

# name -> (restype, argtypes); the authoritative list of exported symbols (tests check it
# against include/ffsr_b200.h)
PROTOTYPES = {
    "ffsr_last_error": (C.c_char_p, []),
    "ffsr_version": (C.c_char_p, []),
    "ffsr_device_check": (_I, []),
    "ffsr_dct_bands": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ffsr_dwt_sub_size": (_I, [_I, _I, C.POINTER(_I), C.POINTER(_I)]),
    "ffsr_dwt_bands": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ffsr_dct_bands_adjoint": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ffsr_dwt_bands_adjoint": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "ffsr_fft_twiddles": (_I, [_I, _P, _P]),
    "ffsr_fft_workspace_bytes": (_SZ, [_I, _I, _I]),
    "ffsr_fft_bands": (_I, [_P, _I, _I, _I, _P, _I, _P, _P, _P, _P, _P, _SZ, _P, _P]),
    "ffsr_crossband_attention": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _I, _P, _I, _P, _P]),
    "ffsr_crossband_out": (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "ffsr_lka_depthwise": (_I, [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P]),
    "ffsr_lka_tail_weight_bytes": (_SZ, []),
    "ffsr_lka_tail_param_floats": (_SZ, []),
    "ffsr_lka_tail64": (_I, [_P, _P, _L, _P, _P, _P, _P, _P, _P]),
    "ffsr_lka_tail128_weight_bytes": (_SZ, []),
    "ffsr_lka_tail128_param_floats": (_SZ, []),
    "ffsr_lka_tail128_mod": (_I, [_P, _P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "ffsr_layernorm": (_I, [_P, _L, _I, _P, _P, _P, _I, _P]),
    "ffsr_layernorm128_bf16": (_I, [_P, _L, _P, _P, _P, _P]),
    "ffsr_lka_depthwise_in": (_I, [_P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P]),
    "ffsr_token_attention": (_I, [_P, _I, _I, _L, _I, _P, _I, _P]),
    "ffsr_align_tokens_weight_bytes": (_SZ, []),
    "ffsr_align_tokens": (_I, [_P, _P, _I, _I, _P, _P, _P, _P]),
    "ffsr_token_attn_weight_bytes": (_SZ, []),
    "ffsr_token_attn_param_floats": (_SZ, []),
    "ffsr_token_attn_chain": (_I, [_P, _I, _I, _P, _P, _P, _P]),
    "ffsr_token_ffn_weight_bytes": (_SZ, []),
    "ffsr_token_ffn_param_floats": (_SZ, []),
    "ffsr_token_ffn_chain": (_I, [_P, _L, _P, _P, _P, _P]),
    "ffsr_gate_finalize": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "ffsr_selector_blob_floats": (_SZ, []),
    "ffsr_selector_fused": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _P, _P]),
    "ffsr_conv2d": (_I, [C.POINTER(ConvParams), _P]),
    "ffsr_conv_params_size": (_SZ, []),
    "ffsr_modulate_hr": (_I, [C.POINTER(_P), _P, _P, _P, _I, _I, _I, _I, _P, _P, _LL, _I, _P]),
    "ffsr_modulate_hr_sized": (_I, [C.POINTER(_P), _P, _I, _I, _P, _P, _I, _I, _I, _I, _P, _P, _LL, _I, _P]),
    "ffsr_modulate_hr_v2": (_I, [C.POINTER(_P), _P, _I, _P, _P, _I, _I, _I, _I, _P, _P, _LL, _I, _P]),
    "ffsr_expert_downsample": (_I, [_P, _I, _I, _I, _P, _LL, _P, _LL, _I, _P]),
    "ffsr_resize_nhwc": (_I, [_P, _I, _I, _I, _I, _LL, _P, _I, _I, _LL, _I, _P]),
    "ffsr_spatial_gate": (_I, [_P, _L, _I, _P, _P, _P, _P, _P, _I, _P]),
    "ffsr_blend_hr": (_I, [_P, _LL, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _LL, _P, _LL, _P]),
    "ffsr_blur_pool": (_I, [_P, _LL, _I, _I, _I, _P, _P, _LL, _P, _LL, _P]),
    "ffsr_blur_pool_backward": (_I, [_P, _LL, _I, _I, _I, _P, _P, _LL, _P]),
    "ffsr_laplacian_sub": (_I, [_P, _LL, _P, _LL, _I, _I, _I, _P, _LL, _P, _LL, _P]),
    "ffsr_edge_attn_upsample": (_I, [_P, _I, _P, _I, _I, _I, _I, _P, _I, _P, _I, _I, _LL, _I, _P]),
    "ffsr_edge_chain_weight_bytes": (_SZ, []),
    "ffsr_edge_chain_param_floats": (_SZ, []),
    "ffsr_edge_refiner_chain": (_I, [_P, _I, _I, _I, _P, _P, _P, _I, _P, _LL, _LL, _LL, _P, _I, _P]),
    "ffsr_nchw_to_nhwc_bf16": (_I, [_P, _I, _I, _L, _P, _LL, _LL, _P]),
    "ffsr_cast_f32_to_bf16": (_I, [_P, _P, _L, _P]),
    "ffsr_final_combine": (_I, [_P, _LL, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P]),
    # ---- train-mode / backward ----
    "ffsr_conv2d_wgrad_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I, _I]),
    "ffsr_conv2d_wgrad": (_I, [C.POINTER(WgradParams), _P, _SZ, _P]),
    "ffsr_wgrad_params_size": (_SZ, []),
    "ffsr_colsum_workspace_bytes": (_SZ, [_I, _I, _I, _I]),
    "ffsr_colsum": (_I, [_P, _I, _I, _I, _I, _I, _LL, _LL, _LL, _P, _P, _SZ, _P]),
    "ffsr_act_forward": (_I, [_P, _P, _L, _I, _I, _P]),
    "ffsr_act_backward": (_I, [_P, _P, _P, _L, _I, _I, _P]),
    "ffsr_layernorm_backward_workspace_bytes": (_SZ, [_L, _I]),
    "ffsr_layernorm_backward": (_I, [_P, _P, _L, _I, _P, _P, _P, _P, _P, _SZ, _P]),
    "ffsr_bn_stats_workspace_bytes": (_SZ, [_I, _L, _I]),
    "ffsr_bn_stats": (_I, [_P, _I, _L, _I, _P, _P, _P, _SZ, _P]),
    "ffsr_bn_apply": (_I, [_P, _I, _L, _I, _P, _P, _P, _P, _P, _P]),
    "ffsr_bn_backward_workspace_bytes": (_SZ, [_I, _L, _I]),
    "ffsr_bn_backward": (_I, [_P, _P, _I, _L, _I, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "ffsr_bn_eval_backward": (_I, [_P, _P, _L, _I, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "ffsr_token_attention_train": (_I, [_P, _I, _I, _L, _I, _P, _P, _F, _U64, _P, _P]),
    "ffsr_token_attention_backward": (_I, [_P, _P, _P, _I, _I, _L, _I, _P, _P, _F, _U64, _P, _P]),
    "ffsr_dwconv_stage": (_I, [_P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "ffsr_dwconv_wgrad_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I]),
    "ffsr_dwconv_wgrad": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _SZ, _P]),
    # ---- fused losses ----
    "ffsr_loss_l1_workspace_bytes": (_SZ, [_L]),
    "ffsr_loss_l1": (_I, [_P, _P, _L, _F, _P, _P, _SZ, _P, _P]),
    "ffsr_loss_swt_workspace_bytes": (_SZ, [_I, _I, _I]),
    "ffsr_loss_swt": (_I, [_P, _P, _I, _I, _I, _F, _P, _P, _SZ, _P, _P]),
    "ffsr_loss_ssim_workspace_bytes": (_SZ, [_I, _I, _I]),
    "ffsr_loss_ssim": (_I, [_P, _P, _I, _I, _I, _F, _P, _P, _SZ, _P, _P]),
    "ffsr_loss_fft_workspace_bytes": (_SZ, [_I, _I, _I]),
    "ffsr_loss_fft": (_I, [_P, _P, _I, _I, _I, _F, _P, _P, _SZ, _P, _P]),
    # ---- bf16 / tcgen05 training path ----
    "ffsr_to_bf16_nhwc": (_I, [_P, _I, _LL, _LL, _LL, _LL, _I, _I, _I, _I, _I, _P, _P]),
    "ffsr_conv2d_wgrad_tc_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I, _I]),
    "ffsr_conv2d_wgrad_tc": (_I, [C.POINTER(WgradParams), _P, _SZ, _P]),
    "ffsr_bilinear_forward": (_I, [_P, _I, _I, _I, _I, _P, _I, _I, _I, _P]),
    "ffsr_bilinear_backward": (_I, [_P, _I, _I, _I, _I, _P, _I, _I, _I, _P]),
    "ffsr_gate_mul_forward": (_I, [_P, _P, _L, _I, _P, _I, _P]),
    "ffsr_gate_mul_backward": (_I, [_P, _P, _P, _L, _I, _P, _P, _I, _P]),
    "ffsr_axpby_forward": (_I, [_P, _P, _P, _L, _P, _P, _L, _I, _P, _I, _P]),
    "ffsr_axpby_backward_workspace_bytes": (_SZ, [_L, _I]),
    "ffsr_axpby_backward": (_I, [_P, _P, _P, _L, _P, _P, _L, _I, _P, _P, _P, _P, _SZ, _I, _P]),
    "ffsr_fft_lowpass_workspace_bytes": (_SZ, [_I, _I, _I]),
    "ffsr_fft_lowpass": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _SZ, _P, _P]),
    "ffsr_fft_lowpass_backward": (_I, [_P, _P, _I, _I, _I, _P, _P, _P, _SZ, _P, _P]),
    # ---- DRCT-L window attention (N1: first kernel of the expert forward) ----
    "ffsr_window_attention": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _I, _P]),
    "ffsr_window_attention_pitched": (_I, [_P, _L, _I, _I, _I, _I, _I, _I, _I, _P, _P, _L, _P]),
    "ffsr_window_attention_head_pad": (_I, [_I]),
    "ffsr_window_attention_headpadded": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _L, _P]),
    "ffsr_layernorm_strided": (_I, [_P, _L, _I, _L, _P, _P, _P, _L, _I, _I, _P]),
    "ffsr_leaky_relu": (_I, [_P, _L, _I, _L, _F, _I, _P]),
    "ffsr_pixel_shuffle2": (_I, [_P, _I, _I, _I, _I, _P, _I, _P]),
    "ffsr_rgb_shift_in": (_I, [_P, _I, _I, _I, _P, _F, _P, _I, _I, _P]),
    "ffsr_rgb_shift_out": (_I, [_P, _I, _I, _I, _I, _P, _F, _P, _I, _P]),
    # ---- cache-shard collate ----
    "ffsr_cache_unpack": (_I, [_P, _SZ, _I, _P, _I, _P, _I, _P]),
    "ffsr_cache_segment_size": (_I, []),
    # ---- fused optimizer ----
    "ffsr_sumsq_workspace_bytes": (_SZ, [_L]),
    "ffsr_sumsq": (_I, [_P, _L, _P, _P, _SZ, _P]),
    "ffsr_adamw_ema_step": (_I, [_P, _P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _I, _P, _P, _P, _F, _F, _F, _P]),
    "ffsr_sum_slots_ordered": (_I, [_P, _I, _L, _L, _P, _P]),
}

_lib = None


def load():
    """dlopen the kernel library (once) and attach prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FusionLibraryError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C image-super-resolution_b200/csrc`). There is no CPU / PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError here == symbol not exported
        fn.restype = res
        fn.argtypes = args
    if lib.ffsr_conv_params_size() != C.sizeof(ConvParams):
        raise FusionLibraryError("ffsr_conv_params layout mismatch between _cabi.py and the built library; rebuild")
    if lib.ffsr_wgrad_params_size() != C.sizeof(WgradParams):
        raise FusionLibraryError("ffsr_wgrad_params layout mismatch between _cabi.py and the built library; rebuild")
    if lib.ffsr_cache_segment_size() != C.sizeof(CacheSegment):
        raise FusionLibraryError("ffsr_cache_segment layout mismatch between _cabi.py and the built library; rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().ffsr_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libffsr_b200 {what} failed (code {rc}): {msg}")
