"""ctypes binding of ``libe2fgvi_b200.so`` (declared in ``include/e2fgvi_b200.h``).

There is NO fallback: if the library is missing or a call fails the caller gets an exception.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libe2fgvi_b200.so")

_c = ctypes
_vp, _fp, _i, _f = _c.c_void_p, _c.c_void_p, _c.c_int, _c.c_float

# name -> (restype, argtypes); kept in the same order as the header so tests can diff them.
SIGNATURES = {
    "e2f_version": (_c.c_char_p, []),
    "e2f_last_error": (_c.c_char_p, []),
    "e2f_flow_warp": (_i, [_vp, _fp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "e2f_flow_warp_nchw": (_i, [_fp, _fp, _fp, _i, _i, _i, _i, _i, _vp]),
    "e2f_dcn_pack_weight": (_i, [_fp, _vp, _i, _i, _i, _vp]),
    "e2f_modulated_deform_conv2d": (_i, [_vp, _fp, _fp, _vp, _fp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "e2f_dcn_pack_input": (_i, [_fp, _fp, _vp, _i, _i, _i, _i, _i, _vp]),
    "e2f_deform_align_fused": (_i, [_vp, _fp, _fp, _fp, _vp, _fp, _vp, _i, _i, _i, _i, _i, _i, _f, _i, _i, _vp]),
    "e2f_deform_align_fused_split": (_i, [_vp, _fp, _fp, _fp, _vp, _fp, _fp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _i, _vp]),
    "e2f_focal_window_attention": (_i, [_vp, _vp, _vp] + [_i] * 13 + [_f, _i, _vp]),
    "e2f_t2t_unfold": (_i, [_fp, _fp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "e2f_upsample2x_split": (_i, [_fp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "e2f_layernorm_split": (_i, [_fp, _fp, _fp, _fp, _vp, _vp, _c.c_int64, _i, _f, _vp]),
    "e2f_t2t_fold_nhwc": (_i, [_fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "e2f_t2t_unfold_nhwc": (_i, [_fp, _fp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "e2f_t2t_fold_unfold": (_i, [_fp, _fp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "e2f_t2t_fold": (_i, [_fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "e2f_split_bf16": (_i, [_fp, _vp, _vp, _c.c_int64, _vp]),
    "e2f_linear_bf16x3": (_i, [_vp, _vp, _vp, _vp, _fp, _fp, _vp, _i, _i, _i, _i, _i, _vp]),
    "e2f_conv3x3_bf16x3": (_i, [_i, _c.POINTER(_vp), _c.POINTER(_vp), _c.POINTER(_i), _vp, _vp, _fp, _fp, _fp, _vp, _vp,
                                _i, _i, _i, _i, _i, _f, _vp]),
    "e2f_conv2d_bf16x3": (_i, [_i, _c.POINTER(_vp), _c.POINTER(_vp), _c.POINTER(_i), _vp, _vp, _fp, _fp, _fp, _vp, _vp,
                               _i, _i, _i, _i, _i, _f, _i, _i, _i, _vp]),
    "e2f_conv2d_rows_bf16x3": (_i, [_i, _c.POINTER(_vp), _c.POINTER(_vp), _c.POINTER(_i), _i, _vp, _vp, _fp, _fp, _fp, _vp,
                                    _vp, _i, _i, _i, _i, _i, _i, _f, _i, _i, _i, _vp]),
    "e2f_conv3x3_tanh_nchw": (_i, [_vp, _vp, _i, _vp, _vp, _fp, _fp, _i, _i, _i, _i, _vp]),
    "e2f_conv_kxn_bf16x3": (_i, [_i, _c.POINTER(_vp), _c.POINTER(_vp), _c.POINTER(_i), _vp, _vp, _fp, _fp, _fp, _vp, _vp, _i, _i,
                                 _i, _i, _i, _i, _i, _f, _i, _vp]),
    "e2f_conv_gather_bf16x3": (_i, [_i, _c.POINTER(_vp), _c.POINTER(_vp), _c.POINTER(_i), _vp, _vp, _fp, _fp, _fp, _fp,
                                    _vp, _vp, _i, _i, _i, _i, _f, _i, _i, _i, _i, _i, _i, _c.POINTER(_c.c_int8),
                                    _c.POINTER(_c.c_int8), _i, _c.POINTER(_c.c_uint8), _c.POINTER(_c.c_uint8),
                                    _c.POINTER(_c.c_uint8), _i, _i, _i, _c.POINTER(_c.c_int64), _c.c_int64, _vp]),
    "e2f_conv_rows_tail": (_i, [_i, _i]),
    "e2f_conv_rows_pitch": (_i, [_i, _i, _i]),
    "e2f_pack_rows_bf16": (_i, [_fp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "e2f_layernorm_pool_split": (_i, [_fp, _fp, _fp, _fp, _fp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "e2f_window_pool": (_i, [_vp, _vp, _fp, _fp, _fp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "e2f_prop_prologue": (_i, [_fp, _fp, _fp, _c.c_int64, _fp, _c.c_int64, _vp, _vp, _vp, _vp, _fp, _fp, _vp, _vp, _vp,
                               _i, _i, _i, _i, _vp]),
    "e2f_spynet_pyramid": (_i, [_fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _fp, _fp, _vp]),
    "e2f_spynet_level_input": (_i, [_fp, _fp, _vp, _vp, _fp, _i, _i, _i, _i, _i, _vp]),
    "e2f_spynet_final": (_i, [_fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _vp]),
    "e2f_peer_alloc": (_i, [_c.c_size_t, _c.POINTER(_c.c_void_p), _c.c_char_p]),
    "e2f_peer_open": (_i, [_c.c_char_p, _c.POINTER(_c.c_void_p)]),
    "e2f_peer_close": (_i, [_vp]),
    "e2f_peer_free": (_i, [_vp]),
    "e2f_peer_copy": (_i, [_vp, _vp, _c.c_size_t, _vp]),
    "e2f_peer_signal": (_i, [_vp, _c.c_uint, _vp]),
    "e2f_peer_wait": (_i, [_vp, _c.c_uint, _vp]),
    "e2f_video_prepare_clip": (_i, [_vp, _vp, _vp, _fp, _i, _i, _i, _i, _i, _vp]),
    "e2f_video_compose": (_i, [_fp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "e2f_video_blend": (_i, [_vp, _vp, _vp, _fp, _i, _c.c_int64, _vp]),
    "e2f_video_finalize": (_i, [_fp, _vp, _c.c_int64, _vp]),
    "e2f_psnr_ssim_workspace_bytes": (_c.c_size_t, [_i, _i, _i, _i]),
    "e2f_psnr_ssim": (_i, [_vp, _fp, _vp, _vp, _i, _i, _i, _i, _c.c_double, _vp, _vp]),
    "e2f_launch_count": (_c.c_int64, []),
}

_lib = None


class ExtensionMissing(RuntimeError):
    pass


def load():
    """Load (once) and return the ctypes library. Raises ExtensionMissing if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ExtensionMissing(
            f"{LIB_PATH} not found: build it with `python -m e2fgvi_b200.build` "
            "(there is no CPU or PyTorch fallback for the hot-path kernels)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, what):
    if status == 0:
        return
    msg = load().e2f_last_error().decode("utf-8", "replace")
    if status == -1:
        raise ValueError(f"{what}: {msg}")
    raise RuntimeError(f"{what} failed (status {status}): {msg}")
