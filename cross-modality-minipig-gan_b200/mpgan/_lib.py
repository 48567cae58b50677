"""ctypes binding of libmpgan_sm100.so (the C ABI declared in include/mpgan.h).

No CPU fallback: every compute wrapper raises if the library is missing or the process has no sm_100 device.
"""
import ctypes
import os
import re
from ctypes import (c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint32, c_void_p, POINTER,
                    Structure)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "libmpgan_sm100.so")
HEADER_PATH = os.path.join(os.path.dirname(os.path.dirname(_HERE)), "include", "mpgan.h")

F32, BF16 = 0, 1
ACT_NONE, ACT_PRELU, ACT_LEAKY, ACT_TANH = 0, 1, 2, 3


class ConvGeom(Structure):
    _fields_ = [("rank", c_int32), ("n", c_int32), ("xs", c_int32 * 3), ("ys", c_int32 * 3), ("cx", c_int32),
                ("cy", c_int32), ("k", c_int32 * 3), ("stride", c_int32 * 3), ("pad", c_int32 * 3)]


_G = POINTER(ConvGeom)
_P = c_void_p
_SIGS = {
    "mpgan_version": (c_int, []),
    "mpgan_last_error": (c_char_p, []),
    "mpgan_device_ok": (c_int, []),
    "mpgan_conv_fprop": (c_int, [_G, c_int, _P, c_int64, _P, _P, _P, c_int64, _P]),
    "mpgan_conv_bprop": (c_int, [_G, c_int, _P, c_int64, _P, _P, _P, c_int64, _P]),
    "mpgan_conv_wgrad": (c_int, [_G, c_int, _P, c_int64, _P, c_int64, _P, _P]),
    "mpgan_c1_supported": (c_int, [_G, c_int]),
    "mpgan_c1_conv_fprop": (c_int, [_G, c_int, _P, c_int64, _P, _P, _P, c_int64, _P, _P]),
    "mpgan_c1_conv_act": (c_int, [_G, c_int, _P, c_int64, _P, _P, _P, _P, c_int64, _P]),
    "mpgan_c1_conv_bprop": (c_int, [_G, c_int, _P, c_int64, _P, _P, _P, c_int64, _P, _P]),
    "mpgan_c1_conv_wgrad": (c_int, [_G, c_int, _P, c_int64, _P, c_int64, _P, _P]),
    "mpgan_tc_supported": (c_int, [_G, c_int]),
    "mpgan_tc_conv_fprop": (c_int, [_G, _P, c_int64, _P, _P, _P, c_int64, _P, _P]),
    "mpgan_tc_conv_bprop": (c_int, [_G, _P, c_int64, _P, _P, _P, c_int64, _P, _P]),
    "mpgan_tc_conv_act": (c_int, [_G, c_int, _P, c_int64, _P, _P, _P, _P, c_int64, _P, c_int64, _P]),
    "mpgan_tc_convt_to1": (c_int, [_G, _P, c_int64, _P, _P, _P, _P, _P]),
    "mpgan_tc_conv_bprop_c1out": (c_int, [_G, _P, c_int64, _P, _P, c_int64, _P, c_int64, _P]),
    "mpgan_tc_conv_bprop_res": (c_int, [_G, _P, c_int64, _P, _P, _P, c_int64, _P, c_int64, _P, _P]),
    "mpgan_tc_conv_wgrad_workspace": (c_size_t, [_G]),
    "mpgan_tc_conv_wgrad": (c_int, [_G, _P, c_int64, _P, c_int64, _P, _P, c_size_t, _P]),
    "mpgan_bn_stats": (c_int, [c_int, _P, c_int64, c_int64, c_int32, _P, _P]),
    "mpgan_bn_finalize": (c_int, [_P, c_int64, c_int32, _P, _P, c_float, c_float, c_int, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mpgan_bn_act_apply": (c_int, [c_int, _P, c_int64, c_int64, c_int32, _P, _P, c_int, _P, c_float, _P, c_int64, _P,
                                   c_int64, _P]),
    "mpgan_bn_train_apply": (c_int, [c_int, _P, c_int64, c_int64, c_int32, _P, _P, _P, c_float, c_float, _P, _P, _P,
                                     _P, _P, _P, _P, c_int, _P, c_float, _P, c_int64, _P, c_int64, _P]),
    "mpgan_bn_act_bwd_reduce": (c_int, [c_int, _P, c_int64, _P, c_int64, c_int64, c_int32, _P, _P, _P, _P, c_int, _P,
                                        c_float, _P, _P]),
    "mpgan_bn_act_bwd_apply": (c_int, [c_int, _P, c_int64, _P, c_int64, c_int64, c_int32, _P, _P, _P, _P, c_int, _P,
                                       c_float, _P, _P, _P, _P, _P, _P, c_int64, _P]),
    "mpgan_add_copy": (c_int, [c_int, _P, c_int64, _P, c_int64, c_int, _P, c_int64, c_int64, c_int32, _P]),
    "mpgan_tanh_fwd": (c_int, [c_int, _P, c_int, _P, c_int64, _P]),
    "mpgan_tanh_bwd": (c_int, [c_int, _P, _P, _P, c_int64, _P]),
    "mpgan_colsum": (c_int, [c_int, _P, c_int64, c_int64, c_int32, _P, _P]),
    "mpgan_linear_fwd": (c_int, [c_int, _P, _P, _P, _P, c_int32, c_int64, c_int32, _P]),
    "mpgan_linear_bwd": (c_int, [c_int, _P, _P, _P, _P, _P, _P, c_int32, c_int64, c_int32, _P]),
    "mpgan_permute_flatten": (c_int, [c_int, _P, c_int, _P, c_int32, c_int32, c_int64, c_int, c_int, _P]),
    "mpgan_sigmoid_fwd": (c_int, [_P, _P, c_int32, _P]),
    "mpgan_sigmoid_bwd": (c_int, [_P, _P, _P, c_int32, _P]),
    "mpgan_bce_fwd": (c_int, [_P, _P, c_float, _P, c_int32, _P]),
    "mpgan_bce_bwd": (c_int, [_P, _P, c_float, _P, _P, c_int32, _P]),
    "mpgan_l1_fwd": (c_int, [c_int, _P, _P, c_int64, c_float, _P, _P]),
    "mpgan_l1_bwd": (c_int, [c_int, _P, _P, c_int64, c_float, _P, _P, c_int, _P]),
    "mpgan_l1_fwd_bwd": (c_int, [c_int, _P, _P, c_int64, c_float, _P, _P, _P, _P, c_int, _P]),
    "mpgan_adam_step": (c_int, [_P, _P, _P, _P, c_int64, c_float, c_float, c_float, c_float, _P, _P, _P]),
    "mpgan_cast": (c_int, [c_int, _P, c_int, _P, c_int64, _P]),
    "mpgan_weight_transpose": (c_int, [c_int, _P, c_int, _P, c_int32, c_int32, c_int32, _P]),
    "mpgan_weight_transpose_batch": (c_int, [_P, c_int32, c_int32, _P]),
    "mpgan_patch_gather": (c_int, [c_int, _P, c_int32, c_int32, _P, c_int32, _P, c_int32, c_int32, _P, _P]),
    "mpgan_patch_scatter_add": (c_int, [c_int, _P, c_int32, c_int32, _P, c_int32, _P, c_int32, c_int32, _P, _P]),
    "mpgan_c1_tail_fwd": (c_int, [_P, c_int32, c_int32, c_int32, _P, _P, _P, c_float, c_float, _P, _P, _P, _P, _P, _P,
                                  _P, _P, _P, _P, _P, _P, _P]),
    "mpgan_c1_tail_bwd_reduce": (c_int, [_P, _P, c_int32, c_int32, c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mpgan_im2col_c1": (c_int, [_P, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P]),
    "mpgan_fold_dw16": (c_int, [_P, c_int32, _P, _P]),
    "mpgan_im2col_c1_vol": (c_int, [_P, c_int32, POINTER(c_int32), POINTER(c_int32), c_int32, c_int32, _P, _P]),
    "mpgan_col2im_c1_vol": (c_int, [_P, c_int32, POINTER(c_int32), POINTER(c_int32), c_int32, c_int32, _P, _P, _P, _P]),
    "mpgan_fold_dw32": (c_int, [_P, c_int32, _P, _P]),
    "mpgan_stencil27": (c_int, [c_int, c_int, _P, c_int32, c_int32, c_int32, c_int32, _P, _P, _P, _P, _P]),
    "mpgan_stencil27_wgrad": (c_int, [c_int, _P, _P, c_int32, c_int32, c_int32, c_int32, _P, _P, _P]),
    "mpgan_order_stats_workspace": (c_size_t, [c_int32]),
    "mpgan_order_stats": (c_int, [_P, c_int64, _P, c_int32, _P, _P, c_size_t, _P]),
    "mpgan_minmax": (c_int, [_P, c_int64, _P, c_int32, _P, _P, c_size_t, _P]),
    "mpgan_rescale_intensity": (c_int, [_P, c_int64, c_float, c_float, c_float, c_float, c_int, c_float, c_float, c_int,
                                        c_int, _P, _P]),
    "mpgan_err_sums": (c_int, [_P, _P, c_int64, _P, _P]),
    "mpgan_ssim_sums": (c_int, [_P, _P, c_int32, c_int32, c_int32, c_int32, c_int32, POINTER(c_double), c_int32, c_double,
                                c_double, c_double, _P, _P]),
    "mpgan_mutual_info_workspace": (c_size_t, [c_int32]),
    "mpgan_mutual_info": (c_int, [_P, _P, c_int32, c_int64, c_int32, _P, _P, _P, _P, c_size_t, _P]),
    "mpgan_err_sums_masked": (c_int, [_P, _P, _P, c_int64, _P, _P]),
    "mpgan_ssim_sums_masked": (c_int, [_P, _P, _P, c_int32, c_int32, c_int32, c_int32, c_int32, POINTER(c_double),
                                       c_int32, c_double, c_double, c_double, _P, _P, _P]),
    "mpgan_mutual_info_masked": (c_int, [_P, _P, _P, c_int32, c_int64, c_int32, _P, _P, _P, _P, c_size_t, _P]),
    "mpgan_otsu_threshold_workspace": (c_size_t, [c_int32, c_int32]),
    "mpgan_otsu_threshold": (c_int, [_P, c_int32, c_int64, c_int32, _P, _P, c_size_t, _P]),
    "mpgan_threshold_mask": (c_int, [_P, _P, c_int32, c_int64, _P, _P]),
    "mpgan_morphology_workspace": (c_size_t, [c_int32, c_int32, c_int32, c_int32]),
    "mpgan_label": (c_int, [_P, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P, _P, c_size_t, _P]),
    "mpgan_largest_component": (c_int, [_P, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P, c_size_t, _P]),
    "mpgan_fill_holes": (c_int, [_P, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P, c_size_t, _P]),
    "mpgan_binary_morphology": (c_int, [_P, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, _P,
                                        _P, c_size_t, _P]),
    "mpgan_distance_transform_workspace": (c_size_t, [c_int32, c_int32, c_int32, c_int32]),
    "mpgan_distance_transform": (c_int, [_P, c_int32, c_int32, c_int32, c_int32, c_int32, c_double, c_double, c_double,
                                         _P, _P, c_size_t, _P]),
    "mpgan_mask_agreement_workspace": (c_size_t, [c_int32, c_int32, c_int32, c_int32]),
    "mpgan_mask_agreement": (c_int, [_P, _P, c_int32, c_int32, c_int32, c_int32, c_int32, c_double, c_double, c_double,
                                     c_int32, c_double, _P, _P, c_size_t, _P]),
    "mpgan_window_gather":(c_int, [_P, c_int32, c_int32, _P, _P, c_int64, c_int64, c_int64, c_float, _P, _P]),
    "mpgan_window_blend": (c_int, [_P, c_int32, c_int32, _P, _P, c_int64, _P, _P]),
    "mpgan_resample_linear": (c_int, [_P, c_int64, c_int32, POINTER(c_int32), POINTER(c_int32), POINTER(c_double),
                                      c_float, _P, _P]),
    "mpgan_resample_nearest": (c_int, [_P, c_int32, c_int64, c_int32, POINTER(c_int32), POINTER(c_int32),
                                       POINTER(c_double), c_uint32, _P, _P]),
    "mpgan_bspline_coefficients": (c_int, [_P, c_int64, c_int32, POINTER(c_int32), _P, _P]),
    "mpgan_resample_bspline": (c_int, [_P, c_int64, c_int32, POINTER(c_int32), POINTER(c_int32), POINTER(c_double),
                                       c_float, _P, _P]),
    "mpgan_resample_linear_maps": (c_int, [_P, c_int64, c_int32, POINTER(c_int32), POINTER(c_int32), _P, c_float, _P,
                                           _P]),
    "mpgan_resample_nearest_maps": (c_int, [_P, c_int32, c_int64, c_int32, POINTER(c_int32), POINTER(c_int32), _P,
                                            c_uint32, _P, _P]),
    "mpgan_resample_bspline_maps": (c_int, [_P, c_int64, c_int32, POINTER(c_int32), POINTER(c_int32), _P, c_float, _P,
                                            _P]),
    "mpgan_gaussian_filter_workspace": (c_size_t, [c_int64, POINTER(c_int32)]),
    "mpgan_gaussian_filter": (c_int, [_P, c_int64, c_int32, POINTER(c_int32), POINTER(c_int32), POINTER(c_double), _P,
                                      _P, c_size_t, _P]),
    "mpgan_rigid_maps": (c_int, [_P, c_int64, c_int32, POINTER(c_double), POINTER(c_double), _P, _P]),
    "mpgan_rigid_level": (c_int, [_P, _P, c_int64, c_int32, POINTER(c_double), POINTER(c_double), _P,
                                  POINTER(c_double), c_int32, c_double, _P]),
    "mpgan_rigid_step": (c_int, [_P, _P, c_int64, c_int32, POINTER(c_double), POINTER(c_double), c_double, c_int32,
                                 _P]),
    "mpgan_mattes_workspace": (c_size_t, [c_int64, POINTER(c_int32), POINTER(c_int32), c_int32]),
    "mpgan_mattes_prepare": (c_int, [_P, _P, _P, c_int64, c_int32, POINTER(c_int32), POINTER(c_int32), c_int32, c_int32,
                                     POINTER(c_double), c_double, _P, _P, _P, c_size_t, _P]),
    "mpgan_mattes_evaluate": (c_int, [_P, _P, _P, c_int64, c_int32, POINTER(c_int32), POINTER(c_int32), c_int32,
                                      c_int32, c_int32, c_int32, _P, _P, _P, _P, _P, c_size_t, _P]),
}

_lib = None


def header_symbols():
    """Every function name declared in include/mpgan.h."""
    text = open(HEADER_PATH).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mpgan_[a-z0-9_]+)\s*\(", text)))


def load():
    """Load the shared library (works without a GPU; compute calls then fail with MPGAN_ERR_CUDA)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)")
        import torch  # noqa: F401  (loads libcudart.so.12 with the right search path first)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def last_error():
    return load().mpgan_last_error().decode()


ABI_CALLS = 0  # compute entry points invoked by this process (each launches >= 1 kernel of ours)


def check(rc, what):
    global ABI_CALLS
    ABI_CALLS += 1
    if rc != 0:
        raise RuntimeError(f"{what} failed (rc={rc}): {last_error()}")


def require_device():
    lib = load()
    if not lib.mpgan_device_ok():
        raise RuntimeError("libmpgan_sm100 needs a CUDA device of compute capability 10.x (B200); no CPU fallback exists")
    return lib
