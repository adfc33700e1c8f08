"""ctypes binding of libbcad.so (the C-ABI declared in include/bcad.h).

Fails loudly when the library is missing: there is no CPU or PyTorch fallback in this package.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libbcad.so")

MAX_CONV = 8
MAX_DENSE = 8

OK, ERR_INVALID, ERR_CUDA, ERR_STATE, ERR_NOMEM = 0, -1, -2, -3, -4
FLATTEN = {"hwc": 0, "chw": 1}
TIES = {"dup": 0, "all": 0, "first": 1}
HEAD = {"softmax": 0, "logits": 1}
PRECISION = {"fp32": 0, "fp16": 1, "fp16x3": 2}
GRAD_MODE = {"logit": 0, "softmax_ce": 1}
TARGET = {"conv": 0, "conv_act": 0, "conv_preact": 1}
T_CONV_OUT, T_POOL_OUT, T_DENSE_Z, T_ALPHA, T_CAM_LOWRES = 0, 1, 2, 3, 4
MAX_EXPLAIN_CLASSES = 8


class Config(C.Structure):
    _fields_ = [
        ("in_h", C.c_int32), ("in_w", C.c_int32), ("in_c", C.c_int32),
        ("num_classes", C.c_int32),
        ("n_conv", C.c_int32),
        ("conv_filters", C.c_int32 * MAX_CONV),
        ("conv_ksize", C.c_int32 * MAX_CONV),
        ("n_hidden", C.c_int32),
        ("hidden_units", C.c_int32 * MAX_DENSE),
        ("alpha_conv", C.c_float), ("alpha_dense", C.c_float),
        ("pad", C.c_int32), ("flatten_order", C.c_int32), ("pool_ties", C.c_int32),
        ("head", C.c_int32), ("precision", C.c_int32), ("max_batch", C.c_int32),
        ("keep_all_activations", C.c_int32), ("device", C.c_int32),
        ("refine_margin", C.c_float), ("refine_capacity", C.c_int32),
    ]


_P = C.c_void_p
_SIGNATURES = {
    "bcad_create": (C.c_int, [C.POINTER(Config), C.POINTER(_P)]),
    "bcad_destroy": (None, [_P]),
    "bcad_last_error": (C.c_char_p, []),
    "bcad_version": (C.c_char_p, []),
    "bcad_set_conv_weights": (C.c_int, [_P, C.c_int, _P, _P]),
    "bcad_set_dense_weights": (C.c_int, [_P, C.c_int, _P, _P]),
    "bcad_fold_batchnorm": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.c_float]),
    "bcad_commit": (C.c_int, [_P]),
    "bcad_set_fast_training": (C.c_int, [_P, C.c_int]),
    "bcad_predict": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P]),
    "bcad_predict_explain": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P, _P, _P, _P]),
    "bcad_predict_explain_sized": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P, _P, C.c_int, C.c_int, _P, _P]),
    "bcad_predict_explain_classes": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, C.c_int, _P, _P, _P, C.c_int, C.c_int, _P, _P]),
    "bcad_gradcam_overlays_host": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, _P, _P, _P, _P, _P]),
    "bcad_gradcam_overlays_classes_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P, _P, _P,
                                                     _P, _P]),
    "bcad_saliency_overlays_classes_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P, _P, _P,
                                                      _P, _P, _P]),
    "bcad_saliency_overlay_resized": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "bcad_gray_resize_preprocess": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "bcad_overlay_classes": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "bcad_explain_backward": (C.c_int, [_P, C.c_int, _P, C.c_int, C.POINTER(_P), _P, _P]),
    "bcad_predict_saliency_classes": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, C.c_int, _P, _P, _P, _P, _P, _P]),
    "bcad_saliency_overlay": (C.c_int, [_P, C.c_int, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "bcad_get_tensor": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "bcad_tensor_elems": (C.c_int64, [_P, C.c_int, C.c_int]),
    "bcad_predict_explain_host": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P, _P, _P]),
    "bcad_predict_explain_host_u8": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P, _P, _P]),
    "bcad_predict_explain_host_u8in": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P, _P, _P, _P]),
    "bcad_gradcam_tail": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "bcad_overlay": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "bcad_conv_block": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int, C.c_int, C.c_int, C.c_float,
                                  C.c_int, _P, _P, _P]),
    "bcad_avg_pool": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "bcad_unet_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "bcad_unet_destroy": (None, [_P]),
    "bcad_unet_set_kernels": (C.c_int, [_P, _P, _P, _P]),
    "bcad_unet_out_shape": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "bcad_unet_forward": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P]),
    "bcad_unet_launch_count": (C.c_int64, [_P]),
    "bcad_unet_set_profiling": (C.c_int, [_P, C.c_int]),
    "bcad_unet_profile_get": (C.c_int, [_P, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_float)]),
    "bcad_gray_preprocess": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "bcad_bottleneck_resize": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "bcad_grad_elems": (C.c_int64, [_P]),
    "bcad_grad_layout": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                   C.POINTER(C.c_int64)]),
    "bcad_train_backward": (C.c_int, [_P, _P, _P, C.c_int, _P, _P, _P]),
    "bcad_train_backward_part": (C.c_int, [_P, _P, _P, C.c_int, _P, _P, C.c_int, _P]),
    "bcad_set_dropout_masks": (C.c_int, [_P, _P, C.c_int, C.c_int, _P]),
    "bcad_apply_update": (C.c_int, [_P, _P, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _P]),
    "bcad_get_conv_weights": (C.c_int, [_P, C.c_int, _P, _P]),
    "bcad_get_dense_weights": (C.c_int, [_P, C.c_int, _P, _P]),
    "bcad_set_explain_target": (C.c_int, [_P, C.c_int]),
    "bcad_refine_stats": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "bcad_launch_count": (C.c_int64, [_P]),
    "bcad_uses_tensor_path": (C.c_int, [_P]),
    "bcad_set_profiling": (C.c_int, [_P, C.c_int]),
    "bcad_selftest_umma": (C.c_int, [_P, C.c_int, _P, C.c_int, _P, _P, _P]),
    "bcad_selftest_umma_bench": (C.c_int, [_P, _P, _P]),
    "bcad_profile_count": (C.c_int, [_P]),
    "bcad_profile_get": (C.c_int, [_P, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_float)]),
}

_lib = None


def exported_symbols():
    return sorted(_SIGNATURES)


def load() -> C.CDLL:
    """dlopen libbcad.so (built in-tree by build.py); raises if absent -- no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("BCAD_LIB", LIB_PATH)       # developer override: an experimental build of the same ABI
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: build it with `python vision-xai-breast-cancer-cad_b200/build.py` "
            "(or __graft_entry__.build()). This package has no CPU / PyTorch fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().bcad_last_error().decode("utf-8", "replace")


def check(rc: int):
    """C status -> the exception classes the reference's callers already catch (SURVEY 8b)."""
    if rc == OK:
        return
    msg = last_error()
    if rc == ERR_INVALID:
        raise ValueError(msg)
    if rc == ERR_NOMEM:
        raise MemoryError(msg)
    raise RuntimeError(msg)
