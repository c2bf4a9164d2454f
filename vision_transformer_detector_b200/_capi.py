"""ctypes binding of include/vitdet_b200.h.

The CUDA library is the only implementation of the path: if it is missing or fails to load, importing
this module raises — there is no CPU or PyTorch fallback behind these entry points.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

MODE_BF16 = 0
MODE_FP32 = 1
MODES = {"bf16": MODE_BF16, "fp32": MODE_FP32, "float32": MODE_FP32, "bfloat16": MODE_BF16}

E_INVALID, E_NO_DEVICE, E_CUDA, E_NOT_FOUND, E_SHAPE, E_UNSET = -1, -2, -3, -4, -5, -6


class VitdetError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"vitdet_b200 error {code}: {message}")
        self.code = code


class Config(C.Structure):
    """struct vitdet_config — kwargs of create_vision_transformer_detector (det.py:498-506)."""
    _fields_ = [
        ("image_h", C.c_int32), ("image_w", C.c_int32),
        ("patch_size", C.c_int32), ("embedding_dim", C.c_int32),
        ("num_heads", C.c_int32), ("key_dim", C.c_int32),
        ("mlp_quantities", C.c_int32), ("repeat_times", C.c_int32),
        ("head_last_units", C.c_int32), ("head_dense_layers", C.c_int32), ("head_block_repeats", C.c_int32),
        ("use_mish", C.c_int32), ("num_slots", C.c_int32), ("classes", C.c_int32),
        ("ln_epsilon", C.c_float),
    ]


class DecodeParams(C.Structure):
    """struct vitdet_decode_params."""
    _fields_ = [
        ("objectness_threshold", C.c_float), ("classification_threshold", C.c_float),
        ("strict", C.c_int32),
        ("image_h", C.c_float), ("image_w", C.c_float),
        ("classes", C.c_int32),
        ("use_transform_predictions", C.c_int32),
        ("corner_scale", C.c_float),
    ]


class DenseEx(C.Structure):
    """struct vitdet_dense_ex — extras of the tensor-core Dense epilogue (operator-level tests)."""
    _fields_ = [
        ("pos", C.c_void_p), ("pos_period", C.c_int32),
        ("ln_gamma", C.c_void_p), ("ln_beta", C.c_void_p), ("ln_eps", C.c_float), ("ln_out", C.c_void_p),
        ("store_bf16", C.c_int32), ("pair", C.c_int32),
    ]


class Detections(C.Structure):
    """struct vitdet_detections (device or host pointers depending on the call)."""
    _fields_ = [
        ("decoded", C.c_void_p), ("class_id", C.c_void_p), ("class_conf", C.c_void_p),
        ("keep", C.c_void_p), ("corners", C.c_void_p), ("packed", C.c_void_p),
    ]


class Image(C.Structure):
    """struct vitdet_image — one uint8 (height, width, 3) image of a ragged batch (device or host pixels)."""
    _fields_ = [("pixels", C.c_void_p), ("height", C.c_int32), ("width", C.c_int32)]


class Jpeg(C.Structure):
    """struct vitdet_jpeg — the host bytes of one JPEG file."""
    _fields_ = [("data", C.c_void_p), ("bytes", C.c_int64)]


# every symbol include/vitdet_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "vitdet_abi_version": (C.c_int, []),
    "vitdet_last_error": (C.c_char_p, []),
    "vitdet_default_config": (None, [C.POINTER(Config)]),
    "vitdet_create": (C.c_int, [C.POINTER(Config), C.POINTER(_P)]),
    "vitdet_destroy": (None, [_P]),
    "vitdet_tokens": (C.c_int, [_P]),
    "vitdet_patch_dim": (C.c_int, [_P]),
    "vitdet_count_params": (C.c_int64, [_P]),
    "vitdet_num_weights": (C.c_int, [_P]),
    "vitdet_weight_info": (C.c_int, [_P, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int64)]),
    "vitdet_set_weight": (C.c_int, [_P, C.c_char_p, _P, C.c_int, C.POINTER(C.c_int64)]),
    "vitdet_get_weight": (C.c_int, [_P, C.c_char_p, _P, C.c_int64]),
    "vitdet_set_chunk": (C.c_int, [_P, C.c_int]),
    "vitdet_workspace_bytes": (C.c_size_t, [_P, C.c_int, C.c_int]),
    "vitdet_profile_enable": (C.c_int, [_P, C.c_uint32]),
    "vitdet_profile_num_categories": (C.c_int, [_P]),
    "vitdet_profile_category_name": (C.c_char_p, [C.c_int]),
    "vitdet_profile_read": (C.c_int, [_P, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int]),
    "vitdet_launch_count": (C.c_int64, [_P, C.c_int]),
    "vitdet_forward": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P]),
    "vitdet_decode": (C.c_int, [_P, C.c_int, C.POINTER(DecodeParams), C.POINTER(Detections), _P]),
    "vitdet_decode_host": (C.c_int, [_P, C.c_int, C.POINTER(DecodeParams), C.POINTER(Detections)]),
    "vitdet_preprocess_image": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P]),
    "vitdet_preprocess_image_host": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_int, C.c_int]),
    "vitdet_resize_with_pad_geometry": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int] + [C.POINTER(C.c_int)] * 4),
    "vitdet_iou": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P, _P]),
    "vitdet_iou_host": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P]),
    "vitdet_forward_u8": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.POINTER(DecodeParams), C.POINTER(Detections), _P]),
    "vitdet_predict_host_u8": (C.c_int, [_P, _P, C.c_int, C.c_int, C.POINTER(DecodeParams), _P, C.POINTER(Detections), _P]),
    "vitdet_map_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "vitdet_map_destroy": (None, [_P]),
    "vitdet_map_reset": (C.c_int, [_P, _P]),
    "vitdet_map_update": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(DecodeParams), _P]),
    "vitdet_map_update_host": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(DecodeParams)]),
    "vitdet_map_result": (C.c_int, [_P, _P, _P, _P, _P]),
    "vitdet_map_state": (C.c_int, [_P, _P, _P, _P, _P]),
    "vitdet_map_iou_thresholds": (C.c_int, [_P, _P]),
    "vitdet_map_launch_count": (C.c_uint64, [_P]),
    "vitdet_forward_decode": (C.c_int, [_P, _P, C.c_int, C.c_int, C.POINTER(DecodeParams), _P, C.POINTER(Detections), _P]),
    "vitdet_predict_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.POINTER(DecodeParams), _P, C.POINTER(Detections), _P]),
    "vitdet_op_dense": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "vitdet_op_layernorm": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_float, _P]),
    "vitdet_op_attention": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "vitdet_op_patchify": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "vitdet_op_dense_ex": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(DenseEx), _P]),
    "vitdet_op_mlp_tail": (C.c_int, [_P] * 8 + [_P, _P, C.c_float, _P] + [C.c_int] * 6 + [_P]),
    "vitdet_op_head_slots": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "vitdet_submit_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.POINTER(DecodeParams), C.c_int, _P, C.POINTER(C.c_int)]),
    "vitdet_collect": (C.c_int, [_P, C.c_int, _P, C.POINTER(Detections)]),
    "vitdet_forward_images": (C.c_int, [_P, C.POINTER(Image), C.c_int, C.c_int, C.POINTER(DecodeParams), _P, C.POINTER(Detections), _P, _P]),
    "vitdet_submit_images_host": (C.c_int, [_P, C.POINTER(Image), C.c_int, C.c_int, C.POINTER(DecodeParams), C.c_int, _P, _P,
                                            C.POINTER(C.c_int)]),
    "vitdet_jpeg_info": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vitdet_decode_jpeg": (C.c_int, [_P, C.POINTER(Jpeg), C.c_int, _P, _P, _P]),
    "vitdet_submit_jpeg_host": (C.c_int, [_P, C.POINTER(Jpeg), C.c_int, C.c_int, C.POINTER(DecodeParams), C.c_int, _P, _P,
                                          C.POINTER(C.c_int)]),
    "vitdet_decode_jpeg_scaled": (C.c_int, [_P, C.POINTER(Jpeg), _P, C.c_int, _P, _P, _P]),
    "vitdet_submit_jpeg_host_scaled": (C.c_int, [_P, C.POINTER(Jpeg), _P, C.c_int, C.c_int, C.POINTER(DecodeParams), C.c_int, _P,
                                                 _P, C.POINTER(C.c_int)]),
    "vitdet_jpeg_auto_ratio": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "vitdet_jpeg_stats": (C.c_int, [_P, _P]),
    "vitdet_gather_detections": (C.c_int, [_P, _P, C.c_int, _P, _P]),
    "vitdet_nccl_unique_id": (C.c_int, [C.c_char_p]),
    "vitdet_nccl_comm_create": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.POINTER(_P)]),
    "vitdet_nccl_comm_destroy": (C.c_int, [_P]),
    "vitdet_set_option": (C.c_int, [_P, C.c_char_p, C.c_int]),
    "vitdet_get_option": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_int)]),
    "vitdet_debug_taps": (C.c_int, [_P, C.c_int]),
    "vitdet_debug_read": (C.c_int, [_P, C.c_char_p, _P, C.c_int64]),
}

_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load() -> C.CDLL:
    """Loads libvitdet_b200.so (built in-tree by build.py).  Raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: build it with `python -m vision_transformer_detector_b200.build` "
            "(needs nvcc). There is no CPU fallback for this path.")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)   # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.vitdet_abi_version() != 2:
        raise ImportError(f"{path}: ABI version {lib.vitdet_abi_version()} != 2")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().vitdet_last_error()
        raise VitdetError(rc, msg.decode("utf-8", "replace") if msg else "")


def default_config() -> Config:
    cfg = Config()
    load().vitdet_default_config(C.byref(cfg))
    return cfg


def np_ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)
