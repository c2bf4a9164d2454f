"""Host-side mirror of the part of the reference's `vision_transformer_utilities.py` that sits immediately before the
hot path: turning an image file (or a decoded uint8 array) into the model's input tensor.  The COCO dataset plumbing of
the reference module (annotation parsing at import time from hard-coded D:\\ paths, tf.data pipeline) is out of scope.

    _get_image_tensor_coco(one_image_path)        vision_transformer_utilities.py:418-449
    preprocess_image(image_uint8)                 the arithmetic of that function: resize_with_pad, clip, /127.5 - 1
    decode_jpeg(files, ratio=1)                   tf.image.decode_jpeg(ratio=) on the GPU, bit-identical to PIL / libjpeg-turbo
    jpeg_auto_ratio(height, width)                the decode ratio PIL's draft() picks for the model's letterbox

The arithmetic runs on the GPU (vitdet_preprocess_image*); only the file decode is host work (PIL)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi
from .vision_transformer_detector import (Constants, DetectorConfig, _is_torch_cuda, _jpeg_arrays, _jpeg_ratios, _jpeg_table,
                                          _torch_stream_ptr)

MODEL_IMAGE_HEIGHT, MODEL_IMAGE_WIDTH = Constants.MODEL_IMAGE_SIZE.value       # vision_transformer_utilities.py:23-24


def resize_with_pad_geometry(height: int, width: int, target_height: int, target_width: int) -> tuple[int, int, int, int]:
    """(resized_height, resized_width, pad_top, pad_left) of tf.image.resize_with_pad, in TF's float32 arithmetic."""
    v = [C.c_int() for _ in range(4)]
    _capi.check(_capi.load().vitdet_resize_with_pad_geometry(int(height), int(width), int(target_height), int(target_width),
                                                             *[C.byref(x) for x in v]))
    return tuple(x.value for x in v)


def preprocess_image(image, target_size=None):
    """uint8 (h, w, 3) -> float32 (H, W, 3) in [-1, 1]: resize_with_pad + clip + /127.5 - 1, on the GPU.
    numpy in -> numpy out; torch CUDA uint8 tensor in -> torch CUDA tensor out (asynchronous on torch's stream)."""
    th, tw = (MODEL_IMAGE_HEIGHT, MODEL_IMAGE_WIDTH) if target_size is None else (int(target_size[0]), int(target_size[1]))
    lib = _capi.load()
    if _is_torch_cuda(image):
        import torch
        x = image.contiguous()
        if x.dtype != torch.uint8 or x.dim() != 3 or x.shape[2] != 3:
            raise ValueError(f"image must be a uint8 tensor of shape (h, w, 3), got {x.dtype} {tuple(x.shape)}")
        out = torch.empty((th, tw, 3), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _capi.check(lib.vitdet_preprocess_image(C.c_void_p(x.data_ptr()), int(x.shape[0]), int(x.shape[1]),
                                                    C.c_void_p(out.data_ptr()), th, tw, _torch_stream_ptr(x.device)))
        return out
    x = np.ascontiguousarray(np.asarray(image))
    if x.dtype != np.uint8 or x.ndim != 3 or x.shape[2] != 3:
        raise ValueError(f"image must be a uint8 array of shape (h, w, 3), got {x.dtype} {x.shape}")
    out = np.empty((th, tw, 3), np.float32)
    _capi.check(lib.vitdet_preprocess_image_host(_capi.np_ptr(x), int(x.shape[0]), int(x.shape[1]), _capi.np_ptr(out), th, tw))
    return out


def _get_image_tensor_coco(one_image_path):
    """vision_transformer_utilities.py:418-449: (image_tensor (H, W, 3) float32 in [-1, 1], (original_height, original_width)).
    tf.io.read_file + tf.image.decode_image(channels=3) become a PIL decode; everything after it runs on the GPU."""
    from PIL import Image
    with Image.open(one_image_path) as im:
        arr = np.asarray(im.convert("RGB"), dtype=np.uint8)
    return preprocess_image(arr), (int(arr.shape[0]), int(arr.shape[1]))


_decoders: dict = {}      # device index -> a handle of a tiny model, whose JPEG decode scratch decode_jpeg uses


def _decoder(index: int) -> C.c_void_p:
    h = _decoders.get(index)
    if h is None:
        cfg = DetectorConfig(input_shape=(16, 16, 3), encoder_num_heads=1, encoder_mlp_quantities=1, encoder_repeat_times=1,
                             mlp_head_last_units=8, mlp_head_dense_layers_quantity=1).to_c()
        h = C.c_void_p()
        _capi.check(_capi.load().vitdet_create(C.byref(cfg), C.byref(h)))
        _decoders[index] = h
    return h


def jpeg_auto_ratio(height: int, width: int, target_size=None) -> int:
    """The decode ratio detect_jpeg(ratio="auto") uses for a height x width file: what PIL's draft("RGB", (rw, rh)) picks
    for the size (rh, rw) resize_with_pad gives it at target_size (default: the model's 608 x 608), i.e. the largest of 8,
    4, 2, 1 that is at most min(width // rw, height // rh)."""
    th, tw = (MODEL_IMAGE_HEIGHT, MODEL_IMAGE_WIDTH) if target_size is None else (int(target_size[0]), int(target_size[1]))
    rc = _capi.load().vitdet_jpeg_auto_ratio(int(height), int(width), th, tw)
    if rc < 0:
        _capi.check(rc)
    return rc


def decode_jpeg(files, device=None, ratio=1) -> list:
    """Baseline JPEG files -> a list of torch CUDA uint8 (h, w, 3) RGB tensors, decoded on the GPU bit-identically to
    np.asarray(PIL.Image.open(f).convert("RGB")) (libjpeg-turbo's ISLOW IDCT and fancy upsampling, which
    tf.image.decode_jpeg also uses).  files: bytes-like objects or paths.  Asynchronous on torch's current stream of
    `device` (default: the current CUDA device).  A file outside baseline JPEG raises VitdetError (E_INVALID) naming it.
    ratio: 1, 2, 4 or 8, or one of them per file: decode at 1 / ratio scale in the DCT domain, (ceil(h / ratio),
    ceil(w / ratio), 3), bit-identical to tf.image.decode_jpeg(ratio=) and to PIL after im.draft("RGB", (w // ratio,
    h // ratio))."""
    import torch
    arrs = _jpeg_arrays(files)
    ratios = _jpeg_ratios(ratio, len(arrs), allow_auto=False)
    lib = _capi.load()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise ValueError(f"device must be a CUDA device, got {dev}")
    index = dev.index if dev.index is not None else torch.cuda.current_device()
    shapes, offs, total = [], [], 0
    for i, a in enumerate(arrs):
        v = [C.c_int() for _ in range(3)]
        rc = lib.vitdet_jpeg_info(C.c_void_p(a.ctypes.data), int(a.size), *[C.byref(x) for x in v])
        if rc:
            msg = lib.vitdet_last_error()
            raise _capi.VitdetError(rc, f"file {i}: " + (msg.decode("utf-8", "replace") if msg else ""))
        h, w = -(-v[0].value // ratios[i]), -(-v[1].value // ratios[i])
        shapes.append((h, w, 3))
        offs.append(total)
        total += (h * w * 3 + 255) // 256 * 256
    with torch.cuda.device(index):
        buf = torch.empty(total, dtype=torch.uint8, device=dev)
        _capi.check(lib.vitdet_decode_jpeg_scaled(_decoder(index), _jpeg_table(arrs), (C.c_int32 * len(arrs))(*ratios), len(arrs),
                                                  C.c_void_p(buf.data_ptr()), (C.c_int64 * len(arrs))(*offs), _torch_stream_ptr(dev)))
    return [buf[o:o + h * w * 3].view(h, w, 3) for o, (h, w, _) in zip(offs, shapes)]
