"""Host-side mirror of the reference module `vision_transformer_detector.py` for ONE path: build the
detector, run prediction, decode the anchor-free head.

Same entry points, argument names, defaults and error behaviour as the reference:

    Constants                                   det.py:19-43
    transformer_preprocessor / transformer_encoder / mlp_head      det.py:239, :312, :417
    create_vision_transformer_detector(...)     det.py:498-583
    model.predict(x) / model(x, training=False) / get_weights / set_weights / weights / count_params
    transform_predictions(inputs)               det.py:586-647
    threshold rule                              det.py:2257-2283 (visualise), det.py:1359-1384 (metric)

Nothing here computes: every number comes from the sm_100a CUDA library behind include/vitdet_b200.h,
called through ctypes (`_capi`).  numpy arrays go through the library's host entry points; torch CUDA
tensors (torch is only a tensor carrier) are passed by device pointer on torch's current stream.
There is no CPU fallback: without the library or without a B200 these functions raise.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import os
from enum import Enum
from typing import Any, Iterable, Sequence

import numpy as np

from . import _capi
from . import keras_init


class Constants(Enum):
    """Module constants of the reference (det.py:19-43)."""
    CLASSES = 80
    MODEL_IMAGE_SIZE = 608, 608          # height, width
    EPSILON = 1e-8
    MAX_DETECT_OBJECTS_QUANTITY = 17
    LATEST_RELATED_IMAGES = 3
    BBOXES_PER_IMAGE = 14
    OBJECTNESS_THRESHOLD = 0.5
    CLASSIFICATION_CONFIDENCE_THRESHOLD = 0.5


# ------------------------------------------------------------------------------------------------
# configuration and the Keras weight table
# ------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class DetectorConfig:
    """Keyword arguments of create_vision_transformer_detector (det.py:498-506)."""
    input_shape: tuple = (*Constants.MODEL_IMAGE_SIZE.value, 3)
    patch_size: int = 17
    embedding_dim: int = 28
    encoder_num_heads: int = 8
    encoder_key_dim: int = 40
    dropout: Any = None
    encoder_mlp_quantities: int = 8
    encoder_repeat_times: int = 8
    mlp_head_last_units: int = 136
    mlp_head_dense_layers_quantity: int = 7
    mlp_head_dense_mish_block_repeats: int = 1
    use_mish: bool = True
    max_weight: float = 10          # training-time constraint only (det.py:209-236): accepted, unused
    clip_weight: bool = True        # idem
    training: Any = None

    @property
    def grid(self) -> tuple[int, int]:
        h, w = int(self.input_shape[0]), int(self.input_shape[1])
        p = int(self.patch_size)
        return -(-h // p), -(-w // p)      # ceil: extract_patches padding='SAME' (det.py:195-197)

    @property
    def tokens(self) -> int:
        gh, gw = self.grid
        return gh * gw

    @property
    def patch_dim(self) -> int:
        return 3 * self.patch_size * self.patch_size

    def encoder_mlp_units(self) -> list[int]:
        # det.py:385-386: last_dimensionality * 2 ** arange(q-1, -1, -1)
        q = self.encoder_mlp_quantities
        return [self.embedding_dim * 2 ** (q - 1 - j) for j in range(q)]

    def head_units(self) -> list[int]:
        # det.py:465-470: reversed(last_units * 2 ** arange(n)), each repeated `block_repeats` times
        out = []
        for k in reversed(range(self.mlp_head_dense_layers_quantity)):
            out += [self.mlp_head_last_units * 2 ** k] * self.mlp_head_dense_mish_block_repeats
        return out

    def to_c(self) -> _capi.Config:
        c = _capi.Config()
        c.image_h, c.image_w = int(self.input_shape[0]), int(self.input_shape[1])
        c.patch_size = int(self.patch_size)
        c.embedding_dim = int(self.embedding_dim)
        c.num_heads = int(self.encoder_num_heads)
        c.key_dim = int(self.encoder_key_dim)
        c.mlp_quantities = int(self.encoder_mlp_quantities)
        c.repeat_times = int(self.encoder_repeat_times)
        c.head_last_units = int(self.mlp_head_last_units)
        c.head_dense_layers = int(self.mlp_head_dense_layers_quantity)
        c.head_block_repeats = int(self.mlp_head_dense_mish_block_repeats)
        c.use_mish = 1 if self.use_mish else 0
        c.num_slots = Constants.MAX_DETECT_OBJECTS_QUANTITY.value
        c.classes = Constants.CLASSES.value
        c.ln_epsilon = 1e-3
        return c


def _keras_name(base: str, index: int) -> str:
    # keras.backend.clear_session() (det.py:548) resets the auto-name counters: first instance is
    # un-suffixed, instance i >= 1 is "<base>_<i>".
    return base if index == 0 else f"{base}_{index}"


def weight_specs(cfg: DetectorConfig) -> list[tuple[str, tuple[int, ...]]]:
    """(name, shape) of every Keras variable of the model, in `model.weights` order.

    Names are the Keras variable names without ':0'.  The C library enumerates the same table
    (vitdet_weight_info); tests check that the two agree."""
    D, H, d, T, P = cfg.embedding_dim, cfg.encoder_num_heads, cfg.encoder_key_dim, cfg.tokens, cfg.patch_dim
    S = Constants.MAX_DETECT_OBJECTS_QUANTITY.value
    out: list[tuple[str, tuple[int, ...]]] = []
    out.append(("linear_projection/kernel", (P, D)))
    out.append(("linear_projection/bias", (D,)))
    out.append(("position_encoding/position_embedding/embeddings", (T, 1)))
    for i in range(cfg.encoder_repeat_times):
        ln1, ln2 = _keras_name("layer_normalization", 2 * i), _keras_name("layer_normalization", 2 * i + 1)
        mha = _keras_name("multi_head_attention", i)
        out += [(f"{ln1}/gamma", (D,)), (f"{ln1}/beta", (D,))]
        for sel in ("query", "key", "value"):
            out += [(f"{mha}/{sel}/kernel", (D, H, d)), (f"{mha}/{sel}/bias", (H, d))]
        out += [(f"{mha}/attention_output/kernel", (H, d, D)), (f"{mha}/attention_output/bias", (D,))]
        out += [(f"{ln2}/gamma", (D,)), (f"{ln2}/beta", (D,))]
        fan_in = D
        for j, units in enumerate(cfg.encoder_mlp_units()):
            out += [(f"MLP_{i + 1}_{j + 1}/kernel", (fan_in, units)), (f"MLP_{i + 1}_{j + 1}/bias", (units,))]
            fan_in = units
    dense_idx = 0
    nm = _keras_name("dense", dense_idx); dense_idx += 1
    out += [(f"{nm}/kernel", (D, S)), (f"{nm}/bias", (S,))]
    fan_in = T
    for units in cfg.head_units():
        nm = _keras_name("dense", dense_idx); dense_idx += 1
        out += [(f"{nm}/kernel", (fan_in, units)), (f"{nm}/bias", (units,))]
        fan_in = units
    out += [("MLP_Head_no_Sigmoid/kernel", (fan_in, 6)), ("MLP_Head_no_Sigmoid/bias", (6,))]
    return out


def random_weights(cfg: DetectorConfig, seed: int = 0, spread: bool = False) -> dict[str, np.ndarray]:
    """Keras-default random initialisation of every variable (see keras_init)."""
    rng = np.random.default_rng(seed)
    return {name: keras_init.init_weight(rng, name, shape, spread=spread) for name, shape in weight_specs(cfg)}


# ------------------------------------------------------------------------------------------------
# graph-builder helpers: same names / arguments as the reference; they thread a symbolic description
# of the model instead of Keras tensors.
# ------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class SymbolicTensor:
    """Stand-in for a Keras symbolic tensor: the static shape (batch dimension None) plus the
    configuration accumulated by the builder functions so far."""
    shape: tuple
    spec: dict


def Input(shape: Sequence[int], name: str = "images") -> SymbolicTensor:
    return SymbolicTensor(shape=(None, *shape), spec={"input_shape": tuple(int(s) for s in shape), "input_name": name})


def _check_inference_only(dropout, training) -> None:
    if dropout is not None:
        raise NotImplementedError("dropout layers exist only for training (det.py:404-405, :485-486); "
                                  "this build implements the inference path (dropout=None)")
    if training:
        raise NotImplementedError("training=True is outside the predict/decode path")


def transformer_preprocessor(inputs: SymbolicTensor, patch_size, embedding_dim, max_weight, clip_weight) -> SymbolicTensor:
    """det.py:239-309: split into patches (SAME padding), Dense(embedding_dim), + learned scalar position."""
    h, w = inputs.shape[1], inputs.shape[2]
    tokens = (-(-h // patch_size)) * (-(-w // patch_size))
    spec = dict(inputs.spec, patch_size=int(patch_size), embedding_dim=int(embedding_dim),
                max_weight=max_weight, clip_weight=clip_weight)
    return SymbolicTensor(shape=(None, tokens, embedding_dim), spec=spec)


def transformer_encoder(embedded_image_patches: SymbolicTensor, use_mish, num_heads, key_dim, dropout,
                        mlp_quantities, repeat_times, max_weight, clip_weight, training=None) -> SymbolicTensor:
    """det.py:312-414: repeat_times x [LN, MHA, +res, LN, mlp_quantities x (Dense + Mish|GELU), +res]."""
    _check_inference_only(dropout, training)
    spec = dict(embedded_image_patches.spec, use_mish=bool(use_mish), encoder_num_heads=int(num_heads),
                encoder_key_dim=int(key_dim), encoder_mlp_quantities=int(mlp_quantities),
                encoder_repeat_times=int(repeat_times))
    return SymbolicTensor(shape=embedded_image_patches.shape, spec=spec)


def mlp_head(encoder_outputs: SymbolicTensor, use_mish, mlp_head_last_units, dense_layers_quantity,
             dense_mish_block_repeats, dropout, max_weight, clip_weight, training=None) -> SymbolicTensor:
    """det.py:417-495: Dense(17) -> Reshape((17, -1)) -> Dense+act pyramid -> Dense(6)."""
    _check_inference_only(dropout, training)
    if bool(use_mish) != encoder_outputs.spec.get("use_mish", bool(use_mish)):
        raise NotImplementedError("encoder and head must use the same activation in this build")
    spec = dict(encoder_outputs.spec, use_mish=bool(use_mish), mlp_head_last_units=int(mlp_head_last_units),
                mlp_head_dense_layers_quantity=int(dense_layers_quantity),
                mlp_head_dense_mish_block_repeats=int(dense_mish_block_repeats))
    return SymbolicTensor(shape=(None, Constants.MAX_DETECT_OBJECTS_QUANTITY.value, 6), spec=spec)


# ------------------------------------------------------------------------------------------------
# decode results
# ------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class DetectionRecords:
    """Per-slot records of the decode, shapes (B, 17, ...).  numpy arrays or torch CUDA tensors."""
    logits: Any        # (B,17,6) f32 raw head output
    decoded: Any       # (B,17,6) f32 transform_predictions output
    class_id: Any      # (B,17)   i32 round-half-even(class)
    class_conf: Any    # (B,17)   f32 (0.5 - |class - id|) / 0.5
    keep: Any          # (B,17)   u8  both thresholds passed
    corners: Any       # (B,17,4) i32 x0, y0, x1, y1
    packed: Any = None  # (B*17,13) f32 the same record as one row (what the ranks all-gather); only with packed=True
    boxes_original: Any = None  # (B,17,4) f32 x0, y0, x1, y1 on each source image; only from detect_images / submit_images

    def detections(self) -> list[list[dict]]:
        """Kept slots per image as plain records (what the visualise loop iterates, det.py:2260-2325)."""
        to_np = lambda a: a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        dec, cid, cc, keep, cor = map(to_np, (self.decoded, self.class_id, self.class_conf, self.keep, self.corners))
        out = []
        for b in range(dec.shape[0]):
            rows = []
            for s in np.nonzero(keep[b])[0]:
                rows.append({"slot": int(s), "class_id": int(cid[b, s]), "objectness": float(dec[b, s, 0]),
                             "class_confidence": float(cc[b, s]), "cx": float(dec[b, s, 2]), "cy": float(dec[b, s, 3]),
                             "h": float(dec[b, s, 4]), "w": float(dec[b, s, 5]),
                             "corners": tuple(int(v) for v in cor[b, s])})
            out.append(rows)
        return out


def _decode_params(objectness_threshold, classification_threshold, strict, image_size,
                   use_transform_predictions=True, corner_scale=1.0) -> _capi.DecodeParams:
    p = _capi.DecodeParams()
    p.objectness_threshold = Constants.OBJECTNESS_THRESHOLD.value if objectness_threshold is None else float(objectness_threshold)
    p.classification_threshold = (Constants.CLASSIFICATION_CONFIDENCE_THRESHOLD.value
                                  if classification_threshold is None else float(classification_threshold))
    p.strict = 1 if strict else 0
    ih, iw = Constants.MODEL_IMAGE_SIZE.value if image_size is None else image_size
    p.image_h, p.image_w = float(ih), float(iw)
    p.classes = Constants.CLASSES.value
    p.use_transform_predictions = 1 if use_transform_predictions else 0
    p.corner_scale = float(corner_scale)
    return p


def _is_uint8(x) -> bool:
    return str(getattr(x, "dtype", "")).endswith("uint8")


def _is_torch_cuda(x) -> bool:
    return type(x).__module__.startswith("torch") and hasattr(x, "is_cuda") and x.is_cuda


def _model_input(x, normalize_uint8: bool):
    """(x as a contiguous numpy array or torch CUDA tensor, u8).  u8: `x` holds uint8 pixels AND the caller asked for the
    fused input normalisation x / 127.5 - 1 (vision_transformer_utilities.py:446-447, done inside the patch kernel), and
    stays uint8.  Otherwise x is cast to float32, which is what keras Model.predict does with a uint8 array."""
    u8 = bool(normalize_uint8) and _is_uint8(x)
    if _is_torch_cuda(x):
        import torch
        return (x.contiguous() if u8 else x.to(torch.float32).contiguous()), u8
    return (np.ascontiguousarray(x) if u8 else np.ascontiguousarray(np.asarray(x, dtype=np.float32))), u8


def _torch_stream_ptr(device) -> C.c_void_p:
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _jpeg_arrays(files) -> list:
    """The bytes of every file as a 1-D uint8 numpy array (a view of bytes-like objects, the contents of paths); ValueError
    for an empty list, an empty file or an item that is neither."""
    if isinstance(files, (bytes, bytearray, memoryview, str, os.PathLike)):
        raise ValueError("files must be a sequence of JPEG files, not a single one")
    items = list(files)
    if not items:
        raise ValueError("files must be a non-empty sequence of bytes-like objects or paths")
    out = []
    for i, f in enumerate(items):
        if isinstance(f, (str, os.PathLike)):
            with open(f, "rb") as fh:
                a = np.frombuffer(fh.read(), np.uint8)
        elif isinstance(f, np.ndarray):
            if f.dtype != np.uint8 or f.ndim != 1 or not f.flags.c_contiguous:
                raise ValueError(f"file {i}: a numpy array must be 1-D contiguous uint8, got {f.dtype} {f.shape}")
            a = f
        elif isinstance(f, (bytes, bytearray, memoryview)):
            a = np.frombuffer(f, np.uint8)
        else:
            raise ValueError(f"file {i}: {type(f).__name__} is neither bytes-like nor a path")
        if a.size == 0:
            raise ValueError(f"file {i} is empty")
        out.append(a)
    return out


def _jpeg_table(arrs) -> C.Array:
    return (_capi.Jpeg * len(arrs))(*[_capi.Jpeg(a.ctypes.data, int(a.size)) for a in arrs])


JPEG_RATIOS = (1, 2, 4, 8)


def _jpeg_ratios(ratio, B: int, allow_auto: bool) -> list:
    """The decode scale of B files as the library's int32 codes: ratio is 1, 2, 4, 8 ("auto", code 0, where allowed) or a
    sequence of B of them.  ValueError for anything else."""
    def code(r, where):
        if allow_auto and isinstance(r, str) and r == "auto":
            return 0
        if isinstance(r, (int, np.integer)) and not isinstance(r, (bool, np.bool_)) and int(r) in JPEG_RATIOS:
            return int(r)
        allowed = '1, 2, 4, 8 or "auto"' if allow_auto else "1, 2, 4 or 8"
        raise ValueError(f"{where}ratio must be {allowed}, got {r!r}")
    if isinstance(ratio, (str, int, np.integer)):
        return [code(ratio, "")] * B
    if not isinstance(ratio, (list, tuple, np.ndarray)):
        raise ValueError(f"ratio must be a ratio or a sequence of one per file, got {type(ratio).__name__}")
    if len(ratio) != B:
        raise ValueError(f"ratio holds {len(ratio)} ratios for {B} files")
    return [code(r, f"file {i}: ") for i, r in enumerate(ratio)]


def _alloc_records_np(B: int, S: int):
    return (np.empty((B, S, 6), np.float32), np.empty((B, S, 6), np.float32), np.empty((B, S), np.int32),
            np.empty((B, S), np.float32), np.empty((B, S), np.uint8), np.empty((B, S, 4), np.int32))


def _alloc_records_torch(B: int, S: int, device):
    import torch
    return (torch.empty((B, S, 6), dtype=torch.float32, device=device),
            torch.empty((B, S, 6), dtype=torch.float32, device=device),
            torch.empty((B, S), dtype=torch.int32, device=device),
            torch.empty((B, S), dtype=torch.float32, device=device),
            torch.empty((B, S), dtype=torch.uint8, device=device),
            torch.empty((B, S, 4), dtype=torch.int32, device=device))


def _records_struct(decoded, class_id, class_conf, keep, corners, packed=None) -> _capi.Detections:
    ptr = (lambda a: C.c_void_p(a.data_ptr())) if hasattr(decoded, "data_ptr") else _capi.np_ptr
    d = _capi.Detections()
    d.decoded, d.class_id, d.class_conf, d.keep, d.corners = ptr(decoded), ptr(class_id), ptr(class_conf), ptr(keep), ptr(corners)
    if packed is not None:
        d.packed = ptr(packed)
    return d


def _alloc_records(B: int, S: int, packed: bool = False, device=None) -> tuple[DetectionRecords, _capi.Detections]:
    """Empty records of B images of S slots, the (B*S, 13) packed array only when asked for, and the Detections struct
    that points at them: numpy arrays, or torch tensors on `device`."""
    if device is None:
        arrs = [*_alloc_records_np(B, S), np.empty((B * S, 13), np.float32) if packed else None]
    else:
        import torch
        arrs = [*_alloc_records_torch(B, S, device), torch.empty((B * S, 13), dtype=torch.float32, device=device) if packed else None]
    return DetectionRecords(*arrs), _records_struct(*arrs[1:])


def decode_predictions(predictions, objectness_threshold=None, classification_threshold=None, strict=True,
                       image_size=None, use_transform_predictions=True, corner_scale=1.0) -> DetectionRecords:
    """transform_predictions + the score thresholds + class ids + corner boxes, on the GPU.

    predictions: raw logits (..., 17, 6) — numpy (host) or torch CUDA tensor.
    strict=True is the metric rule (`>`, det.py:1381-1384); strict=False the visualise rule
    (kept unless `<`, det.py:2264, :2282).  image_size defaults to Constants.MODEL_IMAGE_SIZE, as in
    the reference, which scales by the module constant and not by the model's input shape
    (det.py:637-640).  use_transform_predictions=False treats `predictions` as already decoded rows
    (the flag of MeanAveragePrecision.update_state, det.py:1340-1341)."""
    lib = _capi.load()
    params = _decode_params(objectness_threshold, classification_threshold, strict, image_size,
                            use_transform_predictions, corner_scale)
    if _is_torch_cuda(predictions):
        import torch
        x = predictions.to(torch.float32).contiguous()
        lead = tuple(x.shape[:-1])
        R = int(np.prod(lead)) if lead else 1
        with torch.cuda.device(x.device):
            r, st = _alloc_records(R, 1, device=x.device)
            _capi.check(lib.vitdet_decode(C.c_void_p(x.data_ptr()), R, C.byref(params), C.byref(st), _torch_stream_ptr(x.device)))
        return DetectionRecords(predictions, r.decoded.reshape(*lead, 6), r.class_id.reshape(lead), r.class_conf.reshape(lead),
                                r.keep.reshape(lead), r.corners.reshape(*lead, 4))
    x = np.ascontiguousarray(np.asarray(predictions, dtype=np.float32))
    if x.shape[-1] != 6:
        raise ValueError(f"predictions must have a last dimension of 6, got shape {x.shape}")
    lead = x.shape[:-1]
    R = int(np.prod(lead)) if lead else 1
    r, st = _alloc_records(R, 1)
    _capi.check(lib.vitdet_decode_host(_capi.np_ptr(x), R, C.byref(params), C.byref(st)))
    return DetectionRecords(x, r.decoded.reshape(*lead, 6), r.class_id.reshape(lead), r.class_conf.reshape(lead),
                            r.keep.reshape(lead), r.corners.reshape(*lead, 4))


def transform_predictions(inputs, image_size=None):
    """det.py:586-647: sigmoid, clip the last four to [0, 1], scale class by CLASSES-1 and the box by
    the image size.  Returns an array/tensor of the same shape and kind as `inputs`."""
    return decode_predictions(inputs, image_size=image_size).decoded


def iou_calculator(label_bbox, prediction_bbox):
    """det.py:761-875: element-wise IoU of two equally shaped box arrays whose last axis ends with
    (center_x, center_y, height, width) in pixels; returns the array without its last axis.  numpy in ->
    numpy out, torch CUDA tensors in -> torch CUDA tensor out (computed on the GPU either way)."""
    lib = _capi.load()
    if _is_torch_cuda(label_bbox) or _is_torch_cuda(prediction_bbox):
        import torch
        a = label_bbox.to(torch.float32).contiguous()
        b = prediction_bbox.to(device=a.device, dtype=torch.float32).contiguous()
        if a.shape != b.shape or a.shape[-1] < 4:
            raise ValueError(f"label_bbox {tuple(a.shape)} and prediction_bbox {tuple(b.shape)} must have the same shape (..., >= 4)")
        out = torch.empty(a.shape[:-1], dtype=torch.float32, device=a.device)
        with torch.cuda.device(a.device):
            _capi.check(lib.vitdet_iou(C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), out.numel(), int(a.shape[-1]),
                                       C.c_void_p(out.data_ptr()), _torch_stream_ptr(a.device)))
        return out
    a = np.ascontiguousarray(np.asarray(label_bbox, dtype=np.float32))
    b = np.ascontiguousarray(np.asarray(prediction_bbox, dtype=np.float32))
    if a.shape != b.shape or a.shape[-1] < 4:
        raise ValueError(f"label_bbox {a.shape} and prediction_bbox {b.shape} must have the same shape (..., >= 4)")
    out = np.empty(a.shape[:-1], np.float32)
    _capi.check(lib.vitdet_iou_host(_capi.np_ptr(a), _capi.np_ptr(b), out.size, int(a.shape[-1]), _capi.np_ptr(out)))
    return out


# ------------------------------------------------------------------------------------------------
# evaluation metric
# ------------------------------------------------------------------------------------------------
class MeanAveragePrecision:
    """det.py:1268-2060 (tf.keras.metrics.Metric in the reference): the COCO-style AP — mean over ten IoU
    thresholds of the mean class AP — over the latest LATEST_RELATED_IMAGES related images per class with at most
    BBOXES_PER_IMAGE (confidence, IoU) rows each.  State and arithmetic live on the GPU (csrc/metric.cu); the three
    state attributes of the reference are exposed as read-only numpy copies in the reference's layout.

    update_state takes numpy arrays or torch CUDA tensors of shape (batch, slots, 6); with torch CUDA tensors nothing
    leaves the device, so `metric.update_state(labels, model(images))` evaluates straight from the head's output.
    """

    def __init__(self, name: str = "AP", classes: int | None = None, latest_related_images: int | None = None,
                 bboxes_per_image: int | None = None, image_size=None, **kwargs):
        self.name = name
        self.classes = Constants.CLASSES.value if classes is None else int(classes)
        self.latest_related_images = Constants.LATEST_RELATED_IMAGES.value if latest_related_images is None else int(latest_related_images)
        self.bboxes_per_image = Constants.BBOXES_PER_IMAGE.value if bboxes_per_image is None else int(bboxes_per_image)
        self.image_size = tuple(Constants.MODEL_IMAGE_SIZE.value if image_size is None else image_size)
        self._lib = _capi.load()
        self._h = C.c_void_p()
        _capi.check(self._lib.vitdet_map_create(self.classes, self.latest_related_images, self.bboxes_per_image, C.byref(self._h)))

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.vitdet_map_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _params(self, use_transform_predictions: bool) -> _capi.DecodeParams:
        p = _decode_params(None, None, True, self.image_size, use_transform_predictions)
        p.classes = self.classes
        return p

    def update_state(self, y_true, y_pred, sample_weight=None, use_transform_predictions=True) -> None:
        """det.py:1310-1862.  `sample_weight` is accepted and ignored, as in the reference."""
        p = self._params(bool(use_transform_predictions))
        if _is_torch_cuda(y_true) or _is_torch_cuda(y_pred):
            import torch
            dev = y_pred.device if _is_torch_cuda(y_pred) else y_true.device
            a = torch.as_tensor(y_true).to(device=dev, dtype=torch.float32).contiguous()
            b = torch.as_tensor(y_pred).to(device=dev, dtype=torch.float32).contiguous()
            if a.ndim != 3 or a.shape[-1] != 6 or a.shape != b.shape:
                raise ValueError(f"y_true {tuple(a.shape)} and y_pred {tuple(b.shape)} must both be (batch, slots, 6)")
            with torch.cuda.device(dev):
                _capi.check(self._lib.vitdet_map_update(self._h, C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), int(a.shape[0]),
                                                        int(a.shape[1]), C.byref(p), _torch_stream_ptr(dev)))
            # the kernels read a / b asynchronously on the current stream; torch's caching allocator only reuses their
            # memory for work queued later on that same stream, so letting them go out of scope here is safe
            return
        a = np.ascontiguousarray(np.asarray(y_true, dtype=np.float32))
        b = np.ascontiguousarray(np.asarray(y_pred, dtype=np.float32))
        if a.ndim != 3 or a.shape[-1] != 6 or a.shape != b.shape:
            raise ValueError(f"y_true {a.shape} and y_pred {b.shape} must both be (batch, slots, 6)")
        _capi.check(self._lib.vitdet_map_update_host(self._h, _capi.np_ptr(a), _capi.np_ptr(b), int(a.shape[0]), int(a.shape[1]), C.byref(p)))

    def _result(self):
        mean = np.zeros(1, np.float32)
        per_iou = np.zeros(10, np.float32)
        per_class = np.zeros((10, self.classes), np.float32)
        _capi.check(self._lib.vitdet_map_result(self._h, _capi.np_ptr(mean), _capi.np_ptr(per_iou), _capi.np_ptr(per_class), self._stream()))
        return mean[0], per_iou, per_class

    def result(self) -> np.float32:
        """det.py:1865-2049: the mean average precision as a float32 scalar."""
        return self._result()[0]

    def average_precision_per_iou(self) -> np.ndarray:
        """AP averaged over the classes seen so far, one value per IoU threshold (det.py:2024-2045)."""
        return self._result()[1]

    def average_precisions(self) -> np.ndarray:
        """(10, classes) AP per IoU threshold and class; classes that never showed up hold 0 (det.py:1879-2022)."""
        return self._result()[2]

    def reset_state(self) -> None:
        """det.py:2052-2060."""
        _capi.check(self._lib.vitdet_map_reset(self._h, self._stream()))

    reset_states = reset_state      # keras' older spelling

    def _stream(self) -> C.c_void_p:
        # numpy-only callers never import torch: the legacy stream (NULL), which is also what the *_host entry points use
        import sys
        torch = sys.modules.get("torch")
        if torch is None or not torch.cuda.is_available():
            return C.c_void_p()
        return _torch_stream_ptr(torch.device("cuda", torch.cuda.current_device()))

    def _state(self):
        bboxes = np.zeros((self.classes, self.latest_related_images, self.bboxes_per_image, 2), np.float32)
        labels = np.zeros((self.classes, self.latest_related_images), np.float32)
        showed = np.zeros((self.classes,), np.uint8)
        _capi.check(self._lib.vitdet_map_state(self._h, _capi.np_ptr(bboxes), _capi.np_ptr(labels), _capi.np_ptr(showed), self._stream()))
        return bboxes, labels, showed.astype(bool)

    @property
    def latest_positive_bboxes(self) -> np.ndarray:          # det.py:1286-1292
        return self._state()[0]

    @property
    def labels_quantity_per_image(self) -> np.ndarray:       # det.py:1296-1299
        return self._state()[1]

    @property
    def showed_up_classes(self) -> np.ndarray:               # det.py:1303-1305
        return self._state()[2]

    @property
    def iou_thresholds(self) -> np.ndarray:
        out = np.zeros(10, np.float32)
        _capi.check(self._lib.vitdet_map_iou_thresholds(self._h, _capi.np_ptr(out)))
        return out

    def launch_count(self) -> int:
        return int(self._lib.vitdet_map_launch_count(self._h))


# ------------------------------------------------------------------------------------------------
# the model object
# ------------------------------------------------------------------------------------------------
class Weight:
    """What `model.weights` yields: a named, shaped variable (keras: tf.Variable)."""

    def __init__(self, model: "VisionTransformerDetector", name: str, shape: tuple[int, ...]):
        self._model, self._name, self.shape = model, name, tuple(shape)

    @property
    def name(self) -> str:
        return self._name + ":0"

    def numpy(self) -> np.ndarray:
        return self._model._get_weight(self._name, self.shape)

    def assign(self, value) -> None:
        self._model._set_weight(self._name, np.asarray(value, dtype=np.float32))

    def __repr__(self) -> str:
        return f"<Weight '{self.name}' shape={self.shape} dtype=float32>"


class VisionTransformerDetector:
    """The object create_vision_transformer_detector returns (keras.Model in the reference,
    det.py:579-583).  All arithmetic happens in the CUDA library; this class owns the handle."""

    name = "vision_transformer_detector"

    def __init__(self, config: DetectorConfig, seed: int | None = 0, compute_mode: str | None = None):
        _check_inference_only(config.dropout, config.training)
        self.config = config
        self._lib = _capi.load()
        self._h = C.c_void_p()
        self._inflight = {}     # ticket -> (B, packed, the submitted buffers, boxes_original or None)
        cfg_c = config.to_c()
        _capi.check(self._lib.vitdet_create(C.byref(cfg_c), C.byref(self._h)))
        self.compute_mode = compute_mode or os.environ.get("VITDET_MODE", "bf16")
        self._specs = self._enumerate_weights()
        if seed is not None:
            for name, value in random_weights(config, seed).items():
                self._set_weight(name, value)

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.vitdet_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- shape facts ------------------------------------------------------------------------------
    @property
    def input_shape(self) -> tuple:
        return (None, *self.config.input_shape)

    @property
    def output_shape(self) -> tuple:
        return (None, Constants.MAX_DETECT_OBJECTS_QUANTITY.value, 6)

    @property
    def tokens(self) -> int:
        return int(self._lib.vitdet_tokens(self._h))

    def count_params(self) -> int:
        return int(self._lib.vitdet_count_params(self._h))

    def get_config(self) -> dict:
        return dataclasses.asdict(self.config)

    @classmethod
    def from_config(cls, config: dict, **kw) -> "VisionTransformerDetector":
        return cls(DetectorConfig(**config), **kw)

    # -- weights ----------------------------------------------------------------------------------
    def _enumerate_weights(self) -> list[tuple[str, tuple[int, ...]]]:
        n = self._lib.vitdet_num_weights(self._h)
        out = []
        buf = C.create_string_buffer(256)
        ndim = C.c_int()
        shape = (C.c_int64 * 4)()
        for i in range(n):
            _capi.check(self._lib.vitdet_weight_info(self._h, i, buf, 256, C.byref(ndim), shape))
            out.append((buf.value.decode(), tuple(int(shape[k]) for k in range(ndim.value))))
        return out

    def _set_weight(self, name: str, value: np.ndarray) -> None:
        v = np.ascontiguousarray(value, dtype=np.float32)
        shape = (C.c_int64 * max(v.ndim, 1))(*v.shape)
        _capi.check(self._lib.vitdet_set_weight(self._h, name.encode(), _capi.np_ptr(v), v.ndim, shape))

    def _get_weight(self, name: str, shape: tuple[int, ...]) -> np.ndarray:
        out = np.empty(shape, np.float32)
        _capi.check(self._lib.vitdet_get_weight(self._h, name.encode(), _capi.np_ptr(out), out.size))
        return out

    @property
    def weights(self) -> list[Weight]:
        return [Weight(self, n, s) for n, s in self._specs]

    def get_weights(self) -> list[np.ndarray]:
        return [self._get_weight(n, s) for n, s in self._specs]

    def set_weights(self, weights) -> None:
        """Accepts the Keras `get_weights()` list (positional, `model.weights` order) or a mapping
        from variable name (with or without ':0') to array."""
        if isinstance(weights, dict):
            known = {n for n, _ in self._specs}
            for name, value in weights.items():
                key = name[:-2] if name.endswith(":0") else name
                if key not in known:
                    raise ValueError(f"unknown weight name {name!r}")
                self._set_weight(key, value)
            return
        weights = list(weights)
        if len(weights) != len(self._specs):
            raise ValueError(f"You called `set_weights(weights)` on model {self.name!r} with a weight list of "
                             f"length {len(weights)}, but the model was expecting {len(self._specs)} weights.")
        for (name, shape), value in zip(self._specs, weights):
            value = np.asarray(value)
            if tuple(value.shape) != shape:
                raise ValueError(f"weight {name!r}: shape {tuple(value.shape)} is not compatible with {shape}")
            self._set_weight(name, value)

    def save_weights(self, path: str) -> None:
        np.savez(path, **{n: self._get_weight(n, s) for n, s in self._specs})

    def load_weights(self, path: str) -> None:
        with np.load(path) as z:
            self.set_weights({k: z[k] for k in z.files})

    def set_chunk(self, images_per_chunk: int) -> None:
        _capi.check(self._lib.vitdet_set_chunk(self._h, int(images_per_chunk)))

    def workspace_bytes(self, batch: int, compute_mode: str | None = None) -> int:
        return int(self._lib.vitdet_workspace_bytes(self._h, int(batch), self._mode(compute_mode)))

    # -- run-time switches and debug taps (parity tests, A/B measurements) ---------------------------
    def set_option(self, key: str, value: int) -> None:
        """'fuse_ln', 'fuse_tail', 'gemm_pair' (0/1/2), 'fp32_tc' — see include/vitdet_b200.h."""
        _capi.check(self._lib.vitdet_set_option(self._h, key.encode(), int(value)))

    def get_option(self, key: str) -> int:
        v = C.c_int()
        _capi.check(self._lib.vitdet_get_option(self._h, key.encode(), C.byref(v)))
        return int(v.value)

    def debug_taps(self, enable: bool = True) -> None:
        _capi.check(self._lib.vitdet_debug_taps(self._h, 1 if enable else 0))

    def debug_read(self, name: str, batch: int) -> np.ndarray:
        """One tap of the last forward (taps enabled): 'embedded_patches', 'block_<i>' -> (batch, tokens, D) float32;
        'head_last' -> (batch, 17, mlp_head_last_units)."""
        if name == "head_last":
            out = np.empty((batch, Constants.MAX_DETECT_OBJECTS_QUANTITY.value, self.config.head_units()[-1]), np.float32)
        else:
            out = np.empty((batch, self.config.tokens, self.config.embedding_dim), np.float32)
        _capi.check(self._lib.vitdet_debug_read(self._h, name.encode(), _capi.np_ptr(out), out.size))
        return out

    # -- measurement hooks ------------------------------------------------------------------------
    def profile_categories(self) -> list[str]:
        n = self._lib.vitdet_profile_num_categories(self._h)
        return [self._lib.vitdet_profile_category_name(i).decode() for i in range(n)]

    def profile_enable(self, categories: Iterable[str] | None) -> None:
        """CUDA-event timing around every launch of the named kernel categories (None / [] = off)."""
        names = self.profile_categories()
        mask = 0
        for c in categories or ():
            mask |= 1 << names.index(c)
        _capi.check(self._lib.vitdet_profile_enable(self._h, mask))

    def profile_read(self, reset: bool = True) -> dict[str, tuple[float, int]]:
        """{category: (total device ms, launches)} accumulated since the last reset."""
        out = {}
        ms, n = C.c_double(), C.c_int64()
        for i, name in enumerate(self.profile_categories()):
            _capi.check(self._lib.vitdet_profile_read(self._h, i, C.byref(ms), C.byref(n), 1 if reset else 0))
            if n.value:
                out[name] = (ms.value, n.value)
        return out

    def launch_count(self, reset: bool = True) -> int:
        return int(self._lib.vitdet_launch_count(self._h, 1 if reset else 0))

    # -- forward ----------------------------------------------------------------------------------
    def _mode(self, compute_mode: str | None = None) -> int:
        m = compute_mode or self.compute_mode
        if m not in _capi.MODES:
            raise ValueError(f"compute_mode must be one of {sorted(_capi.MODES)}, got {m!r}")
        return _capi.MODES[m]

    def _check_images(self, shape) -> int:
        want = tuple(self.config.input_shape)
        if len(shape) != 4 or tuple(shape[1:]) != want:
            raise ValueError(f'Input 0 of layer "{self.name}" is incompatible with the layer: expected '
                             f"shape=(None, {', '.join(map(str, want))}), found shape={tuple(shape)}")
        return int(shape[0])

    def detect(self, x, objectness_threshold=None, classification_threshold=None, strict=True, image_size=None,
               compute_mode: str | None = None, packed: bool = False, normalize_uint8: bool = False) -> DetectionRecords:
        """predict + transform_predictions + thresholds in one call (the decode is fused into the
        head's last Dense).  image_size defaults to the model's own input size.  packed=True also returns the
        (B*17, 13) float32 record block that the multi-GPU gather exchanges (parallel.RECORD_WIDTH).
        normalize_uint8=True: `x` holds uint8 pixels, normalised x / 127.5 - 1 inside the patch kernel (a quarter of the
        float32 copy); by default a uint8 array is cast to float32 like any other dtype, as Keras does."""
        B = self._check_images(x.shape)
        S = Constants.MAX_DETECT_OBJECTS_QUANTITY.value
        if image_size is None:
            image_size = self.config.input_shape[:2]
        params = _decode_params(objectness_threshold, classification_threshold, strict, image_size)
        mode = self._mode(compute_mode)
        xi, u8 = _model_input(x, normalize_uint8)
        if _is_torch_cuda(xi):
            import torch
            with torch.cuda.device(xi.device):
                recs, st = _alloc_records(B, S, packed, xi.device)
                logits = C.c_void_p(recs.logits.data_ptr())
                if u8:
                    _capi.check(self._lib.vitdet_forward_u8(self._h, C.c_void_p(xi.data_ptr()), B, logits, mode, C.byref(params),
                                                            C.byref(st), _torch_stream_ptr(xi.device)))
                else:
                    _capi.check(self._lib.vitdet_forward_decode(self._h, C.c_void_p(xi.data_ptr()), B, mode, C.byref(params), logits,
                                                                C.byref(st), _torch_stream_ptr(xi.device)))
            return recs
        recs, st = _alloc_records(B, S, packed)
        fn = self._lib.vitdet_predict_host_u8 if u8 else self._lib.vitdet_predict_host
        _capi.check(fn(self._h, _capi.np_ptr(xi), B, mode, C.byref(params), _capi.np_ptr(recs.logits), C.byref(st), None))
        return recs

    def submit(self, x, objectness_threshold=None, classification_threshold=None, strict=True, image_size=None,
               compute_mode: str | None = None, packed: bool = False, normalize_uint8: bool = False) -> int:
        """Asynchronous detect() for HOST arrays (vitdet_submit_host): stages and copies `x`, enqueues forward + decode +
        read-back and returns a ticket for collect().  Two submissions may be in flight; the copy of the second overlaps
        the compute of the first.  A page-locked `x` must stay alive until its ticket is collected."""
        B = self._check_images(np.shape(x))
        if image_size is None:
            image_size = self.config.input_shape[:2]
        params = _decode_params(objectness_threshold, classification_threshold, strict, image_size)
        xi, u8 = _model_input(x, normalize_uint8)
        ticket = C.c_int(-1)
        _capi.check(self._lib.vitdet_submit_host(self._h, _capi.np_ptr(xi), 1 if u8 else 0, B, self._mode(compute_mode), C.byref(params),
                                                 1 if packed else 0, None, C.byref(ticket)))
        return self._in_flight(ticket, B, packed, xi)

    def _in_flight(self, ticket: C.c_int, B: int, packed: bool, sources, boxes=None) -> int:
        """Registers a submission for collect(); `sources` stay alive until then, as a page-locked buffer is read
        asynchronously."""
        self._inflight[ticket.value] = (B, packed, sources, boxes)
        return ticket.value

    def collect(self, ticket: int) -> DetectionRecords:
        """Waits for a submit() ticket and returns its records as numpy arrays."""
        entry = self._inflight.pop(ticket, None)
        if entry is None:
            # not (or no longer) in flight: fail with the library's error type, like vitdet_collect itself does
            raise _capi.VitdetError(_capi.E_INVALID, f"collect: ticket {ticket} is not in flight")
        B, packed, _, boxes = entry
        recs, st = _alloc_records(B, Constants.MAX_DETECT_OBJECTS_QUANTITY.value, packed)
        recs.boxes_original = boxes
        _capi.check(self._lib.vitdet_collect(self._h, int(ticket), _capi.np_ptr(recs.logits), C.byref(st)))
        return recs

    # -- decoded images of any size ------------------------------------------------------------------
    @staticmethod
    def _image_list(images) -> tuple[list, bool]:
        """(the images as contiguous uint8 (h, w, 3) arrays or CUDA tensors, whether they are CUDA tensors); ValueError for
        anything the library would not take as it is."""
        imgs = list(images)
        if not imgs:
            raise ValueError("images must be a non-empty sequence of uint8 (h, w, 3) images")
        on_gpu = [_is_torch_cuda(im) for im in imgs]
        if any(on_gpu) and not all(on_gpu):
            raise ValueError("images mixes host arrays and CUDA tensors; pass one kind")
        out = []
        for i, im in enumerate(imgs):
            im = im if on_gpu[0] else np.asarray(im)
            if not _is_uint8(im):
                raise ValueError(f"image {i}: dtype {im.dtype}, expected uint8")
            if im.ndim != 3 or im.shape[2] != 3:
                raise ValueError(f"image {i}: shape {tuple(im.shape)}, expected (height, width, 3)")
            out.append(im.contiguous() if on_gpu[0] else np.ascontiguousarray(im))
        if on_gpu[0] and len({im.device for im in out}) != 1:
            raise ValueError("the images are on more than one device")
        return out, on_gpu[0]

    @staticmethod
    def _image_table(imgs, ptr) -> C.Array:
        return (_capi.Image * len(imgs))(*[_capi.Image(ptr(im), int(im.shape[0]), int(im.shape[1])) for im in imgs])

    def detect_images(self, images, objectness_threshold=None, classification_threshold=None, strict=True,
                      compute_mode: str | None = None, packed: bool = False) -> DetectionRecords:
        """detect() on decoded images of any size, what _get_image_tensor_coco (vision_transformer_utilities.py:418-449) feeds
        the model: every image is letterboxed to the model's input size (resize_with_pad, clip, / 127.5 - 1) inside the patch
        kernel.  images: a sequence of uint8 (h, w, 3) numpy arrays (one synchronous call) or of torch CUDA uint8 tensors on
        one device (asynchronous on torch's current stream, torch outputs).  Boxes are decoded at the model's input size;
        `boxes_original` (B, 17, 4) holds x0, y0, x1, y1 of every slot's box on its source image, in source pixels."""
        imgs, on_gpu = self._image_list(images)
        if not on_gpu:
            return self.collect(self.submit_images(imgs, objectness_threshold, classification_threshold, strict, compute_mode, packed))
        import torch
        B, S = len(imgs), Constants.MAX_DETECT_OBJECTS_QUANTITY.value
        params = _decode_params(objectness_threshold, classification_threshold, strict, self.config.input_shape[:2])
        table = self._image_table(imgs, lambda t: t.data_ptr())
        dev = imgs[0].device
        with torch.cuda.device(dev):
            recs, st = _alloc_records(B, S, packed, dev)
            recs.boxes_original = torch.empty((B, S, 4), dtype=torch.float32, device=dev)
            _capi.check(self._lib.vitdet_forward_images(self._h, table, B, self._mode(compute_mode), C.byref(params),
                                                        C.c_void_p(recs.logits.data_ptr()), C.byref(st),
                                                        C.c_void_p(recs.boxes_original.data_ptr()), _torch_stream_ptr(dev)))
        return recs

    def submit_images(self, images, objectness_threshold=None, classification_threshold=None, strict=True,
                      compute_mode: str | None = None, packed: bool = False) -> int:
        """Asynchronous detect_images() for host arrays (vitdet_submit_images_host), completed by collect(ticket); shares the
        two submission slots of submit().  Page-locked arrays must stay alive until their ticket is collected."""
        imgs, on_gpu = self._image_list(images)
        if on_gpu:
            raise ValueError("submit_images takes host arrays; detect_images runs CUDA tensors asynchronously already")
        B, S = len(imgs), Constants.MAX_DETECT_OBJECTS_QUANTITY.value
        params = _decode_params(objectness_threshold, classification_threshold, strict, self.config.input_shape[:2])
        boxes = np.empty((B, S, 4), np.float32)
        ticket = C.c_int(-1)
        _capi.check(self._lib.vitdet_submit_images_host(self._h, self._image_table(imgs, lambda a: a.ctypes.data), B,
                                                        self._mode(compute_mode), C.byref(params), 1 if packed else 0,
                                                        _capi.np_ptr(boxes), None, C.byref(ticket)))
        return self._in_flight(ticket, B, packed, imgs, boxes)

    # -- JPEG files ---------------------------------------------------------------------------------
    def detect_jpeg(self, files, objectness_threshold=None, classification_threshold=None, strict=True,
                    compute_mode: str | None = None, packed: bool = False, ratio=1) -> DetectionRecords:
        """detect_images() on JPEG files, decoded on the GPU bit-identically to PIL's Image.open(f).convert("RGB") (and
        tf.image.decode_jpeg): the same records, boxes_original included, as detect_images on the PIL-decoded images.
        files: a sequence of bytes-like objects (bytes, bytearray, memoryview, 1-D uint8 numpy arrays) or paths.  One
        synchronous call; a file outside baseline JPEG fails the call, naming it (VitdetError E_INVALID).
        ratio: 1, 2, 4, 8, "auto" or one of them per file: decode at 1 / ratio scale in the DCT domain, as
        tf.image.decode_jpeg(ratio=) and PIL's draft() do; "auto" picks what draft() picks for the letterbox size
        (jpeg_auto_ratio; 1 for every image up to about twice the model's input size).  The records are those of
        detect_images on the reduced decode, except boxes_original, which stays in the file's pixels."""
        return self.collect(self.submit_jpeg(files, objectness_threshold, classification_threshold, strict, compute_mode, packed,
                                             ratio))

    def submit_jpeg(self, files, objectness_threshold=None, classification_threshold=None, strict=True,
                    compute_mode: str | None = None, packed: bool = False, ratio=1) -> int:
        """Asynchronous detect_jpeg() (vitdet_submit_jpeg_host_scaled), completed by collect(ticket); shares the two
        submission slots of submit().  Page-locked files are read directly and must stay alive until their ticket is
        collected."""
        arrs = _jpeg_arrays(files)
        B, S = len(arrs), Constants.MAX_DETECT_OBJECTS_QUANTITY.value
        ratios = _jpeg_ratios(ratio, B, allow_auto=True)
        params = _decode_params(objectness_threshold, classification_threshold, strict, self.config.input_shape[:2])
        boxes = np.empty((B, S, 4), np.float32)
        ticket = C.c_int(-1)
        _capi.check(self._lib.vitdet_submit_jpeg_host_scaled(self._h, _jpeg_table(arrs), (C.c_int32 * B)(*ratios), B,
                                                             self._mode(compute_mode), C.byref(params), 1 if packed else 0,
                                                             _capi.np_ptr(boxes), None, C.byref(ticket)))
        return self._in_flight(ticket, B, packed, arrs, boxes)

    def predict(self, x, batch_size=None, verbose="auto", steps=None, callbacks=None, normalize_uint8: bool = False, **kwargs):
        """keras Model.predict: host array in, numpy (B, 17, 6) raw logits out.  `batch_size` only
        chunks the work in Keras; here the engine's own encoder micro-batch bounds memory, so it is
        accepted and ignored.  normalize_uint8: see detect()."""
        if _is_torch_cuda(x):
            return self(x, normalize_uint8=normalize_uint8).cpu().numpy()
        B = self._check_images(np.shape(x))
        xi, u8 = _model_input(x, normalize_uint8)
        logits = np.empty((B, Constants.MAX_DETECT_OBJECTS_QUANTITY.value, 6), np.float32)
        params = _decode_params(None, None, True, self.config.input_shape[:2])
        fn = self._lib.vitdet_predict_host_u8 if u8 else self._lib.vitdet_predict_host
        _capi.check(fn(self._h, _capi.np_ptr(xi), B, self._mode(), C.byref(params), _capi.np_ptr(logits), None, None))
        return logits

    def __call__(self, x, training=False, compute_mode: str | None = None, normalize_uint8: bool = False):
        """model(x, training=False): torch CUDA tensor in -> torch CUDA tensor out (asynchronous on
        torch's current stream); numpy in -> numpy out."""
        if training:
            raise NotImplementedError("training=True is outside the predict/decode path")
        if not _is_torch_cuda(x):
            return self.predict(x, normalize_uint8=normalize_uint8)
        import torch
        B = self._check_images(x.shape)
        xi, u8 = _model_input(x, normalize_uint8)
        with torch.cuda.device(xi.device):
            logits = torch.empty((B, Constants.MAX_DETECT_OBJECTS_QUANTITY.value, 6), dtype=torch.float32, device=xi.device)
            if u8:
                _capi.check(self._lib.vitdet_forward_u8(self._h, C.c_void_p(xi.data_ptr()), B, C.c_void_p(logits.data_ptr()),
                                                        self._mode(compute_mode), None, None, _torch_stream_ptr(xi.device)))
            else:
                _capi.check(self._lib.vitdet_forward(self._h, C.c_void_p(xi.data_ptr()), B, C.c_void_p(logits.data_ptr()),
                                                     self._mode(compute_mode), _torch_stream_ptr(xi.device)))
        return logits


def create_vision_transformer_detector(
        input_shape=None, patch_size=17, embedding_dim=28,
        encoder_num_heads=8, encoder_key_dim=40, dropout=None,
        encoder_mlp_quantities=8,
        encoder_repeat_times=8,
        mlp_head_last_units=136, mlp_head_dense_layers_quantity=7,
        mlp_head_dense_mish_block_repeats=1,
        use_mish=True,
        max_weight=10, clip_weight=True, training=None,
        *, seed: int | None = 0, compute_mode: str | None = None) -> VisionTransformerDetector:
    """Same signature and defaults as the reference (det.py:498-506).  Returns a model whose weights
    are Keras-default random-initialised (seed=None leaves them unset, for set_weights)."""
    if input_shape is None:
        input_shape = (*Constants.MODEL_IMAGE_SIZE.value, 3)
    if len(input_shape) != 3 or int(input_shape[2]) != 3:
        raise ValueError(f"input_shape must be (height, width, 3), got {tuple(input_shape)}")
    image_inputs = Input(shape=input_shape, name="images")
    embedded = transformer_preprocessor(inputs=image_inputs, patch_size=patch_size, embedding_dim=embedding_dim,
                                        max_weight=max_weight, clip_weight=clip_weight)
    encoded = transformer_encoder(embedded, use_mish=use_mish, num_heads=encoder_num_heads, key_dim=encoder_key_dim,
                                  dropout=dropout, mlp_quantities=encoder_mlp_quantities,
                                  repeat_times=encoder_repeat_times, max_weight=max_weight, clip_weight=clip_weight,
                                  training=training)
    head = mlp_head(encoder_outputs=encoded, use_mish=use_mish, mlp_head_last_units=mlp_head_last_units,
                    dense_layers_quantity=mlp_head_dense_layers_quantity,
                    dense_mish_block_repeats=mlp_head_dense_mish_block_repeats, dropout=dropout,
                    max_weight=max_weight, clip_weight=clip_weight, training=training)
    s = head.spec
    cfg = DetectorConfig(
        input_shape=tuple(s["input_shape"]), patch_size=s["patch_size"], embedding_dim=s["embedding_dim"],
        encoder_num_heads=s["encoder_num_heads"], encoder_key_dim=s["encoder_key_dim"], dropout=None,
        encoder_mlp_quantities=s["encoder_mlp_quantities"], encoder_repeat_times=s["encoder_repeat_times"],
        mlp_head_last_units=s["mlp_head_last_units"],
        mlp_head_dense_layers_quantity=s["mlp_head_dense_layers_quantity"],
        mlp_head_dense_mish_block_repeats=s["mlp_head_dense_mish_block_repeats"], use_mish=s["use_mish"],
        max_weight=max_weight, clip_weight=clip_weight, training=None)
    return VisionTransformerDetector(cfg, seed=seed, compute_mode=compute_mode)
