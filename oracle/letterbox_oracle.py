"""CPU ORACLE — test infrastructure, not product code (see vitdet_oracle.py for the rules).

The back-projection of detections made on letterboxed input onto the image the caller gave: the inverse of
tf.image.resize_with_pad as _get_image_tensor_coco (vision_transformer_utilities.py:418-449) applies it, whose geometry
vitdet_oracle.resize_with_pad_geometry restates.
"""
from __future__ import annotations

import numpy as np

from vitdet_oracle import MODEL_IMAGE_SIZE, resize_with_pad_geometry


def boxes_original(decoded: np.ndarray, source_size, target=MODEL_IMAGE_SIZE) -> np.ndarray:
    """Boxes of decoded slots (..., 6) of letterboxed input (cx, cy, h, w in target pixels) on the (height, width) source
    image: x0 = (cx - w/2 - pad_left) * (width / resized_width), likewise x1, y0, y1, then clipped to [0, width] /
    [0, height].  float32 with one rounding per operation in this order (no fused multiply-add), the library's decode
    restated bit for bit.  Returns (..., 4): x0, y0, x1, y1."""
    f = np.float32
    dec = np.asarray(decoded, dtype=f)
    h, w = (int(v) for v in source_size)
    rh, rw, ph, pw = resize_with_pad_geometry(h, w, int(target[0]), int(target[1]))
    hs, ws = f(h) / f(rh), f(w) / f(rw)
    cx, cy, bh, bw = dec[..., 2], dec[..., 3], dec[..., 4], dec[..., 5]
    half_h, half_w = bh / f(2), bw / f(2)

    def clip(v, hi):            # fmaxf / fminf: a NaN operand yields the other one
        return np.fmin(np.fmax(v, f(0)), f(hi))

    x0 = clip(((cx - half_w) - f(pw)) * ws, w)
    y0 = clip(((cy - half_h) - f(ph)) * hs, h)
    x1 = clip(((cx + half_w) - f(pw)) * ws, w)
    y1 = clip(((cy + half_h) - f(ph)) * hs, h)
    return np.stack([x0, y0, x1, y1], axis=-1).astype(f)


def letterbox_box(box, source_size, target=MODEL_IMAGE_SIZE) -> np.ndarray:
    """The forward map: a source-pixel box (x0, y0, x1, y1) -> (cx, cy, h, w) in letterboxed target pixels, float64
    (resize_with_pad scales by resized / source size, then shifts by the bar)."""
    h, w = (int(v) for v in source_size)
    rh, rw, ph, pw = resize_with_pad_geometry(h, w, int(target[0]), int(target[1]))
    x0, y0, x1, y1 = (float(v) for v in box)
    sx, sy = rw / w, rh / h
    return np.array([(x0 + x1) / 2 * sx + pw, (y0 + y1) / 2 * sy + ph, (y1 - y0) * sy, (x1 - x0) * sx])
