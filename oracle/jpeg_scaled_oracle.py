"""CPU ORACLE — test infrastructure, not product code (see vitdet_oracle.py for the rules).

The JPEG decode at 1/2, 1/4 and 1/8 scale in the DCT domain, as csrc/jpeg.cu runs it: libjpeg-turbo's scaled decode (its
scale_num / scale_denom = 1 / ratio), which is what PIL gives after Image.draft() and tf.image.decode_jpeg(ratio=) returns.
It builds on jpeg_oracle.py's header parse, entropy decode, ISLOW IDCT, upsampling and colour conversion.  Stages:
  auto_ratio()        the ratio PIL's draft() picks for the letterbox size (detect_jpeg(ratio="auto"))
  scaled_geometry()   jdmaster.c: output size and each component's DCT scaled size, scaled size and expansion factors
  idct_4x4/2x2/1x1()  jidctred.c's reduced IDCTs
  scaled_planes()     the component planes at each component's scaled block size
  scaled_upsample()   jdsample.c at reduced scale: fancy only where the luma's scaled size is above 1
  decode()            the whole decode; ratio 1 is jpeg_oracle.decode
  boxes_to_file()     boxes_original of a reduced decode carried to the file's pixels
"""
from __future__ import annotations

import numpy as np

from jpeg_oracle import coefficients, idct_islow, parse, pixels_from_coefficients, range_limit, upsample, ycc_to_rgb


def decode(data: bytes, ratio=1, L=None) -> np.ndarray:
    """uint8 RGB of an accepted file decoded at 1 / ratio scale, (ceil(h / ratio), ceil(w / ratio), 3): what PIL gives after
    im.draft("RGB", (w // ratio, h // ratio)) and tf.image.decode_jpeg(ratio=ratio) returns.  ratio 1 is the full decode."""
    if ratio not in (1, 2, 4, 8):
        raise ValueError(f"ratio must be 1, 2, 4 or 8, got {ratio!r}")
    j = parse(data)
    if ratio == 1:
        return pixels_from_coefficients(j, coefficients(j, L))
    return scaled_pixels_from_coefficients(j, coefficients(j, L), ratio)


def auto_ratio(height: int, width: int, resized_height: int, resized_width: int) -> int:
    """The ratio PIL's draft(mode, (resized_width, resized_height)) picks: the largest of 8, 4, 2, 1 that is at most
    min(width // resized_width, height // resized_height); 1 when a resized size is not positive."""
    if resized_height <= 0 or resized_width <= 0:
        return 1
    scale = min(width // resized_width, height // resized_height)
    return next(s for s in (8, 4, 2, 1) if s <= max(scale, 1))


def scaled_geometry(j, ratio):
    """jdmaster.c jpeg_core_output_dimensions at scale 1 / ratio: the output size ceil(h / ratio) x ceil(w / ratio) and,
    per component, its DCT scaled size (the luma's k = 8 / ratio, doubled while both sampling ratios allow it: so 4:2:0
    chroma takes 8 x 8 blocks at ratio 2 and is not upsampled), its scaled ("downsampled") size and its expansion
    factors to the output (jdsample.c h_out_group / h_in_group)."""
    H, W = j["height"], j["width"]
    hmax, vmax = j["hmax"], j["vmax"]
    k = 8 // ratio
    comps = []
    for c in range(j["ncomp"]):
        h, v = j["hs"][c], j["vs"][c]
        ss = k
        while ss < 8 and (hmax * k) % (h * ss * 2) == 0 and (vmax * k) % (v * ss * 2) == 0:
            ss *= 2
        comps.append(dict(size=ss, dw=-(-W * h * ss // (hmax * 8)), dh=-(-H * v * ss // (vmax * 8)),
                          he=hmax * k // (h * ss), ve=vmax * k // (v * ss)))
    return dict(height=-(-H // ratio), width=-(-W // ratio), k=k, comps=comps)


def idct_4x4(coef, qtab):
    """[n, 64] coefficients -> [n, 4, 4] uint8: jidctred.c jpeg_idct_4x4 (rows and columns 0-3, 5-7; 4 is not read)."""
    x = (np.asarray(coef, np.int64) * np.asarray(qtab, np.int64)).reshape(-1, 8, 8)

    def one(s0, s1, s2, s3, s5, s6, s7, shift):
        tmp0 = s0 << 14                                                     # CONST_BITS + 1
        tmp2 = s2 * 15137 + s6 * -6270
        t10, t12 = tmp0 + tmp2, tmp0 - tmp2
        z1, z2, z3, z4 = s7, s5, s3, s1
        o0 = z1 * -1730 + z2 * 11893 + z3 * -17799 + z4 * 8697
        o2 = z1 * -4176 + z2 * -4926 + z3 * 7373 + z4 * 20995
        r = 1 << (shift - 1)
        return [(t10 + o2 + r) >> shift, (t12 + o0 + r) >> shift, (t12 - o0 + r) >> shift, (t10 - o2 + r) >> shift]

    cols = one(*[x[:, r, :] for r in (0, 1, 2, 3, 5, 6, 7)], 12)             # CONST_BITS - PASS1_BITS + 1
    ws = np.stack(cols, 1)                                                  # [n, 4 rows, 8 columns]
    rows = one(*[ws[:, :, c] for c in (0, 1, 2, 3, 5, 6, 7)], 19)           # CONST_BITS + PASS1_BITS + 3 + 1
    return np.stack([range_limit(r) for r in rows], 2)


def idct_2x2(coef, qtab):
    """[n, 64] coefficients -> [n, 2, 2] uint8: jidctred.c jpeg_idct_2x2 (rows and columns 0, 1, 3, 5, 7)."""
    x = (np.asarray(coef, np.int64) * np.asarray(qtab, np.int64)).reshape(-1, 8, 8)

    def one(s0, s1, s3, s5, s7, shift):
        t10 = s0 << 15                                                      # CONST_BITS + 2
        t0 = s7 * -5906 + s5 * 6967 + s3 * -10426 + s1 * 29692
        r = 1 << (shift - 1)
        return [(t10 + t0 + r) >> shift, (t10 - t0 + r) >> shift]

    ws = np.stack(one(*[x[:, r, :] for r in (0, 1, 3, 5, 7)], 13), 1)       # CONST_BITS - PASS1_BITS + 2
    rows = one(*[ws[:, :, c] for c in (0, 1, 3, 5, 7)], 20)                 # CONST_BITS + PASS1_BITS + 3 + 2
    return np.stack([range_limit(r) for r in rows], 2)


def idct_1x1(coef, qtab):
    """[n, 64] coefficients -> [n, 1, 1] uint8: jidctred.c jpeg_idct_1x1, the DC alone: range_limit((dc q0 + 4) >> 3)."""
    dc = np.asarray(coef, np.int64)[:, 0] * int(qtab[0])
    return range_limit((dc + 4) >> 3).reshape(-1, 1, 1)


IDCT = {8: idct_islow, 4: idct_4x4, 2: idct_2x2, 1: idct_1x1}


def scaled_planes(j, coef, g):
    """Component planes [c] of (mcuy * v * size, mcux * h * size) uint8 at each component's DCT scaled size."""
    out = []
    bpm = len(j["blocks"])
    for c in range(j["ncomp"]):
        h, v, k = j["hs"][c], j["vs"][c], g["comps"][c]["size"]
        pl = np.zeros((j["mcuy"] * v * k, j["mcux"] * h * k), np.uint8)
        for u, (bc, bx, by) in enumerate(j["blocks"]):
            if bc != c:
                continue
            px = IDCT[k](coef[u::bpm], j["quant"][c]).reshape(j["mcuy"], j["mcux"], k, k)
            for my in range(j["mcuy"]):
                for mx in range(j["mcux"]):
                    y0, x0 = (my * v + by) * k, (mx * h + bx) * k
                    pl[y0:y0 + k, x0:x0 + k] = px[my, mx]
        out.append(pl)
    return out


def scaled_upsample(plane, comp, H, W, fancy):
    """One chroma plane to the (H, W) output: as upsample(), with the component's own expansion factors and scaled
    size.  jinit_upsampler upsamples fancily only when the luma's scaled size is above 1 and the component is more than 2
    samples wide; otherwise it replicates."""
    he, ve, dw = comp["he"], comp["ve"], comp["dw"]
    if he == 1 and ve == 1:
        return plane[:H, :W]
    assert he == 2 and ve in (1, 2)
    if not fancy or dw <= 2:
        return plane[(np.arange(H) // ve)[:, None], (np.arange(W) >> 1)[None, :]]
    # dw = ceil(W / he) and dh = ceil(H / ve): upsample() at an image of the output's size, sampled (he, ve) : (1, 1)
    return upsample(dict(height=H, width=W, hmax=he, vmax=ve, hs=[1, 1], vs=[1, 1]), plane, 1)


def scaled_pixels_from_coefficients(j, coef, ratio):
    g = scaled_geometry(j, ratio)
    pl = scaled_planes(j, coef, g)
    H, W = g["height"], g["width"]
    if j["ncomp"] == 1:
        y = pl[0][:H, :W]
        return np.stack([y, y, y], -1)
    fancy = g["k"] > 1
    y = pl[0][:H, :W]
    cb, cr = (scaled_upsample(pl[c], g["comps"][c], H, W, fancy) for c in (1, 2))
    if j["space"] == "rgb":
        return np.stack([y, cb, cr], -1)
    return ycc_to_rgb(y, cb, cr)


def boxes_to_file(boxes, decoded_size, file_size) -> np.ndarray:
    """boxes_original of a JPEG decoded at reduced scale (detect_jpeg(ratio=...)): the boxes on the (height, width)
    decoded image, as letterbox_oracle.boxes_original() gives them, carried to the file's (height, width) pixels: x times
    float32(width) / float32(decoded width) (y likewise), one rounding each, then clipped to [0, width] / [0, height].
    At ratio 1 the factor is exactly 1 and the boxes come back unchanged."""
    f = np.float32
    b = np.asarray(boxes, dtype=f)
    (dh, dw), (h, w) = ((int(v) for v in decoded_size), (int(v) for v in file_size))
    sx, sy = f(w) / f(dw), f(h) / f(dh)
    scale = np.array([sx, sy, sx, sy], f)
    hi = np.array([w, h, w, h], f)
    return np.fmin(np.fmax(b * scale, f(0)), hi).astype(f)
