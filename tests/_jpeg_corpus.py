"""Seeded JPEG test files, encoded by PIL: every accepted layout, the files the decoder must reject, and a file with
corrupt entropy data (tests/test_jpeg_oracle.py on the CPU, tests/test_gpu_jpeg.py on the GPU)."""
import io

import numpy as np
from PIL import Image

SIZES = [(1, 1), (3, 7), (8, 8), (16, 16), (9, 17), (47, 33), (48, 64), (90, 120), (131, 97)]     # (height, width)
MODES = {"444": 0, "422": 1, "420": 2, "grey": None}                                            # PIL subsampling
QUALITIES = (50, 75, 95, 100)


def photo(h, w, seed):
    """Smooth colour gradients with noise: photo-like content that exercises every DCT frequency."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    f = rng.uniform(0.05, 0.5, (3, 2))
    base = np.stack([128 + 90 * np.sin(xx * f[c, 0] + c) * np.cos(yy * f[c, 1] + 2 * c) for c in range(3)], -1)
    return np.clip(base + rng.normal(0, 18, (h, w, 3)), 0, 255).astype(np.uint8)


def contrast(h, w):
    """A black / white checkerboard of 1-pixel cells with saturated colour bars: the IDCT overshoots [0, 255]."""
    yy, xx = np.mgrid[0:h, 0:w]
    im = np.where(((yy + xx) & 1)[..., None] == 1, 255, 0).astype(np.uint8).repeat(3, -1)
    im[: h // 3, :, 1:] = 0
    im[h // 3: 2 * h // 3, :, ::2] = 0
    return im


def encode(img, mode, quality, **kw):
    b = io.BytesIO()
    if mode == "grey":
        Image.fromarray(img).convert("L").save(b, "JPEG", quality=quality, **kw)
    else:
        Image.fromarray(img).save(b, "JPEG", quality=quality, subsampling=MODES[mode], **kw)
    return b.getvalue()


def segments(data):
    """[(offset of the marker's FF, marker, payload start, payload end)] up to and including SOS."""
    out, p = [], 2
    while p < len(data):
        m = data[p + 1]
        ln = data[p + 2] << 8 | data[p + 3]
        out.append((p, m, p + 4, p + 2 + ln))
        if m == 0xDA:
            break
        p += 2 + ln
    return out


def rgb_ids(data):
    """The file without its JFIF APP0 and with component ids 'R', 'G', 'B': libjpeg then reads the samples as RGB."""
    d = bytearray(data)
    for p, m, a, e in reversed(segments(data)):
        if m == 0xC0:
            for c in range(3):
                d[a + 6 + 3 * c] = b"RGB"[c]
        elif m == 0xDA:
            for c in range(3):
                d[a + 1 + 2 * c] = b"RGB"[c]
        elif m == 0xE0:
            del d[p:e]
    return bytes(d)


def fill_before_stuffed_zero(data):
    """The file with a fill byte before its first stuffed zero (FF 00 -> FF FF 00): the same pixels for libjpeg."""
    sos_end = [e for _, m, _, e in segments(data) if m == 0xDA][0]
    p = data.index(b"\xFF\x00", sos_end)
    return data[:p] + b"\xFF" + data[p:]


def all_ones_code(data):
    """The file with a DHT before its scan that redefines DC table 0 so that its last code is all ones (3 bits: 111),
    which jpeg_make_d_derived_tbl refuses."""
    sos = [p for p, m, _, _ in segments(data) if m == 0xDA][0]
    table = bytes([0x00]) + bytes([0, 1, 6] + [0] * 13) + bytes(range(7))
    dht = b"\xFF\xC4" + (2 + len(table)).to_bytes(2, "big") + table
    return data[:sos] + dht + data[sos:]


def corpus():
    """[(name, bytes)] of accepted files."""
    files = []
    for i, (h, w) in enumerate(SIZES):
        for j, mode in enumerate(MODES):
            q = QUALITIES[(i + j) % len(QUALITIES)]
            files.append((f"{h}x{w}-{mode}-q{q}", encode(photo(h, w, 100 * i + j), mode, q)))
    for mode in MODES:
        files.append((f"48x64-{mode}-q100", encode(photo(48, 64, 7), mode, 100)))
        files.append((f"16x16-{mode}-contrast", encode(contrast(16, 16), mode, 100)))
        files.append((f"47x33-{mode}-optimize", encode(photo(47, 33, 8), mode, 75, optimize=True)))
    files.append(("47x33-420-contrast", encode(contrast(47, 33), "420", 95)))
    files.append(("48x64-420-restart-blocks", encode(photo(48, 64, 9), "420", 85, restart_marker_blocks=3)))
    files.append(("47x33-444-restart-rows", encode(photo(47, 33, 10), "444", 90, restart_marker_rows=1)))
    files.append(("9x17-grey-restart-blocks", encode(photo(9, 17, 11), "grey", 80, restart_marker_blocks=1)))
    files.append(("131x97-422-restart-rows-optimize", encode(photo(131, 97, 12), "422", 60, restart_marker_rows=2, optimize=True)))
    files.append(("47x33-444-rgb-ids", rgb_ids(encode(photo(47, 33, 13), "444", 90))))
    files.append(("48x64-420-rgb-ids", rgb_ids(encode(photo(48, 64, 14), "420", 90))))
    files.append(("48x64-420-fill-before-stuffed-zero", fill_before_stuffed_zero(encode(photo(48, 64, 15), "420", 95))))
    return files


def _patch_sof(data, offset, value):
    d = bytearray(data)
    for p, m, a, e in segments(data):
        if m == 0xC0:
            d[a + offset] = value
    return bytes(d)


def rejected():
    """[(name, bytes, a fragment of the reason)] of files outside baseline JPEG."""
    base = encode(photo(48, 64, 21), "420", 85)
    b = io.BytesIO()
    Image.fromarray(photo(48, 64, 22)).save(b, "JPEG", quality=85, progressive=True)
    progressive = b.getvalue()
    b = io.BytesIO()
    Image.fromarray(photo(48, 64, 23)).convert("CMYK").save(b, "JPEG", quality=85)
    cmyk = b.getvalue()
    sof9 = bytearray(base)
    sof9[[p for p, m, _, _ in segments(base) if m == 0xC0][0] + 1] = 0xC9
    sos = [p for p, m, _, _ in segments(base) if m == 0xDA][0]
    b = io.BytesIO()
    Image.fromarray(photo(8, 8, 24)).save(b, "PNG")
    return [
        ("progressive", progressive, "progressive"),
        ("cmyk", cmyk, "4 components"),
        ("sof9", bytes(sof9), "arithmetic"),
        ("12-bit", _patch_sof(base, 0, 12), "12-bit"),
        ("sampling-1x2", _patch_sof(base, 7, 0x12), "sampling"),
        ("truncated-before-sos", base[:sos], "truncated"),
        ("not-a-jpeg", b.getvalue(), "not a JPEG"),
        ("all-ones-huffman-code", all_ones_code(base), "bad Huffman table"),
    ]


def flipped():
    """A 4:2:0 file with bytes flipped inside its entropy-coded data; no marker is created or destroyed."""
    d = bytearray(encode(photo(48, 64, 31), "420", 85))
    sos_end = [e for _, m, _, e in segments(bytes(d)) if m == 0xDA][0]
    rng = np.random.default_rng(5)
    for p in sorted(rng.choice(np.arange(sos_end + 4, len(d) - 8), 12, replace=False)):
        if d[p - 1] != 0xFF and d[p] != 0xFF and d[p] ^ 0x5A != 0xFF and d[p + 1] != 0x00:
            d[p] ^= 0x5A
    return bytes(d)
