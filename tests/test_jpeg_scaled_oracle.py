"""CPU tests of the JPEG decode at 1/2, 1/4 and 1/8 scale: the numpy oracle (jpeg_scaled_oracle.decode(data, ratio=r)) against
PIL's draft decode (libjpeg-turbo's scaled IDCTs, what tf.image.decode_jpeg(ratio=r) returns) bit for bit, the library's
auto ratio against PIL's draft choice, the boxes_original factor of a reduced decode, and a clean sm_100a compile."""
import io
import os
import subprocess

import numpy as np
import pytest
from PIL import Image

from _util import oracle  # noqa: F401  (puts oracle/ on the path)
import _jpeg_corpus as jc
import jpeg_oracle as jo
import jpeg_scaled_oracle as js
import letterbox_oracle as lb
from vitdet_oracle import resize_with_pad_geometry
from vision_transformer_detector_b200 import _capi, build
from vision_transformer_detector_b200.vision_transformer_detector import _jpeg_ratios
from vision_transformer_detector_b200.vision_transformer_utilities import jpeg_auto_ratio

RATIOS = (2, 4, 8)


def boundary_files():
    """4:2:2 and 4:2:0 files whose chroma, at some ratio, is 1, 2 or 3 samples wide: replication up to 2, fancy
    upsampling from 3 (4:2:2 chroma at ratio r is ceil(w / 2r) wide)."""
    out = []
    for w in (4, 8, 12, 16, 24, 17, 33, 40, 48):
        for mode in ("422", "420"):
            out.append((f"20x{w}-{mode}", jc.encode(jc.photo(20, w, w), mode, 90)))
    return out


FILES = jc.corpus() + boundary_files()


def pil_draft(data, r):
    """PIL's decode after draft("RGB", (max(1, w // r), max(1, h // r))), and the scale PIL chose."""
    im = Image.open(io.BytesIO(data))
    w, h = im.size
    im.draft("RGB", (max(1, w // r), max(1, h // r)))
    return np.asarray(im.convert("RGB")), im.decoderconfig[0]


def test_oracle_scaled_decode_equals_pil_draft():
    compared, skipped = 0, 0
    for name, data in FILES:
        for r in RATIOS:
            ref, scale = pil_draft(data, r)
            if scale != r:                   # the image is too small for PIL to be asked for this scale
                skipped += 1
                continue
            got = js.decode(data, ratio=r)
            assert got.shape == ref.shape and np.array_equal(got, ref), (name, r)
            compared += 1
    # every file at least 8 pixels on each side is compared at every ratio; only tiny ones are skipped
    assert compared >= 3 * sum(1 for _, d in FILES if min(jo.info(d)[:2]) >= 8), compared
    assert skipped == sum(1 for _, d in FILES for r in RATIOS if min(jo.info(d)[:2]) < r), skipped


def test_boundary_files_cover_replication_and_fancy_upsampling():
    widths = set()
    for _, data in boundary_files():
        j = jo.parse(data)
        for r in RATIOS:
            g = js.scaled_geometry(j, r)
            if g["comps"][1]["he"] == 2 and g["k"] > 1:
                widths.add(g["comps"][1]["dw"])
    assert {1, 2, 3} <= widths


def test_scaled_geometry_follows_jdmaster():
    j420 = jo.parse(jc.encode(jc.photo(48, 64, 1), "420", 90))
    j422 = jo.parse(jc.encode(jc.photo(48, 64, 1), "422", 90))
    # 4:2:0 chroma takes 8 x 8 blocks at ratio 2, 4 x 4 at 4 and 2 x 2 at 8, and is never upsampled
    assert [js.scaled_geometry(j420, r)["comps"][1]["size"] for r in RATIOS] == [8, 4, 2]
    assert all(js.scaled_geometry(j420, r)["comps"][1]["he"] == 1 for r in RATIOS)
    # 4:2:2 chroma keeps the luma's size and is upsampled horizontally
    assert [js.scaled_geometry(j422, r)["comps"][1]["size"] for r in RATIOS] == [4, 2, 1]
    assert all((js.scaled_geometry(j422, r)["comps"][1]["he"], js.scaled_geometry(j422, r)["comps"][1]["ve"]) == (2, 1)
               for r in RATIOS)


def test_one_eighth_luma_is_the_dc_alone():
    data = jc.encode(jc.photo(64, 48, 5), "grey", 85)
    j = jo.parse(data)
    coef = jo.coefficients(j)
    dc = coef[:, 0].reshape(j["mcuy"], j["mcux"]) * j["quant"][0][0]
    assert np.array_equal(js.decode(data, ratio=8)[..., 0], jo.range_limit((dc + 4) >> 3))


def _size_sweep():
    edges = [1, 2, 7, 100, 303, 304, 607, 608, 609, 1215, 1216, 1217, 2431, 2432, 2433, 3024, 4032, 4863, 4864, 4865, 6000, 8000]
    sizes = {(h, w) for h in edges for w in edges if h <= 6000 and w <= 8000}
    sizes |= {(w, h) for h, w in sizes if w <= 6000}                                       # both orientations
    for s in (2, 4, 8):                  # sizes landing exactly on s * resized size, and one pixel either side
        for d in (-1, 0, 1):
            sizes |= {(608 * s + d, 608 * s + d), (456 * s + d, 608 * s + d), (608 * s + d, 456 * s + d)}
    return sorted(sizes)


def _pil_draft_scale(h, w, rh, rw):
    """The scale PIL's draft("RGB", (rw, rh)) picks for an h x w file: a small file with its frame header patched."""
    d = bytearray(jc.encode(jc.photo(8, 8, 0), "420", 90))
    for _, m, a, _ in jc.segments(bytes(d)):
        if m == 0xC0:
            d[a + 1:a + 3] = h.to_bytes(2, "big")
            d[a + 3:a + 5] = w.to_bytes(2, "big")
    im = Image.open(io.BytesIO(bytes(d)))
    assert im.size == (w, h)
    im.draft("RGB", (rw, rh))
    return im.decoderconfig[0]


@pytest.mark.parametrize("target", [(608, 608), (60, 130)])
def test_auto_ratio_equals_pil_draft_choice(target):
    seen = set()
    for h, w in _size_sweep():
        rh, rw, _, _ = resize_with_pad_geometry(h, w, *target)
        got = jpeg_auto_ratio(h, w, target)
        assert got == js.auto_ratio(h, w, rh, rw), (h, w)
        if rh > 0 and rw > 0:
            assert got == _pil_draft_scale(h, w, rh, rw), (h, w)
        seen.add(got)
    assert seen == {1, 2, 4, 8}
    # COCO-size files stay at ratio 1 for the default model
    assert jpeg_auto_ratio(480, 640) == jpeg_auto_ratio(640, 640) == jpeg_auto_ratio(1000, 1200) == 1


def test_auto_ratio_rejects_non_positive_sizes():
    assert _capi.load().vitdet_jpeg_auto_ratio(0, 10, 608, 608) == _capi.E_INVALID
    assert _capi.load().vitdet_jpeg_auto_ratio(10, 10, 608, -1) == _capi.E_INVALID


def test_boxes_original_factor():
    rng = np.random.default_rng(3)
    boxes = np.stack([rng.uniform(0, 600, 50), rng.uniform(0, 450, 50), rng.uniform(0, 600, 50), rng.uniform(0, 450, 50)],
                     -1).astype(np.float32)
    # ratio 1: the factor is exactly 1, the boxes come back bit for bit
    assert np.array_equal(js.boxes_to_file(boxes, (450, 600), (450, 600)), boxes)
    # ratio 4 on a 1799 x 2400 file decoded to 450 x 600: scaled by the size ratio and clipped to the file
    got = js.boxes_to_file(boxes, (450, 600), (1799, 2400))
    assert np.all(got >= 0) and np.all(got[:, 0::2] <= 2400) and np.all(got[:, 1::2] <= 1799)
    sx, sy = np.float32(2400) / np.float32(600), np.float32(1799) / np.float32(450)
    back = got / np.array([sx, sy, sx, sy], np.float32)
    np.testing.assert_allclose(back, boxes, rtol=1e-6, atol=1e-4)
    # through the letterbox: a box on the reduced decode, mapped into its letterbox, back, and on to the file's pixels
    dec = np.zeros((1, 6), np.float32)
    dec[0, 2:] = lb.letterbox_box([50, 30, 300, 225], (450, 600))
    on_file = js.boxes_to_file(lb.boxes_original(dec, (450, 600)), (450, 600), (1799, 2400))
    np.testing.assert_allclose(on_file[0], np.array([50, 30, 300, 225]) * [4, 1799 / 450, 4, 1799 / 450], rtol=1e-5)


@pytest.mark.parametrize("bad", [3, 0, "x", True, 2.0, None, [1, 2]])
def test_malformed_ratio_raises_value_error(bad):
    with pytest.raises(ValueError):
        _jpeg_ratios(bad, 3, allow_auto=True)


def test_auto_is_not_a_decode_jpeg_ratio():
    with pytest.raises(ValueError):
        _jpeg_ratios("auto", 2, allow_auto=False)
    assert _jpeg_ratios([1, "auto", 8], 3, allow_auto=True) == [1, 0, 8]


def test_jpeg_source_compiles_for_sm100a_without_warnings():
    nvcc = build._nvcc()
    csrc = os.path.join(os.path.dirname(build.__file__), "csrc")
    out = subprocess.run([nvcc, *build.NVCC_FLAGS, "-Xptxas", "-v", "-I", build.INCLUDE, "-I", csrc, "-cubin", "-o", os.devnull,
                          os.path.join(csrc, "jpeg.cu")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    log = out.stdout + out.stderr
    assert "warning" not in log.lower(), log
    lines = log.splitlines()
    i = next(n for n, line in enumerate(lines) if "Compiling entry function" in line and "jpeg_idct_kernel" in line)
    assert " 0 bytes spill stores" in lines[i + 2], lines[i:i + 4]
