"""GPU tests of the JPEG decode at 1/2, 1/4 and 1/8 scale (vitdet_decode_jpeg_scaled, vitdet_submit_jpeg_host_scaled):
decode_jpeg(ratio=r) must give PIL's draft decode bit for bit, and detect_jpeg / submit_jpeg(ratio=...) exactly the records
of detect_images on that decode, with boxes_original carried to the file's pixels as the oracle states."""
import ctypes as C
import io

import numpy as np
import pytest
from PIL import Image

from _util import build_model, tiny_config
import _jpeg_corpus as jc
import jpeg_oracle as jo
import jpeg_scaled_oracle as js
import vision_transformer_detector_b200 as vd
from vision_transformer_detector_b200 import _capi
from vision_transformer_detector_b200.vision_transformer_detector import _jpeg_table
from vision_transformer_detector_b200.vision_transformer_utilities import _decoder, decode_jpeg, jpeg_auto_ratio

pytestmark = pytest.mark.gpu

FIELDS = ("logits", "decoded", "class_id", "class_conf", "keep", "corners", "packed")


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def _assert_same(a, b, fields=FIELDS + ("boxes_original",)):
    for f in fields:
        assert np.array_equal(_np(getattr(a, f)), _np(getattr(b, f))), f


def _size(data):
    return jo.info(data)[:2]


def _reduced(data, r):
    """The reference decode at 1 / r: PIL's draft decode where PIL can be asked for that scale, else the oracle."""
    im = Image.open(io.BytesIO(data))
    if r == 1:
        return np.asarray(im.convert("RGB"))
    w, h = im.size
    im.draft("RGB", (max(1, w // r), max(1, h // r)))
    if im.decoderconfig[0] == r:
        return np.asarray(im.convert("RGB"))
    return js.decode(data, ratio=r)


def _coco_files(seed=0):
    sizes = [((480, 640), "420", 85), ((427, 640), "444", 92), ((612, 612), "grey", 75), ((1000, 1500), "422", 95)]
    return [jc.encode(jc.photo(h, w, seed + i), mode, q) for i, ((h, w), mode, q) in enumerate(sizes)]


def _camera_files():
    """4032 x 3024 4:2:0, 3024 x 4032 4:2:2 and 4000 x 3000 grey (width x height), encoded by PIL."""
    return [jc.encode(jc.photo(3024, 4032, 41), "420", 90), jc.encode(jc.photo(4032, 3024, 42), "422", 85),
            jc.encode(jc.photo(3000, 4000, 43), "grey", 92)]


def test_decode_jpeg_scaled_equals_pil_draft():
    files = [d for _, d in jc.corpus()] + _coco_files() + _camera_files()
    compared = 0
    for r in (2, 4, 8):
        got = decode_jpeg(files, ratio=r)
        for i, (g, d) in enumerate(zip(got, files)):
            h, w = _size(d)
            assert tuple(g.shape) == (-(-h // r), -(-w // r), 3), (i, r)
            assert np.array_equal(g.cpu().numpy(), _reduced(d, r)), (i, r)
            compared += 1
    assert compared == 3 * len(files)


def test_mixed_ratios_equal_per_ratio_calls():
    files = _coco_files(seed=5) + [jc.encode(jc.photo(131, 97, 6), "422", 80, restart_marker_rows=2), jc.flipped()]
    ratios = [8, 1, 4, 2, 2, 4]
    per_ratio = {r: decode_jpeg(files, ratio=r) for r in set(ratios)}
    got = decode_jpeg(files, ratio=ratios)
    for i, r in enumerate(ratios):
        assert np.array_equal(got[i].cpu().numpy(), per_ratio[r][i].cpu().numpy()), i
    # ratio 1 through the scaled entry point, which decode_jpeg calls, is the full-size entry point's decode
    import torch
    full = decode_jpeg(files, ratio=[1] * len(files))
    offs = [0]
    for g in full[:-1]:
        offs.append(offs[-1] + (g.numel() + 255) // 256 * 256)
    buf = torch.zeros(offs[-1] + full[-1].numel(), dtype=torch.uint8, device="cuda")
    arrs = [np.frombuffer(d, np.uint8) for d in files]
    lib = _capi.load()
    _capi.check(lib.vitdet_decode_jpeg(_decoder(torch.cuda.current_device()), _jpeg_table(arrs), len(files), C.c_void_p(buf.data_ptr()),
                                       (C.c_int64 * len(files))(*offs), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    for o, g in zip(offs, full):
        assert np.array_equal(buf[o:o + g.numel()].view(g.shape).cpu().numpy(), g.cpu().numpy())


def _detect_files(seed):
    """B = 5 whose auto ratios are 2, 1, 4, 2 and 1 for a 608 x 608 model."""
    spec = [((1000, 1500), "422", 90), ((480, 640), "420", 85), ((2448, 3264), "420", 88), ((1300, 700), "grey", 80),
            ((47, 33), "420", 90)]
    return [jc.encode(jc.photo(h, w, seed + i), mode, q) for i, ((h, w), mode, q) in enumerate(spec)]


CASES = [("default", "bf16", 1), ("tiny", "fp32", 1), ("tiny", "fp32", 0)]


@pytest.mark.parametrize("which,mode,fp32_tc", CASES, ids=[f"{c[0]}-{c[1]}-tc{c[2]}" for c in CASES])
def test_detect_jpeg_scaled_equals_detect_images_on_draft_decode(which, mode, fp32_tc):
    cfg = vd.DetectorConfig() if which == "default" else tiny_config()
    target = cfg.input_shape[:2]
    m = build_model(cfg, vd.random_weights(cfg, seed=4, spread=True), mode)
    m.set_option("fp32_tc", fp32_tc)
    m.set_chunk(2)                                                     # B = 5 on chunks of 2
    files = _detect_files(seed=len(which))
    auto = [jpeg_auto_ratio(*_size(d), target) for d in files]
    if which == "default":
        assert auto == [2, 1, 4, 2, 1]
    for ratio in ("auto", 2, 8, [8, 4, "auto", 1, 2]):
        rs = ratio if isinstance(ratio, list) else [ratio] * len(files)
        rs = [auto[i] if r == "auto" else r for i, r in enumerate(rs)]
        imgs = [_reduced(d, r) for d, r in zip(files, rs)]
        ref = m.detect_images(imgs, packed=True)
        got = m.detect_jpeg(files, packed=True, ratio=ratio)
        _assert_same(got, ref, FIELDS)
        for b, (d, im) in enumerate(zip(files, imgs)):
            want = js.boxes_to_file(ref.boxes_original[b], im.shape[:2], _size(d))
            assert np.array_equal(got.boxes_original[b], want), (ratio, b)
    # ratio 1 through the scaled entry point is today's detect_jpeg in every field
    _assert_same(m.detect_jpeg(files, packed=True, ratio=[1] * len(files)), m.detect_jpeg(files, packed=True))
    m.close()


def test_submit_jpeg_scaled_in_flight_pageable_and_page_locked():
    import torch
    cfg = tiny_config()
    m = build_model(cfg, vd.random_weights(cfg, seed=6, spread=True), "bf16")
    a = _detect_files(seed=10)
    b = [jc.encode(jc.photo(900, 1200, 11), "420", 80), jc.encode(jc.photo(480, 640, 12), "grey", 95, restart_marker_blocks=2)]
    pinned = [torch.frombuffer(bytearray(d), dtype=torch.uint8).pin_memory().numpy() for d in b]
    for src_b in (b, pinned):
        ta = m.submit_jpeg(a, packed=True, ratio="auto")
        tb = m.submit_jpeg(src_b, packed=True, ratio=[4, 2])
        got_b = m.collect(tb)
        got_a = m.collect(ta)
        _assert_same(got_a, m.detect_jpeg(a, packed=True, ratio="auto"))
        _assert_same(got_b, m.detect_jpeg(b, packed=True, ratio=[4, 2]))
    m.close()


def test_launch_count_does_not_depend_on_the_ratio():
    cfg = tiny_config()
    m = build_model(cfg, vd.random_weights(cfg, seed=7), "bf16")
    m.set_chunk(2)
    files = _detect_files(seed=3)
    m.launch_count(reset=True)
    m.detect_jpeg(files)
    full = m.launch_count(reset=True)
    for ratio in (2, 4, 8, "auto", [8, 1, 4, 2, 2]):
        m.detect_jpeg(files, ratio=ratio)
        assert m.launch_count(reset=True) == full, ratio
    m.close()


def test_rejections():
    cfg = tiny_config()
    m = build_model(cfg, vd.random_weights(cfg, seed=8), "bf16")
    good = jc.encode(jc.photo(33, 47, 1), "420", 85)
    # malformed ratios: ValueError before the library is called
    for bad in (3, 0, "x", True, [2], [2, 2, 2]):
        m.launch_count(reset=True)
        with pytest.raises(ValueError):
            m.detect_jpeg([good, good], ratio=bad)
        with pytest.raises(ValueError):
            decode_jpeg([good, good], ratio=bad)
        assert m.launch_count(reset=True) == 0
    with pytest.raises(ValueError):
        decode_jpeg([good], ratio="auto")                # auto is relative to a model's input size
    # in C: E_INVALID naming the file, nothing launched
    lib = _capi.load()
    arrs = [np.frombuffer(good, np.uint8)] * 3
    params = vd.vision_transformer_detector._decode_params(None, None, True, cfg.input_shape[:2])
    ticket = C.c_int(-1)
    m.launch_count(reset=True)
    rc = lib.vitdet_submit_jpeg_host_scaled(m._h, _jpeg_table(arrs), (C.c_int32 * 3)(1, 3, 1), 3, 0, C.byref(params), 0, None,
                                            None, C.byref(ticket))
    assert rc == _capi.E_INVALID and b"file 1: ratio 3" in lib.vitdet_last_error()
    assert m.launch_count(reset=True) == 0
    # files outside baseline JPEG are still rejected with their reasons, at every ratio
    for name, bad, why in jc.rejected():
        for ratio in (2, 4, 8, "auto"):
            m.launch_count(reset=True)
            with pytest.raises(_capi.VitdetError, match=f"file 1: .*{why}") as e:
                m.detect_jpeg([good, bad, good], ratio=ratio)
            assert e.value.code == _capi.E_INVALID, name
            assert m.launch_count(reset=True) == 0, name
            if ratio != "auto":
                with pytest.raises(_capi.VitdetError, match=why):
                    decode_jpeg([good, bad], ratio=ratio)
    m.close()
