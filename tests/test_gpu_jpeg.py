"""GPU tests of the JPEG decoder (vitdet_decode_jpeg, vitdet_submit_jpeg_host): decode_jpeg must give PIL's pixels bit for
bit, and detect_jpeg / submit_jpeg exactly the records of detect_images on the PIL-decoded images."""
import ctypes as C
import io

import numpy as np
import pytest
from PIL import Image

from _util import build_model, tiny_config
import _jpeg_corpus as jc
import jpeg_oracle as jo
import vision_transformer_detector_b200 as vd
from vision_transformer_detector_b200 import _capi
from vision_transformer_detector_b200.vision_transformer_detector import _jpeg_table
from vision_transformer_detector_b200.vision_transformer_utilities import decode_jpeg

pytestmark = pytest.mark.gpu

FIELDS = ("logits", "decoded", "class_id", "class_conf", "keep", "corners", "packed", "boxes_original")


def _pil(data):
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def _assert_same(a, b):
    for f in FIELDS:
        assert np.array_equal(_np(getattr(a, f)), _np(getattr(b, f))), f


def _coco_files(seed=0):
    """COCO-size files (height x width): 480 x 640, 427 x 640, 612 x 612 and 1000 x 1500, in 4:2:0, 4:4:4, grey, 4:2:2."""
    sizes = [((480, 640), "420", 85), ((427, 640), "444", 92), ((612, 612), "grey", 75), ((1000, 1500), "422", 95)]
    return [jc.encode(jc.photo(h, w, seed + i), mode, q) for i, ((h, w), mode, q) in enumerate(sizes)]


def test_decode_jpeg_equals_pil():
    files = [d for _, d in jc.corpus()] + _coco_files()
    got = decode_jpeg(files)
    for i, (g, d) in enumerate(zip(got, files)):
        assert np.array_equal(g.cpu().numpy(), _pil(d)), i


CASES = [("default", "bf16", 1), ("tiny", "fp32", 1), ("tiny", "fp32", 0)]


@pytest.mark.parametrize("which,mode,fp32_tc", CASES, ids=[f"{c[0]}-{c[1]}-tc{c[2]}" for c in CASES])
def test_detect_jpeg_equals_detect_images_on_pil_decode(which, mode, fp32_tc):
    cfg = vd.DetectorConfig() if which == "default" else tiny_config()
    m = build_model(cfg, vd.random_weights(cfg, seed=4, spread=True), mode)
    m.set_option("fp32_tc", fp32_tc)
    files = _coco_files(seed=len(which)) + [jc.encode(jc.photo(47, 33, 3), "420", 90)]       # B = 5
    m.set_chunk(2)                                                     # B = 5 on chunks of 2
    ref = m.detect_images([_pil(d) for d in files], packed=True)
    _assert_same(m.detect_jpeg(files, packed=True), ref)
    m.close()


def test_submit_jpeg_pageable_and_page_locked_in_flight_equal_detect_jpeg():
    import torch
    cfg = tiny_config()
    m = build_model(cfg, vd.random_weights(cfg, seed=6, spread=True), "bf16")
    a = _coco_files(seed=10)
    b = [jc.encode(jc.photo(90, 120, 11), "420", 80), jc.encode(jc.photo(48, 64, 12), "grey", 95, restart_marker_blocks=2)]
    pinned = [torch.frombuffer(bytearray(d), dtype=torch.uint8).pin_memory().numpy() for d in b]
    ta = m.submit_jpeg(a, packed=True)
    tb = m.submit_jpeg(pinned, packed=True)
    got_b = m.collect(tb)
    got_a = m.collect(ta)
    _assert_same(got_a, m.detect_jpeg(a, packed=True))
    _assert_same(got_b, m.detect_jpeg(b, packed=True))
    # the full-size entry point gives what submit_jpeg gets from the scaled one at ratio 1
    lib = _capi.load()
    S = 17
    recs, st = vd.vision_transformer_detector._alloc_records(len(a), S, packed=True)
    recs.boxes_original = np.empty((len(a), S, 4), np.float32)
    params = vd.vision_transformer_detector._decode_params(None, None, True, cfg.input_shape[:2])
    ticket = C.c_int(-1)
    _capi.check(lib.vitdet_submit_jpeg_host(m._h, _jpeg_table([np.frombuffer(d, np.uint8) for d in a]), len(a), _capi.MODE_BF16,
                                            C.byref(params), 1, _capi.np_ptr(recs.boxes_original), None, C.byref(ticket)))
    _capi.check(lib.vitdet_collect(m._h, ticket.value, _capi.np_ptr(recs.logits), C.byref(st)))
    _assert_same(recs, got_a)
    m.close()


def test_launch_count_is_detect_images_plus_a_constant():
    cfg = tiny_config()
    m = build_model(cfg, vd.random_weights(cfg, seed=7), "bf16")
    m.set_chunk(2)
    extra = []
    for files in ([jc.encode(jc.photo(33, 47, 1), "420", 85)], _coco_files(seed=3) + [jc.encode(jc.photo(9, 17, 2), "grey", 50)]):
        imgs = [_pil(d) for d in files]
        m.launch_count(reset=True)
        m.detect_images(imgs)
        n_images = m.launch_count(reset=True)
        m.detect_jpeg(files)
        extra.append(m.launch_count(reset=True) - n_images)
    assert extra[0] == extra[1] > 0
    m.close()


def test_rejected_files_fail_naming_them_and_launch_nothing():
    cfg = tiny_config()
    m = build_model(cfg, vd.random_weights(cfg, seed=8), "bf16")
    good = jc.encode(jc.photo(33, 47, 1), "420", 85)
    for name, bad, why in jc.rejected():
        m.launch_count(reset=True)
        with pytest.raises(_capi.VitdetError, match=f"file 1: .*{why}") as e:
            m.detect_jpeg([good, bad, good])
        assert e.value.code == _capi.E_INVALID, name
        with pytest.raises(_capi.VitdetError, match=why):
            decode_jpeg([good, bad])
        assert m.launch_count(reset=True) == 0, name
    for bad_list in ([], [good, 3], [good, b""], [good, np.zeros(4, np.float32)]):
        with pytest.raises(ValueError):
            m.detect_jpeg(bad_list)
        with pytest.raises(ValueError):
            decode_jpeg(bad_list)
    with pytest.raises(ValueError):
        m.submit_jpeg(good)                      # one file, not a list
    m.close()


def test_corrupt_file_decodes_as_the_oracle_and_the_next_decode_is_exact():
    # the oracle states what corrupt entropy data decodes to under the clamps
    got = decode_jpeg([jc.flipped()])
    assert np.array_equal(got[0].cpu().numpy(), jo.decode(jc.flipped()))
    good = jc.encode(jc.photo(48, 64, 31), "420", 85)
    assert np.array_equal(decode_jpeg([good])[0].cpu().numpy(), _pil(good))
