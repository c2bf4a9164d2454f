"""GPU tests of detection on decoded images of any size (detect_images / submit_images, vitdet_forward_images /
vitdet_submit_images_host): the letterbox fused into the patch kernel must give exactly what preprocessing every image
and stacking the batch gives, in every arithmetic form, and boxes_original must restate the oracle bit for bit."""
import ctypes as C

import numpy as np
import pytest

from _util import build_model, tiny_config
import letterbox_oracle as lb
import vision_transformer_detector_b200 as vd
from vision_transformer_detector_b200 import _capi

pytestmark = pytest.mark.gpu

FIELDS = ("logits", "decoded", "class_id", "class_conf", "keep", "corners", "packed")


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def _ragged(target, seed=0):
    """Five images: wider than the target, an upscaled tiny one that is taller, a downscaled large one, 480 x 640 (resized
    455 x 608 at 608: TF's float32 floor) and one at the model's size."""
    rng = np.random.default_rng(seed)
    sizes = [(300, 900), (7, 3), (1000, 1500), (480, 640), tuple(target)]
    return [rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for h, w in sizes]


def _assert_same(a, b, fields=FIELDS):
    for f in fields:
        assert np.array_equal(_np(getattr(a, f)), _np(getattr(b, f))), f


def _today(m, imgs, target, **kw):
    """The route without this feature: one preprocess per image, a stacked float32 batch, detect."""
    return m.detect(np.stack([vd.preprocess_image(im, target) for im in imgs]), packed=True, **kw)


CASES = [
    ("default", "bf16", 1), ("default", "fp32", 1),
    ("tiny", "bf16", 1), ("tiny", "fp32", 1), ("tiny", "fp32", 0),     # fp32_tc = 0: the IEEE CUDA-core form
]


@pytest.mark.parametrize("which,mode,fp32_tc", CASES, ids=[f"{c[0]}-{c[1]}-tc{c[2]}" for c in CASES])
def test_images_match_preprocess_then_detect_bit_for_bit(which, mode, fp32_tc):
    cfg = vd.DetectorConfig() if which == "default" else tiny_config()
    target = cfg.input_shape[:2]
    m = build_model(cfg, vd.random_weights(cfg, seed=4, spread=True), mode)
    m.set_option("fp32_tc", fp32_tc)
    imgs = _ragged(target, seed=len(which))
    m.set_chunk(2)                                                # B = 5 on chunks of 2: the table is read across chunks
    ref = _today(m, imgs, target)
    got = m.detect_images(imgs, packed=True)
    _assert_same(got, ref)
    for b, im in enumerate(imgs):
        assert np.array_equal(got.boxes_original[b], lb.boxes_original(got.decoded[b], im.shape[:2], target))
    m.close()


def test_model_size_images_equal_the_fused_uint8_path():
    cfg = tiny_config()
    m = build_model(cfg, vd.random_weights(cfg, seed=5, spread=True), "bf16")
    rng = np.random.default_rng(2)
    x = rng.integers(0, 256, size=(4, *cfg.input_shape), dtype=np.uint8)
    x[0, :3] = 0
    x[1, -3:] = 255
    _assert_same(m.detect_images(list(x), packed=True), m.detect(x, normalize_uint8=True, packed=True))
    m.close()


def test_device_host_and_pipelined_routes_agree():
    import torch
    cfg = vd.DetectorConfig()
    m = build_model(cfg, vd.random_weights(cfg, seed=6, spread=True), "bf16")
    imgs = _ragged(cfg.input_shape[:2], seed=9) + [np.full((900, 300, 3), 7, np.uint8)]
    host = m.detect_images(imgs, packed=True)
    dev = m.detect_images([torch.from_numpy(im).cuda() for im in imgs], packed=True)
    torch.cuda.synchronize()
    _assert_same(dev, host, FIELDS + ("boxes_original",))
    assert dev.boxes_original.shape == (len(imgs), 17, 4) and dev.boxes_original.is_cuda
    # two submissions in flight: one from pageable arrays, one from page-locked ones
    pinned = [torch.from_numpy(im).pin_memory().numpy() for im in imgs]
    t0 = m.submit_images(imgs, packed=True)
    t1 = m.submit_images(pinned, packed=True)
    r0, r1 = m.collect(t0), m.collect(t1)
    _assert_same(r0, host, FIELDS + ("boxes_original",))
    _assert_same(r1, host, FIELDS + ("boxes_original",))
    # non-contiguous arrays are taken as their contiguous copies
    flipped = [im[:, ::-1] for im in imgs[:3]]
    _assert_same(m.detect_images(flipped), m.detect_images([np.ascontiguousarray(im) for im in flipped]),
                 FIELDS[:-1] + ("boxes_original",))
    m.close()


def test_launch_count_equals_detect():
    """The letterbox replaces patchify one for one and boxes_original is computed by the fused head tail: no extra launch."""
    import torch
    cfg = tiny_config()
    m = build_model(cfg, vd.random_weights(cfg, seed=7), "bf16")
    imgs = _ragged(cfg.input_shape[:2])
    m.set_chunk(2)
    x = torch.from_numpy(np.stack([vd.preprocess_image(im, cfg.input_shape[:2]) for im in imgs])).cuda()
    m.launch_count(reset=True)
    m.detect(x)
    n_detect = m.launch_count(reset=True)
    m.detect_images([torch.from_numpy(im).cuda() for im in imgs])
    assert m.launch_count(reset=True) == n_detect
    m.detect_images(imgs)
    assert m.launch_count(reset=True) == n_detect
    m.close()


def test_invalid_inputs_are_rejected():
    import torch
    cfg = tiny_config()
    m = build_model(cfg, vd.random_weights(cfg, seed=8), "bf16")
    good = np.zeros((10, 12, 3), np.uint8)
    for bad in ([], [good.astype(np.float32)], [good[..., 0]], [np.zeros((10, 12, 4), np.uint8)],
                [good, torch.from_numpy(good).cuda()]):
        with pytest.raises(ValueError):
            m.detect_images(bad)
        with pytest.raises(ValueError):
            m.submit_images(bad)
    lib = _capi.load()
    params = vd.vision_transformer_detector._decode_params(None, None, True, cfg.input_shape[:2])
    S = 17

    def forward_images(table, B, p=params, boxes=True):
        logits, *recs = vd.vision_transformer_detector._alloc_records_torch(max(B, 1), S, "cuda")
        st = vd.vision_transformer_detector._records_struct(*recs)
        bx = torch.empty((max(B, 1), S, 4), device="cuda")
        return lib.vitdet_forward_images(m._h, table, B, _capi.MODE_BF16, C.byref(p), C.c_void_p(logits.data_ptr()), C.byref(st),
                                         C.c_void_p(bx.data_ptr()) if boxes else None, None)

    dev_good = torch.from_numpy(good).cuda()
    flat = torch.zeros((1, 2000, 3), dtype=torch.uint8, device="cuda")    # resizes to 0 rows at 60 x 130
    m.launch_count(reset=True)
    cases = [
        ((_capi.Image * 2)(_capi.Image(dev_good.data_ptr(), 10, 12), _capi.Image(flat.data_ptr(), 1, 2000)), 2, "image 1"),
        ((_capi.Image * 2)(_capi.Image(dev_good.data_ptr(), 10, 12), _capi.Image(dev_good.data_ptr(), 0, 12)), 2, "image 1"),
        ((_capi.Image * 1)(_capi.Image(None, 10, 12)), 1, "image 0"),
        ((_capi.Image * 1)(_capi.Image(dev_good.data_ptr(), 10, 12)), 0, "B must be positive"),
    ]
    for table, B, text in cases:
        rc = forward_images(table, B)
        assert rc == _capi.E_INVALID and text in lib.vitdet_last_error().decode()
        ticket = C.c_int(-1)
        host = (_capi.Image * len(table))(*[_capi.Image(good.ctypes.data if t.pixels else None, t.height, t.width) for t in table])
        assert lib.vitdet_submit_images_host(m._h, host, B, _capi.MODE_BF16, C.byref(params), 0, None, None, C.byref(ticket)) == _capi.E_INVALID
        assert text in lib.vitdet_last_error().decode()
    one = (_capi.Image * 1)(_capi.Image(dev_good.data_ptr(), 10, 12))
    wrong = vd.vision_transformer_detector._decode_params(None, None, True, (608, 608))
    assert forward_images(one, 1, wrong) == _capi.E_INVALID and "boxes_original" in lib.vitdet_last_error().decode()
    assert m.launch_count(reset=True) == 0
    assert forward_images(one, 1, wrong, boxes=False) == 0                 # without boxes any decode size is allowed
    torch.cuda.synchronize()
    m.close()


def test_rejected_degenerate_image_launches_nothing():
    import torch
    cfg = tiny_config()
    m = build_model(cfg, vd.random_weights(cfg, seed=8), "bf16")
    flat = torch.zeros((1, 2000, 3), dtype=torch.uint8, device="cuda")
    m.launch_count(reset=True)
    with pytest.raises(_capi.VitdetError) as ei:
        m.detect_images([torch.zeros((5, 5, 3), dtype=torch.uint8, device="cuda"), flat])
    assert ei.value.code == _capi.E_INVALID and "image 1" in str(ei.value)
    with pytest.raises(_capi.VitdetError):
        m.detect_images([np.zeros((1, 2000, 3), np.uint8)])
    assert m.launch_count(reset=True) == 0
    m.close()
