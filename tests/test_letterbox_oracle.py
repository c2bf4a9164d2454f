"""CPU tests of the back-projection oracle (oracle/letterbox_oracle.py): boxes drawn on a source image survive the trip
through resize_with_pad's geometry and back, and the clip to the source image holds."""
import numpy as np
import pytest

from _util import oracle  # noqa: F401  (puts oracle/ on the path)
import letterbox_oracle as lb

SIZES = [(480, 640), (640, 480), (427, 640), (608, 608), (7, 3), (1000, 1500), (60, 130)]


def _decoded(cx, cy, h, w):
    return np.array([0.9, 3.0, cx, cy, h, w], np.float32)


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("target", [(608, 608), (60, 130)])
def test_box_round_trips_through_the_letterbox(size, target):
    h, w = size
    rng = np.random.default_rng(h * 31 + w)
    for _ in range(20):
        x0, x1 = np.sort(rng.uniform(0, w, 2))
        y0, y1 = np.sort(rng.uniform(0, h, 2))
        cx, cy, bh, bw = lb.letterbox_box((x0, y0, x1, y1), size, target)
        got = lb.boxes_original(_decoded(cx, cy, bh, bw), size, target)
        assert got.dtype == np.float32 and got.shape == (4,)
        # float32 rounding of the decoded row and of each operation, magnified by the source / resized scale
        rh, rw, _, _ = oracle.resize_with_pad_geometry(h, w, *target)
        tol = 1e-5 * max(target) * max(h / rh, w / rw) + 1e-4
        assert np.allclose(got, [x0, y0, x1, y1], rtol=0, atol=tol), (got, (x0, y0, x1, y1))


def test_boxes_are_clipped_to_the_source_image():
    size = (480, 640)                               # 608 wide, 455 high (TF's float32 floor), a bar of 76 rows on top
    rh, rw, ph, pw = oracle.resize_with_pad_geometry(*size, 608, 608)
    assert (rh, rw, ph, pw) == (455, 608, 76, 0)
    whole = lb.boxes_original(_decoded(304, 304, 608, 608), size)       # the whole model image, bars included
    assert np.array_equal(whole, np.array([0, 0, 640, 480], np.float32))
    in_bar = lb.boxes_original(_decoded(100, 20, 10, 10), size)          # inside the top bar: collapses onto row 0
    assert in_bar[1] == 0 and in_bar[3] == 0
    nan = lb.boxes_original(_decoded(np.nan, 300, 10, 10), size)        # fmaxf / fminf: NaN coordinates clip to 0
    assert nan[0] == 0 and nan[2] == 0 and np.isfinite(nan).all()


def test_operation_order_is_the_documented_one():
    """x0 = (cx - w/2 - pad_left) * (width / resized_width) with a float32 rounding after every operation."""
    f = np.float32
    size = (333, 500)
    rh, rw, ph, pw = oracle.resize_with_pad_geometry(*size, 608, 608)
    dec = np.random.default_rng(5).uniform(0, 608, (64, 6)).astype(f)
    got = lb.boxes_original(dec, size)
    ws, hs = f(f(500) / f(rw)), f(f(333) / f(rh))
    for r in range(64):
        cx, cy, bh, bw = (f(v) for v in dec[r, 2:])
        x0 = f(f(f(cx - f(bw / f(2))) - f(pw)) * ws)
        y1 = f(f(f(cy + f(bh / f(2))) - f(ph)) * hs)
        assert got[r, 0] == min(max(x0, f(0)), f(500))
        assert got[r, 3] == min(max(y1, f(0)), f(333))
