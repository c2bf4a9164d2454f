"""CPU tests of the JPEG decoder's semantics: the numpy oracle (oracle/jpeg_oracle.py) against PIL / libjpeg-turbo bit for
bit, its subsequence decode against its sequential decode, the clamps for corrupt data, and the library's host header
check (vitdet_jpeg_info)."""
import ctypes as C
import io

import numpy as np
import pytest
from PIL import Image

from _util import oracle  # noqa: F401  (puts oracle/ on the path)
import _jpeg_corpus as jc
import jpeg_oracle as jo
from vision_transformer_detector_b200 import _capi

CORPUS = jc.corpus()


def _pil(data):
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))


@pytest.mark.parametrize("name,data", CORPUS, ids=[n for n, _ in CORPUS])
def test_oracle_pixels_equal_pil(name, data):
    assert np.array_equal(jo.decode(data), _pil(data))


@pytest.mark.parametrize("L", [64, 256])
def test_subsequence_decode_equals_sequential(L):
    repaired = 0
    for name, data in CORPUS:
        j = jo.parse(data)
        for s in range(len(j["segments"])):
            stats = {}
            got = jo.decode_subsequences(j, s, L, stats)
            assert np.array_equal(got, jo.decode_sequential(j, s)), (name, s)
            repaired += stats.get("subsequences", 0)
    assert repaired > 0          # the repair path ran


def test_corrupt_entropy_data_decodes_under_the_clamps():
    data = jc.flipped()
    j = jo.parse(data)
    px = jo.decode(data)
    assert px.shape == (48, 64, 3)
    for s in range(len(j["segments"])):
        assert np.array_equal(jo.decode_subsequences(j, s, 64), jo.decode_sequential(j, s))
    clean = jo.decode(jc.encode(jc.photo(48, 64, 31), "420", 85))
    assert not np.array_equal(px, clean)


def test_range_limit_table():
    # jdmaster.c prepare_range_limit_table for 8-bit samples, then idct range_limit = sample_range_limit + CENTERJSAMPLE
    buf = np.zeros(5 * 256 + 128, np.int64)      # sample_range_limit = buf + 256
    buf[256:512] = np.arange(256)                # limit[x] = x
    buf[512:896] = 255                           # rest of the first half of the post-IDCT table
    buf[896:1280] = 0                            # second half ...
    buf[1280:1408] = np.arange(128)              # ... ending with a copy of limit[0 .. 127]
    v = np.arange(-4096, 4096)
    assert np.array_equal(jo.range_limit(v), buf[256 + 128 + (v & 1023)])


def test_fill_byte_before_a_stuffed_zero_is_one_ff():
    data = jc.encode(jc.photo(48, 64, 15), "420", 95)
    patched = jc.fill_before_stuffed_zero(data)
    assert len(patched) == len(data) + 1
    assert np.array_equal(_pil(patched), _pil(data))
    assert np.array_equal(jo.decode(patched), _pil(data))


def test_pil_refuses_an_all_ones_huffman_code():
    with pytest.raises(OSError):
        _pil(jc.all_ones_code(jc.encode(jc.photo(48, 64, 21), "420", 85)))


def test_segment_longer_than_the_device_bit_positions_is_rejected():
    # a restart segment of 2^28 bytes has bit positions past int32; the header check rejects it
    data = jc.encode(jc.photo(16, 16, 3), "420", 85)
    sos_end = [e for _, m, _, e in jc.segments(data) if m == 0xDA][0]
    big = data[:sos_end] + bytes(1 << 28) + b"\xFF\xD9"
    rc, _, msg = _info(big)
    assert rc == _capi.E_INVALID and "restart segment" in msg, msg
    with pytest.raises(jo.JpegError, match="restart segment"):
        jo.parse(big)
    ok = data[:sos_end] + bytes(jo.MAX_SEGMENT_BYTES) + b"\xFF\xD9"   # the longest accepted segment
    assert _info(ok)[0] == 0


def _info(data):
    v = [C.c_int() for _ in range(3)]
    rc = _capi.load().vitdet_jpeg_info(data, len(data), *[C.byref(x) for x in v])
    return rc, [x.value for x in v], (_capi.load().vitdet_last_error() or b"").decode()


@pytest.mark.parametrize("name,data", CORPUS, ids=[n for n, _ in CORPUS])
def test_jpeg_info_agrees_with_pil(name, data):
    rc, (h, w, c), _ = _info(data)
    im = Image.open(io.BytesIO(data))
    assert rc == 0
    assert (h, w) == (im.height, im.width)
    assert c == {"L": 1, "RGB": 3}[im.mode]
    assert (h, w, c) == jo.info(data)


@pytest.mark.parametrize("name,data,why", jc.rejected(), ids=[r[0] for r in jc.rejected()])
def test_jpeg_info_rejects(name, data, why):
    rc, _, msg = _info(data)
    assert rc == _capi.E_INVALID
    assert why in msg, msg
    with pytest.raises(jo.JpegError, match=why):
        jo.parse(data)
