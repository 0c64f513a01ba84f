"""CPU: the host side of a cropped decode (crop_plan.h through tests/native/libb2jcrop.so) and the crop calls' argument
checks. The box mapping under all eight EXIF codes against a numpy model -- orient(a)[box] == orient(a[mapped box]) --
and its refusals; the crop tile list for boxes at every offset inside an MCU and across MCU borders, which must cover the
window's MCUs plus the halo and nothing more, in runs of at most one tile."""
import ctypes
import os

import numpy as np
import pytest

from conftest import ROOT
from test_orientation_parse import orient

TILE_BLOCKS = 192


@pytest.fixture(scope="module")
def lib(built):
    L = ctypes.CDLL(os.path.join(ROOT, "tests", "native", "libb2jcrop.so"))
    u32p, i32p = ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_int32)
    L.chk_crop_window.argtypes = [ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, i32p, u32p]
    L.chk_crop_tiles.argtypes = [ctypes.c_uint32] * 6 + [u32p, ctypes.c_uint32, ctypes.c_uint32, u32p, ctypes.c_int, ctypes.POINTER(ctypes.c_long)]
    return L


def _window(lib, fw, fh, code, box):
    b = (ctypes.c_int32 * 4)(*box)
    w = (ctypes.c_uint32 * 4)()
    return tuple(w) if lib.chk_crop_window(fw, fh, code, b, w) else None


def _tiles(lib, mcw, mch, yh, yv, tot, win, scale, halo, blk_first=1000):
    cap = mcw * mch + 8
    out = (ctypes.c_uint32 * (3 * cap))()
    mx = ctypes.c_long()
    n = lib.chk_crop_tiles(mcw, mch, yh, yv, tot, blk_first, (ctypes.c_uint32 * 4)(*win), scale, halo, out, cap, ctypes.byref(mx))
    return [tuple(out[3 * k:3 * k + 3]) for k in range(n)], mx.value


def test_box_mapping_under_every_code(lib):
    rng = np.random.default_rng(5)
    for fw, fh in ((1, 1), (1, 9), (7, 1), (13, 8), (40, 23)):
        a = rng.integers(0, 255, (fh, fw, 3), np.uint8)
        for code in range(1, 9):
            o = orient(a, code)
            oh, ow = o.shape[:2]
            boxes = [(0, 0, ow, oh), (ow - 1, oh - 1, 1, 1), (0, oh - 1, ow, 1), (ow - 1, 0, 1, oh)]
            for _ in range(40):
                x, y = int(rng.integers(0, ow)), int(rng.integers(0, oh))
                boxes.append((x, y, int(rng.integers(1, ow - x + 1)), int(rng.integers(1, oh - y + 1))))
            for x, y, w, h in boxes:
                win = _window(lib, fw, fh, code, (x, y, w, h))
                assert win is not None, (fw, fh, code, (x, y, w, h))
                x0, y0, ww, wh = win
                assert x0 + ww <= fw and y0 + wh <= fh
                assert np.array_equal(orient(a[y0:y0 + wh, x0:x0 + ww], code), o[y:y + h, x:x + w]), (fw, fh, code, (x, y, w, h))


def test_box_mapping_refuses_what_does_not_fit(lib):
    # 13 x 8 unoriented: the frame is 8 x 13 for codes 5..8
    for code in range(1, 9):
        ow, oh = (8, 13) if code >= 5 else (13, 8)
        assert _window(lib, 13, 8, code, (0, 0, ow, oh)) is not None
        for box in ((0, 0, ow + 1, oh), (0, 0, ow, oh + 1), (ow, 0, 1, 1), (0, oh, 1, 1), (1, 0, ow, 1), (0, 1, 1, oh),
                    (-1, 0, 1, 1), (0, -1, 1, 1), (0, 0, 0, 1), (0, 0, 1, 0), (2 ** 31 - 1, 0, 1, 1), (0, 0, 2 ** 31 - 1, 1)):
            assert _window(lib, 13, 8, code, box) is None, (code, box)


# (yh, yv, blocks per MCU): 4:2:0, 4:2:2, 4:4:4, a generic 2x2 layout with 2x1 chroma, gray, 4:4:0
LAYOUTS = [(2, 2, 6), (2, 1, 4), (1, 1, 3), (2, 2, 8), (1, 1, 1), (1, 2, 4)]


@pytest.mark.parametrize("scale", [1, 2, 4, 8])
def test_crop_tiles_cover_the_window_and_halo_only(lib, scale):
    for yh, yv, tot in LAYOUTS:
        mw, mh = yh * 8 // scale, yv * 8 // scale
        per_tile = TILE_BLOCKS // tot
        for mcw, mch in ((1, 1), (5, 4), (per_tile + 3, 3), (2 * per_tile + 1, 2)):
            fw, fh = mcw * mw, mch * mh
            wins = [(0, 0, fw, fh), (fw - 1, fh - 1, 1, 1)]
            # a box starting and ending at every offset inside an MCU, across up to three MCU borders
            for o in range(mw):
                for span in (1, mw - o, mw - o + 1, 2 * mw + 1):
                    x0 = min(o + (mw if mcw > 2 else 0), fw - 1)
                    wins.append((x0, min(o, fh - 1), max(1, min(span, fw - x0)), max(1, min(span, fh - min(o, fh - 1)))))
            for halo in (0, 1):
                for win in wins:
                    tiles, mx = _tiles(lib, mcw, mch, yh, yv, tot, win, scale, halo)
                    x0, y0, w, h = win
                    c0, c1, r0, r1 = x0 // mw, (x0 + w - 1) // mw, y0 // mh, (y0 + h - 1) // mh
                    want = {r * mcw + c for r in range(max(r0 - halo, 0), min(r1 + halo, mch - 1) + 1)
                            for c in range(max(c0 - halo, 0), min(c1 + halo, mcw - 1) + 1)}
                    full_rows = max(c0 - halo, 0) == 0 and min(c1 + halo, mcw - 1) == mcw - 1
                    got = []
                    for m, n, row in tiles:
                        assert 1 <= n <= per_tile and row == 1000 + m * tot
                        assert (m % mcw) + n <= mcw or full_rows   # inside one MCU row, unless whole rows meet
                        got.extend(range(m, m + n))
                    assert len(got) == len(set(got)) and set(got) == want, (yh, yv, tot, scale, mcw, mch, win, halo)
                    assert len(tiles) <= mx


def test_crop_calls_refuse_bad_arguments(built):
    import ocljpegdecoder_b200 as b2j
    L = b2j.load_library()
    boxes = np.array([[0, 0, 1, 1]], np.int32)
    assert L.b2j_batch_set_crops(None, boxes.ctypes.data) == -1
    assert L.b2j_batch_set_crops(None, None) == -1
    opts = b2j.HostOpts(pixel_model=b2j.PIXELS_LIBJPEG)
    f = (ctypes.c_char_p * 1)(b"\xff\xd8")
    ln = (ctypes.c_size_t * 1)(2)
    out = (ctypes.c_void_p * 1)()
    st = np.zeros(1, np.int32)
    assert L.b2j_decode_host_crop(None, 1, f, ln, ctypes.byref(opts), boxes.ctypes.data, out, st.ctypes.data) == -1
    with pytest.raises(ValueError):
        b2j.api._crop_boxes([[0, 0, 1]], 1)
    with pytest.raises(ValueError):
        b2j.api._crop_boxes([[0, 0, 1, 1]] * 2, 1)


def test_crop_frame_is_scale_then_orientation(built, fixture_jpeg):
    import ocljpegdecoder_b200 as b2j
    rc, d = b2j.parse_header(fixture_jpeg)
    assert rc == 0
    for scale in (1, 2, 4, 8):
        w, h = -(-d.width // scale), -(-d.height // scale)
        for code in range(1, 9):
            assert b2j.crop_frame(d, scale, code) == ((h, w) if code >= 5 else (w, h))
            assert b2j.api._out_shape(d, b2j.OUT_RGB24, scale, code, (1, 2, 3, 4)) == (4, 3, 3)
            assert b2j.api._out_shape(d, b2j.OUT_RGB_PLANAR, scale, code, (1, 2, 3, 4)) == (3, 4, 3)
