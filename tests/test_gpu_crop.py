"""GPU: a crop window per image in the libjpeg pixel model (b2j_batch_set_crops, b2j_decode_host_crop).

The batch of test_gpu_orientation -- 4:2:0, 4:2:2, 4:4:4, a generic layout with multi-block chroma, gray, 1xN and Nx1
images, an image of many tiles -- six times over, in every format at scales 1, 2, 4 and 8: each crop is the slice of a
different batch's uncropped decode of the same files, bit-exact. The boxes hold the full frame, 1x1 at each corner,
one-pixel strips along each edge, boxes starting and ending at every offset inside an MCU and widths 1..40. Each cropped
batch is built on a Decoder whose pools hold a just-closed batch of the same geometry and other pixels, and its first
decode is the cropped one, so a missing halo MCU shows as wrong pixels instead of reading an earlier correct decode.
Then every EXIF code with crops; Pillow, OpenCV and torchvision on tagged files; switching crops on and off; refusals;
the host call into one pinned arena with guard bytes; and 65537 cropped images."""
import numpy as np
import pytest

import synth
from test_gpu_libjpeg import _craft
from test_gpu_orientation import ITEMS, TAGGED, _gate
from test_gray_model import _draft_gray
from test_libjpeg_model import _gray_jpeg
from test_orientation_parse import orient
from test_scaled_model import _draft_rgb

pytestmark = pytest.mark.gpu

SCALES = (1, 2, 4, 8)
COPIES = 6
FILES = ITEMS * COPIES


def _poison_items():
    """ITEMS' geometry with other pixels."""
    return [
        synth.synth_jpeg(131, 77, 101, 85, "420", 3),
        synth.synth_jpeg(203, 99, 104, 95, "422", 2),
        synth.synth_jpeg(96, 41, 102, 90, "444", 0),
        _craft(((2, 2), (2, 1), (2, 1)), 45, 37, 108, ri=1),
        _gray_jpeg(99, 61, 111, 80, 2),
        synth.synth_jpeg(1, 37, 121, 90, "420", 0),
        synth.synth_jpeg(29, 1, 122, 90, "444", 0),
        _gray_jpeg(1, 23, 123, 85),
        _gray_jpeg(17, 1, 124, 85),
        synth.synth_jpeg(701, 477, 125, 90, "420", 0),
        _craft((2, 1), 3, 11, 110),
    ]


POISON = _poison_items() * COPIES
FORMATS = ("OUT_BGRA", "OUT_RGB24", "OUT_RGB_PLANAR", "OUT_GRAY8")


def _crop(a, box, fmt):
    import ocljpegdecoder_b200 as b2j
    x, y, w, h = (int(v) for v in box)
    return a[:, y:y + h, x:x + w] if fmt == b2j.OUT_RGB_PLANAR else a[y:y + h, x:x + w]


def _mcu(d, scale):
    """An MCU's size in output pixels at `scale`."""
    return d.mcu_width // scale, d.mcu_height // scale


def _box_lists(descs, scale, frames):
    """Every box the test asks for, per image of `frames` ((w, h) per image)."""
    out = []
    for d, (fw, fh) in zip(descs, frames):
        mw, mh = _mcu(d, scale)
        boxes = [(0, 0, fw, fh), (0, 0, 1, 1), (fw - 1, 0, 1, 1), (0, fh - 1, 1, 1), (fw - 1, fh - 1, 1, 1),
                 (0, 0, fw, 1), (0, fh - 1, fw, 1), (0, 0, 1, fh), (fw - 1, 0, 1, fh)]
        for o in range(max(mw, mh)):   # start at every offset inside an MCU, end at every offset too
            x, y = min(mw + o % mw, fw - 1), min(mh + o % mh, fh - 1)
            for span in (mw - o % mw, 2 * mw + 1 - o % mw):
                boxes.append((x, y, max(1, min(span, fw - x)), max(1, min(span + 3, fh - y))))
        for w in range(1, 41):
            x = (7 * w) % fw
            boxes.append((min(x, max(fw - w, 0)), (3 * w) % fh, min(w, fw), min(1 + w % 9, fh - (3 * w) % fh)))
        out.append(list(dict.fromkeys((int(x), int(y), int(w), int(h)) for x, y, w, h in boxes)))
    return out


def _rounds(box_lists):
    """Boxes for one batch of FILES per round: copy k of image j takes its boxes k, k + COPIES, ..."""
    n = len(ITEMS)
    rounds = max(-(-len(b) // COPIES) for b in box_lists[:n])
    out = []
    for r in range(rounds):
        out.append([box_lists[j][(r * COPIES + k) % len(box_lists[j])] for k in range(COPIES) for j in range(n)])
    return out


@pytest.fixture(scope="module")
def full(decoder):
    """The uncropped decodes of FILES' first copy, per (format, scale), from a batch of its own."""
    import ocljpegdecoder_b200 as b2j
    b = decoder.batch(ITEMS, gate=_gate())
    out = {}
    try:
        b.upload()
        b.set_pixel_model(b2j.PIXELS_LIBJPEG)
        for name in FORMATS:
            b.set_output_format(getattr(b2j, name))
            for s in SCALES:
                b.set_scale(s)
                b.decode()
                assert not b.status().any()
                out[name, s] = b.read_all_pixels()
        yield out
    finally:
        b.close()


@pytest.fixture(scope="module")
def fresh():
    """A Decoder of its own, so that its pools hold only what this file puts there."""
    import ocljpegdecoder_b200 as b2j
    d = b2j.Decoder(0)
    yield d
    d.close()


def _poisoned_batch(dec, fmt, scale):
    """A batch of FILES on `dec`, right after a batch of POISON decoded at these settings was closed on it."""
    import ocljpegdecoder_b200 as b2j
    p = dec.batch(POISON, gate=_gate())
    p.upload()
    p.set_pixel_model(b2j.PIXELS_LIBJPEG)
    p.set_output_format(b2j.OUT_RGB24 if fmt == b2j.OUT_GRAY8 else fmt)
    p.set_scale(scale)
    p.decode()
    p.sync()
    p.close()
    b = dec.batch(FILES, gate=_gate())
    b.upload()
    b.set_pixel_model(b2j.PIXELS_LIBJPEG)
    b.set_output_format(fmt)
    b.set_scale(scale)
    return b


@pytest.mark.parametrize("scale", SCALES)
@pytest.mark.parametrize("fmt_name", FORMATS)
def test_crops_are_slices_of_the_uncropped_decode(fresh, full, fmt_name, scale):
    import ocljpegdecoder_b200 as b2j
    fmt = getattr(b2j, fmt_name)
    descs = [b2j.parse_header(f, _gate())[1] for f in ITEMS]
    frames = [b2j.crop_frame(d, scale) for d in descs]
    ref = full[fmt_name, scale]
    for r, boxes in enumerate(_rounds(_box_lists(descs, scale, frames))):
        b = _poisoned_batch(fresh, fmt, scale)
        try:
            b.set_crops(boxes)
            b.decode()
            assert not b.status().any()
            got = b.read_all_pixels()
            for i, box in enumerate(boxes):
                want = _crop(ref[i % len(ITEMS)], box, fmt)
                assert got[i].shape == want.shape and np.array_equal(got[i], want), (fmt_name, scale, r, i, box)
                _, nbytes = b.pixels_device(i)
                assert nbytes == want.nbytes
        finally:
            b.close()


@pytest.mark.parametrize("scale", (1, 4))
def test_every_code_with_crops(decoder, scale):
    import ocljpegdecoder_b200 as b2j
    rng = np.random.default_rng(scale)
    ref = decoder.batch(ITEMS, gate=_gate())
    b = decoder.batch(ITEMS, gate=_gate())
    try:
        for x in (ref, b):
            x.upload()
            x.set_pixel_model(b2j.PIXELS_LIBJPEG)
            x.set_scale(scale)
        for name in FORMATS:
            fmt = getattr(b2j, name)
            ref.set_output_format(fmt)
            b.set_output_format(fmt)
            for code in range(1, 9):
                codes = np.array([code if i % 4 else 1 for i in range(len(ITEMS))], np.uint8)
                ref.set_orientations(codes)
                ref.decode()
                want_full = ref.read_all_pixels()
                b.set_crops(None)
                b.set_orientations(codes)
                boxes = []
                for i in range(b.n):
                    fw, fh = b.crop_frame(i)
                    x, y = int(rng.integers(0, fw)), int(rng.integers(0, fh))
                    boxes.append((x, y, int(rng.integers(1, fw - x + 1)), int(rng.integers(1, fh - y + 1))))
                b.set_crops(boxes)
                b.decode()
                assert not b.status().any()
                for i, g in enumerate(b.read_all_pixels()):
                    want = _crop(want_full[i], boxes[i], fmt)
                    assert g.shape == want.shape and np.array_equal(g, want), (name, scale, code, i, boxes[i])
    finally:
        ref.close()
        b.close()


@pytest.mark.parametrize("scale", SCALES)
def test_host_crop_equals_pillow_opencv_and_torchvision(decoder, scale):
    cv2 = pytest.importorskip("cv2")
    import torch
    from PIL import Image
    from torchvision.io import ImageReadMode, decode_jpeg
    import ocljpegdecoder_b200 as b2j
    cv_rgb = {1: cv2.IMREAD_COLOR, 2: cv2.IMREAD_REDUCED_COLOR_2, 4: cv2.IMREAD_REDUCED_COLOR_4, 8: cv2.IMREAD_REDUCED_COLOR_8}[scale]
    cv_gray = {1: cv2.IMREAD_GRAYSCALE, 2: cv2.IMREAD_REDUCED_GRAYSCALE_2, 4: cv2.IMREAD_REDUCED_GRAYSCALE_4,
               8: cv2.IMREAD_REDUCED_GRAYSCALE_8}[scale]
    rng = np.random.default_rng(40 + scale)
    boxes = []
    for data in TAGGED:
        fw, fh = b2j.crop_frame(b2j.parse_header(data, _gate())[1], scale, b2j.parse_orientation(data))
        x, y = int(rng.integers(0, fw)), int(rng.integers(0, fh))
        boxes.append((x, y, int(rng.integers(1, fw - x + 1)), int(rng.integers(1, fh - y + 1))))
    kw = dict(gate=_gate(), pixel_model=b2j.PIXELS_LIBJPEG, scale=scale, exif_orientation=True, group=5, crops=boxes)
    rgb, st = decoder.decode_host_ex(TAGGED, out_format=b2j.OUT_RGB24, **kw)
    assert not st.any()
    gray, st = decoder.decode_host_ex(TAGGED, out_format=b2j.OUT_GRAY8, **kw)
    assert not st.any()
    for k, data in enumerate(TAGGED):
        x, y, w, h = boxes[k]
        buf = np.frombuffer(data, np.uint8)
        assert np.array_equal(rgb[k], cv2.imdecode(buf, cv_rgb)[y:y + h, x:x + w, ::-1]), (k, scale)
        assert np.array_equal(gray[k], cv2.imdecode(buf, cv_gray)[y:y + h, x:x + w]), (k, scale)
        code = b2j.parse_orientation(data)
        # Pillow: draft(), exif_transpose(), crop()
        assert np.array_equal(rgb[k], np.asarray(Image.fromarray(orient(_draft_rgb(data, scale), code)).crop((x, y, x + w, y + h)))), (k, scale)
        assert np.array_equal(gray[k], orient(_draft_gray(data, scale), code)[y:y + h, x:x + w]), (k, scale)
        if scale == 1:
            t = torch.frombuffer(bytearray(data), dtype=torch.uint8)
            tv = decode_jpeg(t, mode=ImageReadMode.RGB, apply_exif_orientation=True)[:, y:y + h, x:x + w]
            assert np.array_equal(rgb[k], tv.permute(1, 2, 0).numpy()), k


def test_switching_crops_on_and_off(decoder):
    import ocljpegdecoder_b200 as b2j
    never = decoder.batch(ITEMS, gate=_gate())
    b = decoder.batch(ITEMS, gate=_gate())
    try:
        for x in (never, b):
            x.upload()
            x.set_pixel_model(b2j.PIXELS_LIBJPEG)
            x.set_output_format(b2j.OUT_RGB24)
        never.decode()
        plain, plain_info, plain_st = never.read_all_pixels(), never.info(), never.status()
        plain_coefs = [never.coefs(i) for i in range(never.n)]
        b.decode()
        boxes = [(w // 3, h // 4, max(1, w // 2), max(1, h // 2)) for w, h in (b.crop_frame(i) for i in range(b.n))]
        for k in range(3):
            b.set_crops(boxes if k != 1 else None)
            info = b.info()
            assert info.kernel_launches == plain_info.kernel_launches
            if k == 1:
                assert info.device_bytes == plain_info.device_bytes
            else:
                assert info.device_bytes > plain_info.device_bytes
            b.decode()
            assert np.array_equal(b.status(), plain_st)
            assert all(np.array_equal(b.coefs(i), c) for i, c in enumerate(plain_coefs))
            got = b.read_all_pixels()
            wants = plain if k == 1 else [_crop(p, bx, b2j.OUT_RGB24) for p, bx in zip(plain, boxes)]
            assert all(np.array_equal(g, w) for g, w in zip(got, wants)), k
        # the reference model and downscale are refused
        with pytest.raises(b2j.B2JError) as e:
            b.downscale(2)
        assert e.value.code == -1 and "crop" in str(e.value)
        b.set_pixel_model(b2j.PIXELS_REFERENCE)
        with pytest.raises(b2j.B2JError) as e:
            b.decode()
        assert e.value.code == -1 and "crop" in str(e.value)
        b.set_pixel_model(b2j.PIXELS_LIBJPEG)
        # a box that stops fitting after set_scale or set_orientations: the decode and the reads refuse, naming the image
        big = [(0, 0) + b.crop_frame(i) for i in range(b.n)]
        b.set_crops(big)
        b.set_scale(2)
        with pytest.raises(b2j.B2JError) as e:
            b.decode()
        assert e.value.code == -1 and "image 0" in str(e.value)
        with pytest.raises(b2j.B2JError):
            b.pixels(0)
        b.set_scale(1)
        b.decode()
        assert all(np.array_equal(g, w) for g, w in zip(b.read_all_pixels(), plain))
        tall = next(i for i in range(b.n) if big[i][2] != big[i][3])
        b.set_orientations([6 if i == tall else 1 for i in range(b.n)])
        with pytest.raises(b2j.B2JError) as e:
            b.decode()
        assert e.value.code == -1 and ("image %d" % tall) in str(e.value)
        b.set_orientations(None)
        b.decode()
        assert all(np.array_equal(g, w) for g, w in zip(b.read_all_pixels(), plain))
        # the setter's refusals change nothing
        launches, held = b.info().kernel_launches, b.info().device_bytes
        for bad in ((-1, 0, 1, 1), (0, -1, 1, 1), (0, 0, 0, 1), (0, 0, 1, 0)):
            arr = np.array([(0, 0, 1, 1)] * (b.n - 1) + [bad], np.int32)
            assert b.lib.b2j_batch_set_crops(b._h, arr.ctypes.data) == -1
        assert (b.info().kernel_launches, b.info().device_bytes) == (launches, held)
        b.decode()
        assert all(np.array_equal(g, w) for g, w in zip(b.read_all_pixels(), plain))
    finally:
        never.close()
        b.close()


@pytest.mark.parametrize("fmt_name", FORMATS)
def test_host_crop_into_one_arena_with_guards(decoder, full, fmt_name):
    """Neighbours in one pinned arena, so that downloads merge, with guard bytes: full-frame and cropped boxes mixed,
    one box outside its frame (status B2J_E_ARG, its neighbours decoded, its bytes untouched), and b2j_decode_host_ex
    unchanged."""
    import ocljpegdecoder_b200 as b2j
    fmt = getattr(b2j, fmt_name)
    for scale in (1, 2):
        ref = full[fmt_name, scale]
        frames = [(p.shape[-1], p.shape[-2]) if fmt == b2j.OUT_RGB_PLANAR else (p.shape[1], p.shape[0]) for p in ref]
        boxes = [(0, 0, fw, fh) if i % 2 else (fw // 5, fh // 3, max(1, fw - fw // 5 - 1), max(1, fh // 2)) for i, (fw, fh) in enumerate(frames)]
        bad = 4
        boxes[bad] = (1, 0) + frames[bad]   # one column too far
        wants = [_crop(p, bx, fmt) if i != bad else p[..., :0, :0] for i, (p, bx) in enumerate(zip(ref, boxes))]
        sizes = [w.nbytes for w in wants]
        guard = 37
        arena = b2j.PinnedBuffer(sum(sizes) + 2 * guard)
        try:
            arena.array[:] = 0xA5
            offs = guard + np.cumsum([0] + sizes)
            outs = [arena.address + int(o) for o in offs[:-1]]
            _, st = decoder.decode_host_ex(ITEMS, outs=outs, gate=_gate(), out_format=fmt, pixel_model=b2j.PIXELS_LIBJPEG, scale=scale, group=4,
                                           crops=boxes)
            assert st[bad] == -1 and not np.delete(st, bad).any(), st
            for i, w in enumerate(wants):
                got = arena.array[offs[i]:offs[i + 1]].reshape(w.shape)
                assert np.array_equal(got, w), (fmt_name, scale, i)
            assert (arena.array[:guard] == 0xA5).all() and (arena.array[-guard:] == 0xA5).all()
        finally:
            arena.close()
        plain, st = decoder.decode_host_ex(ITEMS, gate=_gate(), out_format=fmt, pixel_model=b2j.PIXELS_LIBJPEG, scale=scale, group=4)
        assert not st.any() and all(np.array_equal(g, w) for g, w in zip(plain, ref))
    # crops need the libjpeg model
    with pytest.raises(b2j.B2JError) as e:
        decoder.decode_host_ex(ITEMS[:1], gate=_gate(), out_format=b2j.OUT_RGB24, crops=[(0, 0, 1, 1)])
    assert e.value.code == -1


def test_65537_cropped_images(decoder):
    import ocljpegdecoder_b200 as b2j
    from test_gpu_libjpeg_limits import MANY_FILES, N_MANY
    c = len(MANY_FILES)
    files = [MANY_FILES[i % c] for i in range(N_MANY)]
    b = decoder.batch(files, gate=_gate())
    try:
        b.upload()
        b.set_pixel_model(b2j.PIXELS_LIBJPEG)
        for fmt in (b2j.OUT_RGB24, b2j.OUT_GRAY8):
            b.set_output_format(fmt)
            b.set_crops(None)
            b.decode()
            plain = [b.pixels(k) for k in range(c)]
            boxes = []
            for i in range(N_MANY):
                fw, fh = b.crop_frame(i)
                x, y = (i * 7) % fw, (i * 3) % fh
                boxes.append((x, y, 1 + (i % (fw - x)), 1 + ((i // 5) % (fh - y))))
            b.set_crops(boxes)
            b.decode()
            assert not b.status().any()
            got = b.read_all_pixels()
            bad = [i for i in range(N_MANY) if not np.array_equal(got[i], _crop(plain[i % c], boxes[i], fmt))]
            assert not bad, (fmt, len(bad), bad[:8])
    finally:
        b.close()
