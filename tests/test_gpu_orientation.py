"""GPU: EXIF orientation (b2j_batch_set_orientations, k_orient, b2j_host_opts.exif_orientation).

One batch of mixed layouts -- 4:2:0, 4:2:2, 4:4:4, a generic layout and gray, odd sizes, 1xN and Nx1 images, images of
many tiles -- with code-1 images interleaved with oriented ones, in every format at scales 1, 2, 4 and 8 in the libjpeg
model and at scale 1 in the reference model, for every code: each result is the numpy transform of the same batch's
unoriented decode. Then EXIF-tagged files against OpenCV's imdecode (default flags, IMREAD_GRAYSCALE, IMREAD_REDUCED_*),
torchvision's decode_jpeg(apply_exif_orientation=True) and Pillow's exif_transpose() of draft(); switching codes, the way
back to None (launches, device bytes, pixels), downscale's refusal; the host calls into one pinned arena with guard bytes;
and 65537 images cycling the eight codes."""
import ctypes
import io

import numpy as np
import pytest

import synth
from test_gpu_libjpeg import _craft
from test_gray_model import _draft_gray
from test_libjpeg_model import _gray_jpeg
from test_orientation_parse import orient
from test_scaled_model import _draft_rgb

pytestmark = pytest.mark.gpu

SCALES = (1, 2, 4, 8)


def _items():
    return [
        synth.synth_jpeg(131, 77, 1, 85, "420", 3),
        synth.synth_jpeg(203, 99, 4, 95, "422", 2),
        synth.synth_jpeg(96, 41, 2, 90, "444", 0),
        _craft(((2, 2), (2, 1), (2, 1)), 45, 37, 8, ri=1),
        _gray_jpeg(99, 61, 11, 80, 2),
        synth.synth_jpeg(1, 37, 21, 90, "420", 0),
        synth.synth_jpeg(29, 1, 22, 90, "444", 0),
        _gray_jpeg(1, 23, 23, 85),
        _gray_jpeg(17, 1, 24, 85),
        synth.synth_jpeg(701, 477, 25, 90, "420", 0),   # 11 x 8 tiles at full size
        _craft((2, 1), 3, 11, 10),
    ]


ITEMS = _items()


def _gate():
    import ocljpegdecoder_b200 as b2j
    return b2j.GATE_EXTENDED | b2j.GATE_GRAY


def _codes(code, n):
    """`code` for most images, 1 for every third (interleaved)."""
    return np.array([code if (i + code) % 3 else 1 for i in range(n)], np.uint8)


def _oriented(a, code, fmt):
    import ocljpegdecoder_b200 as b2j
    if fmt == b2j.OUT_RGB_PLANAR:
        return np.stack([orient(p, code) for p in a])
    return orient(a, code)


@pytest.fixture(scope="module")
def batch(decoder):
    b = decoder.batch(ITEMS, gate=_gate())
    b.upload()
    yield b
    b.close()


def _settings():
    import ocljpegdecoder_b200 as b2j
    lj, ref = b2j.PIXELS_LIBJPEG, b2j.PIXELS_REFERENCE
    out = [(lj, f, s) for s in SCALES for f in (b2j.OUT_BGRA, b2j.OUT_RGB24, b2j.OUT_RGB_PLANAR, b2j.OUT_GRAY8)]
    return out + [(ref, f, 1) for f in (b2j.OUT_BGRA, b2j.OUT_RGB24, b2j.OUT_RGB_PLANAR)]


@pytest.mark.parametrize("setting", range(19))
def test_every_code_is_the_transform_of_the_unoriented_decode(batch, setting):
    import ocljpegdecoder_b200 as b2j
    model, fmt, scale = _settings()[setting]
    batch.set_pixel_model(model)
    batch.set_output_format(fmt)
    batch.set_scale(scale)
    try:
        batch.set_orientations(None)
        batch.decode()
        assert not batch.status().any()
        base = batch.read_all_pixels()
        launches = batch.info().kernel_launches
        for code in range(1, 9):
            codes = _codes(code, batch.n)
            batch.set_orientations(codes)
            assert batch.info().kernel_launches == launches + (code != 1)
            batch.decode()
            assert not batch.status().any()
            got = batch.read_all_pixels()
            for i in range(batch.n):
                want = _oriented(base[i], int(codes[i]), fmt)
                assert got[i].shape == want.shape and np.array_equal(got[i], want), (setting, code, i)
                _, nbytes = batch.pixels_device(i)
                assert nbytes == want.nbytes
            for i in (0, batch.n - 1):
                assert np.array_equal(batch.pixels(i), got[i])
    finally:
        batch.set_orientations(None)
        batch.set_scale(1)
        batch.set_output_format(b2j.OUT_BGRA)
        batch.set_pixel_model(b2j.PIXELS_REFERENCE)


def test_switching_codes_and_going_back(decoder, batch):
    import ocljpegdecoder_b200 as b2j
    batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
    batch.set_output_format(b2j.OUT_RGB24)
    try:
        batch.decode()
        before = batch.info()
        base = batch.read_all_pixels()
        rng = np.random.default_rng(3)
        for k in range(6):
            codes = rng.integers(1, 9, batch.n).astype(np.uint8)
            batch.set_orientations(codes)
            if k == 3:   # a format change moves the copies and rebuilds the tile table
                batch.set_output_format(b2j.OUT_GRAY8)
                batch.decode()
                gray = batch.read_all_pixels()
                batch.set_orientations(None)
                batch.decode()
                assert all(np.array_equal(orient(g, int(c)), w) for g, c, w in zip(batch.read_all_pixels(), codes, gray))
                batch.set_orientations(codes)
                batch.set_output_format(b2j.OUT_RGB24)
            assert batch.info().kernel_launches == before.kernel_launches + 1
            assert batch.info().device_bytes > before.device_bytes
            batch.decode()
            for i, g in enumerate(batch.read_all_pixels()):
                assert np.array_equal(g, orient(base[i], int(codes[i]))), (k, i)
            with pytest.raises(b2j.B2JError) as e:
                batch.downscale(2)
            assert e.value.code == -1 and "orient" in str(e.value)
        # codes all 1 is the unoriented decode; a bad code changes nothing
        for bad in (0, 9, 255):
            with pytest.raises(b2j.B2JError):
                batch.set_orientations([bad] * batch.n)
        assert batch.info().kernel_launches == before.kernel_launches + 1
        for codes in (np.ones(batch.n, np.uint8), None):
            batch.set_orientations(codes)
            after = batch.info()
            assert (after.kernel_launches, after.device_bytes) == (before.kernel_launches, before.device_bytes)
            batch.decode()
            assert all(np.array_equal(g, w) for g, w in zip(batch.read_all_pixels(), base))
        batch.downscale(2)
        assert batch.downscaled(0).shape == (39, 66, 3)
    finally:
        batch.set_orientations(None)
        batch.set_output_format(b2j.OUT_BGRA)
        batch.set_pixel_model(b2j.PIXELS_REFERENCE)


def test_timed_decode_counts_the_pass(batch):
    import ocljpegdecoder_b200 as b2j
    batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
    batch.set_output_format(b2j.OUT_RGB24)
    try:
        batch.set_orientations(_codes(6, batch.n))
        t = batch.decode_timed()
        assert t.idct_ms > 0 and t.total_ms >= t.idct_ms
        per, total = batch.decode_steps(3)
        assert all(p.idct_ms > 0 for p in per) and total > 0
    finally:
        batch.set_orientations(None)
        batch.set_output_format(b2j.OUT_BGRA)
        batch.set_pixel_model(b2j.PIXELS_REFERENCE)


# ---- the libraries, on EXIF-tagged files ------------------------------------------------------------------------------
def _tagged(code, layout, w, h, seed):
    from PIL import Image
    px = synth.synth_pixels(w, h, seed)
    im = Image.fromarray(px[:, :, 0], "L") if layout == "gray" else Image.fromarray(px)
    ex = Image.Exif()
    ex[0x0112] = code
    b = io.BytesIO()
    im.save(b, "JPEG", quality=90, exif=ex.tobytes(), **({} if layout == "gray" else dict(subsampling=layout)))
    return b.getvalue()


TAGGED = [_tagged(code, layout, w, h, 30 + code)
          for code in range(0, 10) for layout, (w, h) in ((2, (53, 37)), (1, (41, 29)), (0, (37, 53)), ("gray", (45, 31)))]


@pytest.mark.parametrize("scale", SCALES)
def test_host_call_equals_opencv_torchvision_and_pillow(decoder, scale):
    cv2 = pytest.importorskip("cv2")
    import torch
    from PIL import Image, ImageOps
    from torchvision.io import ImageReadMode, decode_jpeg
    import ocljpegdecoder_b200 as b2j
    cv_rgb = {1: cv2.IMREAD_COLOR, 2: cv2.IMREAD_REDUCED_COLOR_2, 4: cv2.IMREAD_REDUCED_COLOR_4, 8: cv2.IMREAD_REDUCED_COLOR_8}[scale]
    cv_gray = {1: cv2.IMREAD_GRAYSCALE, 2: cv2.IMREAD_REDUCED_GRAYSCALE_2, 4: cv2.IMREAD_REDUCED_GRAYSCALE_4,
               8: cv2.IMREAD_REDUCED_GRAYSCALE_8}[scale]
    kw = dict(gate=_gate(), pixel_model=b2j.PIXELS_LIBJPEG, scale=scale, exif_orientation=True, group=5)
    rgb, st = decoder.decode_host_ex(TAGGED, out_format=b2j.OUT_RGB24, **kw)
    assert not st.any()
    gray, st = decoder.decode_host_ex(TAGGED, out_format=b2j.OUT_GRAY8, **kw)
    assert not st.any()
    for k, data in enumerate(TAGGED):
        buf = np.frombuffer(data, np.uint8)
        assert np.array_equal(rgb[k], cv2.imdecode(buf, cv_rgb)[..., ::-1]), (k, scale)
        assert np.array_equal(gray[k], cv2.imdecode(buf, cv_gray)), (k, scale)
        code = b2j.parse_orientation(data)
        assert np.array_equal(rgb[k], orient(_draft_rgb(data, scale), code)), (k, scale)
        assert np.array_equal(gray[k], orient(_draft_gray(data, scale), code)), (k, scale)
        if scale == 1:
            t = torch.frombuffer(bytearray(data), dtype=torch.uint8)
            assert np.array_equal(rgb[k], decode_jpeg(t, mode=ImageReadMode.RGB, apply_exif_orientation=True).permute(1, 2, 0).numpy()), k
            assert np.array_equal(gray[k], decode_jpeg(t, mode=ImageReadMode.GRAY, apply_exif_orientation=True)[0].numpy()), k
            assert np.array_equal(rgb[k], np.asarray(ImageOps.exif_transpose(Image.open(io.BytesIO(data))).convert("RGB"))), k


@pytest.mark.parametrize("fmt_name", ["OUT_RGB24", "OUT_GRAY8", "OUT_RGB_PLANAR", "OUT_BGRA"])
def test_host_calls_into_one_arena_with_guards(decoder, batch, fmt_name):
    """Odd-sized neighbours in one pinned arena, so that downloads merge, with guard bytes in front and behind: every
    output is the oriented image, no guard byte changes; with exif_orientation off the outputs are the unoriented ones."""
    import ocljpegdecoder_b200 as b2j
    fmt = getattr(b2j, fmt_name)
    files = [f for f in TAGGED[::3]] + ITEMS
    codes = [b2j.parse_orientation(f) for f in files]
    assert len(set(codes)) == 8
    ref = decoder.batch(files, gate=_gate())
    try:
        ref.upload()
        ref.set_pixel_model(b2j.PIXELS_LIBJPEG)
        ref.set_output_format(fmt)
        for scale in (1, 4):
            ref.set_scale(scale)
            ref.decode()
            plain = ref.read_all_pixels()
            for on in (True, False):
                wants = [_oriented(p, c, fmt) if on else p for p, c in zip(plain, codes)]
                sizes = [w.nbytes for w in wants]
                guard = 37
                arena = b2j.PinnedBuffer(sum(sizes) + 2 * guard)
                try:
                    arena.array[:] = 0xA5
                    offs = guard + np.cumsum([0] + sizes)
                    outs = [arena.address + int(o) for o in offs[:-1]]
                    kw = dict(outs=outs, gate=_gate(), out_format=fmt, pixel_model=b2j.PIXELS_LIBJPEG, scale=scale, exif_orientation=on)
                    for call in range(2):
                        arena.array[guard:-guard] = 0
                        if call == 0:
                            _, st = decoder.decode_host_args(b2j.HostArgs(files, group=6, **kw))
                        else:
                            _, st = b2j.decode_host_multi([decoder], files, group=4, **kw)
                        assert not st.any(), st
                        for i, w in enumerate(wants):
                            got = arena.array[offs[i]:offs[i + 1]].reshape(w.shape)
                            assert np.array_equal(got, w), (fmt_name, scale, on, call, i)
                        assert (arena.array[:guard] == 0xA5).all() and (arena.array[-guard:] == 0xA5).all()
                finally:
                    arena.close()
    finally:
        ref.close()
    # b2j_decode_host_ex refuses an exif_orientation other than 0 and 1
    args = b2j.HostArgs(files[:1], gate=_gate())
    args.opts.exif_orientation = 2
    with pytest.raises(b2j.B2JError) as e:
        decoder.decode_host_args(args)
    assert e.value.code == -1


# ---- more than 65535 oriented images ----------------------------------------------------------------------------------
def test_65537_images_cycling_the_codes(decoder):
    import ocljpegdecoder_b200 as b2j
    from test_gpu_libjpeg_limits import MANY_FILES, N_MANY
    c = len(MANY_FILES)
    files = [MANY_FILES[i % c] for i in range(N_MANY)]
    codes = np.array([i % 8 + 1 for i in range(N_MANY)], np.uint8)
    b = decoder.batch(files, gate=_gate())
    try:
        b.upload()
        b.set_pixel_model(b2j.PIXELS_LIBJPEG)
        for fmt in (b2j.OUT_RGB24, b2j.OUT_GRAY8):
            b.set_output_format(fmt)
            b.set_orientations(None)
            b.decode()
            plain = [b.pixels(k) for k in range(c)]
            b.set_orientations(codes)
            b.decode()
            assert not b.status().any()
            got = b.read_all_pixels()
            bad = [i for i in range(N_MANY) if not np.array_equal(got[i], orient(plain[i % c], int(codes[i])))]
            assert not bad, (fmt, len(bad), bad[:8])
    finally:
        b.close()


def test_refusals_change_nothing(batch):
    L = batch.lib
    assert L.b2j_batch_set_orientations(None, None) == -1
    launches, held = batch.info().kernel_launches, batch.info().device_bytes
    codes = np.full(batch.n, 6, np.uint8)
    codes[-1] = 0
    assert L.b2j_batch_set_orientations(batch._h, codes.ctypes.data) == -1
    assert (batch.info().kernel_launches, batch.info().device_bytes) == (launches, held)
    with pytest.raises(ValueError):
        batch.set_orientations([6] * (batch.n + 1))
    batch.decode()
    assert not batch.status().any() and batch.pixels(0).shape == (77, 131, 4)
