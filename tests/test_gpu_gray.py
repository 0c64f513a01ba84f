"""GPU: B2J_OUT_GRAY8 in the libjpeg pixel model (libjpeg's grayscale output, k_idct_gray) on the mixed batch of
test_gpu_libjpeg.py -- everyday, generic and gray tiles, restart-interval and self-synchronising streams, a 3x11 image, a
1080p 4:2:0 and a 4K 4:4:4 frame and streams of extreme coefficients -- at scales 1, 2, 4 and 8, against the numpy model and
Pillow's draft("L"); status and coefficients, the launch count, the sample plane that GRAY8 does not allocate, switching
formats and scales, downscale, the host calls and the refusals."""
import numpy as np
import pytest

import libjpeg_gray_model
import libjpeg_model
from test_gpu_libjpeg import ITEMS, _gate
from test_gray_model import _draft_gray

pytestmark = pytest.mark.gpu

SCALES = (1, 2, 4, 8)


@pytest.fixture(scope="module")
def expected(oracle):
    """{scale: [(model gray, Pillow draft("L") or None)]}, the model's RGB at scale 1, and the oracle's coefficients per item."""
    from oracle import GATE_EXTENDED, GATE_GRAY
    gate = GATE_EXTENDED | GATE_GRAY
    px = {s: [] for s in SCALES}
    rgb, coefs = [], []
    for name, data, _ in ITEMS:
        img, coef = libjpeg_gray_model.oracle_coefs(oracle, data, gate)
        dims = (img.width, img.height, list(img.sampling), img.mcu_count_w, img.mcu_count_h)
        for s in SCALES:
            px[s].append((libjpeg_gray_model.decode_gray(coef, *dims, s), None if name.startswith("x") else _draft_gray(data, s)))
        rgb.append(libjpeg_model.decode_rgb(coef, *dims))
        coefs.append(coef)
    return px, rgb, coefs


def _libjpeg_batch(decoder):
    import ocljpegdecoder_b200 as b2j
    b = decoder.batch([it[1] for it in ITEMS], gate=_gate())
    b.upload()
    b.set_pixel_model(b2j.PIXELS_LIBJPEG)
    return b


@pytest.fixture(scope="module")
def batch(decoder):
    b = _libjpeg_batch(decoder)
    yield b
    b.close()


@pytest.mark.parametrize("scale", SCALES)
def test_gray8_equals_model_and_pillow_draft(batch, expected, scale):
    import ocljpegdecoder_b200 as b2j
    px, _, coefs = expected
    batch.set_scale(scale)
    batch.set_output_format(b2j.OUT_GRAY8)
    try:
        batch.decode()
        st = batch.status()
        assert not st.any(), [(ITEMS[i][0], int(st[i])) for i in np.nonzero(st)[0]]
        outs = batch.read_all_pixels()
        for i, (name, _, _) in enumerate(ITEMS):
            got = batch.pixels(i)
            model, pil = px[scale][i]
            assert got.shape == model.shape, (name, got.shape, model.shape)
            assert np.array_equal(got, outs[i]), name
            _, nbytes = batch.pixels_device(i)
            assert nbytes == got.nbytes == got.shape[0] * got.shape[1], name
            assert np.array_equal(got, model), (name, scale, int((got != model).sum()))
            assert pil is None or np.array_equal(got, pil), (name, scale)
            if scale == 1:
                assert np.array_equal(batch.coefs(i), coefs[i]), name
    finally:
        batch.set_scale(1)
        batch.set_output_format(b2j.OUT_BGRA)


def test_gray8_runs_one_kernel_and_no_sample_plane(decoder, expected):
    import ocljpegdecoder_b200 as b2j
    _, rgb, _ = expected
    b = _libjpeg_batch(decoder)
    try:
        held = b.info().device_bytes   # what a batch holds for the reference model
        b.set_output_format(b2j.OUT_RGB24)
        launches_rgb = b.info().kernel_launches
        b.set_output_format(b2j.OUT_GRAY8)
        assert b.info().kernel_launches == launches_rgb - 1
        for s in (1, 8, 2):
            b.set_scale(s)
            b.decode()
            assert not b.status().any()
        # a batch decoded only in GRAY8 holds what a reference-model batch holds: no sample plane
        assert b.info().device_bytes == held
        b.set_scale(1)
        b.set_output_format(b2j.OUT_RGB24)
        assert b.info().kernel_launches == launches_rgb
        b.decode()   # the first decode in a colour format allocates the sample plane
        assert not b.status().any()
        assert b.info().device_bytes >= held + 64 * b.info().total_blocks
        for i in range(len(ITEMS)):
            assert np.array_equal(b.pixels(i), rgb[i]), ITEMS[i][0]
    finally:
        b.close()


def test_alternating_formats_and_scales_gives_a_fresh_batch_pixels(decoder, batch, expected):
    import ocljpegdecoder_b200 as b2j
    px, rgb, _ = expected
    fresh = _libjpeg_batch(decoder)
    try:
        fresh.set_output_format(b2j.OUT_GRAY8)
        fresh.set_scale(2)
        fresh.decode()
        want = fresh.read_all_pixels()
        for fmt, s in ((b2j.OUT_GRAY8, 4), (b2j.OUT_RGB24, 1), (b2j.OUT_GRAY8, 2)):
            batch.set_output_format(fmt)
            batch.set_scale(s)
            batch.decode()
            assert not batch.status().any()
            if fmt == b2j.OUT_RGB24:
                for i in range(len(ITEMS)):
                    assert np.array_equal(batch.pixels(i), rgb[i]), ITEMS[i][0]
        for i in range(len(ITEMS)):
            got = batch.pixels(i)
            assert np.array_equal(got, want[i]) and np.array_equal(got, px[2][i][0]), ITEMS[i][0]
    finally:
        batch.set_scale(1)
        batch.set_output_format(b2j.OUT_BGRA)
        fresh.close()


def test_downscale_of_gray8(batch, expected):
    import ocljpegdecoder_b200 as b2j
    px, _, _ = expected
    batch.set_output_format(b2j.OUT_GRAY8)
    try:
        batch.decode()
        for factor in (2, 4, 8):
            batch.downscale(factor)
            for i, (name, _, _) in enumerate(ITEMS):
                want = libjpeg_model.box_filter(px[1][i][0], factor)
                got = batch.downscaled(i)
                assert got.shape == want.shape and np.array_equal(got, want), (name, factor)
    finally:
        batch.set_output_format(b2j.OUT_BGRA)


def test_host_calls_in_gray8(decoder, expected):
    import ocljpegdecoder_b200 as b2j
    px, _, _ = expected
    files = [it[1] for it in ITEMS]
    for s in (1, 2):
        # small groups: several batches, each with a packed pixel plane and merged downloads of neighbouring images
        outs, st = decoder.decode_host_ex(files, gate=_gate(), out_format=b2j.OUT_GRAY8, pixel_model=b2j.PIXELS_LIBJPEG, group=4, scale=s)
        assert not st.any(), st
        for i, o in enumerate(outs):
            assert np.array_equal(o, px[s][i][0]), (ITEMS[i][0], s)
    outs, st = b2j.decode_host_multi([decoder], files, gate=_gate(), out_format=b2j.OUT_GRAY8, pixel_model=b2j.PIXELS_LIBJPEG, group=3, scale=4)
    assert not st.any(), st
    for i, o in enumerate(outs):
        assert np.array_equal(o, px[4][i][0]), ITEMS[i][0]
    # one pinned arena whose outputs are neighbours at odd offsets: the downloads of a group merge
    for s in (1, 8):
        shapes = [px[s][i][0].shape for i in range(len(files))]
        sizes = [int(np.prod(sh)) for sh in shapes]
        assert any(n % 4 for n in sizes)
        arena = b2j.PinnedBuffer(sum(sizes) + 1)
        try:
            arena.array[-1] = 0xA5   # one guard byte behind the last image
            offs = np.cumsum([0] + sizes)
            args = b2j.HostArgs(files, outs=[arena.address + int(o) for o in offs[:-1]], gate=_gate(), out_format=b2j.OUT_GRAY8,
                                pixel_model=b2j.PIXELS_LIBJPEG, group=5, scale=s)
            _, st = decoder.decode_host_args(args)
            assert not st.any(), st
            for i, sh in enumerate(shapes):
                o = arena.array[offs[i]:offs[i + 1]].reshape(sh)
                assert np.array_equal(o, px[s][i][0]), (ITEMS[i][0], s)
            assert arena.array[-1] == 0xA5
        finally:
            arena.close()


def test_gray8_refusals_leave_the_batch_decoding(decoder, batch, expected):
    import ocljpegdecoder_b200 as b2j
    px, _, _ = expected
    data = ITEMS[0][1]
    out = [np.zeros(1 << 20, np.uint8)]

    def still_decodes():
        batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
        batch.set_output_format(b2j.OUT_GRAY8)
        batch.decode()
        assert not batch.status().any()
        assert np.array_equal(batch.pixels(0), px[1][0][0])

    try:
        for bad in (4, -1):
            with pytest.raises(b2j.B2JError) as e:
                batch.set_output_format(bad)
            assert e.value.code == -1
            with pytest.raises(b2j.B2JError) as e:
                decoder.decode_host_ex([data], outs=out, gate=_gate(), out_format=bad, pixel_model=b2j.PIXELS_LIBJPEG)
            assert e.value.code == -1
            still_decodes()
        # the reference pixel model has no grayscale output: accepted as a format, refused at decode
        with pytest.raises(b2j.B2JError) as e:
            decoder.decode_host_ex([data], outs=out, gate=_gate(), out_format=b2j.OUT_GRAY8, pixel_model=b2j.PIXELS_REFERENCE)
        assert e.value.code == -1
        still_decodes()
        batch.set_pixel_model(b2j.PIXELS_REFERENCE)
        with pytest.raises(b2j.B2JError) as e:
            batch.decode()
        assert e.value.code == -1 and "libjpeg pixel model" in str(e.value)
        still_decodes()
    finally:
        batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
        batch.set_output_format(b2j.OUT_BGRA)
