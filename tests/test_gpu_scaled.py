"""GPU: the libjpeg pixel model's scaled decode (b2j_batch_set_scale 2, 4, 8) on the mixed batch of test_gpu_libjpeg.py --
everyday, generic and gray tiles, restart-interval and self-synchronising streams, a 3x11 image, a 1080p 4:2:0 and a 4K
4:4:4 frame and streams of extreme coefficients -- in every output format, against the numpy model and Pillow's draft();
coefficients and status as at full size, the return to scale 1, the host calls with a scale, and the refusals."""
import io

import numpy as np
import pytest

import libjpeg_model
from test_gpu_libjpeg import ITEMS, _as_rgb, _gate

pytestmark = pytest.mark.gpu

SCALES = (2, 4, 8)


def _draft(data, s):
    """Pillow's scaled decode, or None where draft() cannot ask for this scale (image narrower or shorter than s)."""
    from PIL import Image
    im = Image.open(io.BytesIO(data))
    w, h = im.size
    if w < s or h < s:
        return None
    im.draft("RGB", (w // s, h // s))
    assert im.size == (-(-w // s), -(-h // s))
    return np.asarray(im.convert("RGB"))


@pytest.fixture(scope="module")
def expected(oracle):
    """{scale: [(model RGB, Pillow draft RGB or None)]} and the oracle's coefficients per item."""
    from oracle import GATE_EXTENDED, GATE_GRAY
    gate = GATE_EXTENDED | GATE_GRAY
    px = {s: [] for s in SCALES}
    coefs = []
    for name, data, _ in ITEMS:
        for s in SCALES:
            pil = None if name.startswith("x") else _draft(data, s)
            px[s].append((libjpeg_model.decode_oracle(oracle, data, gate, s), pil))
        oracle.set_strict(False)
        try:
            rc, _, coef, _ = oracle.decode(data, gate=gate, want_pixels=False)
        finally:
            oracle.set_strict(True)
        assert rc == 0, name
        coefs.append(coef)
    return px, coefs


@pytest.fixture(scope="module")
def batch(decoder):
    import ocljpegdecoder_b200 as b2j
    b = decoder.batch([it[1] for it in ITEMS], gate=_gate())
    b.upload()
    b.set_pixel_model(b2j.PIXELS_LIBJPEG)
    b.decode()   # the first decode in this model allocates the sample plane; the scaled decodes add nothing to it
    yield b
    b.close()


@pytest.mark.parametrize("scale", SCALES)
def test_scaled_decode_equals_model_and_pillow_draft(batch, expected, scale):
    import ocljpegdecoder_b200 as b2j
    px, coefs = expected
    before = batch.info()
    batch.set_scale(scale)
    try:
        for fmt in (b2j.OUT_BGRA, b2j.OUT_RGB24, b2j.OUT_RGB_PLANAR):
            batch.set_output_format(fmt)
            batch.decode()
            st = batch.status()
            assert not st.any(), [(ITEMS[i][0], int(st[i])) for i in np.nonzero(st)[0]]
            outs = batch.read_all_pixels()
            for i, (name, _, _) in enumerate(ITEMS):
                got = batch.pixels(i)
                assert np.array_equal(got, outs[i]), (name, fmt)
                _, nbytes = batch.pixels_device(i)
                assert nbytes == got.nbytes, name
                if fmt == b2j.OUT_BGRA:
                    assert not got[..., 3].any(), name
                got = _as_rgb(got, fmt)
                model, pil = px[scale][i]
                assert np.array_equal(got, model), (name, scale, fmt, int((got != model).any(axis=2).sum()))
                assert pil is None or np.array_equal(got, pil), (name, scale, fmt)
                if fmt == b2j.OUT_RGB24:
                    assert np.array_equal(batch.coefs(i), coefs[i]), name
        after = batch.info()
        assert (after.kernel_launches, after.device_bytes, after.pixel_bytes) == (before.kernel_launches, before.device_bytes, before.pixel_bytes)
    finally:
        batch.set_scale(1)
        batch.set_output_format(b2j.OUT_BGRA)


def test_scale_one_after_a_scaled_decode_gives_a_fresh_batch_pixels(decoder, batch):
    import ocljpegdecoder_b200 as b2j
    files = [it[1] for it in ITEMS]
    fresh = decoder.batch(files, gate=_gate())
    try:
        fresh.upload()
        fresh.set_pixel_model(b2j.PIXELS_LIBJPEG)
        fresh.set_output_format(b2j.OUT_RGB24)
        fresh.decode()
        want = fresh.read_all_pixels()
        batch.set_output_format(b2j.OUT_RGB24)
        batch.set_scale(8)
        batch.decode()
        batch.set_scale(1)
        batch.decode()
        assert not batch.status().any()
        for i in range(len(files)):
            assert np.array_equal(batch.pixels(i), want[i]), ITEMS[i][0]
    finally:
        batch.set_output_format(b2j.OUT_BGRA)
        fresh.close()


def test_host_calls_with_a_scale(decoder, expected):
    import ocljpegdecoder_b200 as b2j
    px, _ = expected
    files = [it[1] for it in ITEMS]
    # small groups: several batches, each with a packed pixel plane and merged downloads of neighbouring images
    outs, st = decoder.decode_host_ex(files, gate=_gate(), out_format=b2j.OUT_RGB24, pixel_model=b2j.PIXELS_LIBJPEG, group=4, scale=2)
    assert not st.any(), st
    for i, o in enumerate(outs):
        assert np.array_equal(o, px[2][i][0]), ITEMS[i][0]
    outs, st = b2j.decode_host_multi([decoder], files, gate=_gate(), out_format=b2j.OUT_BGRA, pixel_model=b2j.PIXELS_LIBJPEG, group=3, scale=4)
    assert not st.any(), st
    for i, o in enumerate(outs):
        assert not o[..., 3].any() and np.array_equal(o[..., 2::-1], px[4][i][0]), ITEMS[i][0]
    # one pinned arena whose outputs are neighbours: the downloads of a group merge
    shapes = [(3,) + px[8][i][0].shape[:2] for i in range(len(files))]
    arena = b2j.PinnedBuffer(sum(int(np.prod(s)) for s in shapes))
    try:
        offs = np.cumsum([0] + [int(np.prod(s)) for s in shapes])
        args = b2j.HostArgs(files, outs=[arena.address + int(o) for o in offs[:-1]], gate=_gate(), out_format=b2j.OUT_RGB_PLANAR,
                            pixel_model=b2j.PIXELS_LIBJPEG, group=5, scale=8)
        _, st = decoder.decode_host_args(args)
        assert not st.any(), st
        for i, s in enumerate(shapes):
            o = arena.array[offs[i]:offs[i + 1]].reshape(s)
            assert np.array_equal(np.moveaxis(o, 0, 2), px[8][i][0]), ITEMS[i][0]
    finally:
        arena.close()


def test_refusals_leave_the_batch_decoding(decoder, batch):
    import ocljpegdecoder_b200 as b2j
    data = ITEMS[0][1]
    out = [np.zeros(1 << 20, np.uint8)]
    for bad in (0, 3, 16, -1):
        with pytest.raises(b2j.B2JError) as e:
            batch.set_scale(bad)
        assert e.value.code == -1
        if bad:   # 0 in the host options means 1
            with pytest.raises(b2j.B2JError) as e:
                decoder.decode_host_ex([data], outs=out, gate=_gate(), pixel_model=b2j.PIXELS_LIBJPEG, scale=bad)
            assert e.value.code == -1
    # the reference pixel model has no scaled decode
    with pytest.raises(b2j.B2JError) as e:
        decoder.decode_host_ex([data], outs=out, gate=_gate(), pixel_model=b2j.PIXELS_REFERENCE, scale=2)
    assert e.value.code == -1
    batch.set_scale(2)
    try:
        batch.set_pixel_model(b2j.PIXELS_REFERENCE)
        with pytest.raises(b2j.B2JError) as e:
            batch.decode()
        assert e.value.code == -1 and "libjpeg pixel model" in str(e.value)
        batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
        batch.decode()
        with pytest.raises(b2j.B2JError) as e:
            batch.downscale(2)
        assert e.value.code == -1
    finally:
        batch.set_scale(1)
        batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
    outs, st = decoder.decode_host_ex([data], gate=_gate(), pixel_model=b2j.PIXELS_LIBJPEG, scale=0)
    _, d = b2j.parse_header(data, _gate())
    assert not st.any() and outs[0].shape == (d.height, d.width, 4)
    batch.decode()
    assert not batch.status().any()
    batch.downscale(2)
