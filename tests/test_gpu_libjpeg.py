"""GPU: the libjpeg pixel model (B2J_PIXELS_LIBJPEG) against Pillow and the numpy model (tests/libjpeg_model.py) on one
mixed batch -- everyday, gray and generic tiles, restart-interval and self-synchronising streams, a 1080p 4:2:0 and a 4K
4:4:4 frame whose tiles span MCU rows, and streams of extreme coefficients (against the model only: default Pillow's SIMD
IDCT differs there) -- in every output format; coefficients and status as in the reference model, switching back,
downscale, the host calls, caller-built gray descriptors and the refusal of an unknown model."""
import io

import numpy as np
import pytest

import jpegcraft
import libjpeg_model
import synth
from test_libjpeg_model import _gray_jpeg, extreme_streams

pytestmark = pytest.mark.gpu


def _craft(samp, w, h, seed, ri=0):
    q = [[2 + (i % 9) for i in range(64)], [3 + (i % 7) for i in range(64)]]
    return jpegcraft.encode_pixels(synth.synth_pixels(w, h, seed), samp, q, restart_interval=ri)[0]


def _items():
    """[(name, file bytes, gray)]; the names of files default Pillow is not compared with start with "x"."""
    return [
        ("s420_ri", synth.synth_jpeg(131, 77, 1, 85, "420", 3), False),
        ("s420_sync", synth.synth_jpeg(320, 200, 3, 75, "420", 0), False),
        ("s444", synth.synth_jpeg(96, 41, 2, 90, "444", 0), False),
        ("s422_ri", synth.synth_jpeg(203, 99, 4, 95, "422", 2), False),
        ("c440", _craft((1, 2), 57, 45, 5), False),
        ("c411_ri", _craft((4, 1), 77, 30, 6, ri=2), False),
        ("c14", _craft((1, 4), 35, 70, 7), False),
        ("c222121", _craft(((2, 2), (2, 1), (2, 1)), 45, 37, 8, ri=1), False),
        ("c221212", _craft(((2, 2), (1, 2), (1, 2)), 50, 33, 9), False),
        ("c21_narrow", _craft((2, 1), 3, 11, 10), False),
        ("gray_ri", _gray_jpeg(99, 61, 11, 80, 2), True),
        ("gray", _gray_jpeg(64, 33, 12, 90), True),
        ("hd420", synth.synth_jpeg(1920, 1080, 13, 90, "420", 0), False),
        ("uhd444", synth.synth_jpeg(3840, 2160, 14, 95, "444", 16), False),
    ] + [("x%d" % k, data, False) for k, data in enumerate(extreme_streams())]


ITEMS = _items()


def _gate():
    import ocljpegdecoder_b200 as b2j
    return b2j.GATE_EXTENDED | b2j.GATE_GRAY


@pytest.fixture(scope="module")
def expected(oracle):
    """Per item: (model RGB, Pillow RGB or None, oracle coefficients)."""
    from oracle import GATE_EXTENDED, GATE_GRAY
    from PIL import Image
    out = []
    for name, data, gray in ITEMS:
        model = libjpeg_model.decode_oracle(oracle, data, GATE_EXTENDED | GATE_GRAY)
        pil = None if name.startswith("x") else np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))
        oracle.set_strict(False)
        try:
            rc, _, coef, _ = oracle.decode(data, gate=GATE_EXTENDED | GATE_GRAY, want_pixels=False)
        finally:
            oracle.set_strict(True)
        assert rc == 0, name
        out.append((model, pil, coef))
    return out


@pytest.fixture(scope="module")
def batch(decoder):
    b = decoder.batch([it[1] for it in ITEMS], gate=_gate())
    b.upload()
    yield b
    b.close()


def _as_rgb(px, fmt):
    import ocljpegdecoder_b200 as b2j
    if fmt == b2j.OUT_BGRA:
        return px[..., 2::-1]
    if fmt == b2j.OUT_RGB_PLANAR:
        return np.moveaxis(px, 0, 2)
    return px


def test_model_equals_pillow_in_every_format(batch, expected):
    import ocljpegdecoder_b200 as b2j
    before = batch.info()
    batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
    try:
        for fmt in (b2j.OUT_BGRA, b2j.OUT_RGB24, b2j.OUT_RGB_PLANAR):
            batch.set_output_format(fmt)
            batch.decode()
            st = batch.status()
            assert not st.any(), [(ITEMS[i][0], int(st[i])) for i in np.nonzero(st)[0]]
            for i, (name, _, _) in enumerate(ITEMS):
                px = batch.pixels(i)
                if fmt == b2j.OUT_BGRA:
                    assert not px[..., 3].any(), name
                got = _as_rgb(px, fmt)
                model, pil, coef = expected[i]
                assert np.array_equal(got, model), (name, fmt, int((got != model).any(axis=2).sum()))
                assert pil is None or np.array_equal(got, pil), (name, fmt)
                assert np.array_equal(batch.coefs(i), coef), name
        after = batch.info()
        # two kernels instead of one per tile kind (three kinds here); the sample plane: 64 bytes per block
        assert before.kernel_launches - 3 + 2 == after.kernel_launches
        assert after.device_bytes >= before.device_bytes + 64 * before.total_blocks
    finally:
        batch.set_pixel_model(b2j.PIXELS_REFERENCE)
        batch.set_output_format(b2j.OUT_BGRA)
    assert batch.info().kernel_launches == before.kernel_launches


def test_switching_back_gives_the_reference_pixels(decoder, batch):
    import ocljpegdecoder_b200 as b2j
    files = [it[1] for it in ITEMS]
    fresh = decoder.batch(files, gate=_gate())
    try:
        fresh.upload()
        for fmt in (b2j.OUT_BGRA, b2j.OUT_RGB24):
            fresh.set_output_format(fmt)
            fresh.decode()
            want = [fresh.pixels(i) for i in range(len(files))]
            batch.set_output_format(fmt)
            batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
            batch.decode()
            batch.set_pixel_model(b2j.PIXELS_REFERENCE)
            batch.decode()
            assert not batch.status().any()
            for i in range(len(files)):
                assert np.array_equal(batch.pixels(i), want[i]), ITEMS[i][0]
                assert np.array_equal(batch.coefs(i), fresh.coefs(i)), ITEMS[i][0]
    finally:
        batch.set_output_format(b2j.OUT_BGRA)
        fresh.close()


@pytest.mark.parametrize("factor", [2, 8])
def test_downscale_in_the_libjpeg_model(batch, expected, factor):
    import ocljpegdecoder_b200 as b2j
    batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
    try:
        for fmt in (b2j.OUT_BGRA, b2j.OUT_RGB24):
            batch.set_output_format(fmt)
            batch.decode()
            batch.downscale(factor)
            for i, (name, _, _) in enumerate(ITEMS):
                want = libjpeg_model.box_filter(expected[i][0], factor)
                got = _as_rgb(batch.downscaled(i), fmt)
                assert np.array_equal(got, want), (name, fmt)
    finally:
        batch.set_pixel_model(b2j.PIXELS_REFERENCE)
        batch.set_output_format(b2j.OUT_BGRA)


def test_host_calls_in_the_libjpeg_model(decoder, expected):
    import ocljpegdecoder_b200 as b2j
    files = [it[1] for it in ITEMS]
    outs, st = decoder.decode_host_ex(files, gate=_gate(), out_format=b2j.OUT_RGB24, pixel_model=b2j.PIXELS_LIBJPEG, group=4)
    assert not st.any(), st
    for i, o in enumerate(outs):
        assert np.array_equal(o, expected[i][0]), ITEMS[i][0]
    outs, st = b2j.decode_host_multi([decoder], files, gate=_gate(), out_format=b2j.OUT_BGRA, pixel_model=b2j.PIXELS_LIBJPEG)
    assert not st.any(), st
    for i, o in enumerate(outs):
        assert np.array_equal(o[..., 2::-1], expected[i][0]), ITEMS[i][0]
    args = b2j.HostArgs(files, gate=_gate(), out_format=b2j.OUT_RGB_PLANAR, pixel_model=b2j.PIXELS_LIBJPEG)
    outs, st = decoder.decode_host_args(args)
    assert not st.any(), st
    for i, o in enumerate(outs):
        assert np.array_equal(np.moveaxis(o, 0, 2), expected[i][0]), ITEMS[i][0]


def test_unknown_pixel_model_is_refused(decoder, batch):
    import ocljpegdecoder_b200 as b2j
    for bad in (2, -1):
        with pytest.raises(b2j.B2JError) as e:
            batch.set_pixel_model(bad)
        assert e.value.code == -1
        with pytest.raises(b2j.B2JError) as e:
            decoder.decode_host_ex([ITEMS[0][1]], gate=_gate(), pixel_model=bad)
        assert e.value.code == -1
    # the batch still decodes the reference's pixels
    batch.decode()
    assert not batch.status().any()


def test_gray_descriptor_with_chroma_sampling_bytes(decoder, expected):
    """b2j_batch_create takes caller-built descriptors. A gray frame's sampling[1..2] carry nothing, and a descriptor
    with 0x11 there (the gray images last in the batch, so that a misplaced block would land behind the sample plane)
    decodes to the same pixels as the one b2j_parse_header builds, in both models."""
    import ocljpegdecoder_b200 as b2j
    k = [i for i, it in enumerate(ITEMS) if it[2]]
    files = [ITEMS[i][1] for i in k]
    plain = decoder.batch(files, gate=_gate())
    descs = (b2j.ImageDesc * len(files))()
    for j, f in enumerate(files):
        rc, d = b2j.parse_header(f, _gate())
        assert rc == 0 and list(d.sampling) == [0x11, 0, 0]
        d.sampling[1] = d.sampling[2] = 0x11
        descs[j] = d
    odd = b2j.Batch(decoder, files, descs)
    try:
        for b in (plain, odd):
            b.upload()
        for model in (b2j.PIXELS_REFERENCE, b2j.PIXELS_LIBJPEG):
            want = []
            for b in (plain, odd):
                b.set_pixel_model(model)
                b.decode()
                assert not b.status().any()
                want.append([b.pixels(j) for j in range(len(files))])
            for j, i in enumerate(k):
                assert np.array_equal(want[1][j], want[0][j]), (ITEMS[i][0], model)
                if model == b2j.PIXELS_LIBJPEG:
                    assert np.array_equal(want[1][j][..., 2::-1], expected[i][0]), ITEMS[i][0]
    finally:
        plain.close()
        odd.close()
