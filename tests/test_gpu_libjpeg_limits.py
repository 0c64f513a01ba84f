"""GPU: the libjpeg pixel model (B2J_PIXELS_LIBJPEG) at the edges of its geometry and of a batch, against the numpy model
(tests/libjpeg_model.py, tests/libjpeg_gray_model.py) fed the oracle's coefficients, and against Pillow's draft() on
encoder-written files (crafted blocks may meet the SIMD caveat of b2j.h, so those are compared with the model only).

- Every layout the extended gate admits: luma factors of 3 and 4, 2x3 and 2x4, Cb and Cr on layouts of their own; gray
  images of many tiles, one of them 99 pixels wide so that a tile covers fifteen MCU rows with partial first and last
  rows; generic and gray images whose tiles start in the middle of an MCU row; and runs of widths 1..40 that give
  ceil(W / s) every residue mod 4 at every scale. In BGRA, RGB24, RGB_PLANAR and GRAY8 at scales 1, 2, 4 and 8. The
  batch's descriptors are checked to contain what the test is about.
- 65537 images in one batch, more than a grid's y dimension (65535) holds: the upsampling and downscale kernels stride
  over images. RGB24 and GRAY8 at scales 1 and 8, downscale in both pixel models, and a host call whose last pipeline
  group holds 65536 images.
- One batch whose sample plane and pixel plane both extend past 2^32 bytes (125 4:4:4 frames of about 12 MP, about 21 GB
  of device memory; skipped when less is free), compared image by image in both pixel models.

The module took 47 s on an NVIDIA B200 at a 1000 W power limit, 30 s of it the 4 GiB test. Most of that time is the
numpy model, Pillow and the host-side comparisons.
"""
import ctypes

import numpy as np
import pytest

import libjpeg_gray_model
import libjpeg_model
import synth
from test_gpu_libjpeg import _as_rgb, _gate
from test_gray_model import _draft_gray
from test_layout_streams import GENERIC_LAYOUTS, MULTI_CHROMA_LAYOUTS, large_411_stream, layout_streams, make_stream
from test_libjpeg_model import _gray_jpeg
from test_scaled_model import _draft_rgb

pytestmark = pytest.mark.gpu

SCALES = (1, 2, 4, 8)
TILE_BLOCKS = 192   # kTileBlocks (ocljpegdecoder_b200/csrc/b2j_internal.h): a tile holds 192 // blocks-per-MCU MCUs


def _fmts():
    import ocljpegdecoder_b200 as b2j
    return (b2j.OUT_BGRA, b2j.OUT_RGB24, b2j.OUT_RGB_PLANAR, b2j.OUT_GRAY8)


def _model(oracle, data, scales):
    """{scale: (model RGB, model gray)} and the oracle's coefficients of one file."""
    img, coef = libjpeg_gray_model.oracle_coefs(oracle, data, _gate())
    dims = (img.width, img.height, list(img.sampling), img.mcu_count_w, img.mcu_count_h)
    return {s: (libjpeg_model.decode_rgb(coef, *dims, s), libjpeg_gray_model.decode_gray(coef, *dims, s)) for s in scales}, coef


# ---- every layout, many tiles, every output width residue -------------------------------------------------------------
EXTRA_LAYOUTS = [((2, 3), (1, 1), (1, 1))]   # admitted, and in neither list of test_layout_streams.py
RUN_LAYOUTS = [(2, 2), (3, 1), ((2, 2), (2, 1), (1, 2)), "gray"]


def _layout_items():
    """[(name, file bytes, encoder-written)]"""
    out = []
    for samp in GENERIC_LAYOUTS + MULTI_CHROMA_LAYOUTS + EXTRA_LAYOUTS:
        out += [(s.name, s.data, s.kind == "photo") for s in layout_streams(samp)]
    s = large_411_stream()
    out.append((s.name, s.data, True))
    out += [("s420", synth.synth_jpeg(333, 250, 31, 85, "420", 0), True),
            ("s422_ri3", synth.synth_jpeg(517, 77, 32, 90, "422", 3), True),
            ("s444", synth.synth_jpeg(250, 190, 33, 75, "444", 0), True),
            ("gray_99x1000", _gray_jpeg(99, 1000, 34, 85), True),
            ("gray_99x1000_ri7", _gray_jpeg(99, 1000, 35, 70, 7), True),
            ("gray_1920x1080", _gray_jpeg(1920, 1080, 36, 90), True)]
    for k, lay in enumerate(RUN_LAYOUTS):
        for w in range(1, 41):
            h, seed = 3 + (5 * w) % 19, 1000 * k + w
            if lay == "gray":
                out.append(("run_gray_w%d" % w, _gray_jpeg(w, h, seed, 80), True))
            else:
                s = make_stream("run_%d_w%d" % (k, w), lay, w, h, "photo", seed)
                out.append((s.name, s.data, True))
    return out


@pytest.fixture(scope="module")
def layout_items():
    return _layout_items()   # built on first use: writing the 1080p frames takes seconds


def _is_gray(d):
    return d.sampling[1] == 0


def _is_generic(d):
    return not _is_gray(d) and not (d.sampling[1] == d.sampling[2] == 0x11 and d.sampling[0] in (0x11, 0x21, 0x22, 0x12))


def _tiles(d):
    """The tiles b2j_batch_create cuts from an image, as (first MCU, last MCU)."""
    per = TILE_BLOCKS // d.tot_blks_per_mcu
    return [(m, min(m + per, d.mcu_count) - 1) for m in range(0, d.mcu_count, per)]


@pytest.fixture(scope="module")
def layout_expected(oracle, layout_items):
    """Per item: ({scale: (model RGB, model gray, Pillow RGB or None, Pillow gray or None)}, oracle coefficients)."""
    out = []
    for name, data, photo in layout_items:
        px, coef = _model(oracle, data, SCALES)
        out.append(({s: px[s] + ((_draft_rgb(data, s), _draft_gray(data, s)) if photo else (None, None)) for s in SCALES}, coef))
    return out


@pytest.fixture(scope="module")
def layout_batch(decoder, layout_items):
    import ocljpegdecoder_b200 as b2j
    b = decoder.batch([it[1] for it in layout_items], gate=_gate())
    b.upload()
    b.set_pixel_model(b2j.PIXELS_LIBJPEG)
    yield b
    b.close()


def test_layout_batch_covers_what_it_claims(layout_batch):
    """From the descriptors: generic and gray images with a tile that starts mid-row, tiles over three and more MCU rows
    (over ten in a gray image), every layout the model distinguishes, and every residue of ceil(W / s) mod 4 at every
    scale among generic and among gray images."""
    descs = [layout_batch.descs[i] for i in range(layout_batch.n)]
    mid = lambda d: any(m0 % d.mcu_count_w for m0, _ in _tiles(d))
    span = lambda d: max(m1 // d.mcu_count_w - m0 // d.mcu_count_w + 1 for m0, m1 in _tiles(d))
    assert any(mid(d) for d in descs if _is_generic(d)) and any(mid(d) for d in descs if _is_gray(d))
    assert any(span(d) >= 3 for d in descs if _is_generic(d)) and any(span(d) >= 10 for d in descs if _is_gray(d))
    assert any(len(_tiles(d)) >= 3 for d in descs if _is_generic(d))
    layouts = {tuple(d.sampling) for d in descs}
    for want in [(0x31, 0x11, 0x11), (0x13, 0x11, 0x11), (0x32, 0x11, 0x11), (0x23, 0x11, 0x11), (0x24, 0x11, 0x11),
                 (0x41, 0x21, 0x21), (0x22, 0x21, 0x12), (0x11, 0, 0)]:
        assert want in layouts, want
    for s in SCALES:
        for kind in (_is_generic, _is_gray):
            assert {-(-d.width // s) % 4 for d in descs if kind(d)} == {0, 1, 2, 3}, (s, kind.__name__)


@pytest.mark.parametrize("scale", SCALES)
def test_every_layout_in_every_format(layout_items, layout_batch, layout_expected, scale):
    import ocljpegdecoder_b200 as b2j
    layout_batch.set_scale(scale)
    try:
        for fmt in _fmts():
            layout_batch.set_output_format(fmt)
            layout_batch.decode()
            st = layout_batch.status()
            assert not st.any(), [(layout_items[i][0], int(st[i])) for i in np.nonzero(st)[0]]
            outs = layout_batch.read_all_pixels()
            for i, (name, _, _) in enumerate(layout_items):
                rgb, gray, pil_rgb, pil_gray = layout_expected[i][0][scale]
                got = outs[i]
                if fmt == b2j.OUT_GRAY8:
                    assert np.array_equal(got, gray), (name, scale, int((got != gray).sum()))
                    assert pil_gray is None or np.array_equal(got, pil_gray), (name, scale)
                    continue
                if fmt == b2j.OUT_BGRA:
                    assert not got[..., 3].any(), name
                got = _as_rgb(got, fmt)
                assert np.array_equal(got, rgb), (name, scale, fmt, int((got != rgb).any(axis=2).sum()))
                assert pil_rgb is None or np.array_equal(got, pil_rgb), (name, scale, fmt)
                if fmt == b2j.OUT_RGB24 and scale == 1:
                    assert np.array_equal(layout_batch.coefs(i), layout_expected[i][1]), name
    finally:
        layout_batch.set_scale(1)
        layout_batch.set_output_format(b2j.OUT_BGRA)


# ---- more than 65535 images -------------------------------------------------------------------------------------------
N_MANY = 65537
N_HOST = 131070   # groups of 2, 4, ..., 32768 images (65534), then one of 65536


def _many_files():
    """Seven distinct small files (a prime cycle), every one a different size: everyday, factor-3 and mixed-chroma
    layouts, gray, with and without restart markers."""
    return [synth.synth_jpeg(17, 9, 41, 85, "420", 0),
            _gray_jpeg(13, 7, 42, 80),
            make_stream("many_31", (3, 1), 29, 11, "photo", 43).data,
            synth.synth_jpeg(21, 6, 44, 90, "422", 1),
            make_stream("many_22_21_12", ((2, 2), (2, 1), (1, 2)), 19, 18, "photo", 45, 2).data,
            _gray_jpeg(5, 3, 46, 95, 1),
            synth.synth_jpeg(11, 13, 47, 75, "444", 0)]


MANY_FILES = _many_files()


def _cycled(n, shapes):
    """Output arrays for n images whose shapes cycle through `shapes`: one array [count, *shape] per distinct file, and
    the address of every image's place in them."""
    c = len(shapes)
    arrs = [np.full(((n - k + c - 1) // c,) + tuple(shapes[k]), 0xA5, np.uint8) for k in range(c)]
    return arrs, [arrs[i % c].ctypes.data + (i // c) * arrs[i % c].strides[0] for i in range(n)]


def _assert_cycled(arrs, wants, what):
    c = len(arrs)
    for k, (a, w) in enumerate(zip(arrs, wants)):
        assert a.shape[1:] == w.shape, (what, k, a.shape, w.shape)
        bad = np.nonzero((a != w[None]).reshape(len(a), -1).any(axis=1))[0]
        assert len(bad) == 0, (what, "file %d" % k, "%d images differ, first" % len(bad), [k + c * int(j) for j in bad[:8]])


@pytest.fixture(scope="module")
def many_expected(oracle):
    """Per distinct file: {scale: (model RGB, model gray)} at 1 and 8, the model RGB box-filtered by 2, the oracle's
    BGRA (the reference model) box-filtered by 2, and the oracle's coefficients."""
    from oracle import GATE_EXTENDED, GATE_GRAY
    out = []
    for data in MANY_FILES:
        px, coef = _model(oracle, data, (1, 8))
        rc, _, _, bgra = oracle.decode(data, gate=GATE_EXTENDED | GATE_GRAY)
        assert rc == 0
        out.append((px, libjpeg_model.box_filter(px[1][0], 2), libjpeg_model.box_filter(bgra, 2), coef))
    return out


@pytest.fixture(scope="module")
def many_batch(decoder):
    b = decoder.batch([MANY_FILES[i % len(MANY_FILES)] for i in range(N_MANY)], gate=_gate())
    b.upload()
    yield b
    b.close()


@pytest.mark.parametrize("scale", [1, 8])
def test_more_than_65535_images(many_batch, many_expected, scale):
    import ocljpegdecoder_b200 as b2j
    b = many_batch
    b.set_pixel_model(b2j.PIXELS_LIBJPEG)
    b.set_scale(scale)
    try:
        for fmt in (b2j.OUT_RGB24, b2j.OUT_GRAY8):
            b.set_output_format(fmt)
            b.decode()
            st = b.status()
            assert not st.any(), np.nonzero(st)[0][:8]
            wants = [e[0][scale][0 if fmt == b2j.OUT_RGB24 else 1] for e in many_expected]
            arrs, addrs = _cycled(N_MANY, [w.shape for w in wants])
            b.read_all_pixels(addrs)
            _assert_cycled(arrs, wants, (scale, fmt))
        c = len(MANY_FILES)
        for i in list(range(c)) + list(range(N_MANY - c, N_MANY)):
            assert np.array_equal(b.coefs(i), many_expected[i % c][3]), i
    finally:
        b.set_scale(1)
        b.set_output_format(b2j.OUT_BGRA)
        b.set_pixel_model(b2j.PIXELS_REFERENCE)


def test_downscale_of_more_than_65535_images(many_batch, many_expected):
    """b2j_batch_downscale(2) over every image in both pixel models: a grid of one row of CTAs per image would exceed
    CUDA's limit on gridDim.y."""
    import ocljpegdecoder_b200 as b2j
    b = many_batch
    try:
        for model, fmt, k in ((b2j.PIXELS_LIBJPEG, b2j.OUT_RGB24, 1), (b2j.PIXELS_REFERENCE, b2j.OUT_BGRA, 2)):
            b.set_pixel_model(model)
            b.set_output_format(fmt)
            b.decode()
            assert not b.status().any()
            b.downscale(2)
            wants = [e[k] for e in many_expected]
            arrs, addrs = _cycled(N_MANY, [w.shape for w in wants])
            for i, a in enumerate(addrs):
                rc = b.lib.b2j_batch_read_downscaled(b._h, None, i, ctypes.c_void_p(a))
                assert rc == 0, (i, rc)
            _assert_cycled(arrs, wants, ("downscale", model))
    finally:
        b.set_output_format(b2j.OUT_BGRA)
        b.set_pixel_model(b2j.PIXELS_REFERENCE)


def test_host_call_with_a_group_of_65536_images(decoder, many_expected):
    """b2j_decode_host_ex ramps its first groups up (2, 4, 8, ... images); with no bound on images or bytes per group
    its last group here holds 65536 images, decoded as one batch."""
    import ocljpegdecoder_b200 as b2j
    c = len(MANY_FILES)
    wants = [e[0][1][0] for e in many_expected]
    arrs, addrs = _cycled(N_HOST, [w.shape for w in wants])
    args = b2j.HostArgs([MANY_FILES[i % c] for i in range(N_HOST)], outs=addrs, gate=_gate(), out_format=b2j.OUT_RGB24, group=N_HOST,
                        group_mb=4096, pixel_model=b2j.PIXELS_LIBJPEG)
    _, st = decoder.decode_host_args(args)
    assert not st.any(), np.nonzero(st)[0][:8]
    _assert_cycled(arrs, wants, "host")


# ---- planes past 4 GiB ------------------------------------------------------------------------------------------------
BIG_SIZES = [(4001, 2999), (3967, 3011), (4093, 2897)]   # unequal and not powers of two: a wrapped offset lands elsewhere
N_BIG = 125
BIG_DEVICE_BYTES = 24 << 30


def test_planes_past_4_gib(oracle):
    """125 4:4:4 frames of about 12 MP, cycling three files: 70 M blocks, so the sample plane (64 bytes per block) and
    the pixel plane (4 bytes per pixel) extend past 2^32 bytes. The reference model's BGRA goes first, so that a byte
    the libjpeg model's decode does not write differs from what it should be."""
    torch = pytest.importorskip("torch")
    free, _ = torch.cuda.mem_get_info()
    if free < BIG_DEVICE_BYTES:
        pytest.skip("needs %.1f GB of free device memory, %.1f GB free" % (BIG_DEVICE_BYTES / 1e9, free / 1e9))
    import ocljpegdecoder_b200 as b2j
    from oracle import GATE_EXTENDED, GATE_GRAY
    files = [synth.synth_jpeg(w, h, 50 + k, 75, "444", 0) for k, (w, h) in enumerate(BIG_SIZES)]
    want = []
    for data in files:
        px, coef = _model(oracle, data, (1, 8))
        rc, _, _, bgra = oracle.decode(data, gate=GATE_EXTENDED | GATE_GRAY)
        assert rc == 0
        want.append(dict(bgra=bgra, rgb1=px[1][0], rgb8=px[8][0], gray1=px[1][1], box=libjpeg_model.box_filter(px[1][0], 2), coef=coef))
    c = len(files)
    dec = b2j.Decoder(0)   # its own context: the pool's 21 GB go back when it closes
    b = dec.batch([files[i % c] for i in range(N_BIG)], gate=_gate())
    try:
        b.upload()
        b.decode()
        assert not b.status().any()
        first, _ = b.pixels_device(0)
        last, _ = b.pixels_device(N_BIG - 1)
        info = b.info()
        print("blocks %d, sample plane %.2f GB, last image's pixels at byte %.2f G" % (info.total_blocks, 64 * info.total_blocks / 1e9, (last - first) / 1e9))
        assert 64 * info.total_blocks > 1 << 32 and last - first > 1 << 32

        def check(key, read):
            for i in range(N_BIG):
                got, w = read(i), want[i % c][key]
                assert got.shape == w.shape and np.array_equal(got, w), (key, i, int((got != w).sum()))

        check("bgra", b.pixels)
        b.set_pixel_model(b2j.PIXELS_LIBJPEG)
        b.set_output_format(b2j.OUT_RGB24)
        b.decode()
        assert not b.status().any()
        assert b.info().device_bytes >= info.device_bytes + 64 * info.total_blocks   # the sample plane
        check("rgb1", b.pixels)
        b.downscale(2)
        check("box", b.downscaled)
        b.set_scale(8)
        b.decode()
        assert not b.status().any()
        check("rgb8", b.pixels)
        b.set_scale(1)
        b.set_output_format(b2j.OUT_GRAY8)
        b.decode()
        assert not b.status().any()
        check("gray1", b.pixels)
        for i in range(N_BIG - c, N_BIG):   # past 2^32 bytes of the coefficient plane too
            assert np.array_equal(b.coefs(i), want[i % c]["coef"]), i
    finally:
        b.close()
        dec.close()
