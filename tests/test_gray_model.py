"""CPU: the numpy model of the libjpeg pixel model's grayscale output (B2J_OUT_GRAY8, libjpeg's JCS_GRAYSCALE:
libjpeg_gray_model) at scales 1, 2, 4 and 8, against Pillow's draft("L") on Pillow-written 4:4:4, 4:2:2, 4:2:0 and
gray files with and without restart markers, on jpegcraft layouts and on a 1080p frame; against OpenCV's IMREAD_GRAYSCALE /
IMREAD_REDUCED_GRAYSCALE_* and torchvision's decode_jpeg(mode=GRAY) on the Pillow files; and against libjpeg-turbo's C code
(JSIMD_FORCENONE=1) on streams of extreme coefficients. The GPU tests of GRAY8 take this model as their reference."""
import io
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import jpegcraft
import libjpeg_gray_model
import libjpeg_model
import synth
from test_libjpeg_model import _gray_jpeg, _ijg_tables, extreme_streams
from test_scaled_model import CRAFT_LAYOUTS, SIZES, _gate

PIL = pytest.importorskip("PIL.Image")

SCALES = (1, 2, 4, 8)


def _pillow_files():
    """[(name, bytes)]: the Pillow-written files of test_scaled_model.py, every sampling, with and without restart markers."""
    out = []
    for sub in ("444", "422", "420", "gray"):
        for ri in (0, 2):
            for k, (w, h) in enumerate(SIZES):
                q = (50, 75, 90, 100)[k % 4]
                seed = 100 * k + q
                data = _gray_jpeg(w, h, seed, q, ri) if sub == "gray" else synth.synth_jpeg(w, h, seed, q, sub, ri)
                out.append(("%s_ri%d_%dx%d" % (sub, ri, w, h), data))
    return out


def _draft_gray(data, scale):
    """Pillow's draft("L") decode, or None when the image is narrower or shorter than the scale (draft() cannot ask for it)."""
    from PIL import Image
    im = Image.open(io.BytesIO(data))
    w, h = im.size
    if w < scale or h < scale:
        return None
    im.draft("L", (w // scale, h // scale))
    assert im.mode == "L" and im.size == (-(-w // scale), -(-h // scale))
    return np.asarray(im)


def _check(oracle, data, scales=SCALES):
    from PIL import Image
    w, h = Image.open(io.BytesIO(data)).size
    for s in scales:
        got = libjpeg_gray_model.decode_oracle_gray(oracle, data, _gate(), s)
        assert got.dtype == np.uint8 and got.shape == (-(-h // s), -(-w // s)), (s, got.shape)
        want = _draft_gray(data, s)
        if want is not None:
            assert np.array_equal(got, want), (s, w, h, int((got != want).sum()))


@pytest.mark.parametrize("ri", [0, 2])
@pytest.mark.parametrize("sub", ["444", "422", "420", "gray"])
def test_gray_model_equals_pillow_draft_on_pillow_files(oracle, sub, ri):
    for k, (w, h) in enumerate(SIZES):
        q = (50, 75, 90, 100)[k % 4]
        seed = 100 * k + q
        _check(oracle, _gray_jpeg(w, h, seed, q, ri) if sub == "gray" else synth.synth_jpeg(w, h, seed, q, sub, ri))


def test_gray_model_equals_pillow_draft_on_a_1080p_frame(oracle):
    _check(oracle, synth.synth_jpeg(1920, 1080, 5, 90, "420", 0))


@pytest.mark.parametrize("ri", [0, 3])
@pytest.mark.parametrize("samp", CRAFT_LAYOUTS, ids=lambda s: "".join("%d%d" % x for x in jpegcraft._layout(s)))
def test_gray_model_equals_pillow_draft_on_jpegcraft_files(oracle, samp, ri):
    for k, (w, h) in enumerate([(5, 9), (35, 70), (77, 45), (203, 99)]):
        q = (60, 85, 95, 75)[k]
        data, _ = jpegcraft.encode_pixels(synth.synth_pixels(w, h, 11 * k + 3), samp, _ijg_tables(q), restart_interval=ri)
        _check(oracle, data)


def test_gray_model_is_the_luma_plane_of_the_rgb_model(oracle):
    """For a one-component file the RGB model repeats the gray plane in all three channels."""
    data = _gray_jpeg(99, 61, 11, 80, 2)
    for s in SCALES:
        rgb = libjpeg_model.decode_oracle(oracle, data, _gate(), s)
        assert np.array_equal(libjpeg_gray_model.decode_oracle_gray(oracle, data, _gate(), s), rgb[..., 0]), s


def test_gray_model_equals_opencv_reduced_grayscale(oracle):
    cv2 = pytest.importorskip("cv2")
    flags = {1: cv2.IMREAD_GRAYSCALE, 2: cv2.IMREAD_REDUCED_GRAYSCALE_2, 4: cv2.IMREAD_REDUCED_GRAYSCALE_4,
             8: cv2.IMREAD_REDUCED_GRAYSCALE_8}
    for name, data in _pillow_files():
        for s in SCALES:
            want = cv2.imdecode(np.frombuffer(data, np.uint8), flags[s])
            got = libjpeg_gray_model.decode_oracle_gray(oracle, data, _gate(), s)
            assert np.array_equal(got, want), (name, s, got.shape, want.shape)


def test_gray_model_equals_torchvision_decode_jpeg_gray(oracle):
    torch = pytest.importorskip("torch")
    io_ = pytest.importorskip("torchvision.io")
    for name, data in _pillow_files():
        want = io_.decode_jpeg(torch.frombuffer(bytearray(data), dtype=torch.uint8), mode=io_.ImageReadMode.GRAY).numpy()
        got = libjpeg_gray_model.decode_oracle_gray(oracle, data, _gate())
        assert want.shape == (1,) + got.shape and np.array_equal(got, want[0]), name


_DRAFT_CHILD = r"""
import json, sys
import numpy as np
from PIL import Image
for p, s in json.loads(sys.argv[1]):
    im = Image.open(p)
    im.draft("L", (im.size[0] // s, im.size[1] // s))
    np.save("%s.%d.npy" % (p, s), np.asarray(im))
"""


def test_gray_model_equals_libjpeg_c_code_on_extreme_coefficients(oracle, tmp_path):
    streams = extreme_streams()
    jobs = []
    for k, data in enumerate(streams):
        p = str(tmp_path / ("x%d.jpg" % k))
        with open(p, "wb") as f:
            f.write(data)
        jobs += [(p, s) for s in SCALES]
    env = dict(os.environ, JSIMD_FORCENONE="1")
    subprocess.check_call([sys.executable, "-c", _DRAFT_CHILD, json.dumps(jobs)], env=env)
    for k, data in enumerate(streams):
        for s in SCALES:
            want = np.load("%s.%d.npy" % (str(tmp_path / ("x%d.jpg" % k)), s))
            got = libjpeg_gray_model.decode_oracle_gray(oracle, data, _gate(), s)
            assert np.array_equal(got, want), (k, s, int((got != want).sum()))


def test_gray8_output_shapes(built):
    import ocljpegdecoder_b200 as b2j
    from ocljpegdecoder_b200.api import _out_shape
    assert b2j.OUT_GRAY8 == 3
    d = b2j.ImageDesc()
    d.width, d.height = 203, 99
    assert _out_shape(d, b2j.OUT_GRAY8) == (99, 203)
    assert [_out_shape(d, b2j.OUT_GRAY8, s) for s in (2, 4, 8)] == [(50, 102), (25, 51), (13, 26)]
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "b2j.h")) as f:
        assert "#define B2J_OUT_GRAY8 3" in f.read()
