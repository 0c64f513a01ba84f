"""CPU: the numpy model of the libjpeg pixel model's scaled decode (tests/libjpeg_model.py) against
Pillow's draft() (libjpeg-turbo's scale_denom 2, 4, 8) on Pillow-written 4:4:4, 4:2:2, 4:2:0 and gray files with and without
restart markers and on jpegcraft layouts, and against libjpeg-turbo's C code (JSIMD_FORCENONE=1) on streams of extreme
coefficients. The GPU tests of the scaled decode take this model as their reference."""
import io
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import jpegcraft
import libjpeg_model
import synth
from test_libjpeg_model import _gray_jpeg, _ijg_tables, extreme_streams

PIL = pytest.importorskip("PIL.Image")

SCALES = (2, 4, 8)
SIZES = [(1, 1), (3, 7), (9, 5), (17, 33), (131, 77), (203, 99), (640, 480)]
# 4:2:2, 4:4:0, 4:1:1, 2x2, 1x4, 4x2, (22,12,12), (22,21,21);
# then what else the extended gate admits: luma factors of 3 (chroma replicated by 3, a DCT size that never doubles),
# 2x3, 2x4 (chroma h1v2 at 1/2), and Cb and Cr on layouts of their own, (41,21,21) and (22,21,12) (h2v1 beside h1v2)
CRAFT_LAYOUTS = [(2, 1), (1, 2), (4, 1), (2, 2), (1, 4), (4, 2), ((2, 2), (1, 2), (1, 2)), ((2, 2), (2, 1), (2, 1)),
                 (3, 1), (1, 3), (3, 2), (2, 3), (2, 4), ((4, 1), (2, 1), (2, 1)), ((2, 2), (2, 1), (1, 2))]


def _gate():
    from oracle import GATE_EXTENDED, GATE_GRAY
    return GATE_EXTENDED | GATE_GRAY


def _draft_rgb(data, scale):
    """Pillow's scaled decode, or None when the image is narrower or shorter than the scale (draft() cannot ask for it)."""
    from PIL import Image
    im = Image.open(io.BytesIO(data))
    w, h = im.size
    if w < scale or h < scale:
        return None
    im.draft("RGB", (w // scale, h // scale))
    assert im.size == (-(-w // scale), -(-h // scale))
    return np.asarray(im.convert("RGB"))


def _check(oracle, data, scales=SCALES):
    from PIL import Image
    w, h = Image.open(io.BytesIO(data)).size
    for s in scales:
        got = libjpeg_model.decode_oracle(oracle, data, _gate(), s)
        assert got.shape == (-(-h // s), -(-w // s), 3), (s, got.shape)
        want = _draft_rgb(data, s)
        if want is not None:
            assert np.array_equal(got, want), (s, w, h, int((got != want).any(axis=2).sum()))


@pytest.mark.parametrize("ri", [0, 2])
@pytest.mark.parametrize("sub", ["444", "422", "420", "gray"])
def test_scaled_model_equals_pillow_draft_on_pillow_files(oracle, sub, ri):
    for k, (w, h) in enumerate(SIZES):
        q = (50, 75, 90, 100)[k % 4]
        seed = 100 * k + q
        _check(oracle, _gray_jpeg(w, h, seed, q, ri) if sub == "gray" else synth.synth_jpeg(w, h, seed, q, sub, ri))


def test_scaled_model_equals_pillow_draft_on_a_1080p_frame(oracle):
    _check(oracle, synth.synth_jpeg(1920, 1080, 5, 90, "420", 0))


@pytest.mark.parametrize("ri", [0, 3])
@pytest.mark.parametrize("samp", CRAFT_LAYOUTS, ids=lambda s: "".join("%d%d" % x for x in jpegcraft._layout(s)))
def test_scaled_model_equals_pillow_draft_on_jpegcraft_files(oracle, samp, ri):
    for k, (w, h) in enumerate([(5, 9), (35, 70), (77, 45), (203, 99)]):
        q = (60, 85, 95, 75)[k]
        data, _ = jpegcraft.encode_pixels(synth.synth_pixels(w, h, 11 * k + 3), samp, _ijg_tables(q), restart_interval=ri)
        _check(oracle, data)


_DRAFT_CHILD = r"""
import io, json, sys
import numpy as np
from PIL import Image
for p, s in json.loads(sys.argv[1]):
    im = Image.open(p)
    im.draft("RGB", (im.size[0] // s, im.size[1] // s))
    np.save("%s.%d.npy" % (p, s), np.asarray(im.convert("RGB")))
"""


def test_scaled_model_equals_libjpeg_c_code_on_extreme_coefficients(oracle, tmp_path):
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
            got = libjpeg_model.decode_oracle(oracle, data, _gate(), s)
            assert np.array_equal(got, want), (k, s, int((got != want).any(axis=2).sum()))


def test_host_opts_scale_field(built):
    import ctypes
    import ocljpegdecoder_b200 as b2j
    assert b2j.HostOpts.pixel_model.offset == 20 and b2j.HostOpts.scale.offset == 24 and ctypes.sizeof(b2j.HostOpts) == 32
    assert "b2j_batch_set_scale" in b2j.EXPORTED_SYMBOLS
