"""CPU: the numpy libjpeg pixel model (tests/libjpeg_model.py) against Pillow (libjpeg-turbo), fed the oracle's
coefficients: Pillow-written and jpegcraft-written files of every layout the model distinguishes, odd sizes, several
qualities, with and without restart markers; and streams with extreme coefficients against libjpeg-turbo's C code paths
(Pillow with JSIMD_FORCENONE=1). The GPU tests take this model as their reference."""
import io
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import jpegcraft
import libjpeg_model
import synth
from conftest import ROOT

PIL = pytest.importorskip("PIL.Image")

SIZES = [(1, 1), (3, 7), (4, 5), (5, 9), (6, 2), (17, 33), (200, 151), (313, 234), (640, 480)]
SMALL_SIZES = SIZES[:7]

# jpegcraft layouts: 4:2:2, 4:4:0, 4:1:1, 2x2, 1x4, 4x2, (22,12,12), (22,21,21);
# then what else the extended gate admits: luma factors of 3 (chroma replicated by 3, a DCT size that never doubles),
# 2x3, 2x4 (chroma h1v2 at 1/2), and Cb and Cr on layouts of their own, (41,21,21) and (22,21,12) (h2v1 beside h1v2)
CRAFT_LAYOUTS = [(2, 1), (1, 2), (4, 1), (2, 2), (1, 4), (4, 2), ((2, 2), (1, 2), (1, 2)), ((2, 2), (2, 1), (2, 1)),
                 (3, 1), (1, 3), (3, 2), (2, 3), (2, 4), ((4, 1), (2, 1), (2, 1)), ((2, 2), (2, 1), (1, 2))]


def _gate(gray=False):
    from oracle import GATE_EXTENDED, GATE_GRAY
    return GATE_EXTENDED | (GATE_GRAY if gray else 0)


def _pillow_rgb(data):
    from PIL import Image
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))


def _gray_jpeg(w, h, seed, quality, restart_mcus=0):
    from PIL import Image
    buf = io.BytesIO()
    kw = dict(format="JPEG", quality=quality)
    if restart_mcus:
        kw["restart_marker_blocks"] = restart_mcus
    Image.fromarray(synth.synth_pixels(w, h, seed)[:, :, 1], "L").save(buf, **kw)
    return buf.getvalue()


def _ijg_tables(quality):
    """The Annex K luma / chroma quantisers scaled like libjpeg's jpeg_quality_scaling, in zig-zag order."""
    luma = [16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29, 51, 87, 80, 62,
            18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99]
    chroma = [17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99] + [99] * 32
    scale = 5000 // quality if quality < 50 else 200 - 2 * quality
    out = []
    for t in (luma, chroma):
        nat = [min(max((q * scale + 50) // 100, 1), 255) for q in t]
        out.append([nat[z] for z in jpegcraft.ZIGZAG])
    return out


def _check(oracle, data, gray=False):
    want = _pillow_rgb(data)
    got = libjpeg_model.decode_oracle(oracle, data, _gate(gray))
    assert got.shape == want.shape
    assert np.array_equal(got, want), int((got != want).any(axis=2).sum())


@pytest.mark.parametrize("ri", [0, 2])
@pytest.mark.parametrize("sub", ["444", "422", "420", "gray"])
def test_model_equals_pillow_on_pillow_files(oracle, sub, ri):
    for k, (w, h) in enumerate(SIZES):
        for q in (50, 75, 90, 100):
            seed = 100 * k + q
            if sub == "gray":
                _check(oracle, _gray_jpeg(w, h, seed, q, ri), gray=True)
            else:
                _check(oracle, synth.synth_jpeg(w, h, seed, q, sub, ri))


@pytest.mark.parametrize("ri", [0, 3])
@pytest.mark.parametrize("samp", CRAFT_LAYOUTS, ids=lambda s: "".join("%d%d" % x for x in jpegcraft._layout(s)))
def test_model_equals_pillow_on_jpegcraft_files(oracle, samp, ri):
    sizes = SMALL_SIZES + ([(200, 151)] if ri else [(313, 234)])
    for k, (w, h) in enumerate(sizes):
        q = (50, 60, 75, 85, 90, 95, 100, 80)[k % 8]
        data, _ = jpegcraft.encode_pixels(synth.synth_pixels(w, h, 7 * k + 1), samp, _ijg_tables(q), restart_interval=ri)
        _check(oracle, data)


def extreme_streams():
    """Nine streams of random coefficients (AC up to +-300, +-600 and +-1023) in 4:4:4, 4:2:2 and 4:2:0, two of them with
    every quantiser 255: the values for which libjpeg-turbo's SIMD IDCT overflows its 16-bit lanes."""
    out = []
    for k, (samp, amp, q) in enumerate([((1, 1), 300, None), ((2, 1), 300, None), ((2, 2), 300, None),
                                        ((1, 1), 600, None), ((2, 1), 600, 255), ((2, 2), 600, None),
                                        ((1, 1), 1023, 255), ((2, 1), 1023, None), ((2, 2), 1023, None)]):
        rng = np.random.RandomState(900 + k)
        w, h = 24 + 5 * k, 17 + 3 * k
        mw, mh = 8 * samp[0], 8 * samp[1]
        n = -(-w // mw) * -(-h // mh) * (samp[0] * samp[1] + 2)
        blocks = rng.randint(-amp, amp + 1, size=(n, 64))
        blocks[:, 0] = rng.randint(-1000, 1001, size=n)
        qtabs = [[q] * 64] * 2 if q else [list(rng.randint(1, 256, size=64)) for _ in range(2)]
        out.append(jpegcraft.build_jpeg(w, h, samp, blocks, qtabs))
    return out


_DECODE_CHILD = r"""
import io, json, sys
import numpy as np
from PIL import Image
paths = json.loads(sys.argv[1])
for p in paths:
    with open(p, "rb") as f:
        a = np.asarray(Image.open(io.BytesIO(f.read())).convert("RGB"))
    np.save(p + ".npy", a)
"""


def _pillow_in_child(paths, simd):
    env = dict(os.environ)
    env.pop("JSIMD_FORCENONE", None)
    if not simd:
        env["JSIMD_FORCENONE"] = "1"
    subprocess.check_call([sys.executable, "-c", _DECODE_CHILD, json.dumps(paths)], env=env)
    return [np.load(p + ".npy") for p in paths]


def test_model_equals_libjpeg_c_code_on_extreme_coefficients(oracle, tmp_path, record_property):
    streams = extreme_streams()
    paths = []
    for k, data in enumerate(streams):
        p = str(tmp_path / ("x%d.jpg" % k))
        with open(p, "wb") as f:
            f.write(data)
        paths.append(p)
    c_path = _pillow_in_child(paths, simd=False)
    simd_path = _pillow_in_child(paths, simd=True)
    differ = 0
    for data, want, simd in zip(streams, c_path, simd_path):
        got = libjpeg_model.decode_oracle(oracle, data, _gate())
        assert np.array_equal(got, want), int((got != want).any(axis=2).sum())
        differ += int(not np.array_equal(simd, want))
    # the caveat the header states: with these coefficients default (SIMD) Pillow is not libjpeg-turbo's C code
    record_property("default_pillow_differs_on", "%d of %d streams" % (differ, len(streams)))
    with open("/proc/cpuinfo") as f:
        avx2 = " avx2" in f.read()
    if avx2:
        assert differ > 0


def test_abi_constants_and_host_opts_layout(built):
    import ctypes
    import ocljpegdecoder_b200 as b2j
    with open(os.path.join(ROOT, "include", "b2j.h")) as f:
        src = f.read()
    defines = dict(re.findall(r"#define (B2J_PIXELS_\w+) (\d+)", src))
    assert defines == {"B2J_PIXELS_REFERENCE": "0", "B2J_PIXELS_LIBJPEG": "1"}
    assert (b2j.PIXELS_REFERENCE, b2j.PIXELS_LIBJPEG) == (0, 1)
    assert b2j.HostOpts.pixel_model.offset == 20 and ctypes.sizeof(b2j.HostOpts) == 32
    assert "b2j_batch_set_pixel_model" in b2j.EXPORTED_SYMBOLS
