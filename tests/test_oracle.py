"""CPU: pins the oracle (oracle/oracle.c) against the reference's own fixture hashes, the committed
golden vectors, and the stored digests of the unmodified reference's output (tests/golden/reference_digests.json)."""
import hashlib
import json
import os

import numpy as np
import pytest

import jpegcraft
import synth
from conftest import GOLDEN

with open(os.path.join(GOLDEN, "golden.json")) as f:
    GOLD = json.load(f)


def _load(name):
    with open(os.path.join(GOLDEN, name + ".jpg"), "rb") as f:
        return f.read()


def test_fixture_hashes_match_survey(oracle, fixture_jpeg):
    # SURVEY.md 8(c): hashes of the reference CPU path on its own fixture
    rc, img, coef, bgra = oracle.decode(fixture_jpeg, gate=0)
    assert rc == 0
    assert (img.width, img.height, img.blk_count, img.mcu_count) == (313, 234, 1800, 300)
    assert hashlib.sha256(coef.tobytes()).hexdigest() == "c25806f5238c8ec7c2a4846cf6b67c5b567fd268599591392baf77e91023924e"
    assert hashlib.sha256(bgra.tobytes()).hexdigest() == "efb49cf99f2f6c583c546d6ef24c5d26ae339955c8bbe467341933aafa9b16e5"


@pytest.mark.parametrize("name", sorted(GOLD))
def test_oracle_matches_golden(oracle, name):
    data = _load(name)
    g = GOLD[name]
    assert hashlib.sha256(data).hexdigest() == g["file_sha256"]
    rc, img, coef, bgra = oracle.decode(data, gate=1 if g["needs_extended_gate"] else 0)
    assert rc == 0
    assert (img.width, img.height, img.blk_count) == (g["width"], g["height"], g["blk_count"])
    assert hashlib.sha256(coef.tobytes()).hexdigest() == g["coef_sha256"]
    assert hashlib.sha256(bgra.tobytes()).hexdigest() == g["pixel_sha256"]


def test_reference_gate_rejects_422(oracle):
    data = _load("g422_q85")
    rc, _ = oracle.parse(data, gate=0)
    assert rc == -2          # decoder.cpp:58-69 admits only 4:2:0 and 4:4:4
    rc, _ = oracle.parse(data, gate=1)
    assert rc == 0


def test_zigzag_is_standard(oracle):
    zz = oracle.zigzag()
    assert sorted(zz.tolist()) == list(range(64))
    assert zz[:10].tolist() == [0, 1, 8, 16, 9, 2, 3, 10, 17, 24] and zz[63] == 63


CASES = [(64, 48, "444", 75, 0, False), (67, 45, "420", 90, 0, False), (67, 45, "420", 90, 1, False),
         (200, 120, "420", 50, 3, True), (130, 70, "422", 85, 0, False), (130, 70, "422", 85, 2, True),
         (500, 375, "420", 75, 0, False), (333, 211, "444", 95, 5, True), (16, 16, "420", 100, 0, False),
         (640, 360, "420", 90, 16, False)]


def _sha(a):
    return hashlib.sha256(a if isinstance(a, bytes) else a.tobytes()).hexdigest()


def case_key(case):
    return "%dx%d_%s_q%d_ri%d%s" % (case[0], case[1], case[2], case[3], case[4], "_opt" if case[5] else "")


def case_jpeg(case):
    w, h, ss, q, ri, opt = case
    return synth.synth_jpeg(w, h, 500 + w + h, q, ss, ri, opt)


@pytest.mark.parametrize("case", CASES)
def test_oracle_matches_reference_build(oracle, reference_digests, case):
    want = reference_digests["oracle_cases"][case_key(case)]
    data = case_jpeg(case)
    assert _sha(data) == want["file_sha256"]
    rc, img, coef, bgra = oracle.decode(data, gate=1)
    assert want["ok"] == (rc == 0)
    if want["ok"]:
        assert _sha(coef) == want["coef_sha256"]
        assert _sha(bgra) == want["pixel_sha256"]


def rst_defect_jpegs():
    return [synth.synth_jpeg(640, 480, 900 + i, 90, "420", 1) for i in range(24)]   # 1200 restart markers per image


def test_oracle_reproduces_reference_rst_defect(oracle, reference_digests):
    """The reference drops an RSTn whose FF is the last byte of one of its 2 KiB reads and then
    aborts (decoder.cpp:118-131). strict mode predicts exactly those files; non-strict decodes them."""
    want = reference_digests["rst_defect"]
    files = rst_defect_jpegs()
    assert len(files) == len(want)
    n_fail = 0
    for data, w in zip(files, want):
        assert _sha(data) == w["file_sha256"]
        oracle.set_strict(True)
        rc_s, _, coef_s, _ = oracle.decode(data, want_pixels=False)
        oracle.set_strict(False)
        rc_n, _, coef_n, _ = oracle.decode(data, want_pixels=False)
        oracle.set_strict(True)
        assert w["ok"] == (rc_s == 0)
        assert rc_n == 0
        if w["ok"]:
            assert _sha(coef_s) == w["coef_sha256"] and _sha(coef_n) == w["coef_sha256"]
        else:
            n_fail += 1
    assert n_fail > 0   # with 1200 markers per image the defect shows up in this sample


def crafted_streams():
    """[(jpeg, blocks, quantisers, blocks per MCU, luma blocks per MCU)] in a fixed order."""
    rng = np.random.RandomState(5)
    out = []
    for sampling, (w, h) in (((2, 2), (48, 32)), ((1, 1), (24, 16)), ((2, 1), (48, 16))):
        ny = sampling[0] * sampling[1]
        tot = ny + 2
        n_mcu = ((w + 8 * sampling[0] - 1) // (8 * sampling[0])) * ((h + 8 * sampling[1] - 1) // (8 * sampling[1]))
        blocks = np.zeros((n_mcu * tot, 64), np.int64)
        for b in range(len(blocks)):
            kind = b % 5
            if kind == 0:      # full block, no EOB
                blocks[b, 1:] = rng.randint(1, 4, 63) * rng.choice([-1, 1], 63)
            elif kind == 1:    # ZRL chains: one coefficient far out
                blocks[b, 50 + b % 13] = rng.randint(-30, 30) or 7
            elif kind == 2:    # DC only
                pass
            elif kind == 3:    # big magnitudes
                blocks[b, 1:6] = rng.randint(-1023, 1023, 5)
            else:              # last coefficient set
                blocks[b, 63] = -1
        blocks[:, 0] = np.clip(np.cumsum(rng.randint(-300, 300, len(blocks))), -1000, 1000)
        q = [[1 + (i % 7) for i in range(64)], [2 + (i % 5) for i in range(64)]]
        for ri, fill in ((0, 0), (1, 0), (2, 3)):
            data = jpegcraft.build_jpeg(w, h, sampling, blocks, q, restart_interval=ri, fill_before_rst=fill)
            out.append((data, blocks, q, tot, ny))
    return out


def test_crafted_streams_oracle_vs_reference(oracle, reference_digests):
    want = reference_digests["crafted"]
    streams = crafted_streams()
    assert len(streams) == len(want)
    zz = oracle.zigzag()
    for (data, blocks, q, tot, ny), w in zip(streams, want):
        assert _sha(data) == w["file_sha256"]
        rc, img, coef, _ = oracle.decode(data, gate=1, want_pixels=False)
        assert rc == 0 and w["ok"]
        assert _sha(coef) == w["coef_sha256"]
        exp = np.zeros_like(coef)
        for b in range(len(blocks)):
            qq = np.array(q[0] if b % tot < ny else q[1])
            exp[b, zz] = blocks[b] * qq
        assert np.array_equal(coef, exp)


def test_grayscale_extension_against_pillow(oracle):
    """The oracle's one-component extension (GATE_GRAY; the reference refuses such files): the reference's loops
    with the chroma components absent. Pillow (libjpeg) is the independent check: same coefficients after
    dequantisation would be ideal, but libjpeg does not expose them -- pixels agree within +-2 (IDCT rounding)."""
    import io
    from PIL import Image
    import synth
    from oracle import GATE_GRAY, GATE_EXTENDED
    oracle.set_strict(False)
    try:
        for i, (w, h, q, ri) in enumerate([(131, 77, 75, 0), (64, 64, 50, 1), (9, 200, 95, 3), (320, 240, 90, 16)]):
            buf = io.BytesIO()
            kw = dict(format="JPEG", quality=q)
            if ri:
                kw["restart_marker_blocks"] = ri
            Image.fromarray(synth.synth_pixels(w, h, 60 + i)[:, :, 2], "L").save(buf, **kw)
            f = buf.getvalue()
            assert oracle.decode(f, gate=GATE_EXTENDED)[0] != 0
            rc, img, coef, bgra = oracle.decode(f, gate=GATE_EXTENDED | GATE_GRAY)
            assert rc == 0 and img.tot_blks_per_mcu == 1
            assert coef.shape == (((w + 7) // 8) * ((h + 7) // 8), 64)
            pil = np.asarray(Image.open(io.BytesIO(f)).convert("L"), dtype=np.int16)
            assert np.abs(bgra[..., 0].astype(np.int16) - pil).max() <= 2
            assert np.array_equal(bgra[..., 0], bgra[..., 1]) and np.array_equal(bgra[..., 1], bgra[..., 2]) and not bgra[..., 3].any()
    finally:
        oracle.set_strict(True)


GENERIC_LAYOUTS = [((4, 1), (1, 1), (1, 1)), ((1, 4), (1, 1), (1, 1)), ((3, 1), (1, 1), (1, 1)), ((4, 2), (1, 1), (1, 1)),
                   ((2, 4), (1, 1), (1, 1)), ((1, 3), (1, 1), (1, 1)), ((3, 2), (1, 1), (1, 1))]


def _random_blocks(n, seed):
    rng = np.random.RandomState(seed)
    blocks = np.zeros((n, 64), np.int64)
    blocks[:, 0] = np.clip(np.cumsum(rng.randint(-40, 40, n)), -500, 500)
    for b in range(n):
        k = rng.randint(0, 12)
        idx = rng.choice(np.arange(1, 64), k, replace=False)
        blocks[b, idx] = rng.randint(-30, 30, k)
    return blocks


def generic_luma_key(samp, ri):
    return "%d%d_ri%d" % (samp[0] + (ri,))


def generic_luma_jpeg(samp, ri):
    (h, v) = samp[0]
    w, hgt = 8 * h * 3 - 3, 8 * v * 2 - 1            # 3 x 2 MCUs, ragged right and bottom edges
    n = 6 * (h * v + 2)
    return jpegcraft.build_jpeg(w, hgt, samp, _random_blocks(n, 7 * h + v + ri), [[2 + (i % 5) for i in range(64)], [3] * 64], restart_interval=ri)


@pytest.mark.parametrize("samp", GENERIC_LAYOUTS, ids=lambda s: "%d%d" % s[0])
def test_generic_luma_sampling_oracle_vs_reference(oracle, reference_digests, samp):
    """Luma h x v beyond the four everyday layouts (4:1:1 = 41, 14, 31, 42, ...) with 1x1 chroma: the reference's gate
    refuses them, its CPU loops decode them as they are (decoder.cpp:429-495). Oracle (extended gate) against the
    unmodified reference with the gate skipped: coefficients and pixels bit-exact, with and without restart markers."""
    from oracle import GATE_EXTENDED
    for ri in (0, 2):
        want = reference_digests["generic_luma"][generic_luma_key(samp, ri)]
        data = generic_luma_jpeg(samp, ri)
        assert _sha(data) == want["file_sha256"]
        assert oracle.parse(data, 0)[0] != 0         # the reference gate refuses it
        rc, img, coef, bgra = oracle.decode(data, gate=GATE_EXTENDED)
        assert rc == 0
        assert want["ok"]
        assert _sha(coef) == want["coef_sha256"]
        assert _sha(bgra) == want["pixel_sha256"]


def test_multi_block_chroma_is_plain_replication(oracle):
    """Chroma components with several blocks per MCU (22,21,21 and 22,12,12; the reference stops with "Unsupported color
    space", decoder.cpp:486-490): the oracle's extension is the same pixel replication over the component's blocks.
    Checked against an independent numpy restatement built from the oracle's own coefficient tap."""
    import jpegcraft
    from oracle import GATE_EXTENDED
    for samp in (((2, 2), (2, 1), (2, 1)), ((2, 2), (1, 2), (1, 2)), ((4, 1), (2, 1), (2, 1)), ((2, 2), (2, 1), (1, 2))):
        tot = sum(a * b for a, b in samp)
        mw, mh = 8 * samp[0][0], 8 * samp[0][1]
        w, hgt = 2 * mw - 5, 2 * mh - 3
        data = jpegcraft.build_jpeg(w, hgt, samp, _random_blocks(4 * tot, 11), [[1 + (i % 3) for i in range(64)], [2] * 64])
        rc, img, coef, bgra = oracle.decode(data, gate=GATE_EXTENDED)
        assert rc == 0, samp
        # independent restatement: IDCT every block with the oracle's IDCT, assemble planes, replicate, convert
        planes = []
        first = 0
        for (a, b) in samp:
            pl = np.zeros((2 * 8 * b, 2 * 8 * a), np.int32)
            for my in range(2):
                for mx in range(2):
                    base = (my * 2 + mx) * tot + first
                    for k in range(a * b):
                        blk = oracle.idct(coef[base + k]).reshape(8, 8)
                        pl[my * 8 * b + (k // a) * 8:my * 8 * b + (k // a) * 8 + 8, mx * 8 * a + (k % a) * 8:mx * 8 * a + (k % a) * 8 + 8] = blk
            planes.append(pl)
            first += a * b
        Y = planes[0]
        U = np.repeat(np.repeat(planes[1], samp[0][1] // samp[1][1], axis=0), samp[0][0] // samp[1][0], axis=1)
        V = np.repeat(np.repeat(planes[2], samp[0][1] // samp[2][1], axis=0), samp[0][0] // samp[2][0], axis=1)
        for (x, y) in [(0, 0), (w - 1, hgt - 1), (w // 2, hgt // 2), (mw, mh - 1), (mw - 1, mh)]:
            want = oracle.yuv_to_rgb32(int(Y[y, x]), int(U[y, x]), int(V[y, x]))
            got = int(bgra[y, x, 0]) | int(bgra[y, x, 1]) << 8 | int(bgra[y, x, 2]) << 16
            assert got == want, (samp, x, y)
