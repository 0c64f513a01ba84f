"""GPU: parity of the CUDA path (through the C ABI) against the oracle, the golden vectors and
the reference build where it travelled. Bar: coefficients bit-exact; pixels within +-1 per channel
of the cpuIDCT8x8 path (north_star) -- the integer colour path is designed to be exact, so the
tests assert max |d| <= 1 AND report/assert the mismatch fraction (expected 0)."""
import hashlib
import json
import os

import numpy as np
import pytest

import jpegcraft
import synth
from conftest import GOLDEN

pytestmark = pytest.mark.gpu

with open(os.path.join(GOLDEN, "golden.json")) as f:
    GOLD = json.load(f)


def _load(name):
    with open(os.path.join(GOLDEN, name + ".jpg"), "rb") as f:
        return f.read()


def _decode(decoder, files):
    batch = decoder.batch(files)
    batch.upload()
    batch.decode()
    st = batch.status()
    coefs = [batch.coefs(i) for i in range(len(files))]
    pix = [batch.pixels(i) for i in range(len(files))]
    batch.close()
    return st, coefs, pix


def _check_pixels(got, want):
    d = np.abs(got.astype(np.int16) - want.astype(np.int16))
    frac = float((d > 0).mean())
    assert d.max() <= 1, "pixel difference above +-1 (max %d)" % d.max()
    assert frac == 0.0, "pixel mismatch fraction %.3e (within +-1 but the integer path should be exact)" % frac


def test_golden_vectors(decoder):
    names = sorted(GOLD)
    files = [_load(n) for n in names]
    st, coefs, pix = _decode(decoder, files)
    assert not st.any(), st
    for n, c, p in zip(names, coefs, pix):
        g = GOLD[n]
        assert c.shape == (g["blk_count"], 64) and p.shape == (g["height"], g["width"], 4)
        assert hashlib.sha256(c.tobytes()).hexdigest() == g["coef_sha256"], n
        assert hashlib.sha256(p.tobytes()).hexdigest() == g["pixel_sha256"], n


def test_reference_fixture_hashes(decoder, fixture_jpeg):
    st, coefs, pix = _decode(decoder, [fixture_jpeg])
    assert st[0] == 0
    assert hashlib.sha256(coefs[0].tobytes()).hexdigest() == "c25806f5238c8ec7c2a4846cf6b67c5b567fd268599591392baf77e91023924e"
    assert hashlib.sha256(pix[0].tobytes()).hexdigest() == "efb49cf99f2f6c583c546d6ef24c5d26ae339955c8bbe467341933aafa9b16e5"


SPECS = [(64, 48, "444", 75, 0, False), (67, 45, "420", 90, 0, False), (67, 45, "420", 90, 1, False),
         (200, 120, "420", 50, 3, True), (130, 70, "422", 85, 0, False), (130, 70, "422", 85, 2, True),
         (640, 480, "420", 90, 16, False), (640, 480, "444", 95, 7, True), (333, 211, "444", 95, 5, False),
         (500, 375, "420", 75, 0, False), (16, 16, "420", 100, 0, False), (8, 8, "444", 10, 0, False),
         (1, 1, "420", 90, 0, False), (17, 9, "422", 60, 1, False), (1023, 31, "420", 35, 5, True),
         (31, 1023, "444", 99, 2, False), (1920, 1080, "420", 90, 16, False), (1280, 720, "422", 85, 40, False)]


def test_synthetic_mixed_batch_against_oracle(decoder, oracle):
    """All layouts, odd sizes, optimised/standard tables, RI dividing and not dividing the MCU row,
    decoded as ONE batch (one launch per kernel for all of them)."""
    files = [synth.synth_jpeg(w, h, 300 + i, q, ss, ri, opt) for i, (w, h, ss, q, ri, opt) in enumerate(SPECS)]
    st, coefs, pix = _decode(decoder, files)
    assert not st.any(), st
    oracle.set_strict(False)
    try:
        for f, c, p in zip(files, coefs, pix):
            rc, img, coef, bgra = oracle.decode(f)
            assert rc == 0
            assert np.array_equal(c, coef)
            _check_pixels(p, bgra)
    finally:
        oracle.set_strict(True)


def reference_build_jpegs():
    return [synth.synth_jpeg(w, h, 700 + i, q, ss, ri, opt) for i, (w, h, ss, q, ri, opt) in enumerate(SPECS[:12])]


def test_against_reference_build(decoder, reference_digests):
    """Coefficients and pixels against the digests of the unmodified reference's output (pixels: equal digests is the
    exact match that _check_pixels asks for)."""
    want = reference_digests["gpu_batch"]
    files = reference_build_jpegs()
    assert [hashlib.sha256(f).hexdigest() for f in files] == [w["file_sha256"] for w in want]
    st, coefs, pix = _decode(decoder, files)
    assert not st.any()
    n_checked = 0
    for w, c, p in zip(want, coefs, pix):
        if not w["ok"]:
            continue   # the reference's own RSTn-at-chunk-end defect (see test_oracle.py)
        assert hashlib.sha256(c.tobytes()).hexdigest() == w["coef_sha256"]
        assert hashlib.sha256(p.tobytes()).hexdigest() == w["pixel_sha256"]
        n_checked += 1
    assert n_checked >= 8


def _crafted(sampling, w, h, ri, fill, seed, stuffed=False):
    rng = np.random.RandomState(seed)
    ny = sampling[0] * sampling[1]
    tot = ny + 2
    n_mcu = ((w + 8 * sampling[0] - 1) // (8 * sampling[0])) * ((h + 8 * sampling[1] - 1) // (8 * sampling[1]))
    blocks = np.zeros((n_mcu * tot, 64), np.int64)
    for b in range(len(blocks)):
        kind = (b + seed) % 6
        if kind == 0:
            blocks[b, 1:] = rng.randint(1, 4, 63) * rng.choice([-1, 1], 63)      # all 63 AC set, no EOB
        elif kind == 1:
            blocks[b, 50 + b % 13] = int(rng.randint(1, 30))                     # ZRL chains
        elif kind == 3:
            blocks[b, 1:6] = rng.randint(-1023, 1023, 5)                         # maximum baseline magnitudes
        elif kind == 4:
            blocks[b, 63] = -1
        elif kind == 5 and stuffed:
            blocks[b, 1:40] = -1 if b % 2 else 1                                 # long runs of 1 bits -> FF00 stuffing
    dc = np.cumsum(rng.randint(-300, 300, len(blocks)))
    blocks[:, 0] = np.clip(dc, -1000, 1000)
    if len(blocks) > 8:
        src = blocks[1::7, 0].copy()
        blocks[0:7 * len(src):7, 0] = src                                        # DC difference 0 (category 0)
    else:
        blocks[::7, 0] = 0
    q = [[1 + (i % 7) for i in range(64)], [2 + (i % 5) for i in range(64)]]
    return jpegcraft.build_jpeg(w, h, sampling, blocks, q, restart_interval=ri, fill_before_rst=fill)


def test_crafted_edge_streams(decoder, oracle):
    files = []
    for sampling, (w, h) in (((2, 2), (80, 48)), ((1, 1), (40, 24)), ((2, 1), (80, 24)), ((1, 2), (40, 48))):
        for ri, fill in ((0, 0), (1, 0), (2, 3), (9, 1)):
            files.append(_crafted(sampling, w, h, ri, fill, seed=len(files), stuffed=True))
    st, coefs, pix = _decode(decoder, files)
    assert not st.any(), st
    oracle.set_strict(False)
    try:
        for f, c, p in zip(files, coefs, pix):
            rc, img, coef, bgra = oracle.decode(f)
            assert rc == 0
            assert f.count(b"\xff\x00") > 0
            assert np.array_equal(c, coef)
            # crafted blocks drive the IDCT far outside [-256,255]; the reference's clip table only
            # covers +-512 (cpuIDCT8x8.cpp:13-23, undefined beyond), the oracle and the GPU both clamp
            _check_pixels(p, bgra)
    finally:
        oracle.set_strict(True)


def test_many_restart_intervals_wrap_mod8(decoder, oracle):
    # 2400 intervals in one image: RSTn numbering wraps 300 times; several CTAs per image
    f = synth.synth_jpeg(1280, 480, 77, 85, "420", 1)
    st, coefs, pix = _decode(decoder, [f])
    assert st[0] == 0
    oracle.set_strict(False)
    try:
        rc, _, coef, bgra = oracle.decode(f)
    finally:
        oracle.set_strict(True)
    assert rc == 0 and np.array_equal(coefs[0], coef)
    _check_pixels(pix[0], bgra)


def test_corrupt_streams_are_flagged(decoder, oracle):
    good = synth.synth_jpeg(320, 240, 5, 90, "420", 4)
    rc, d = oracle.parse(good)
    off = d.scan_offset
    cases = {}
    # RSTn out of sequence
    b = bytearray(good)
    k = good.index(b"\xff\xd1", off)
    b[k + 1] = 0xD5
    cases["rst_sequence"] = bytes(b)
    # a restart marker removed
    k = good.index(b"\xff\xd2", off)
    cases["rst_missing"] = good[:k] + good[k + 2:]
    # truncated in the middle of the scan
    cases["truncated"] = good[:off + (len(good) - off) // 2]
    # garbage bits in the middle of an interval
    b = bytearray(good)
    mid = off + (len(good) - off) // 3
    for j in range(24):
        if b[mid + j] != 0xFF and b[mid + j - 1] != 0xFF:
            b[mid + j] ^= 0x5A
    cases["bitflips"] = bytes(b)
    names = sorted(cases)
    st, _, _ = _decode(decoder, [cases[n] for n in names] + [good])
    assert st[-1] == 0
    for n, s in zip(names, st[:-1]):
        rc, *_ = oracle.decode(cases[n], want_pixels=False)
        if rc != 0:
            assert s != 0, "%s: the reference path fails but the GPU status is clean" % n


def test_decode_is_idempotent_and_batch_invariant(decoder):
    files = [synth.synth_jpeg(w, h, 20 + i, q, ss, ri) for i, (w, h, ss, q, ri, _) in enumerate(SPECS[:8])]
    batch = decoder.batch(files)
    batch.upload()
    batch.decode()
    a = [batch.pixels(i).copy() for i in range(len(files))]
    batch.decode_steps(3)
    b = [batch.pixels(i) for i in range(len(files))]
    batch.close()
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    # each image alone == the same image inside the batch
    for i in (1, 5):
        st, _, pix = _decode(decoder, [files[i]])
        assert st[0] == 0 and np.array_equal(pix[0], a[i])


def test_decode_host_api(decoder, oracle, fixture_jpeg):
    files = [fixture_jpeg, synth.synth_jpeg(256, 192, 7, 90, "420", 4), b"not a jpeg", synth.synth_jpeg(96, 64, 9, 80, "444", 0)]
    outs, st = decoder.decode_host(files)
    assert st[2] < 0 and st[0] == 0 and st[1] == 0 and st[3] == 0
    for i in (0, 1, 3):
        rc, _, _, bgra = oracle.decode(files[i])
        assert rc == 0
        _check_pixels(outs[i], bgra)


def test_full_size_config2_batch(decoder, oracle):
    """BASELINE configs[1] at full size: 256 x 1080p 4:2:0 q90 RI=16. EVERY image of the batch: coefficients (the
    reference's int32 tap) and pixels against the unmodified reference where it decodes the file, else against the
    non-strict oracle port (SHA-256 per image, computed on a pool of host processes); clean status, idempotence of
    the pixel checksum, and big-batch == small-batch."""
    import cpu_digests
    files = synth.config_batch(1, 256)
    batch = decoder.batch(files)
    batch.upload()
    batch.decode()
    assert not batch.status().any()
    want = cpu_digests.config_digests(1, range(256))
    kinds = [w[0] for w in want]
    assert "failed" not in kinds
    print("256 x 1080p: %d images against the unmodified reference, %d against the oracle port" % (kinds.count("reference"), kinds.count("oracle")))
    sums = []
    for i in range(256):
        hc = hashlib.sha256(batch.coefs(i).tobytes()).hexdigest()
        hp = hashlib.sha256(batch.pixels(i).tobytes()).hexdigest()
        assert hc == want[i][1], "coefficients of image %d differ from the %s" % (i, want[i][0])
        assert hp == want[i][2], "pixels of image %d differ from the %s" % (i, want[i][0])
        sums.append(hp)
    batch.decode_steps(2)
    assert [hashlib.sha256(batch.pixels(i).tobytes()).hexdigest() for i in range(0, 256, 5)] == sums[::5]
    batch.close()
    st, _, pix = _decode(decoder, [files[k] for k in (10, 250)])
    assert not st.any()
    assert hashlib.sha256(pix[0].tobytes()).hexdigest() == sums[10]
    assert hashlib.sha256(pix[1].tobytes()).hexdigest() == sums[250]


@pytest.mark.parametrize("cfg,count", [(2, 2), (3, 1), (4, 64)])
def test_other_baseline_configs(decoder, oracle, cfg, count):
    """configs[2..4] (4K 4:4:4 q95, 8K 4:2:2 q85, 500x375 4:2:0 q75): streams without restart markers."""
    files = synth.config_batch(cfg, count)
    st, coefs, pix = _decode(decoder, files)
    assert not st.any()
    oracle.set_strict(False)
    try:
        for i in sorted(set([0, count - 1])):
            rc, _, coef, bgra = oracle.decode(files[i])
            assert rc == 0
            assert np.array_equal(coefs[i], coef)
            _check_pixels(pix[i], bgra)
    finally:
        oracle.set_strict(True)


@pytest.mark.parametrize("cfg,count,stride", [(2, 64, 7), (4, 8192, 10)])
def test_full_size_selfsync_configs(decoder, oracle, cfg, count, stride):
    """BASELINE configs[2] and configs[4] at full size (64 x 4K 4:4:4 q95, 8192 x 500x375 4:2:0 q75; no restart
    markers: the self-synchronising path). Whole batch: clean status; on every `stride`-th image: the pixel
    checksum is stable over repeated decodes and equals the checksum of the same image decoded in a small
    batch of its own; on a sample: coefficients and pixels equal the oracle's."""
    files = synth.config_batch(cfg, count)
    batch = decoder.batch(files)
    batch.upload()
    batch.decode()
    assert not batch.status().any()
    stats = batch.sync_stats()
    print("config", cfg, "sync stats", stats.tolist())
    idx = list(range(0, count, stride))
    sums = [hashlib.sha256(batch.pixels(i).tobytes()).hexdigest() for i in idx]
    batch.decode_steps(2)
    assert not batch.status().any()
    assert sums == [hashlib.sha256(batch.pixels(i).tobytes()).hexdigest() for i in idx]
    # every `stride`-th image (>= 10 % of the batch) against the reference / the oracle port, coefficients and pixels
    import cpu_digests
    want = cpu_digests.config_digests(cfg, idx)
    for i, w, hp in zip(idx, want, sums):
        assert w[0] != "failed"
        assert hashlib.sha256(batch.coefs(i).tobytes()).hexdigest() == w[1], (cfg, i, w[0])
        assert hp == w[2], (cfg, i, w[0])
    batch.close()
    some = idx[::max(1, len(idx) // 6)]
    st, _, pix = _decode(decoder, [files[k] for k in some])
    assert not st.any()
    for k, p in zip(some, pix):
        assert hashlib.sha256(p.tobytes()).hexdigest() == sums[idx.index(k)]


def test_selfsync_streams_without_restart_markers(decoder, oracle):
    """Streams without DRI take the self-synchronising sub-sequence decoder: quality 100 makes blocks that
    are longer than a whole 1024-bit sub-sequence, quality 5 makes sub-sequences with dozens of blocks."""
    specs = [(257, 129, "420", 100), (257, 129, "444", 100), (640, 360, "422", 5), (640, 360, "420", 5),
             (1024, 768, "444", 92), (333, 777, "420", 60)]
    files = [synth.synth_jpeg(w, h, 900 + i, q, ss, 0, optimize=(i % 2 == 0)) for i, (w, h, ss, q) in enumerate(specs)]
    batch = decoder.batch(files)
    batch.upload()
    batch.decode()
    assert not batch.status().any()
    stats = batch.sync_stats()
    n_sub = sum((len(f) + 127) // 128 for f in files)
    print("sync stats", stats.tolist(), "sub-sequences", n_sub)
    # round 1 corrects guessed states; with blocks longer than a sub-sequence (quality 100) the guesses
    # converge slowly and the in-order sweep -- the correctness safety net -- finishes the job
    assert stats[1] > 0 and stats[7] < n_sub
    oracle.set_strict(False)
    try:
        for i, f in enumerate(files):
            rc, _, coef, bgra = oracle.decode(f)
            assert rc == 0
            assert np.array_equal(batch.coefs(i), coef)
            _check_pixels(batch.pixels(i), bgra)
    finally:
        oracle.set_strict(True)
    batch.close()


def test_selfsync_sweep_repairs_every_chunk_border(decoder, oracle):
    """B2J_SYNC_PRE=0 switches the pre-lanes off: every chunk but the first of an image starts from a bare guess, so
    the in-order sweep -- the safety net correctness rests on -- has to re-run nearly every chunk, and the result must
    not change."""
    specs = [(1600, 1200, "444", 95), (1024, 768, "420", 75), (2048, 640, "422", 85), (500, 375, "420", 75), (640, 480, "420", 100)]
    files = [synth.synth_jpeg(w, h, 950 + i, q, ss, 0, optimize=(i % 2 == 1)) for i, (w, h, ss, q) in enumerate(specs)]
    st0, c0, p0 = _decode(decoder, files)
    assert not st0.any()
    os.environ["B2J_SYNC_PRE"] = "0"
    try:
        batch = decoder.batch(files)
    finally:
        del os.environ["B2J_SYNC_PRE"]
    batch.upload()
    batch.decode()
    assert not batch.status().any()
    stats = batch.sync_stats()
    n_chunks = sum(((len(f) + 127) // 128 + 125) // 126 for f in files)
    print("sync stats without pre-lanes", stats.tolist(), "chunks about", n_chunks)
    assert stats[7] > n_chunks // 4
    for i in range(len(files)):
        assert np.array_equal(batch.coefs(i), c0[i]), i
        assert np.array_equal(batch.pixels(i), p0[i]), i
    batch.close()
    oracle.set_strict(False)
    try:
        rc, _, coef, bgra = oracle.decode(files[0])
    finally:
        oracle.set_strict(True)
    assert rc == 0 and np.array_equal(c0[0], coef)
    _check_pixels(p0[0], bgra)


def test_selfsync_corrupt_streams_are_flagged(decoder, oracle):
    good = synth.synth_jpeg(320, 240, 6, 90, "420", 0)
    rc, d = oracle.parse(good)
    off = d.scan_offset
    cases = {"truncated": good[:off + (len(good) - off) // 2]}
    b = bytearray(good)
    mid = off + (len(good) - off) // 3
    for j in range(24):
        if b[mid + j] != 0xFF and b[mid + j - 1] != 0xFF:
            b[mid + j] ^= 0x5A
    cases["bitflips"] = bytes(b)
    names = sorted(cases)
    st, _, _ = _decode(decoder, [cases[n] for n in names] + [good])
    assert st[-1] == 0
    for n, s in zip(names, st[:-1]):
        rc, *_ = oracle.decode(cases[n], want_pixels=False)
        if rc != 0:
            assert s != 0, "%s: the reference path fails but the GPU status is clean" % n


def test_sixteen_bit_quantisation_tables(decoder, oracle, reference=None):
    """DQT with 16-bit precision: the reference keeps the raw little-endian words (no byte swap), so the
    quantisers exceed 255 and the kernel's generic (non-dp2a) dequantisation runs. Mixed with 8-bit images."""
    rng = np.random.RandomState(3)
    blocks = np.zeros((2 * 6, 64), np.int64)
    blocks[:, 0] = rng.randint(-20, 20, 12)
    blocks[:, 1:4] = rng.randint(-2, 3, (12, 3))
    q16 = [[(1 + (i % 3)) for i in range(64)], [2] * 64]      # big-endian 0x0001.. -> read as 0x0100.. = 256..768
    f16 = jpegcraft.build_jpeg(32, 16, (2, 2), blocks, q16, dqt16=True)
    f8 = synth.synth_jpeg(64, 48, 1, 80, "420", 2)
    st, coefs, pix = _decode(decoder, [f16, f8])
    assert not st.any()
    for f, c, p in zip([f16, f8], coefs, pix):
        rc, img, coef, bgra = oracle.decode(f)
        assert rc == 0
        assert np.array_equal(c, coef)
        _check_pixels(p, bgra)
    assert np.abs(coefs[0]).max() >= 256


def test_robust_mode_decodes_files_with_comments(decoder, oracle):
    """A COM segment (Pillow's comment=) and an extra APP1 make the reference parser stop; in robust mode the
    decode equals the decode of the same image written without them."""
    import ocljpegdecoder_b200 as b2j
    base = synth.synth_jpeg(160, 96, 31, 88, "420", 4)
    com = b"\xff\xfe" + (2 + 7).to_bytes(2, "big") + b"comment"
    k = base.index(b"\xff\xdb")
    dirty = base[:k] + com + base[k:]
    assert oracle.parse(dirty, 1)[0] != 0
    outs, st = decoder.decode_host([dirty, base], gate=b2j.GATE_EXTENDED | b2j.PARSE_ROBUST)
    assert not st.any()
    rc, _, _, bgra = oracle.decode(base)
    assert rc == 0
    _check_pixels(outs[0], bgra)
    _check_pixels(outs[1], bgra)


def test_prepass_and_reader_stress_batch(decoder, oracle):
    """Inputs that stress the single-pass pre-pass and the bit readers, against the oracle: many chunks per image
    (several look-back windows), a stream that ends in the middle of a chunk (dead chunks behind), no restart markers,
    broken restart numbering, stuffed bytes at chunk borders, dense q100 blocks with optimised tables."""
    good = synth.synth_jpeg(320, 240, 5, 90, "420", 4)
    b = bytearray(good)
    k = good.index(b"\xff\xd1")
    b[k + 1] = 0xD5
    big = synth.synth_jpeg(2560, 1600, 91, 97, "444", 7)          # > 64 chunks of 16 KiB
    files = [big, synth.synth_jpeg(1600, 1200, 92, 95, "444", 0), good, bytes(b), big[:len(big) // 2],
             synth.synth_jpeg(640, 480, 93, 75, "420", 0), _crafted((2, 2), 80, 48, 2, 3, seed=3, stuffed=True),
             synth.synth_jpeg(800, 608, 94, 100, "420", 3, optimize=True)]
    assert (len(big) + 16383) // 16384 > 64
    st, coefs, pix = _decode(decoder, files)
    assert st[0] == 0 and st[1] == 0 and st[3] != 0 and st[4] != 0 and st[7] == 0
    st2, coefs2, pix2 = _decode(decoder, files)
    assert st2.tolist() == st.tolist()
    oracle.set_strict(False)
    try:
        for i in (0, 1, 2, 5, 6, 7):
            rc, _, coef, bgra = oracle.decode(files[i])
            assert rc == 0, i
            assert np.array_equal(coefs[i], coef), i
            _check_pixels(pix[i], bgra)
            assert np.array_equal(pix2[i], pix[i])
    finally:
        oracle.set_strict(True)


def test_output_formats(decoder, oracle):
    """RGB24 and planar RGB carry exactly the reference's colour values (decoder.cpp:367-370), rearranged: all
    sampling layouts, widths that are and are not multiples of four, 16-bit quantisers (the generic kernel)."""
    import ocljpegdecoder_b200 as b2j
    specs = [(640, 480, "420", 90, 16), (200, 120, "444", 85, 0), (131, 77, "420", 75, 3), (322, 98, "422", 60, 5), (65, 33, "444", 95, 0)]
    files = [synth.synth_jpeg(w, h, 700 + i, q, ss, ri) for i, (w, h, ss, q, ri) in enumerate(specs)]
    files.append(_crafted((1, 2), 40, 48, 2, 0, seed=9, stuffed=True))
    batch = decoder.batch(files)
    batch.upload()
    batch.decode()
    assert not batch.status().any()
    bgra = [batch.pixels(i).copy() for i in range(len(files))]
    for b in bgra:
        assert not b[..., 3].any()
    batch.set_output_format(b2j.OUT_RGB24)
    batch.decode()
    for i, b in enumerate(bgra):
        rgb = batch.pixels(i)
        assert rgb.shape == b.shape[:2] + (3,)
        assert np.array_equal(rgb, b[..., 2::-1]), i
    batch.set_output_format(b2j.OUT_RGB_PLANAR)
    batch.decode()
    for i, b in enumerate(bgra):
        chw = batch.pixels(i)
        assert chw.shape == (3,) + b.shape[:2]
        assert np.array_equal(chw, np.moveaxis(b[..., 2::-1], 2, 0)), i
    batch.set_output_format(b2j.OUT_BGRA)
    batch.decode()
    for i, b in enumerate(bgra):
        assert np.array_equal(batch.pixels(i), b)
    batch.close()
    oracle.set_strict(False)
    try:
        rc, _, _, want = oracle.decode(files[2])
    finally:
        oracle.set_strict(True)
    assert rc == 0 and np.array_equal(bgra[2], want)
    # 16-bit DQT: the generic (non-dp2a) kernel variant
    rng = np.random.RandomState(5)
    blocks = np.zeros((2 * 6, 64), np.int64)
    blocks[:, 0] = rng.randint(-20, 20, 12)
    blocks[:, 1:4] = rng.randint(-2, 3, (12, 3))
    wide = jpegcraft.build_jpeg(32, 16, (2, 2), blocks, [[(1 + (i % 3)) for i in range(64)], [2] * 64], dqt16=True)
    b2 = decoder.batch([wide])
    b2.upload()
    b2.decode()
    ref = b2.pixels(0).copy()
    b2.set_output_format(b2j.OUT_RGB24)
    b2.decode()
    assert np.array_equal(b2.pixels(0), ref[..., 2::-1])
    b2.close()


def test_randomised_batch_against_oracle(decoder, oracle):
    """One mixed batch of 160 images with random geometry (1..400 px a side), sampling, quality, restart
    interval (none, 1..40 MCUs, longer than the image), standard and optimised tables -- Pillow-encoded and
    hand-crafted -- every image compared with the oracle: coefficients and pixels bit-exact, status clean."""
    rng = np.random.RandomState(20261018)
    files = []
    for i in range(128):
        w, h = int(rng.randint(1, 400)), int(rng.randint(1, 400))
        ss = ["444", "420", "422"][int(rng.randint(0, 3))]
        q = int(rng.choice([5, 25, 50, 75, 90, 95, 100]))
        ri = int(rng.choice([0, 0, 1, 2, 3, 7, 16, 40, 5000]))
        files.append(synth.synth_jpeg(w, h, 5000 + i, q, ss, ri, optimize=bool(rng.randint(0, 2))))
    for i in range(32):
        sampling = [(1, 1), (2, 2), (2, 1), (1, 2)][int(rng.randint(0, 4))]
        w, h = int(rng.randint(1, 100)), int(rng.randint(1, 100))
        files.append(_crafted(sampling, w, h, int(rng.choice([0, 1, 2, 5, 11])), int(rng.randint(0, 3)), seed=100 + i, stuffed=bool(i % 2)))
    st, coefs, pix = _decode(decoder, files)
    assert not st.any(), np.nonzero(st)[0].tolist()
    oracle.set_strict(False)
    try:
        for i, f in enumerate(files):
            rc, _, coef, bgra = oracle.decode(f)
            assert rc == 0, i
            assert np.array_equal(coefs[i], coef), i
            _check_pixels(pix[i], bgra)
    finally:
        oracle.set_strict(True)


def _gray_jpeg(w, h, seed, quality, restart_mcus=0, optimize=False):
    import io
    from PIL import Image
    px = synth.synth_pixels(w, h, seed)[:, :, 1]
    buf = io.BytesIO()
    kw = dict(format="JPEG", quality=quality, optimize=optimize)
    if restart_mcus:
        kw["restart_marker_blocks"] = int(restart_mcus)
    Image.fromarray(px, "L").save(buf, **kw)
    return buf.getvalue()


def test_grayscale_extension(decoder, oracle):
    """One-component frames (B2J_GATE_GRAY; SURVEY.md 8f rank 4). The reference refuses them, so the check is
    the oracle's extension -- the reference's own loops with the chroma components absent (U = V = 0) -- plus
    Pillow as an independent decoder within the +-2 that separates the Chen-Wang IDCT from libjpeg's."""
    import io
    from PIL import Image
    import ocljpegdecoder_b200 as b2j
    from oracle import GATE_GRAY as ORC_GRAY, GATE_EXTENDED as ORC_EXT
    specs = [(640, 480, 90, 16, False), (131, 77, 75, 0, False), (64, 64, 50, 1, True), (1, 1, 90, 0, False),
             (333, 9, 95, 3, False), (1024, 768, 85, 0, True), (200, 120, 100, 0, False)]
    files = [_gray_jpeg(w, h, 40 + i, q, ri, opt) for i, (w, h, q, ri, opt) in enumerate(specs)]
    colour = synth.synth_jpeg(160, 96, 3, 90, "420", 4)
    mix = files + [colour]
    # refused without the flag, like the reference
    rc, _ = b2j.parse_header(files[0], b2j.GATE_EXTENDED)
    assert rc != 0
    batch = decoder.batch(mix, gate=b2j.GATE_EXTENDED | b2j.GATE_GRAY)
    batch.upload()
    batch.decode()
    assert not batch.status().any()
    oracle.set_strict(False)
    try:
        for i, f in enumerate(mix):
            rc, img, coef, bgra = oracle.decode(f, gate=ORC_EXT | ORC_GRAY)
            assert rc == 0, i
            assert np.array_equal(batch.coefs(i), coef), i
            got = batch.pixels(i)
            _check_pixels(got, bgra)
            if i < len(files):
                assert np.array_equal(got[..., 0], got[..., 1]) and np.array_equal(got[..., 1], got[..., 2])
                pil = np.asarray(Image.open(io.BytesIO(f)).convert("L"), dtype=np.int16)
                assert np.abs(got[..., 0].astype(np.int16) - pil).max() <= 2, i
    finally:
        oracle.set_strict(True)
    ref = [batch.pixels(i).copy() for i in range(len(mix))]
    batch.set_output_format(b2j.OUT_RGB_PLANAR)
    batch.decode()
    for i, b in enumerate(ref):
        assert np.array_equal(batch.pixels(i), np.moveaxis(b[..., 2::-1], 2, 0)), i
    batch.close()


def test_dc_category_above_16_is_flagged(decoder, oracle):
    """Documented deviation (include/b2j.h, DESIGN.md): the reference accepts DC categories up to 25 (decoder.cpp:230);
    the coefficient plane here is int16, so a DC table symbol above 16 is no codeword to the decoder: the block is
    flagged B2J_ST_BAD_CODE and the image reported as corrupt instead of decoded with a 17-bit difference."""
    dc_bits = list(jpegcraft.DC_LUMA_BITS)
    dc_vals = list(jpegcraft.DC_LUMA_VALS)
    dc_vals[0] = 17                                  # the 2-bit code now means "category 17"
    tables = dict(jpegcraft.STD_TABLES)
    tables[(0, 0)] = (dc_bits, dc_vals)
    blocks = np.zeros((6, 64), np.int64)             # DC difference 0 everywhere: every luma block starts with that code
    # category 0 is symbol 0 in the standard table; with the swapped table the writer needs the code of symbol 0 to exist
    codes = jpegcraft.canonical_codes(dc_bits, dc_vals)
    assert 0 not in codes and 17 in codes
    # write the stream by hand: luma DC code for symbol 17 followed by 17 value bits, then EOB; chroma as usual
    std = {k: jpegcraft.canonical_codes(*v) for k, v in jpegcraft.STD_TABLES.items()}
    bw = jpegcraft.BitWriter()
    for b in range(6):
        if b < 4:
            code, l = codes[17]
            bw.put(code, l); bw.put(0x10000, 17)     # +65536
            code, l = std[(1, 0)][0x00]
        else:
            code, l = std[(0, 1)][0]
            bw.put(code, l)
            code, l = std[(1, 1)][0x00]
        bw.put(code, l)
    bw.flush()
    shell = jpegcraft.build_jpeg(16, 16, (2, 2), blocks, [[1] * 64, [1] * 64], tables={**tables, (0, 0): (dc_bits, [0] + dc_vals[1:])})
    k = shell.index(b"\xff\xda")
    head = bytearray(shell[:k + 14])
    j = head.index(bytes([0xFF, 0xC4, 0x00, 0x1F, 0x00]))   # the DC luma DHT
    head[j + 5 + 16] = 17
    data = bytes(head) + bytes(bw.out) + b"\xff\xd9"
    good = synth.synth_jpeg(64, 48, 2, 90, "420", 0)
    st, _, _ = _decode(decoder, [data, good])
    assert st[1] == 0
    assert st[0] & 0x01, "DC category 17 must be flagged as B2J_ST_BAD_CODE, status %#x" % st[0]


def test_decode_host_ex_formats_threads_and_groups(decoder, oracle):
    """b2j_decode_host_ex: every output layout, 1 and several host threads, small groups (buffers of finished groups are
    recycled while later groups are still being staged), a refused file in the middle. All against the oracle."""
    import ocljpegdecoder_b200 as b2j
    specs = [(320, 240, "420", 90, 8), (200, 120, "444", 85, 0), (131, 77, "420", 75, 3), (322, 98, "422", 60, 0), (65, 33, "444", 95, 0),
             (500, 375, "420", 75, 0), (96, 64, "444", 80, 2)]
    files = [synth.synth_jpeg(w, h, 900 + i, q, ss, ri) for i, (w, h, ss, q, ri) in enumerate(specs)] * 5
    files.insert(9, b"\xff\xd8 this is not a jpeg")
    want = {}
    oracle.set_strict(False)
    try:
        for i, f in enumerate(files):
            if i == 9:
                continue
            key = hashlib.sha256(f).hexdigest()
            if key not in want:
                rc, _, _, bgra = oracle.decode(f, 1)
                assert rc == 0
                want[key] = bgra
    finally:
        oracle.set_strict(True)
    for fmt, nt, group in [(b2j.OUT_BGRA, 1, 4), (b2j.OUT_RGB24, 4, 3), (b2j.OUT_RGB_PLANAR, 3, 0), (b2j.OUT_BGRA, 0, 0)]:
        outs, st = decoder.decode_host_ex(files, out_format=fmt, n_threads=nt, group=group)
        assert st[9] < 0 and not np.delete(st, 9).any(), st
        for i, f in enumerate(files):
            if i == 9:
                continue
            ref = want[hashlib.sha256(f).hexdigest()]
            if fmt == b2j.OUT_BGRA:
                assert np.array_equal(outs[i], ref), (fmt, i)
            elif fmt == b2j.OUT_RGB24:
                assert np.array_equal(outs[i], ref[..., 2::-1]), (fmt, i)
            else:
                assert np.array_equal(outs[i], np.moveaxis(ref[..., 2::-1], 2, 0)), (fmt, i)
    # caller buffers that are neighbours in memory: the downloads of neighbouring images merge into one copy
    good = [f for i, f in enumerate(files) if i != 9]
    descs = [b2j.parse_header(f)[1] for f in good]
    for fmt, bpp in ((b2j.OUT_BGRA, 4), (b2j.OUT_RGB24, 3)):
        sizes = [d.width * d.height * bpp for d in descs]
        offs = np.concatenate([[0], np.cumsum(sizes)])
        big = np.zeros(int(offs[-1]) + 16, np.uint8)
        base = big.ctypes.data
        _, st = decoder.decode_host_ex(good, outs=[base + int(o) for o in offs[:-1]], out_format=fmt, n_threads=2, group=8)
        assert not st.any()
        assert not big[int(offs[-1]):].any()
        for i, f in enumerate(good):
            ref = want[hashlib.sha256(f).hexdigest()]
            got = big[int(offs[i]):int(offs[i + 1])].reshape(descs[i].height, descs[i].width, bpp)
            assert np.array_equal(got, ref if bpp == 4 else ref[..., 2::-1]), (fmt, i)
    # the plain call is the same path with the defaults
    outs, st = decoder.decode_host(files)
    assert st[9] < 0 and not np.delete(st, 9).any()
    assert np.array_equal(outs[0], want[hashlib.sha256(files[0]).hexdigest()])


def test_decode_host_multi_and_pinned_buffers(decoder, oracle, tmp_path):
    """b2j_decode_host_multi shards one list of files over several contexts (one host thread each; here as many contexts
    as the box has GPUs, at least two -- two contexts on one GPU exercise the same threading), reading the files with
    b2j_read_files into a pinned arena and writing RGB24 into one pinned output buffer (b2j_host_alloc)."""
    import ocljpegdecoder_b200 as b2j
    files = [synth.synth_jpeg(160 + 16 * (i % 5), 120 + 8 * (i % 3), 300 + i, 70 + i % 25, ["420", "444", "422"][i % 3], [0, 4][i % 2]) for i in range(23)]
    paths = []
    for i, f in enumerate(files):
        p = tmp_path / ("f%02d.jpg" % i)
        p.write_bytes(f)
        paths.append(str(p))
    rc, arena, addrs, lens = b2j.read_files(paths, 3)
    assert rc == 0 and lens == [len(f) for f in files]
    rc_bad, arena2, addrs2, lens2 = b2j.read_files(paths[:2] + [str(tmp_path / "missing.jpg")], 2)
    assert rc_bad != 0 and addrs2[2] is None and lens2[:2] == lens[:2]
    b2j.host_free(arena2)
    descs = [b2j.parse_header(f)[1] for f in files]
    sizes = [d.width * d.height * 3 for d in descs]
    offs = np.concatenate([[0], np.cumsum([(s + 255) // 256 * 256 for s in sizes])])
    pinned = b2j.PinnedBuffer(int(offs[-1]))
    ngpu = max(2, min(8, decoder.lib.b2j_device_count()))
    decs = [decoder] + [b2j.Decoder(k % decoder.lib.b2j_device_count()) for k in range(1, ngpu)]
    try:
        outs, st = b2j.decode_host_multi(decs, addrs, lens=lens, outs=[pinned.address + int(o) for o in offs[:-1]], out_format=b2j.OUT_RGB24, n_threads=2, group=4)
        assert not st.any(), st
        oracle.set_strict(False)
        try:
            for i in range(0, len(files), 3):
                rc, _, _, bgra = oracle.decode(files[i], 1)
                assert rc == 0
                got = pinned.array[int(offs[i]):int(offs[i]) + sizes[i]].reshape(descs[i].height, descs[i].width, 3)
                assert np.array_equal(got, bgra[..., 2::-1]), i
        finally:
            oracle.set_strict(True)
    finally:
        for d in decs[1:]:
            d.close()
        pinned.close()
        b2j.host_free(arena)


def test_secondary_boundary_coefficients_in_pixels_out(decoder, oracle):
    """b2j_idct_*: the reference's coefficient tap (int32, dequantised: what its decoder.cpp hands to clidct_transfer_data_to_device)
    in, the pixels of its CPU path out -- 4:4:4 and 4:2:0 as the reference knows them, 4:2:2 / 4:4:0 beyond; odd sizes; upload in
    two pieces; the coefficients read back as they were sent."""
    import ocljpegdecoder_b200 as b2j
    for w, h, ss, hv, q in [(200, 120, "444", (1, 1), 85), (131, 77, "420", (2, 2), 75), (640, 480, "420", (2, 2), 95), (322, 98, "422", (2, 1), 60)]:
        data = synth.synth_jpeg(w, h, 40 + w, q, ss, 0)
        oracle.set_strict(False)
        try:
            rc, img, coef, bgra = oracle.decode(data, 1)
        finally:
            oracle.set_strict(True)
        assert rc == 0
        idct = b2j.Idct(decoder, w, h, hv[0], hv[1])
        assert idct.blk_count == coef.shape[0]
        half = coef.shape[0] // 2
        idct.upload(coef[half:], offset=half)
        idct.upload(coef[:half], offset=0)
        idct.run()
        assert np.array_equal(idct.pixels(), bgra), (w, h, ss)
        assert np.array_equal(idct.coefs(), coef)
        idct.close()


def test_downscaled_output(decoder):
    """b2j_batch_downscale: box-filter reduction by 2, 4, 8 in every output format against numpy: sizes that are and are not
    multiples of the factor (edge means over the pixels that exist), rounding (sum + n/2) // n."""
    import ocljpegdecoder_b200 as b2j
    files = [synth.synth_jpeg(w, h, 60 + w, q, ss, ri) for w, h, ss, q, ri in [(320, 240, "420", 90, 8), (131, 77, "444", 85, 0), (65, 33, "422", 75, 0), (8, 8, "444", 50, 0)]]
    batch = decoder.batch(files)
    batch.upload()

    def box(a, f):   # a: [H, W, C] uint8
        h, w, c = a.shape
        oh, ow = (h + f - 1) // f, (w + f - 1) // f
        pad = np.zeros((oh * f, ow * f, c), np.uint32)
        cnt = np.zeros((oh * f, ow * f, 1), np.uint32)
        pad[:h, :w] = a
        cnt[:h, :w] = 1
        s = pad.reshape(oh, f, ow, f, c).sum(axis=(1, 3))
        n = cnt.reshape(oh, f, ow, f, 1).sum(axis=(1, 3))
        return ((s + n // 2) // n).astype(np.uint8)

    for fmt in (b2j.OUT_BGRA, b2j.OUT_RGB24, b2j.OUT_RGB_PLANAR):
        batch.set_output_format(fmt)
        batch.decode()
        assert not batch.status().any()
        for f in (2, 4, 8):
            batch.downscale(f)
            for i in range(len(files)):
                full = batch.pixels(i)
                got = batch.downscaled(i)
                if fmt == b2j.OUT_RGB_PLANAR:
                    want = np.moveaxis(box(np.moveaxis(full, 0, 2), f), 2, 0)
                else:
                    want = box(full, f)
                assert got.shape == want.shape and np.array_equal(got, want), (fmt, f, i)
    batch.close()
