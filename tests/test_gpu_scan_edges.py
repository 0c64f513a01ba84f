"""The scan pre-pass (k_unstuff_fused) at its borders, behind EOI and on malformed markers.

The pre-pass works on 4-byte words, 16-byte groups, 64-byte thread ranges and 16 KiB chunks (tests/scan_model.py reads
the geometry from b2j_internal.h). The boundary batch puts every kind of special byte pair across every kind of border:
  - split pairs: a stuffed FF 00, a bare FF Dn, a fill run ending in FF Dn, EOI, with the FF the last byte in front of a
    word, group, thread and chunk border, and a fill run crossing each border;
  - fill runs of 1..70 bytes, one across a chunk border, one over a whole thread, one over a whole chunk (it keeps 0 bytes);
  - dense markers: RI = 1 with nearly empty blocks in a gray and a 4:2:0 image, a marker every 3-7 bytes over 5 chunks
    and more (over 4000 in a chunk of the gray one), their phase walking through every offset mod 64;
  - every residue mod 16 of the clean bytes in front of a chunk (the copy-out's misalignment);
  - scans of 16384 m - 1, 16384 m and 16384 m + 1 bytes with EOI last, a file cut behind the FF of EOI at 16384 m;
  - data behind EOI: a second JPEG with restart markers, random bytes, zeros, a trailer starting with FF D0, and 34
    chunks of trailer behind an image of more than 33 chunks; each behind a DRI and a no-DRI image.
Every variant has a canonical file (the same blocks with no fill and no trailer) and must decode as it does. The CPU
tests check, with the model, that the batch holds all of this and that the fixtures are what they claim, before any GPU
time. The malformed batch puts stray and foreign markers and truncations between good images: where the reference
fails, the status must flag it; where the status is clean, the decode must be the reference's.
"""
import numpy as np
import pytest

import jpegcraft
import scan_model as sm
import synth
from scan_model import CHUNK, THREAD

GOOD_Q = [[1 + (i % 3) for i in range(64)], [2] * 64]


def _stuffy_blocks(n, seed):
    """DC differences of +-2047 (eleven value bits of 1 behind a code of eight 1s) and AC values of 1023: FF bytes, so
    stuffed FF 00 pairs, every few bytes."""
    rng = np.random.RandomState(seed)
    b = np.zeros((n, 64), np.int64)
    b[:, 0] = np.where(np.arange(n) % 2 == 0, 2047, 0)
    for k in range(1, 6):
        b[:, k] = rng.randint(-3, 4, n)
    b[rng.rand(n) < 0.3, rng.randint(6, 30)] = 1023
    return b


def _sparse_blocks(n, seed, p):
    """Nearly empty blocks: a DC value of -1 or 1 in a share p of them, 0 elsewhere, and an end-of-block code."""
    rng = np.random.RandomState(seed)
    b = np.zeros((n, 64), np.int64)
    b[:, 0] = rng.choice([-1, 1], n) * (rng.rand(n) < p)
    return b


def _n_blocks(samp, w, h):
    lay = [(1, 1)] if samp == "gray" else jpegcraft._layout(samp)
    mw, mh = 8 * max(a for a, _ in lay), 8 * max(b for _, b in lay)
    return -(-w // mw) * -(-h // mh) * sum(a * b for a, b in lay)


class Base:
    """One image's header and restart intervals (stuffed and before stuffing); files are built from them."""

    def __init__(self, name, samp, w, h, ri, content, seed):
        self.name, self.dri = name, ri > 0
        if content == "photo":
            data, blocks = jpegcraft.encode_pixels(synth.synth_pixels(w, h, seed), samp, GOOD_Q, restart_interval=ri)
        else:
            n = _n_blocks(samp, w, h)
            blocks = _stuffy_blocks(n, seed) if content == "stuffy" else _sparse_blocks(n, seed, content)
        self.head, self.intervals, self.plain = jpegcraft.build_parts(w, h, samp, blocks, GOOD_Q, ri)
        self.n_segs = len(self.intervals)

    def file(self, fills=0, fill_eoi=0, trailer=b""):
        fills = [fills] * (self.n_segs - 1) if isinstance(fills, int) else fills
        return self.head + jpegcraft.join_scan(self.intervals, fills, fill_eoi) + trailer

    def end(self, fills=0):
        """Scan bytes in front of EOI's fill with these marker fills."""
        return len(self.file(fills)) - len(self.head) - 2


def _bases():
    return {
        "420_stuffy": Base("420_stuffy", (2, 2), 320, 160, 2, "stuffy", 1),
        "444_photo": Base("444_photo", (1, 1), 400, 240, 3, "photo", 2),
        "422_stuffy": Base("422_stuffy", (2, 1), 256, 96, 1, "stuffy", 3),
        "31_photo": Base("31_photo", (3, 1), 360, 200, 2, "photo", 4),
        "gray_stuffy": Base("gray_stuffy", "gray", 256, 160, 1, "stuffy", 5),
        "gray_dense": Base("gray_dense", "gray", 1536, 1152, 1, 0.5, 6),
        "420_dense": Base("420_dense", (2, 2), 2048, 1728, 1, 0.0, 7),
        "420_nodri": Base("420_nodri", (2, 2), 400, 300, 0, "photo", 8),
        "gray_nodri": Base("gray_nodri", "gray", 320, 200, 0, "stuffy", 9),
        "444_big": Base("444_big", (1, 1), 800, 800, 0, "photo", 10),
    }


SPLIT_KINDS = ("stuff", "rst", "fillrun", "fillcross")


def boundary_cases():
    """[(name, file, canonical file, base)], canonical files included (name ending in ':canon')."""
    bases = _bases()
    cases = [(b.name + ":canon", b.file(), b.file(), b) for b in bases.values()]

    def add(name, base, **kw):
        cases.append((base.name + ":" + name, base.file(**kw), base.file(), base))

    # split pairs at every border, fill runs crossing them; chunk borders are waited for (a marker close in front of one)
    for key in ("420_stuffy", "444_photo", "422_stuffy", "31_photo", "gray_stuffy"):
        b = bases[key]
        wants = [(k, sb) for sb in (4, 16, THREAD) for k in SPLIT_KINDS] + [(k, CHUNK, 300) for k in SPLIT_KINDS]
        fills, _ = sm.place_fills(b.intervals, wants, default=lambda r: r % 3)
        add("split", b, fills=fills)
    # fill runs of 1..70, and one of 130 (it covers an aligned 64-byte thread range)
    b = bases["422_stuffy"]
    add("fill1to70", b, fills=[1 + r % 70 for r in range(b.n_segs - 1)])
    add("fill130", b, fills=[130 if r == 7 else 0 for r in range(b.n_segs - 1)])
    # dense markers, the per-marker fill cycling so that the marker phase walks through every offset mod 64
    for key in ("gray_dense", "420_dense"):
        b = bases[key]
        add("cycle", b, fills=[(0, 0, 0, 1)[r % 4] for r in range(b.n_segs - 1)])
    # the ends of the scan: EOI split at each border, scan lengths 16384 m + {-1, 0, +1}, fill before EOI over a chunk
    for key in ("420_stuffy", "gray_nodri", "420_nodri"):
        b = bases[key]
        e = b.end()
        for sb in (4, 16, THREAD):
            add("eoi_split_%d" % sb, b, fill_eoi=(sb - 1 - e) % sb)
        for d in (-1, 0, 1):
            add("len_%+d" % d, b, fill_eoi=(CHUNK - 2 + d - e) % CHUNK)
        add("fill_chunk", b, fill_eoi=(CHUNK - e % CHUNK) + CHUNK + 3)   # a chunk of nothing but fill bytes
        f = b.file(fill_eoi=(CHUNK - 1 - e) % CHUNK)                      # EOI's FF the last byte of a chunk ...
        cases.append((b.name + ":cut_after_ff", f[:-1], b.file(), b))     # ... and the file cut behind it
    # data behind EOI, behind a DRI and a no-DRI image
    rng = np.random.RandomState(11)
    second = synth.synth_jpeg(200, 104, 9, 80, "420", 2)
    for key in ("420_stuffy", "420_nodri"):
        b = bases[key]
        add("trail_jpeg", b, trailer=second)
        for n in (1, 777, 100000):
            add("trail_rand_%d" % n, b, trailer=rng.randint(0, 256, n).astype(np.uint8).tobytes())
        add("trail_zeros", b, trailer=bytes(5000))
        add("trail_ffd0", b, trailer=b"\xFF\xD0" + rng.randint(0, 256, 3000).astype(np.uint8).tobytes())
    add("trail_34_chunks", bases["444_big"], trailer=rng.randint(0, 256, 34 * CHUNK + 100).astype(np.uint8).tobytes())
    return cases


_CASES = None


def _cases():
    global _CASES
    if _CASES is None:
        _CASES = boundary_cases()
    return _CASES


def _scan(case):
    return case[1][len(case[3].head):]


def test_boundary_batch_covers_what_it_claims():
    """From the pre-pass model: every pattern the module docstring lists is in the boundary batch."""
    cases = _cases()
    found = set()
    residues = set()
    fill_lengths = set()
    for name, data, canon, base in cases:
        scan = _scan((name, data, canon, base))
        m = sm.Prepass(scan)
        for i, kind in m.specials:
            for border in sm.split_at(i):
                if kind == "stuff":
                    found.add(("stuff", border))
                elif kind == "rst":
                    found.add(("fillrun" if i and scan[i - 1] == 0xFF else "rst", border))
                elif kind == "fill":
                    found.add(("fillcross", border))
                elif kind == "term" and i + 1 < len(scan) and scan[i + 1] == 0xD9:
                    found.add(("eoi", border))
        # fill runs: consecutive fill bytes in front of a marker or the terminator
        run = 0
        for (i, kind), nxt in zip(m.specials, m.specials[1:] + [(None, None)]):
            run = run + 1 if kind == "fill" else 0
            if kind == "fill" and nxt[1] != "fill":
                lo, hi = i - run + 1, i + 1            # fill bytes [lo, hi], the marker's FF at hi
                fill_lengths.add(run)
                if lo // CHUNK != hi // CHUNK:
                    found.add(("fill_over_chunk",))
                if -(-lo // THREAD) * THREAD + THREAD <= hi:
                    found.add(("fill_over_thread",))
        keeps = m.chunk_keeps()
        if 0 in keeps[:-1]:
            found.add(("empty_chunk",))
        residues |= {k % 16 for k in m.kept_before_chunks()[1:]}
        if name.endswith(("dense:cycle",)):
            offs = [i - 1 for i, _, _ in m.markers]
            gaps = np.diff(offs)
            per_chunk = np.bincount(np.array(offs) // CHUNK)
            if len(offs) and m.term >= 5 * CHUNK and gaps.max() <= 7 and gaps.min() >= 3:
                found.add(("dense", base.name, per_chunk.max() > 4000 if base.name.startswith("gray") else True))
            assert {o % THREAD for o in offs} == set(range(THREAD)), name
        # scan ends and trailers
        if m.term == len(scan) - 2 and scan.endswith(b"\xFF\xD9"):
            d = len(scan) % CHUNK
            if d in (CHUNK - 1, 0, 1) and len(scan) > CHUNK:
                found.add(("scan_len", {CHUNK - 1: -1, 0: 0, 1: 1}[d]))
        if scan.endswith(b"\xFF") and m.term == len(scan) and len(scan) % CHUNK == 0:   # the pad's FF ends it
            found.add(("cut_after_ff",))
        if m.term + 2 < len(scan):
            trailer = scan[m.term + 2:]
            kinds = set()
            if trailer.startswith(b"\xFF\xD8") and b"\xFF\xD0" in trailer and b"\xFF\x00" in trailer and trailer.endswith(b"\xFF\xD9"):
                kinds.add("jpeg")
            if trailer.startswith(b"\xFF\xD0"):
                kinds.add("ffd0")
            if not any(trailer):
                kinds.add("zeros")
            if "rand" in name:
                kinds.add("random")
            if len(trailer) > 33 * CHUNK and m.term > 33 * CHUNK:
                kinds.add("big")
            for k in kinds:
                found.add(("trailer", k, base.dri))
    for border in sm.BORDERS:
        for kind in SPLIT_KINDS + ("eoi",):
            assert (kind, border) in found, (kind, border)
    assert set(range(1, 71)) <= fill_lengths
    for want in [("fill_over_chunk",), ("fill_over_thread",), ("empty_chunk",), ("cut_after_ff",),
                 ("dense", "gray_dense", True), ("dense", "420_dense", True),
                 ("scan_len", -1), ("scan_len", 0), ("scan_len", 1)]:
        assert want in found, want
    assert residues == set(range(16)), sorted(residues)
    for k in ("jpeg", "random", "zeros", "ffd0"):
        for dri in (True, False):
            assert ("trailer", k, dri) in found, (k, dri)
    assert ("trailer", "big", False) in found
    # one random trailer of each size 1 B .. 100 KB
    sizes = {len(_scan(c)) - sm.Prepass(_scan(c)).term - 2 for c in cases if "rand" in c[0]}
    assert min(sizes) == 1 and max(sizes) == 100000


GATE = 1 | 4   # B2J_GATE_EXTENDED | B2J_GATE_GRAY (the oracle's gates are the same numbers)


def test_prepass_model_and_oracle_agree_on_the_fixtures(oracle):
    """For every file: the model's clean stream, interval by interval, is what the writer emitted before stuffing, and the
    non-strict oracle decodes it to the canonical file's coefficients."""
    oracle.set_strict(False)
    try:
        canon = {}
        for name, data, cf, base in _cases():
            m = sm.Prepass(_scan((name, data, cf, base)))
            starts, end = m.intervals(base.n_segs, base.dri)
            assert len(m.markers) == (base.n_segs - 1 if base.dri else 0), name
            bounds = starts + [end]
            for r in range(base.n_segs):
                assert m.clean[bounds[r]:bounds[r + 1]] == base.plain[r], (name, r)
            assert end == len(m.clean)
            if cf not in canon:
                rc, _, coef, _ = oracle.decode(cf, gate=GATE, want_pixels=False)
                assert rc == 0, name
                canon[cf] = coef
            rc, _, coef, _ = oracle.decode(data, gate=GATE, want_pixels=False)
            assert rc == 0, name
            assert np.array_equal(coef, canon[cf]), name
    finally:
        oracle.set_strict(True)


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _oracle_ref(oracle, files):
    oracle.set_strict(False)
    try:
        return [oracle.decode(f, gate=GATE) for f in files]
    finally:
        oracle.set_strict(True)


def _decode_batch(decoder, files):
    b = decoder.batch(files, gate=GATE)
    b.upload()
    out = []
    for _ in range(2):
        b.decode()
        out.append((b.status(), [b.coefs(i) for i in range(b.n)], b.read_all_pixels()))
    b.close()
    return out


@pytest.fixture(scope="module")
def boundary_decode(decoder, oracle):
    files = [c[1] for c in _cases()]
    return files, _decode_batch(decoder, files), _oracle_ref(oracle, files)


@pytest.mark.gpu
def test_every_variant_decodes_as_its_canonical_file(boundary_decode):
    files, runs, ref = boundary_decode
    (st, coefs, pix), (st2, coefs2, pix2) = runs
    index = {c[1]: i for i, c in enumerate(_cases()) if c[0].endswith(":canon")}
    bad = [(c[0], hex(s)) for c, s in zip(_cases(), st) if s]
    assert not bad, bad
    assert np.array_equal(st, st2)
    for i, (name, data, canon, base) in enumerate(_cases()):
        rc, _, rcoef, rbgra = ref[i]
        j = index[canon]
        assert rc == 0, name
        assert np.array_equal(coefs[i], rcoef), name
        assert np.array_equal(pix[i], rbgra), name
        assert np.array_equal(coefs[i], coefs[j]) and np.array_equal(pix[i], pix[j]), name
        assert np.array_equal(coefs[i], coefs2[i]) and np.array_equal(pix[i], pix2[i]), name


@pytest.mark.gpu
def test_host_call_on_the_boundary_batch(decoder, boundary_decode):
    """b2j_decode_host_ex in RGB24 with groups of 3 images: the trailers inflate the bytes each group uploads."""
    import ocljpegdecoder_b200 as b2j
    files, runs, _ = boundary_decode
    outs, st = decoder.decode_host_ex(files, gate=GATE, out_format=b2j.OUT_RGB24, group=3)
    assert not st.any(), st
    for i, (o, p) in enumerate(zip(outs, runs[0][2])):
        assert np.array_equal(o, p[..., 2::-1]), _cases()[i][0]


# ---- malformed markers next to good images -------------------------------------------------------------------------------
def _data_pos(f, scan0, frac):
    """A scan offset near frac of the scan that splits no FF xx pair and sits next to no marker byte."""
    k = scan0 + int((len(f) - 2 - scan0) * frac)
    while f[k - 1] == 0xFF or f[k] == 0xFF or 0xD0 <= f[k] <= 0xD7:
        k += 1
    return k


def malformed_cases():
    """[(name, file, good)]: good images (goods alone decode clean) interleaved with malformed ones."""
    goods = [("g420_ri4", synth.synth_jpeg(320, 240, 5, 90, "420", 4)),
             ("g420", synth.synth_jpeg(320, 240, 5, 90, "420", 0)),
             ("g444_ri3", synth.synth_jpeg(200, 136, 6, 85, "444", 3)),
             ("g422", synth.synth_jpeg(512, 384, 7, 95, "422", 0)),
             ("g420_big_ri2", synth.synth_jpeg(640, 480, 8, 95, "420", 2))]
    bad = []
    for name, f in goods:
        scan0 = f.index(b"\xFF\xDA") + 2 + int.from_bytes(f[f.index(b"\xFF\xDA") + 2:f.index(b"\xFF\xDA") + 4], "big")
        eoi = len(f) - 2
        dri = b"\xFF\xDD" in f[:scan0]
        rsts = [i for i in range(scan0, eoi) if f[i] == 0xFF and 0xD0 <= f[i + 1] <= 0xD7]
        k = _data_pos(f, scan0, 0.6)
        bad.append((name + ":stray_rst_60", f[:k] + b"\xFF\xD3" + f[k:]))
        bad.append((name + ":rst_before_eoi", f[:eoi] + b"\xFF\xD5" + f[eoi:]))
        if dri:
            last = rsts[-1] + 2
            k = _data_pos(f, last, 0.5)
            bad.append((name + ":stray_rst_last_interval", f[:k] + bytes([0xFF, 0xD0 + (len(rsts) & 7)]) + f[k:]))
            k = (rsts[len(rsts) // 2] + rsts[len(rsts) // 2 + 1]) // 2
            while f[k - 1] == 0xFF or f[k] == 0xFF:
                k += 1
            bad.append((name + ":extra_rst_mid_interval", f[:k] + b"\xFF\xD6" + f[k:]))
            before_last = last
        else:
            before_last = _data_pos(f, scan0, 0.97)
        for m in (b"\xFF\xFE", b"\xFF\xDC", b"\xFF\x01"):
            bad.append((name + ":foreign_%02x" % m[1], f[:before_last] + m + f[before_last:]))
        for m in range(1, (len(f) - scan0) // CHUNK + 1):
            for d in (-2, -1, 0, 1):
                bad.append((name + ":cut_%d%+d" % (m, d), f[:scan0 + m * CHUNK + d]))
        ffs = [i for i in range(scan0, eoi) if f[i] == 0xFF]
        if ffs:
            i = ffs[len(ffs) // 2]
            bad.append((name + ":cut_after_ff", f[:i + 1]))
    out = []
    for j in range(max(len(goods), len(bad))):
        if j < len(goods):
            out.append(goods[j] + (True,))
        out += [b + (False,) for b in bad[j * len(bad) // len(goods):(j + 1) * len(bad) // len(goods)]] if j < len(goods) else []
    return out


@pytest.mark.gpu
def test_malformed_markers_next_to_good_images(decoder, oracle):
    """(a) where the non-strict oracle fails, the status is not 0; (b) where the status is 0, coefficients and pixels are
    the oracle's; (c) every good image is bit-exact with the oracle and with a batch of the good images alone."""
    cases = malformed_cases()
    files = [c[1] for c in cases]
    (st, coefs, pix), _ = _decode_batch(decoder, files)
    ref = _oracle_ref(oracle, files)
    goods = [c[1] for c in cases if c[2]]
    (gst, gcoefs, gpix), _ = _decode_batch(decoder, goods)
    assert not gst.any()
    fails = []
    g = 0
    for i, (name, f, good) in enumerate(cases):
        rc, _, rcoef, rbgra = ref[i]
        if rc != 0 and st[i] == 0:
            fails.append("(a) %s: the oracle fails (rc %d), status 0" % (name, rc))
        if st[i] == 0 and rc == 0 and not (np.array_equal(coefs[i], rcoef) and np.array_equal(pix[i], rbgra)):
            fails.append("(b) %s: status 0, %d blocks differ from the oracle" % (name, int((coefs[i] != rcoef).any(axis=1).sum())))
        if good:
            if not (st[i] == 0 and rc == 0 and np.array_equal(coefs[i], rcoef) and np.array_equal(pix[i], rbgra)
                    and np.array_equal(coefs[i], gcoefs[g]) and np.array_equal(pix[i], gpix[g])):
                fails.append("(c) %s" % name)
            g += 1
    assert not fails, "\n".join(fails)
