"""GPU: generic sampling layouts, per-component tables, long Huffman codes and the largest decode tables, against the
oracle (extended gate, non-strict) and against the blocks the streams were written from (tests/test_layout_streams.py).
Coefficients bit-exact, pixels exact, status clean."""
import hashlib
import io
import os

import numpy as np
import pytest

import synth
from test_layout_streams import (BIG_MAPPINGS, LAYOUTS, big_table_stream, large_411_stream, layout_streams, long_code_streams,
                                 make_stream, table_streams)
from test_oracle import GENERIC_LAYOUTS, generic_luma_jpeg, generic_luma_key

pytestmark = pytest.mark.gpu


def _gray_jpeg(w, h, seed, quality, restart_mcus=0):
    from PIL import Image
    buf = io.BytesIO()
    kw = dict(format="JPEG", quality=quality)
    if restart_mcus:
        kw["restart_marker_blocks"] = restart_mcus
    Image.fromarray(synth.synth_pixels(w, h, seed)[:, :, 1], "L").save(buf, **kw)
    return buf.getvalue()


def _mixed():
    """[(name, file bytes, Stream or None, gray)]: every generic and multi-block-chroma layout in every variant, the
    reference's generic-luma inputs, a 4:1:1 1080p frame without restart markers, and 4:2:0, 4:4:4 and gray images, so
    that all three tile kinds run in one decode."""
    out = [(s.name, s.data, s, False) for samp in LAYOUTS for s in layout_streams(samp)]
    out += [("ref_" + generic_luma_key(samp, ri), generic_luma_jpeg(samp, ri), None, False) for samp in GENERIC_LAYOUTS for ri in (0, 2)]
    big = large_411_stream()
    out.append((big.name, big.data, big, False))
    out += [("s420", synth.synth_jpeg(131, 77, 1, 85, "420", 3), None, False), ("s444", synth.synth_jpeg(96, 40, 2, 90, "444", 0), None, False),
            ("s420_sync", synth.synth_jpeg(320, 200, 3, 75, "420", 0), None, False)]
    out += [("gray_ri", _gray_jpeg(99, 61, 4, 80, 2), None, True), ("gray", _gray_jpeg(64, 33, 5, 90), None, True)]
    return out


MIXED = _mixed()


def _gate(gray):
    import ocljpegdecoder_b200 as b2j
    return b2j.GATE_EXTENDED | b2j.GATE_GRAY if gray else b2j.GATE_EXTENDED


def _oracle(oracle, data, gray=False):
    from oracle import GATE_EXTENDED, GATE_GRAY
    oracle.set_strict(False)
    try:
        rc, _, coef, bgra = oracle.decode(data, gate=GATE_EXTENDED | (GATE_GRAY if gray else 0))
    finally:
        oracle.set_strict(True)
    assert rc == 0
    return coef, bgra


def _decode(dec, files, gray=False):
    batch = dec.batch(files, gate=_gate(gray))
    batch.upload()
    batch.decode()
    st = batch.status()
    coefs = [batch.coefs(i) for i in range(len(files))]
    pix = [batch.pixels(i) for i in range(len(files))]
    return batch, st, coefs, pix


def _check(oracle, items, st, coefs, pix):
    assert not st.any(), [(items[i][0], int(st[i])) for i in np.nonzero(st)[0]]
    for (name, data, s, gray), c, p in zip(items, coefs, pix):
        want_c, want_p = _oracle(oracle, data, gray)
        assert np.array_equal(c, want_c), name
        if s is not None:
            assert np.array_equal(c, s.expected_coefs()), name
        assert np.array_equal(p, want_p), (name, int((p != want_p).any(axis=2).sum()))


@pytest.fixture(scope="module")
def mixed_default(decoder):
    batch, st, coefs, pix = _decode(decoder, [m[1] for m in MIXED], gray=True)
    yield batch, st, coefs, pix
    batch.close()


def test_generic_layouts_mixed_batch(oracle, mixed_default, reference_digests):
    batch, st, coefs, pix = mixed_default
    _check(oracle, MIXED, st, coefs, pix)
    # the inputs the unmodified reference decoded (gate skipped): its own coefficients and pixels
    want = reference_digests["generic_luma"]
    n = 0
    for (name, data, _, _), c, p in zip(MIXED, coefs, pix):
        if name.startswith("ref_"):
            w = want[name[4:]]
            assert hashlib.sha256(data).hexdigest() == w["file_sha256"]
            assert hashlib.sha256(c.tobytes()).hexdigest() == w["coef_sha256"], name
            assert hashlib.sha256(p.tobytes()).hexdigest() == w["pixel_sha256"], name
            n += 1
    assert n == 2 * len(GENERIC_LAYOUTS)


def test_generic_layouts_other_output_formats(mixed_default):
    import ocljpegdecoder_b200 as b2j
    batch, _, _, bgra = mixed_default
    try:
        batch.set_output_format(b2j.OUT_RGB24)
        batch.decode()
        assert not batch.status().any()
        for i, b in enumerate(bgra):
            assert np.array_equal(batch.pixels(i), b[..., 2::-1]), MIXED[i][0]
        batch.set_output_format(b2j.OUT_RGB_PLANAR)
        batch.decode()
        assert not batch.status().any()
        for i, b in enumerate(bgra):
            assert np.array_equal(batch.pixels(i), np.moveaxis(b[..., 2::-1], 2, 0)), MIXED[i][0]
    finally:
        batch.set_output_format(b2j.OUT_BGRA)


@pytest.mark.parametrize("luma", [(4, 1), (1, 4), (3, 1), (4, 2), (2, 4)], ids=lambda s: "%d%d" % s)
def test_secondary_boundary_generic_luma(decoder, oracle, luma):
    import ocljpegdecoder_b200 as b2j
    s = make_stream("idct", luma, 8 * luma[0] * 3 - 5, 8 * luma[1] * 2 + 3, "photo", 40 + luma[0] * 5 + luma[1])
    coef, bgra = _oracle(oracle, s.data)
    idct = b2j.Idct(decoder, 8 * luma[0] * 3 - 5, 8 * luma[1] * 2 + 3, luma[0], luma[1])
    try:
        assert idct.blk_count == coef.shape[0]
        idct.upload(coef)
        idct.run()
        assert np.array_equal(idct.pixels(), bgra)
        assert np.array_equal(idct.coefs(), coef)
    finally:
        idct.close()


def test_tables_per_component(decoder, oracle):
    """Huffman tables mapped to the components in several ways (ids 2 and 3 included), three and four DQTs with Cr on a
    table of its own; 4:2:0, 4:4:4 and a generic layout, with and without restart markers; in the same batch images that
    share the DHT payloads but map them differently, and images with one mapping and different DQTs."""
    ss = table_streams()
    items = [(s.name, s.data, s, False) for s in ss]
    batch, st, coefs, pix = _decode(decoder, [s.data for s in ss])
    batch.close()
    _check(oracle, items, st, coefs, pix)


def test_long_codes(decoder, oracle):
    """Codes longer than every first-level table: the second-level DC lookup of the decoder, the walk's one-symbol path
    through the decode tables in global memory; once more with the pre-lanes off (every chunk border is repaired by
    the sweep)."""
    ss = long_code_streams()
    items = [(s.name, s.data, s, False) for s in ss]
    batch, st, coefs, pix = _decode(decoder, [s.data for s in ss])
    batch.close()
    _check(oracle, items, st, coefs, pix)
    k = [s.name for s in ss].index("long_photo_22_ri0")
    os.environ["B2J_SYNC_PRE"] = "0"
    try:
        batch = decoder.batch([ss[k].data])
    finally:
        del os.environ["B2J_SYNC_PRE"]
    try:
        batch.upload()
        batch.decode()
        assert not batch.status().any()
        assert np.array_equal(batch.coefs(0), coefs[k]) and np.array_equal(batch.pixels(0), pix[k])
    finally:
        batch.close()


def test_largest_decode_tables(decoder, oracle):
    """Two DC and three AC tables of the largest kind fit the decode CTA's shared memory and decode; three DC tables of
    that kind do not, and the parser refuses those files one by one instead of failing the batch that holds them."""
    import ocljpegdecoder_b200 as b2j
    fits = [big_table_stream("dc2_ac3", ri) for ri in (0, 4)]
    good = synth.synth_jpeg(160, 96, 12, 90, "420", 0)
    items = [(s.name, s.data, s, False) for s in fits] + [("good", good, None, False)]
    batch, st, coefs, pix = _decode(decoder, [it[1] for it in items])
    batch.close()
    _check(oracle, items, st, coefs, pix)
    for name in sorted(BIG_MAPPINGS):
        if name == "dc2_ac3":
            continue
        big = big_table_stream(name)
        assert b2j.parse_header(big.data)[0] == -3   # B2J_E_UNSUPPORTED
        outs, st = decoder.decode_host([big.data, good])
        assert st[0] == -3 and st[1] == 0, st
        assert np.array_equal(outs[1], _oracle(oracle, good)[1])
