"""CPU: the streams of the layout tests (tests/test_gpu_layouts.py), checked without any decoder under test.

The generators write streams the GPU suite had never seen: generic sampling layouts (up to 10 blocks per MCU, chroma
components with several blocks), Huffman and quantisation tables mapped to the components in every way the gate admits
(table ids 2 and 3, Cr on tables of its own), codes long enough to leave every first-level lookup (a 16-bit DC code and
a 16-bit end-of-block code), and Huffman tables whose decode tables are the largest a search over code lengths finds.
For each stream the oracle's coefficient tap must be the written blocks times the quantiser of each block's component
-- a check that depends on no decoder. Streams without restart markers also go through the host emulation of the
self-synchronising path (tests/native/synccheck.cpp), and the long-code streams must reach its one-symbol path through
the decode tables."""
import ctypes
import os

import numpy as np
import pytest

import jpegcraft
import synth
from conftest import ROOT
from test_oracle import GENERIC_LAYOUTS

MULTI_CHROMA_LAYOUTS = [((2, 2), (2, 1), (2, 1)), ((2, 2), (1, 2), (1, 2)), ((4, 1), (2, 1), (2, 1)), ((2, 2), (2, 1), (1, 2))]
LAYOUTS = GENERIC_LAYOUTS + MULTI_CHROMA_LAYOUTS

Q_LUMA = [2 + (i % 5) for i in range(64)]
Q_CHROMA = [3 + (i % 4) for i in range(64)]
Q_THIRD = [1 + (i * 7) % 9 for i in range(64)]
Q_FOURTH = [4 + (i % 3) for i in range(64)]


def layout_id(samp):
    return "_".join("%d%d" % s for s in samp)


class Stream:
    """A crafted file and what it was written from."""

    def __init__(self, name, kind, data, samp, blocks, qtabs, comp_quant):
        self.name, self.kind, self.data, self.samp, self.blocks, self.qtabs, self.comp_quant = name, kind, data, samp, blocks, qtabs, comp_quant

    @property
    def restart_interval(self):
        return _restart_interval(self.data)

    def expected_coefs(self):
        """The coefficient tap a correct decoder produces: blocks x quantiser of the block's component, natural order."""
        nblk = [h * v for h, v in self.samp]
        comp = np.repeat([0, 1, 2], nblk)
        comp = np.tile(comp, len(self.blocks) // sum(nblk))
        q = np.array([self.qtabs[self.comp_quant[c]] for c in range(3)], np.int64)[comp]
        out = np.zeros((len(self.blocks), 64), np.int32)
        out[:, jpegcraft.ZIGZAG] = self.blocks * q
        return out


def _restart_interval(data):
    k = data.find(b"\xff\xdd")
    return int.from_bytes(data[k + 4:k + 6], "big") if 0 <= k < data.find(b"\xff\xda") else 0


def crafted_blocks(n, seed, stuffed=True):
    """Blocks that a photographic encoder rarely writes: all 63 AC set (no end-of-block), ZRL chains, the largest
    baseline magnitudes, the last coefficient alone, runs of ones that produce FF00 stuffing."""
    rng = np.random.RandomState(seed)
    blocks = np.zeros((n, 64), np.int64)
    for b in range(n):
        kind = (b + seed) % 6
        if kind == 0:
            blocks[b, 1:] = rng.randint(1, 4, 63) * rng.choice([-1, 1], 63)
        elif kind == 1:
            blocks[b, 50 + b % 13] = int(rng.randint(1, 30))
        elif kind == 3:
            blocks[b, 1:6] = rng.choice([-1023, 1023, -1, 1, 700], 5)
        elif kind == 4:
            blocks[b, 63] = -1
        elif kind == 5 and stuffed:
            blocks[b, 1:40] = -1 if b % 2 else 1
    blocks[:, 0] = np.clip(np.cumsum(rng.randint(-300, 300, n)), -1000, 1000)
    return blocks


def make_stream(name, samp, w, h, kind, seed, ri=0, qtabs=(Q_LUMA, Q_CHROMA), comp_quant=(0, 1, 1), **kw):
    """kind 'photo': synth.synth_pixels through jpegcraft.encode_pixels; 'crafted': crafted_blocks."""
    samp = jpegcraft._layout(samp)
    qtabs = [list(q) for q in qtabs]
    if kind == "photo":
        data, blocks = jpegcraft.encode_pixels(synth.synth_pixels(w, h, seed), samp, qtabs, comp_quant, restart_interval=ri, **kw)
    else:
        mw, mh = 8 * max(a for a, _ in samp), 8 * max(b for _, b in samp)
        n = -(-w // mw) * -(-h // mh) * sum(a * b for a, b in samp)
        blocks = crafted_blocks(n, seed)
        data = jpegcraft.build_jpeg(w, h, samp, blocks, qtabs, restart_interval=ri, comp_quant=comp_quant, **kw)
    return Stream(name, kind, data, samp, blocks, qtabs, comp_quant)


def layout_streams(samp):
    """Per layout: widths = 0, 1, 2, 3 (mod 4), width 1, a single MCU, three tiles or more (a tile holds 192 // blocks per
    MCU MCUs), restart intervals none, 1, not dividing an MCU row and longer than the image; photographic and crafted."""
    samp = jpegcraft._layout(samp)
    mw, mh = 8 * max(a for a, _ in samp), 8 * max(b for _, b in samp)
    tot = sum(a * b for a, b in samp)
    seed = 10 * samp[0][0] + samp[0][1] + 100 * sum(a * b for a, b in samp[1:])
    specs = [("w2mod4", 2 * mw + 2, 2 * mh + 5, "photo", 0),
             ("w3mod4_ri1", 3 * mw - 1, 2 * mh - 3, "crafted", 1),
             ("tiles_ri5", 13 * mw, 7 * mh - 2, "photo", 5),                 # 13 MCUs a row: RI 5 does not divide it
             ("w1_ri_long", 1, 3 * mh + 1, "crafted", 1000),
             ("one_mcu", mw - 3, mh - 1, "crafted", 0)]
    out = [make_stream("%s_%s" % (layout_id(samp), n), samp, w, h, kind, seed + k, ri) for k, (n, w, h, kind, ri) in enumerate(specs)]
    assert 13 * (-(-(7 * mh - 2) // mh)) >= 2 * (192 // tot) + 1
    return out


# Huffman tables in slots 2 and 3 as well, each with contents of its own
def _all_slot_tables():
    t = dict(jpegcraft.STD_TABLES)
    rev = jpegcraft.reversed_tables()
    t[(0, 2)] = rev[(0, 1)]
    t[(1, 2)] = rev[(1, 0)]
    t[(0, 3)] = (list(jpegcraft.LONG_DC_BITS), list(jpegcraft.LONG_DC_VALS))
    t[(1, 3)] = rev[(1, 1)]
    return t


TABLE_MAPPINGS = [   # (name, comp_tables, qtabs, comp_quant)
    ("y11_cb00_cr10", ((1, 1), (0, 0), (1, 0)), (Q_LUMA, Q_CHROMA), (0, 1, 1)),
    ("ids23", ((2, 2), (0, 1), (3, 3)), (Q_LUMA, Q_CHROMA), (0, 1, 1)),
    ("q012", ((0, 0), (1, 1), (1, 1)), (Q_LUMA, Q_CHROMA, Q_THIRD), (0, 1, 2)),
    ("q3_mixed", ((3, 2), (1, 0), (2, 3)), (Q_LUMA, Q_CHROMA, Q_THIRD, Q_FOURTH), (3, 0, 2)),
]


def table_streams():
    """Every mapping on 4:2:0, 4:4:4 and a generic layout, with and without restart markers; then, for the LUT-set cache,
    a pair with identical DHT payloads and different mappings and a pair with one mapping and different DQTs."""
    out = []
    tables = _all_slot_tables()
    for k, (name, ct, qt, cq) in enumerate(TABLE_MAPPINGS):
        for j, samp in enumerate([(2, 2), (1, 1), ((2, 2), (2, 1), (1, 2))]):
            for ri in (0, 3):
                kind = "photo" if (j + ri) % 2 == 0 else "crafted"
                out.append(make_stream("%s_%s_ri%d" % (name, layout_id(jpegcraft._layout(samp)), ri), samp, 77, 45, kind, 60 + 7 * k + j,
                                       ri, qt, cq, tables=tables, comp_tables=ct))
    px = dict(w=64, h=48, kind="photo", seed=5)
    out.append(make_stream("cache_map_a", (2, 2), tables=tables, comp_tables=((0, 0), (1, 1), (1, 1)), **px))
    out.append(make_stream("cache_map_b", (2, 2), tables=tables, comp_tables=((0, 0), (1, 1), (0, 1)), **px))
    out.append(make_stream("cache_dqt_a", (2, 2), qtabs=(Q_LUMA, Q_CHROMA, Q_THIRD), comp_quant=(0, 1, 2), **px))
    out.append(make_stream("cache_dqt_b", (2, 2), qtabs=(Q_LUMA, Q_FOURTH, Q_CHROMA), comp_quant=(0, 1, 2), **px))
    return out


def long_code_streams():
    """DC codes of 1..11 bits and one of 16 bits, AC tables in reversed Annex K order (end-of-block on a 16-bit code):
    a crafted 2x2 stream, photographic 4:2:0 and a generic layout, with and without restart markers."""
    t = jpegcraft.long_code_tables()
    out = []
    for ri in (0, 2):
        out.append(make_stream("long_crafted_22_ri%d" % ri, (2, 2), 96, 64, "crafted", 3, ri, tables=t))
        out.append(make_stream("long_photo_22_ri%d" % ri, (2, 2), 200, 120, "photo", 4, ri, tables=t))
        out.append(make_stream("long_photo_42_ri%d" % ri, (4, 2), 133, 70, "photo", 5, ri, tables=t))
    return out


# ---- the largest decode tables --------------------------------------------------------------------------------------
LUT_MAX_DECODE = 12288   # kLutMaxDecode (ocljpegdecoder_b200/csrc/b2j_internal.h), u16 entries


def big_tables():
    """Four DC and four AC tables whose two-level decode tables are the largest the search in jpegcraft finds (256 codes
    each, symbols in reversed order so that the symbols a stream uses sit on the longest codes), each slot with a
    different symbol order."""
    dc_bits, ac_bits = jpegcraft.largest_table_bits(6), jpegcraft.largest_table_bits(10)
    t = {}
    for th in range(4):
        vals = list(range(255, -1, -1))
        vals = vals[th:] + vals[:th]
        t[(0, th)] = (list(dc_bits), vals)
        t[(1, th)] = (list(ac_bits), vals)
    return t


def lut_decode_entries(tables, comp_tables):
    """What build_lut_set() puts in the decode part of the set: header + one table per distinct slot, padded to 8."""
    slots = sorted({(0, dc) for dc, _ in comp_tables} | {(1, ac) for _, ac in comp_tables})
    n = 16 + sum(jpegcraft._lut_entries(tables[s][0], 6 if s[0] == 0 else 10) for s in slots)
    return -(-n // 8) * 8


BIG_MAPPINGS = {"dc2_ac3": ((0, 0), (1, 1), (1, 2)), "dc3_ac2": ((0, 0), (1, 1), (2, 1)), "dc3_ac3": ((0, 0), (1, 1), (2, 2))}


def big_table_stream(name, ri=0):
    return make_stream("big_%s_ri%d" % (name, ri), (2, 2), 120, 72, "photo", 8, ri, tables=big_tables(), comp_tables=BIG_MAPPINGS[name])


def all_streams():
    out = [s for samp in LAYOUTS for s in layout_streams(samp)]
    out += table_streams() + long_code_streams()
    out += [big_table_stream("dc2_ac3", ri) for ri in (0, 4)]
    return out


STREAMS = all_streams()


# ---- tests ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def synccheck(built):
    L = ctypes.CDLL(os.path.join(ROOT, "tests", "native", "libb2jsync.so"))
    L.b2j_synccheck.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]

    def run(data, force_sweep=False):
        stats = np.zeros(10, np.uint64)
        rc = L.b2j_synccheck(data, len(data), 1, 1 if force_sweep else 0, stats.ctypes.data)
        return rc, stats
    return run


def test_generators_cover_what_they_claim():
    names = [s.name for s in STREAMS]
    assert len(set(names)) == len(names)
    for samp in LAYOUTS:
        ss = [s for s in STREAMS if s.samp == list(samp)]
        widths = [synth_w(s) for s in ss]
        assert {w % 4 for w in widths} == {0, 1, 2, 3} and 1 in widths
        assert {s.restart_interval for s in ss} >= {0, 1, 5, 1000}
    assert max(sum(a * b for a, b in samp) for samp in LAYOUTS) == 10
    # the crafted blocks carry what they are meant to
    craft = [s for s in STREAMS if s.kind == "crafted"]
    allb = np.concatenate([s.blocks for s in craft])
    assert (np.abs(allb[:, 1:]) == 1023).any() and (allb[:, 1:] != 0).all(axis=1).any()
    assert all(s.data.count(b"\xff\x00") for s in STREAMS if "w3mod4" in s.name)


def synth_w(s):
    k = s.data.index(b"\xff\xc0")
    return int.from_bytes(s.data[k + 7:k + 9], "big")


@pytest.mark.parametrize("s", STREAMS, ids=lambda s: s.name)
def test_oracle_coefficients_are_the_written_blocks(oracle, s):
    """Independent of every decoder: the oracle's tap equals the blocks the writer entropy-coded, dequantised with the
    table of each block's own component."""
    from oracle import GATE_EXTENDED
    oracle.set_strict(False)
    try:
        rc, img, coef, _ = oracle.decode(s.data, gate=GATE_EXTENDED, want_pixels=False)
    finally:
        oracle.set_strict(True)
    assert rc == 0
    assert [img.quant_id[c] for c in range(3)] == list(s.comp_quant)
    assert np.array_equal(coef, s.expected_coefs())


@pytest.mark.parametrize("s", [s for s in STREAMS if s.restart_interval == 0], ids=lambda s: s.name)
def test_self_sync_emulation_agrees(synccheck, s):
    rc, st = synccheck(s.data)
    assert rc == 0, (rc, st.tolist())
    rc, st2 = synccheck(s.data, force_sweep=True)
    assert rc == 0, (rc, st2.tolist())
    if s.name.startswith("long_"):
        assert st[8] > 0, "the walk never took the one-symbol path through the decode tables: %s" % st.tolist()


def test_large_411_frame_stream(oracle, synccheck):
    """4:1:1 at 1920x1080 without restart markers: many synchronisation chunks."""
    s = large_411_stream()
    from oracle import GATE_EXTENDED
    oracle.set_strict(False)
    try:
        rc, _, coef, _ = oracle.decode(s.data, gate=GATE_EXTENDED, want_pixels=False)
    finally:
        oracle.set_strict(True)
    assert rc == 0 and np.array_equal(coef, s.expected_coefs())
    rc, st = synccheck(s.data)
    assert rc == 0 and st[1] >= 8, st.tolist()


def large_411_stream():
    return make_stream("large_411", (4, 1), 1920, 1080, "photo", 21, 0, qtabs=([1 + i % 3 for i in range(64)], [2] * 64))


def test_largest_tables_found(built):
    """The search finds 256-code tables of 2704 (DC) and 2144 (AC) entries; the C++ builder agrees with the count."""
    L = ctypes.CDLL(os.path.join(ROOT, "tests", "native", "libb2jcheck.so"))
    L.chk_lut_decode.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_uint32, ctypes.POINTER(ctypes.c_int)]
    for (tc, th), (bits, vals) in big_tables().items():
        n = ctypes.c_int()
        assert L.chk_lut_decode(bytes(bits), bytes(vals), 1 if tc == 0 else 0, 0, ctypes.byref(n)) >= 0
        assert n.value == jpegcraft._lut_entries(bits, 6 if tc == 0 else 10) == (2704 if tc == 0 else 2144)
    for (tc, _), (bits, vals) in jpegcraft.STD_TABLES.items():   # Annex K: the count agrees there too
        assert L.chk_lut_decode(bytes(bits), bytes(vals), 1 if tc == 0 else 0, 0, ctypes.byref(n)) >= 0
        assert n.value == jpegcraft._lut_entries(bits, 6 if tc == 0 else 10)


@pytest.mark.parametrize("name", sorted(BIG_MAPPINGS))
def test_parser_refuses_tables_that_do_not_fit(built, oracle, name):
    """Three components on distinct 256-code tables need more decode-table space than a decode CTA has: the parser
    refuses the file (per file, so that a batch is not lost); what fits is admitted. The oracle decodes all of them."""
    import ocljpegdecoder_b200 as b2j
    s = big_table_stream(name)
    need = lut_decode_entries(big_tables(), BIG_MAPPINGS[name])
    print(name, "decode-table entries", need)
    assert need == {"dc2_ac3": 11856, "dc3_ac2": 12416, "dc3_ac3": 14560}[name]
    for gate in (b2j.GATE_EXTENDED, b2j.GATE_REFERENCE, b2j.GATE_EXTENDED | b2j.PARSE_ROBUST):
        rc, _ = b2j.parse_header(s.data, gate)
        assert rc == (0 if need <= LUT_MAX_DECODE else -3), (gate, rc)
    from oracle import GATE_EXTENDED
    assert oracle.decode(s.data, gate=GATE_EXTENDED, want_pixels=False)[0] == 0
