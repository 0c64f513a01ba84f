"""A tiny baseline-JPEG *writer* for crafting edge-case streams (test tooling, pure Python).

It entropy-codes caller-supplied QUANTISED coefficient blocks (scan order) with the JPEG Annex K
tables, so tests control exactly which symbols appear: full blocks without EOB, ZRL chains, DC
category 0 and 11, maximum AC magnitudes, stuffed FF bytes, fill bytes before RSTn, restart
interval 1, and so on. Small images only.
"""
import numpy as np

# Annex K.3 typical Huffman tables
DC_LUMA_BITS = [0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0]
DC_LUMA_VALS = list(range(12))
DC_CHROMA_BITS = [0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0]
DC_CHROMA_VALS = list(range(12))
AC_LUMA_BITS = [0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7D]
AC_LUMA_VALS = [
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71,
    0x14, 0x32, 0x81, 0x91, 0xA1, 0x08, 0x23, 0x42, 0xB1, 0xC1, 0x15, 0x52, 0xD1, 0xF0, 0x24, 0x33, 0x62, 0x72,
    0x82, 0x09, 0x0A, 0x16, 0x17, 0x18, 0x19, 0x1A, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2A, 0x34, 0x35, 0x36, 0x37,
    0x38, 0x39, 0x3A, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4A, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
    0x5A, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6A, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7A, 0x83,
    0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8A, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9A, 0xA2, 0xA3,
    0xA4, 0xA5, 0xA6, 0xA7, 0xA8, 0xA9, 0xAA, 0xB2, 0xB3, 0xB4, 0xB5, 0xB6, 0xB7, 0xB8, 0xB9, 0xBA, 0xC2, 0xC3,
    0xC4, 0xC5, 0xC6, 0xC7, 0xC8, 0xC9, 0xCA, 0xD2, 0xD3, 0xD4, 0xD5, 0xD6, 0xD7, 0xD8, 0xD9, 0xDA, 0xE1, 0xE2,
    0xE3, 0xE4, 0xE5, 0xE6, 0xE7, 0xE8, 0xE9, 0xEA, 0xF1, 0xF2, 0xF3, 0xF4, 0xF5, 0xF6, 0xF7, 0xF8, 0xF9, 0xFA]
AC_CHROMA_BITS = [0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77]
AC_CHROMA_VALS = [
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22,
    0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xA1, 0xB1, 0xC1, 0x09, 0x23, 0x33, 0x52, 0xF0, 0x15, 0x62, 0x72, 0xD1,
    0x0A, 0x16, 0x24, 0x34, 0xE1, 0x25, 0xF1, 0x17, 0x18, 0x19, 0x1A, 0x26, 0x27, 0x28, 0x29, 0x2A, 0x35, 0x36,
    0x37, 0x38, 0x39, 0x3A, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4A, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
    0x59, 0x5A, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6A, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7A,
    0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8A, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9A,
    0xA2, 0xA3, 0xA4, 0xA5, 0xA6, 0xA7, 0xA8, 0xA9, 0xAA, 0xB2, 0xB3, 0xB4, 0xB5, 0xB6, 0xB7, 0xB8, 0xB9, 0xBA,
    0xC2, 0xC3, 0xC4, 0xC5, 0xC6, 0xC7, 0xC8, 0xC9, 0xCA, 0xD2, 0xD3, 0xD4, 0xD5, 0xD6, 0xD7, 0xD8, 0xD9, 0xDA,
    0xE2, 0xE3, 0xE4, 0xE5, 0xE6, 0xE7, 0xE8, 0xE9, 0xEA, 0xF2, 0xF3, 0xF4, 0xF5, 0xF6, 0xF7, 0xF8, 0xF9, 0xFA]

STD_TABLES = {
    (0, 0): (DC_LUMA_BITS, DC_LUMA_VALS), (0, 1): (DC_CHROMA_BITS, DC_CHROMA_VALS),
    (1, 0): (AC_LUMA_BITS, AC_LUMA_VALS), (1, 1): (AC_CHROMA_BITS, AC_CHROMA_VALS),
}


def canonical_codes(bits, vals):
    """symbol -> (code, length)"""
    out, code, k = {}, 0, 0
    for l in range(1, 17):
        for _ in range(bits[l - 1]):
            out[vals[k]] = (code, l)
            code += 1
            k += 1
        code <<= 1
    return out


class BitWriter:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def put(self, value, nbits):
        if nbits == 0:
            return
        self.acc = (self.acc << nbits) | (value & ((1 << nbits) - 1))
        self.n += nbits
        while self.n >= 8:
            b = (self.acc >> (self.n - 8)) & 0xFF
            self.out.append(b)
            if b == 0xFF:
                self.out.append(0x00)   # byte stuffing
            self.n -= 8
        self.acc &= (1 << self.n) - 1

    def flush(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)   # pad with ones

    def raw(self, data):
        assert self.n == 0
        self.out += bytes(data)


def _category(v):
    return 0 if v == 0 else int(abs(int(v))).bit_length()


def _value_bits(v, size):
    return v if v >= 0 else v + (1 << size) - 1


def encode_block(bw, blk, pred, dc_codes, ac_codes, zrl_only_tail=False):
    """blk: 64 quantised coefficients in SCAN order; blk[0] is the absolute DC value."""
    diff = int(blk[0]) - pred
    s = _category(diff)
    code, l = dc_codes[s]
    bw.put(code, l)
    bw.put(_value_bits(diff, s), s)
    run = 0
    last_nz = max([i for i in range(1, 64) if blk[i] != 0], default=0)
    for i in range(1, 64):
        v = int(blk[i])
        if v == 0:
            if i > last_nz and not zrl_only_tail:
                code, l = ac_codes[0x00]
                bw.put(code, l)
                return int(blk[0])
            run += 1
            if run == 16:
                code, l = ac_codes[0xF0]
                bw.put(code, l)
                run = 0
            continue
        s = _category(v)
        code, l = ac_codes[(run << 4) | s]
        bw.put(code, l)
        bw.put(_value_bits(v, s), s)
        run = 0
    if run and not zrl_only_tail:
        code, l = ac_codes[0x00]
        bw.put(code, l)
    return int(blk[0])


def _seg(marker, payload):
    return bytes([0xFF, marker]) + (len(payload) + 2).to_bytes(2, "big") + bytes(payload)


def build_jpeg(width, height, sampling, blocks, qtabs, restart_interval=0, fill_before_rst=0,
               tables=None, comp_tables=((0, 0), (1, 1), (1, 1)), with_app0=True, trailing=b"", dqt16=False,
               comp_quant=(0, 1, 1)):
    """sampling: luma (h, v) with 1x1 chroma, or ((hy, vy), (hu, vu), (hv, vv)). blocks: int array [n_blocks, 64] in MCU order and
    SCAN (zig-zag) coefficient order, blocks[:,0] = absolute DC. qtabs: one to four 64-lists (zig-zag order), written as
    DQT tables 0, 1, ...; comp_quant: the table of each component (Y, Cb, Cr). tables: dict like STD_TABLES, keyed
    (class, id); comp_tables: the (DC id, AC id) of each component. Returns the file bytes."""
    tables = tables or STD_TABLES
    if isinstance(sampling[0], (tuple, list)):
        samp = [tuple(x) for x in sampling]          # ((hy, vy), (hu, vu), (hv, vv))
    else:
        samp = [tuple(sampling), (1, 1), (1, 1)]
    h, v = samp[0]
    nblk = [a * b for a, b in samp]
    tot = sum(nblk)
    mcu_w, mcu_h = 8 * max(a for a, _ in samp), 8 * max(b for _, b in samp)
    n_mcu = ((width + mcu_w - 1) // mcu_w) * ((height + mcu_h - 1) // mcu_h)
    blocks = np.asarray(blocks)
    assert blocks.shape == (n_mcu * tot, 64), (blocks.shape, n_mcu * tot)
    out = bytearray(b"\xFF\xD8")
    if with_app0:
        out += _seg(0xE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    assert 1 <= len(qtabs) <= 4 and all(0 <= q < len(qtabs) for q in comp_quant)
    for k, qt in enumerate(qtabs):
        if dqt16:   # precision 1: 64 big-endian 16-bit entries (the reference reads them WITHOUT a byte swap, parser.cpp:81-87)
            out += _seg(0xDB, bytes([0x10 | k]) + b"".join(int(q).to_bytes(2, "big") for q in qt))
        else:
            out += _seg(0xDB, bytes([k]) + bytes(qt))
    sof = bytes([8]) + height.to_bytes(2, "big") + width.to_bytes(2, "big") + bytes([3])
    for c in range(3):
        sof += bytes([c + 1, (samp[c][0] << 4) | samp[c][1], comp_quant[c]])
    out += _seg(0xC0, sof)
    for (tc, th), (bits, vals) in sorted(tables.items()):
        out += _seg(0xC4, bytes([(tc << 4) | th]) + bytes(bits) + bytes(vals))
    if restart_interval:
        out += _seg(0xDD, restart_interval.to_bytes(2, "big"))
    sos = bytes([3])
    for c in range(3):
        sos += bytes([c + 1, (comp_tables[c][0] << 4) | comp_tables[c][1]])
    sos += bytes([0, 0x3F, 0])
    out += _seg(0xDA, sos)
    codes = {k: canonical_codes(*tv) for k, tv in tables.items()}
    bw = BitWriter()
    pred = [0, 0, 0]
    rst = 0
    bi = 0
    for m in range(n_mcu):
        if restart_interval and m and m % restart_interval == 0:
            bw.flush()
            bw.raw(b"\xFF" * fill_before_rst + bytes([0xFF, 0xD0 + (rst & 7)]))
            rst += 1
            pred = [0, 0, 0]
        for c in range(3):
            for _ in range(nblk[c]):
                dc_codes = codes[(0, comp_tables[c][0])]
                ac_codes = codes[(1, comp_tables[c][1])]
                pred[c] = encode_block(bw, blocks[bi], pred[c], dc_codes, ac_codes)
                bi += 1
    bw.flush()
    out += bw.out
    out += b"\xFF\xD9" + trailing
    return bytes(out)


# ---- tables whose codes reach the long-code paths of a decoder ------------------------------------------------------
def reversed_tables():
    """The Annex K code lengths with the symbol order reversed: the most frequent symbols get the longest codes (the AC
    end-of-block code becomes 16 bits long, the DC category 0 code 9 bits for luma and 11 for chroma)."""
    return {k: (list(bits), list(vals)[::-1]) for k, (bits, vals) in STD_TABLES.items()}


# DC code lengths 1..11 and one 16-bit code. With LONG_DC_VALS the 16-bit code is category 0, the longest short code
# category 1, ... so that everyday differences take codes longer than any first-level lookup.
LONG_DC_BITS = [1] * 11 + [0, 0, 0, 0, 1]
LONG_DC_VALS = list(range(11, -1, -1))


def long_code_tables():
    """DC tables with LONG_DC_BITS, AC tables with the Annex K lengths in reversed symbol order."""
    t = reversed_tables()
    t[(0, 0)] = (list(LONG_DC_BITS), list(LONG_DC_VALS))
    t[(0, 1)] = (list(LONG_DC_BITS), list(LONG_DC_VALS[1:]) + [LONG_DC_VALS[0]])
    return t


# ---- a plain photographic encoder for any sampling layout ----------------------------------------------------------
ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
                   28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54,
                   47, 55, 62, 63])   # scan position -> natural (row-major) index


def _layout(sampling):
    if isinstance(sampling[0], (tuple, list)):
        return [tuple(x) for x in sampling]
    return [tuple(sampling), (1, 1), (1, 1)]


def encode_pixels(rgb, sampling, qtabs, comp_quant=(0, 1, 1), **kw):
    """Encodes an RGB image (uint8 [H, W, 3]) as a baseline JPEG in any sampling layout (see build_jpeg): YCbCr in float64
    (JFIF), edges replicated to whole MCUs, chroma box-averaged by its subsampling factors, orthonormal 8x8 DCT-II (which
    is the JPEG FDCT), quantisation by rounding, blocks in MCU and scan order. Returns (file bytes, blocks [n, 64] in
    scan order) -- the blocks are what a decoder's entropy stage must reproduce."""
    from scipy.fft import dctn
    rgb = np.asarray(rgb, np.float64)
    hgt, wid = rgb.shape[:2]
    samp = _layout(sampling)
    hmax, vmax = max(a for a, _ in samp), max(b for _, b in samp)
    mcw, mch = -(-wid // (8 * hmax)), -(-hgt // (8 * vmax))
    r, g, b = rgb[..., 0], rgb[..., 1], rgb[..., 2]
    planes = [0.299 * r + 0.587 * g + 0.114 * b,
              -0.168736 * r - 0.331264 * g + 0.5 * b + 128.0,
              0.5 * r - 0.418688 * g - 0.081312 * b + 128.0]
    pad = ((0, mch * 8 * vmax - hgt), (0, mcw * 8 * hmax - wid))
    coefs = []
    for c, (h, v) in enumerate(samp):
        p = np.pad(planes[c], pad, mode="edge")
        fy, fx = vmax // v, hmax // h
        p = p.reshape(p.shape[0] // fy, fy, p.shape[1] // fx, fx).mean(axis=(1, 3)) - 128.0
        blk = p.reshape(p.shape[0] // 8, 8, p.shape[1] // 8, 8).transpose(0, 2, 1, 3)
        dct = dctn(blk, type=2, norm="ortho", axes=(2, 3)).reshape(blk.shape[0], blk.shape[1], 64)
        q = np.zeros(64)
        q[ZIGZAG] = qtabs[comp_quant[c]]
        quant = np.round(dct / q)[..., ZIGZAG].astype(np.int64)
        quant[..., 1:] = np.clip(quant[..., 1:], -1023, 1023)
        coefs.append(quant)
    blocks = []
    for my in range(mch):
        for mx in range(mcw):
            for c, (h, v) in enumerate(samp):
                for by in range(v):
                    for bx in range(h):
                        blocks.append(coefs[c][my * v + by, mx * h + bx])
    blocks = np.array(blocks, np.int64)
    return build_jpeg(wid, hgt, samp, blocks, qtabs, comp_quant=comp_quant, **kw), blocks


# ---- the largest two-level decode tables ----------------------------------------------------------------------------
def _lut_entries(bits, primary):
    """Entries of the two-level decode table of a code with these BITS (ocljpegdecoder_b200/csrc/huff_lut.cpp): the primary
    table, then one sub-table of 2^(longest code - primary) entries per primary prefix that has longer codes, each
    starting on a multiple of 8 behind the primary table."""
    longest = {}
    code = 0
    for l in range(1, 17):
        for _ in range(bits[l - 1]):
            if l > primary:
                longest[code >> (l - primary)] = l
            code += 1
        code <<= 1
    rel = 0
    for k, prefix in enumerate(sorted(longest)):
        if k:
            rel = -(-rel // 8) * 8
        rel += 1 << (longest[prefix] - primary)
    return (1 << primary) + rel


def largest_table_bits(primary, max_codes=256):
    """BITS (16 counts) of a valid code of at most `max_codes` codes whose two-level decode table is as large as this
    search finds, for a primary table of `primary` bits. Dynamic programme over the primary prefixes, which canonical
    codes fill in order: a prefix whose longest code has length L gets 2^(L - primary) entries and, once its codes are
    no shorter than L0, costs 2^(L0 - primary) codes (all of length L0) or 2^(L0 - primary) + L - L0 codes (L0 ... L-1, L, L).
    The last prefix needs one 16-bit code only."""
    def cost(l0, l):
        return (1 << (l - primary)) if l == l0 else (1 << (l0 - primary)) + l - l0

    def padded(l):
        return -(-(1 << (l - primary)) // 8) * 8

    frontier = {}   # (L of the last full prefix, codes) -> (entries behind the primary table, [L of each full prefix])
    for l in range(primary + 1, 17):
        if cost(primary + 1, l) <= max_codes:
            frontier[(l, cost(primary + 1, l))] = (padded(l), [l])
    best = (0, [])
    for _ in range((1 << primary) - 1):
        nxt = {}
        for (l0, c), (e, seq) in frontier.items():
            if c < max_codes:
                best = max(best, (e + (1 << (16 - primary)), seq + [16]))
            for l in range(l0, 17):
                if c + cost(l0, l) > max_codes:
                    break
                key = (l, c + cost(l0, l))
                if key not in nxt or nxt[key][0] < e + padded(l):
                    nxt[key] = (e + padded(l), seq + [l])
        frontier = nxt
    seq = best[1]
    bits = [0] * 16
    l0 = primary + 1
    for l in seq[:-1]:
        if l == l0:
            bits[l - 1] += 1 << (l - primary)
        else:
            bits[l0 - 1] += (1 << (l0 - primary)) - 1
            for m in range(l0 + 1, l):
                bits[m - 1] += 1
            bits[l - 1] += 2
        l0 = l
    bits[15] += 1
    return bits
