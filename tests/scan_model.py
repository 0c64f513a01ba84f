"""A plain model of the decoder's scan pre-pass (k_unstuff_fused, ocljpegdecoder_b200/csrc/kernels.cu) and a helper that
places fill bytes so that chosen byte patterns land on the pre-pass's borders (test tooling, pure Python).

The pre-pass classifies the raw scan with the host's pad (FF D9 D9 ...) behind it, byte by byte with predecessor p and
successor n:
  FF     : kept iff n == 00; otherwise dropped, and the scan ends here (a terminator) unless n is 00, FF or D0..D7;
  not FF : dropped iff p == FF and it is 00 or D0..D7 (then an RSTn marker); kept otherwise.
Everything at and behind the first terminator is cut. Its borders are 4-byte words, 16-byte groups, a thread's
kScanGroups groups and a chunk of kScanThreads threads; the geometry is read from b2j_internal.h.
"""
import os
import re

_HDR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ocljpegdecoder_b200", "csrc", "b2j_internal.h")


def _constant(name):
    with open(_HDR) as f:
        m = re.search(r"constexpr int %s = (\d+);" % name, f.read())
    assert m, name
    return int(m.group(1))


SCAN_GROUPS = _constant("kScanGroups")
SCAN_THREADS = _constant("kScanThreads")
WORD, GROUP = 4, 16
THREAD = GROUP * SCAN_GROUPS
CHUNK = THREAD * SCAN_THREADS
BORDERS = {"word": WORD, "group": GROUP, "thread": THREAD, "chunk": CHUNK}
PAD = 32   # the host pads a scan with at least this many bytes (FF D9 D9 ...)


def where(i):
    """(chunk, thread, 16-byte group, word) of scan byte i."""
    return i // CHUNK, i % CHUNK // THREAD, i % THREAD // GROUP, i % GROUP // WORD


def split_at(i):
    """The borders between scan bytes i and i + 1, as names of BORDERS."""
    return {name for name, b in BORDERS.items() if (i + 1) % b == 0}


class Prepass:
    """The pre-pass on one raw scan (the bytes from behind SOS to the end of the file).

    clean      : the clean stream (kept bytes up to the first terminator)
    term       : scan offset of the terminator FF
    markers    : [(scan offset of the Dn byte, Dn, clean position)] in front of the terminator
    specials   : [(scan offset, kind)] of every byte that is not plain data: 'stuff' (an FF followed by 00), 'fill' (an FF
                 followed by FF), 'rst' (the FF of FF Dn), 'term' (the terminator FF), 'zero' / 'dn' (the second byte)
    """

    def __init__(self, scan):
        raw = bytes(scan) + b"\xFF" + b"\xD9" * (PAD - 1)
        clean, markers, specials = bytearray(), [], []
        term = None
        for i in range(len(raw) - 1):
            b, p, n = raw[i], raw[i - 1] if i else 0, raw[i + 1]
            if b == 0xFF:
                if n == 0x00:
                    clean.append(b)
                    specials.append((i, "stuff"))
                elif n == 0xFF:
                    specials.append((i, "fill"))
                elif 0xD0 <= n <= 0xD7:
                    specials.append((i, "rst"))
                else:
                    specials.append((i, "term"))
                    term = i
                    break
            elif p == 0xFF and b == 0x00:
                specials.append((i, "zero"))
            elif p == 0xFF and 0xD0 <= b <= 0xD7:
                specials.append((i, "dn"))
                markers.append((i, b, len(clean)))
            else:
                clean.append(b)
        assert term is not None   # the pad always ends the scan
        self.clean, self.term, self.markers, self.specials = bytes(clean), term, markers, specials

    def intervals(self, n_segs, has_dri):
        """(clean start of every restart interval, clean bytes the decoders may read): with DRI the first n_segs - 1 markers
        start intervals; a later one, or any marker without DRI, ends the readable stream (b2j.h)."""
        starting = n_segs - 1 if has_dri else 0
        starts = [0] + [c for _, _, c in self.markers[:starting]]
        stray = [c for _, _, c in self.markers[starting:]]
        return starts, min([len(self.clean)] + stray)

    def kept_before_chunks(self):
        """Clean bytes in front of each chunk the scan reaches (the copy-out's destination offset)."""
        out, kept, k = [], 0, 0
        dropped = {i for i, kind in self.specials if kind in ("fill", "rst", "zero", "dn")}
        for i in range(self.term):
            if i % CHUNK == 0:
                out.append(kept)
            if i not in dropped:
                kept += 1
        return out

    def chunk_keeps(self):
        """Clean bytes each chunk in front of the terminator's contributes."""
        starts = self.kept_before_chunks() + [len(self.clean)]
        return [b - a for a, b in zip(starts, starts[1:])]


def place_fills(intervals, wants, default=0, cap=70):
    """Per-marker fill counts for jpegcraft.join_scan(intervals, fills) that put each wanted pattern on a border.

    wants: [(kind, border size)] or [(kind, border size, cap)] satisfied in order, each by the first marker that can, with kind
      'rst'      : the FF of the marker is the last byte in front of the border (fill any, 0 included)
      'fillrun'  : the same, behind at least one fill byte (a fill run ending in a marker, split between FF and Dn)
      'fillcross': a fill run in front of the marker crosses the border
      'stuff'    : the FF of a stuffed FF 00 in the interval behind the marker is the last byte in front of the border.
    A marker that cannot satisfy the next want with at most `cap` fill bytes gets `default` (an int, or a function of
    the marker's ordinal). Returns (fills, the wants that no marker satisfied)."""
    fills, pending, pos = [], list(wants), len(intervals[0])
    for r, iv in enumerate(intervals[1:]):
        f = None
        if pending:
            kind, b, limit = (pending[0] + (cap,))[:3]
            if kind in ("rst", "fillrun"):
                f = (b - 1 - pos) % b
                if kind == "fillrun" and f == 0:
                    f = b
            elif kind == "fillcross":
                f = (b - pos) % b + 1   # the fill bytes at border - 1 and border
                f = f if f >= 2 else f + b
            elif kind == "stuff":
                offs = [j for j in range(len(iv) - 1) if iv[j] == 0xFF and iv[j + 1] == 0]
                cands = [(b - 1 - (pos + 2 + j)) % b for j in offs]
                f = min(cands) if cands else None
            if f is not None and f <= limit:
                pending.pop(0)
            else:
                f = None
        if f is None:
            f = default(r) if callable(default) else default
        fills.append(f)
        pos += f + 2 + len(iv)
    return fills, pending
