"""CPU: b2j_parse_orientation against Pillow's reading of the EXIF orientation tag (Image.getexif()[0x0112], 1 outside
1..8) on Pillow-written files with every tag value 0..9 and on hand-built files -- big- and little-endian TIFF, an XMP
APP1 in front of the Exif APP1, two Exif APP1s, Exif behind APP0 JFIF and behind a COM; cut and corrupted Exif segments
give 1 or the right code and leave b2j_parse_header's result alone; the ABI of the new symbols and option."""
import ctypes
import io
import struct

import numpy as np
import pytest

import synth


def orient(a, code):
    """The EXIF orientation transform of an (h, w, ...) array (Pillow's exif_transpose table)."""
    return {1: a, 2: a[:, ::-1], 3: a[::-1, ::-1], 4: a[::-1], 5: a.swapaxes(0, 1), 6: a.swapaxes(0, 1)[:, ::-1],
            7: a.swapaxes(0, 1)[::-1, ::-1], 8: a.swapaxes(0, 1)[::-1]}[code]


def tiff(code, big_endian=False, before=(), after=()):
    """A TIFF header and IFD0 with tag 0x0112 = code (SHORT), between extra SHORT entries `before` and `after`."""
    e = ">" if big_endian else "<"
    entries = [(t, v) for t, v in before] + [(0x0112, code)] + [(t, v) for t, v in after]
    out = (b"MM\x00*" if big_endian else b"II*\x00") + struct.pack(e + "I", 8) + struct.pack(e + "H", len(entries))
    for t, v in entries:
        out += struct.pack(e + "HHIHH", t, 3, 1, v, 0)
    return out + struct.pack(e + "I", 0)


def segment(marker, payload):
    return b"\xff" + bytes([marker]) + struct.pack(">H", len(payload) + 2) + payload


def exif_app1(code, big_endian=False):
    return segment(0xE1, b"Exif\x00\x00" + tiff(code, big_endian))


def with_segments(jpeg, *segs):
    """jpeg with the given segments right behind SOI."""
    return jpeg[:2] + b"".join(segs) + jpeg[2:]


def pillow_orientation(data):
    from PIL import Image
    v = Image.open(io.BytesIO(data)).getexif().get(0x0112)
    return v if isinstance(v, int) and 1 <= v <= 8 else 1


@pytest.fixture(scope="module")
def plain():
    """A baseline file without APPn segments."""
    return synth.synth_jpeg(53, 37, 5, 90, "420", 0)


def _parse(data):
    import ocljpegdecoder_b200 as b2j
    return b2j.parse_orientation(data)


def test_pillow_written_tags_0_to_9(built):
    from PIL import Image
    base = Image.fromarray(synth.synth_pixels(53, 37, 3))
    for code in range(10):
        ex = Image.Exif()
        ex[0x0112] = code
        b = io.BytesIO()
        base.save(b, "JPEG", quality=90, exif=ex.tobytes())
        data = b.getvalue()
        want = code if 1 <= code <= 8 else 1
        assert pillow_orientation(data) == want
        assert _parse(data) == want, code


def test_hand_built_files(built, plain):
    app0 = segment(0xE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    xmp = segment(0xE1, b"http://ns.adobe.com/xap/1.0/\x00<x:xmpmeta/>")
    com = segment(0xFE, b"a comment")
    for code in range(1, 9):
        cases = {
            "II": with_segments(plain, exif_app1(code)),
            "MM": with_segments(plain, exif_app1(code, True)),
            "xmp_first": with_segments(plain, xmp, exif_app1(code, True)),
            "two_exif": with_segments(plain, exif_app1(code), exif_app1(9 - code if code != 1 else 6)),
            "after_jfif": with_segments(plain, app0, exif_app1(code)),
            "after_com": with_segments(plain, com, exif_app1(code, True)),
            "after_tables": plain[:plain.index(b"\xff\xc4")] + exif_app1(code) + plain[plain.index(b"\xff\xc4"):],
            "other_tags": with_segments(plain, segment(0xE1, b"Exif\x00\x00" + tiff(code, code % 2 == 0, [(0x010F, 7)], [(0x0131, 2)]))),
        }
        for name, data in cases.items():
            assert pillow_orientation(data) == code, (name, code)
            assert _parse(data) == code, (name, code)
    # no Exif, an XMP APP1 only, a tag behind SOS, out-of-range values
    assert _parse(plain) == 1
    assert _parse(with_segments(plain, xmp)) == 1
    assert _parse(plain[:-2] + exif_app1(6) + plain[-2:]) == 1
    for v in (0, 9, 0x0106, 0xFFFF):
        data = with_segments(plain, exif_app1(v, True))
        assert pillow_orientation(data) == 1 and _parse(data) == 1, v


def test_cut_and_corrupted_exif_give_1_or_the_code(built, plain):
    import ocljpegdecoder_b200 as b2j
    want_rc, want_d = b2j.parse_header(plain, b2j.GATE_EXTENDED | b2j.PARSE_ROBUST)
    for big in (False, True):
        payload = b"Exif\x00\x00" + tiff(6, big, [(0x010F, 7)])
        for n in range(len(payload) + 1):
            cut = payload[:n]
            data = with_segments(plain, segment(0xE1, cut))
            assert _parse(data) in (1, 6), (big, n)
            rc, d = b2j.parse_header(data, b2j.GATE_EXTENDED | b2j.PARSE_ROBUST)
            assert rc == want_rc and d.scan_size == want_d.scan_size and d.width == want_d.width, (big, n)
            # the file itself ends inside the segment, whose length claims the whole payload
            assert _parse(plain[:2] + segment(0xE1, payload)[:4 + n]) in (1, 6), (big, n)
        e = ">" if big else "<"
        for ifd in (0, 1, 2, 7, 9, len(payload) - 6 - 2, len(payload) - 6, 0xFFFFFFFF, 0x7FFFFFFF):
            bad = payload[:10] + struct.pack(e + "I", ifd) + payload[14:]
            assert _parse(with_segments(plain, segment(0xE1, bad))) in (1, 6), (big, ifd)
        for count in (0, 1, 2, 3, 100, 0xFFFF):
            bad = payload[:14] + struct.pack(e + "H", count) + payload[16:]
            got = _parse(with_segments(plain, segment(0xE1, bad)))
            assert got == (6 if count >= 2 else 1) if count <= 3 else got in (1, 6), (big, count)
    # segment lengths below 2, a missing SOI, stray bytes, empty and tiny inputs
    for data in (b"", b"\xff", b"\xff\xd8", b"\xff\xd8\xff\xe1\x00\x01", b"\xff\xd8\xff\xe1\x00", plain[2:], b"\xff\xd8\x00\x00" + plain[2:]):
        assert _parse(data) == 1


def test_null_pointers_are_refused(built):
    import ocljpegdecoder_b200 as b2j
    L = b2j.load_library()
    o = ctypes.c_int32(5)
    assert L.b2j_parse_orientation(None, 10, ctypes.byref(o)) == -1
    assert L.b2j_parse_orientation(b"\xff\xd8", 2, None) == -1
    assert L.b2j_parse_orientation(b"", 0, ctypes.byref(o)) == 0 and o.value == 1


def test_host_opts_abi(built):
    import ocljpegdecoder_b200 as b2j
    assert ctypes.sizeof(b2j.HostOpts) == 32
    assert b2j.HostOpts.exif_orientation.offset == 28 and b2j.HostOpts.scale.offset == 24
    assert "b2j_parse_orientation" in b2j.EXPORTED_SYMBOLS and "b2j_batch_set_orientations" in b2j.EXPORTED_SYMBOLS
    L = ctypes.CDLL(b2j.library_path())
    assert hasattr(L, "b2j_parse_orientation") and hasattr(L, "b2j_batch_set_orientations")


def test_orient_table_matches_pillow(built):
    """orient() above is Pillow's exif_transpose on a plain array, for every code and for odd, 1xN and Nx1 sizes."""
    from PIL import Image, ImageOps
    for h, w in ((37, 53), (1, 7), (7, 1), (2, 3)):
        a = np.arange(h * w * 3, dtype=np.uint32).reshape(h, w, 3).astype(np.uint8) ^ np.uint8(h)
        im = Image.fromarray(a)
        for code in range(1, 9):
            ex = im.getexif()
            ex[0x0112] = code
            im.info["exif"] = ex.tobytes()
            got = np.asarray(ImageOps.exif_transpose(im))
            assert np.array_equal(got, orient(a, code)), (h, w, code)
