"""CPU: the exact integer arithmetic the kernels compile (ocljpegdecoder_b200/csrc/b2j_math.h) and
the host LUT builder, exercised through tests/native/libb2jcheck.so (same header, built with g++),
against the oracle. This is not a CPU decode path: it checks formulas before GPU time is spent."""
import ctypes
import hashlib
import os

import numpy as np
import pytest

import jpegcraft
from conftest import ROOT


@pytest.fixture(scope="module")
def chk(built):
    L = ctypes.CDLL(os.path.join(ROOT, "tests", "native", "libb2jcheck.so"))
    L.chk_csc_pixel.restype = ctypes.c_uint32
    L.chk_csc_pixel.argtypes = [ctypes.c_int32] * 3
    L.chk_extend.restype = ctypes.c_int32
    L.chk_extend.argtypes = [ctypes.c_uint32, ctypes.c_int]
    L.chk_csc_exhaustive.restype = ctypes.c_long
    L.chk_lut_decode.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_uint32, ctypes.POINTER(ctypes.c_int)]
    return L


def test_idct_matches_oracle(chk, oracle):
    rng = np.random.RandomState(1)
    for k in range(400):
        if k % 4 == 0:
            blk = rng.randint(-2048, 2048, 64)
        elif k % 4 == 1:
            blk = np.zeros(64, np.int64)
            blk[rng.randint(0, 64, 5)] = rng.randint(-1500, 1500, 5)
        elif k % 4 == 2:
            blk = np.zeros(64, np.int64)
            blk[0] = rng.randint(-2047, 2047)
        else:
            blk = rng.randint(-300, 300, 64) * (rng.rand(64) < 0.3)
        a = np.ascontiguousarray(blk, dtype=np.int32)
        got = a.copy()
        chk.chk_idct(got.ctypes.data)
        assert np.array_equal(got, oracle.idct(a))


def idct_blocks():
    rng = np.random.RandomState(2)
    return [np.ascontiguousarray(rng.randint(-255, 255, 64) * (rng.rand(64) < 0.4), dtype=np.int32) for _ in range(100)]


def test_idct_matches_reference_build(chk, reference_digests):
    want = reference_digests["idct"]
    blocks = idct_blocks()
    assert len(blocks) == len(want)
    for k, (a, w) in enumerate(zip(blocks, want)):
        assert hashlib.sha256(a.tobytes()).hexdigest() == w["block_sha256"], k
        got = a.copy()
        chk.chk_idct(got.ctypes.data)
        assert hashlib.sha256(got.tobytes()).hexdigest() == w["idct_sha256"], k


def test_colour_exhaustive_against_double_formula(chk):
    # all 2^27 (Y,U,V) in [-256,255]^3 against the reference's double arithmetic (decoder.cpp:367-370)
    first = (ctypes.c_int32 * 3)()
    assert chk.chk_csc_exhaustive(first) == 0, list(first)


def colour_triples():
    rng = np.random.RandomState(3)
    trip = [(-256, -256, -256), (255, 255, 255), (0, 0, 0), (188, -200, 200), (201, -200, 200), (187, -200, 200), (202, -200, 200)]
    trip += [tuple(int(v) for v in rng.randint(-256, 256, 3)) for _ in range(2000)]
    return trip


def test_colour_spot_against_oracle_and_reference(chk, oracle, reference_digests):
    """Every triple against the oracle; all of them at once against the digest of the reference's uint32 results."""
    got = []
    for y, u, v in colour_triples():
        got.append(chk.chk_csc_pixel(y, u, v))
        assert got[-1] == oracle.yuv_to_rgb32(y, u, v)
    assert hashlib.sha256(np.array(got, np.uint32).tobytes()).hexdigest() == reference_digests["colour_spot_sha256"]


def test_extend(chk):
    for n in range(1, 17):
        for v in list(range(min(1 << n, 64))) + [(1 << n) - 1, 1 << (n - 1), (1 << (n - 1)) - 1]:
            top = (v << (32 - n)) & 0xFFFFFFFF
            want = v if v >> (n - 1) else v + 1 - (1 << n)   # decoder.cpp:72-82
            assert chk.chk_extend(top, n) == want
    assert chk.chk_extend(0xFFFFFFFF, 0) == 0 and chk.chk_extend(0, 0) == 0


def test_zigzag_table(chk, oracle):
    assert [chk.chk_zigzag(i) for i in range(64)] == oracle.zigzag().tolist()


def _check_table(chk, bits, vals, is_dc):
    codes = jpegcraft.canonical_codes(bits, vals)
    n = ctypes.c_int()
    rng = np.random.RandomState(7)
    for sym, (code, l) in codes.items():
        for _ in range(3):
            tail = int(rng.randint(0, 1 << 30)) & ((1 << (32 - l)) - 1)
            peek = ((code << (32 - l)) | tail) & 0xFFFFFFFF
            e = chk.chk_lut_decode(bytes(bits), bytes(vals), is_dc, peek, ctypes.byref(n))
            assert e > 0
            ln, size, run = e & 0xFF, (e >> 8) & 0xFF, (e >> 16) & 0xFF
            assert ln == l
            if is_dc:
                assert size == sym and run == 0
            else:
                assert (run << 4 | size) == sym
    return n.value


def test_lut_standard_tables(chk):
    sizes = []
    for (tc, th), (bits, vals) in jpegcraft.STD_TABLES.items():
        sizes.append(_check_table(chk, bits, vals, 1 if tc == 0 else 0))
    assert max(sizes) <= 1024 + 512     # primary 2^10 + a few small sub-tables


def test_lut_invalid_prefix_is_rejected(chk):
    bits, vals = jpegcraft.AC_LUMA_BITS, jpegcraft.AC_LUMA_VALS
    n = ctypes.c_int()
    # sixteen 1-bits is no codeword of the Annex K AC luminance table
    assert chk.chk_lut_decode(bytes(bits), bytes(vals), 0, 0xFFFFFFFF, ctypes.byref(n)) == 0


def test_lut_random_tables(chk):
    rng = np.random.RandomState(11)
    for _ in range(30):
        # random complete-ish length distribution via Kraft budget
        nsym = int(rng.randint(2, 200))
        lens = []
        budget = 1 << 16
        for _k in range(nsym):
            l = int(rng.randint(1, 17))
            while l <= 16 and (1 << (16 - l)) > budget - (nsym - len(lens) - 1):
                l += 1
            if l > 16:
                break
            lens.append(l)
            budget -= 1 << (16 - l)
        lens.sort()
        if len(lens) < 2:
            continue
        bits = [lens.count(l) for l in range(1, 17)]
        vals = [int(v) for v in rng.permutation(256)[:len(lens)]]
        # AC interpretation accepts any symbol byte
        _check_table(chk, bits, vals, 0)
