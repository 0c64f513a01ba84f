"""The libjpeg pixel model (B2J_PIXELS_LIBJPEG) in numpy: what libjpeg-turbo's C code computes from a baseline file's
dequantised coefficients with its default decompression settings at scale_denom 1, 2, 4 or 8 (b2j_batch_set_scale,
Pillow's draft()): jidctint.c's ISLOW IDCT or jidctred.c's reduced IDCTs at the DCT size jdmaster.c chooses per
component, jdsample.c's upsampling ("fancy" chroma filters, none at 1/8), jdcolor.c's fixed-point YCbCr -> RGB.

Test tooling. It is fed the oracle's coefficients (int32 [blk_count, 64], natural order, dequantised, MCU-interleaved) and
is the reference the GPU tests compare the kernels with. tests/test_libjpeg_model.py (full size) and
tests/test_scaled_model.py (1/2, 1/4, 1/8) check it against Pillow and libjpeg-turbo's C code.
"""
import numpy as np

CONST_BITS, PASS1_BITS = 13, 2
# FIX(x) = round(x * 2^13) of the constants jidctint.c names
F0298, F0390, F0541, F0765, F0899, F1175 = 2446, 3196, 4433, 6270, 7373, 9633
F1501, F1847, F1961, F2053, F2562, F3072 = 12299, 15137, 16069, 16819, 20995, 25172


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def _range_limit(y):
    """range_limit[y & RANGE_MASK] of an IDCT output: wraps, does not clamp."""
    m = (y + 128) & 1023
    return np.where(m < 256, m, np.where(m < 640, 255, 0)).astype(np.uint8)


def _wrap32(w):
    """The pass-1 results are stored in the IDCTs' int workspace: 32 bits."""
    return ((w + (1 << 31)) & 0xFFFFFFFF) - (1 << 31)


def _pass(d, n):
    """One 1-D pass of jpeg_idct_islow over the 8 int64 arrays d[0..7] (inputs 0..7 of a column or a row). Returns the 8
    outputs DESCALE(., n). The zero-AC shortcuts of the C code are exact special cases of this and are not needed."""
    z2, z3 = d[2], d[6]
    z1 = (z2 + z3) * F0541
    tmp2 = z1 - z3 * F1847
    tmp3 = z1 + z2 * F0765
    tmp0 = (d[0] + d[4]) << CONST_BITS
    tmp1 = (d[0] - d[4]) << CONST_BITS
    tmp10, tmp13, tmp11, tmp12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    t0, t1, t2, t3 = d[7], d[5], d[3], d[1]
    z1, z2, z3, z4 = t0 + t3, t1 + t2, t0 + t2, t1 + t3
    z5 = (z3 + z4) * F1175
    t0, t1, t2, t3 = t0 * F0298, t1 * F2053, t2 * F3072, t3 * F1501
    z1, z2, z3, z4 = -z1 * F0899, -z2 * F2562, -z3 * F1961 + z5, -z4 * F0390 + z5
    t0 = t0 + z1 + z3
    t1 = t1 + z2 + z4
    t2 = t2 + z2 + z3
    t3 = t3 + z1 + z4
    out = [tmp10 + t3, tmp11 + t2, tmp12 + t1, tmp13 + t0, tmp13 - t0, tmp12 - t1, tmp11 - t2, tmp10 - t3]
    return [_descale(o, n) for o in out]


def idct_islow(blocks):
    """Dequantised coefficients int [n, 64] (natural order) -> samples uint8 [n, 8, 8]. 64-bit arithmetic like libjpeg's
    JLONG; the pass-1 results are stored as C int (32 bits), so they wrap the way the C code's workspace does."""
    x = np.asarray(blocks, np.int64).reshape(-1, 8, 8)
    ws = np.stack([_wrap32(w) for w in _pass([x[:, k, :] for k in range(8)], CONST_BITS - PASS1_BITS)], axis=1)   # [n, r, c]
    return _range_limit(np.stack(_pass([ws[:, :, k] for k in range(8)], CONST_BITS + PASS1_BITS + 3), axis=2))


def _pass4(d, n):
    """One 1-D pass of jpeg_idct_4x4 over d[0..7] (d[4] unused): 4 outputs DESCALE(., n)."""
    tmp0 = d[0] << (CONST_BITS + 1)
    tmp2 = d[2] * 15137 + d[6] * -6270
    t10, t12 = tmp0 + tmp2, tmp0 - tmp2
    z1, z2, z3, z4 = d[7], d[5], d[3], d[1]
    a = z1 * -1730 + z2 * 11893 + z3 * -17799 + z4 * 8697
    b = z1 * -4176 + z2 * -4926 + z3 * 7373 + z4 * 20995
    return [_descale(o, n) for o in (t10 + b, t12 + a, t12 - a, t10 - b)]


def idct_4x4(blocks):
    """jpeg_idct_4x4: int [n, 64] -> uint8 [n, 4, 4], 64-bit products, 32-bit workspace like idct_islow."""
    x = np.asarray(blocks, np.int64).reshape(-1, 8, 8)
    ws = np.stack([_wrap32(w) for w in _pass4([x[:, k, :] for k in range(8)], CONST_BITS - PASS1_BITS + 1)], axis=1)
    return _range_limit(np.stack(_pass4([ws[:, :, k] for k in range(8)], CONST_BITS + PASS1_BITS + 3 + 1), axis=2))


def _pass2(d, n):
    """One 1-D pass of jpeg_idct_2x2 over d[0], d[1], d[3], d[5], d[7]: 2 outputs DESCALE(., n)."""
    t10 = d[0] << (CONST_BITS + 2)
    t0 = d[7] * -5906 + d[5] * 6967 + d[3] * -10426 + d[1] * 29692
    return [_descale(t10 + t0, n), _descale(t10 - t0, n)]


def idct_2x2(blocks):
    """jpeg_idct_2x2: int [n, 64] -> uint8 [n, 2, 2]."""
    x = np.asarray(blocks, np.int64).reshape(-1, 8, 8)
    ws = np.stack([_wrap32(w) for w in _pass2([x[:, k, :] for k in range(8)], CONST_BITS - PASS1_BITS + 2)], axis=1)
    return _range_limit(np.stack(_pass2([ws[:, :, k] for k in range(8)], CONST_BITS + PASS1_BITS + 3 + 2), axis=2))


def idct_1x1(blocks):
    """jpeg_idct_1x1: (DC * q + 4) >> 3 -> uint8 [n, 1, 1]."""
    x = np.asarray(blocks, np.int64).reshape(-1, 64)
    return _range_limit((x[:, 0] + 4) >> 3).reshape(-1, 1, 1)


IDCT_BY_SIZE = {8: idct_islow, 4: idct_4x4, 2: idct_2x2, 1: idct_1x1}


def layout(sampling):
    """Sampling bytes (h << 4 | v, as in SOF0; 0 for absent components) -> [(h, v)] of the components present."""
    return [(s >> 4, s & 15) for s in sampling if s]


def dct_size(h, v, hmax, vmax, min_size):
    """jdmaster.c: a component's DCT size, doubled from min_size = 8 / scale while both factors still divide evenly."""
    ss = min_size
    while ss < 8 and (hmax * min_size) % (h * ss * 2) == 0 and (vmax * min_size) % (v * ss * 2) == 0:
        ss *= 2
    return ss


def _clamp_idx(i, n):
    return np.clip(i, 0, n - 1)


def upsample(plane, rh, rv, dw, dh, width, height, fancy=True):
    """One component's samples (the dw x dh top-left part of its plane) -> width x height, jdsample.c's choice of method.
    jdsample.c has no fancy filter when the smallest DCT size is 1 (fancy=False): every ratio replicates."""
    s = plane[:dh, :dw].astype(np.int32)
    xs = np.arange(width)
    ys = np.arange(height)
    if not fancy or (rh, rv) == (1, 1):
        return s[(ys // rv)[:, None], (xs // rh)[None, :]]
    if (rh, rv) == (2, 1) and dw > 2:
        sx = xs >> 1
        near = s[:, sx] * 3
        far = s[:, _clamp_idx(np.where(xs & 1, sx + 1, sx - 1), dw)]
        return ((near + far + np.where(xs & 1, 2, 1)) >> 2)[:height]
    if (rh, rv) == (1, 2):
        r = ys >> 1
        n = _clamp_idx(np.where(ys & 1, r + 1, r - 1), dh)
        return ((s[r] * 3 + s[n] + np.where(ys & 1, 2, 1)[:, None]) >> 2)[:, :width]
    if (rh, rv) == (2, 2) and dw > 2:
        r = ys >> 1
        n = _clamp_idx(np.where(ys & 1, r + 1, r - 1), dh)
        cs = s[r] * 3 + s[n]                                   # [height, dw]
        sx = xs >> 1
        far = cs[:, _clamp_idx(np.where(xs & 1, sx + 1, sx - 1), dw)]
        return (cs[:, sx] * 3 + far + np.where(xs & 1, 7, 8)) >> 4
    return s[(ys // rv)[:, None], (xs // rh)[None, :]]


def ycc_to_rgb(y, cb, cr):
    """jdcolor.c ycc_rgb_convert: SCALEBITS 16 fixed point, arithmetic shifts, clamped to [0, 255]."""
    y = y.astype(np.int64)
    cb = cb.astype(np.int64) - 128
    cr = cr.astype(np.int64) - 128
    r = y + ((91881 * cr + 32768) >> 16)
    b = y + ((116130 * cb + 32768) >> 16)
    g = y + ((-22554 * cb - 46802 * cr + 32768) >> 16)
    return np.clip(np.stack([r, g, b], axis=-1), 0, 255).astype(np.uint8)


def decode_rgb(coef, width, height, sampling, mcu_count_w, mcu_count_h, scale=1):
    """Dequantised coefficients -> RGB uint8 [ceil(height/scale), ceil(width/scale), 3] in the libjpeg model (gray:
    R = G = B = Y)."""
    samp = layout(sampling)
    hmax, vmax = max(h for h, _ in samp), max(v for _, v in samp)
    mins = 8 // scale
    ow, oh = -(-width // scale), -(-height // scale)
    coef = np.asarray(coef).reshape(mcu_count_h, mcu_count_w, sum(h * v for h, v in samp), 64)
    first, comps = 0, []
    for h, v in samp:
        ss = dct_size(h, v, hmax, vmax, mins)
        px = IDCT_BY_SIZE[ss](coef[:, :, first:first + h * v].reshape(-1, 64)).reshape(mcu_count_h, mcu_count_w, v, h, ss, ss)
        plane = px.transpose(0, 2, 4, 1, 3, 5).reshape(mcu_count_h * v * ss, mcu_count_w * h * ss)   # MCU-padded
        first += h * v
        dw, dh = -(-width * h * ss // (hmax * 8)), -(-height * v * ss // (vmax * 8))
        rh, rv = hmax * mins // (h * ss), vmax * mins // (v * ss)
        comps.append(upsample(plane, rh, rv, dw, dh, ow, oh, fancy=mins > 1))
    if len(comps) == 1:
        g = comps[0].astype(np.uint8)
        return np.stack([g, g, g], axis=-1)
    return ycc_to_rgb(*comps)


def decode_oracle(oracle, data, gate, scale=1):
    """The model's RGB pixels of one file at 1/scale, from the oracle's coefficients (non-strict: the intended decode)."""
    oracle.set_strict(False)
    try:
        rc, img, coef, _ = oracle.decode(data, gate=gate, want_pixels=False)
    finally:
        oracle.set_strict(True)
    assert rc == 0, rc
    return decode_rgb(coef, img.width, img.height, list(img.sampling), img.mcu_count_w, img.mcu_count_h, scale)


def box_filter(px, factor):
    """b2j_batch_downscale's arithmetic on an [H, W, C] array: the rounded mean (sum + n/2) / n over factor x factor
    cells, of the n values that exist in the partial cells at the right and bottom edges."""
    px = np.asarray(px, np.int64)
    h, w = px.shape[0], px.shape[1]
    oh, ow = -(-h // factor), -(-w // factor)
    pad = np.zeros((oh * factor, ow * factor) + px.shape[2:], np.int64)
    cnt = np.zeros((oh * factor, ow * factor), np.int64)
    pad[:h, :w] = px
    cnt[:h, :w] = 1
    s = pad.reshape(oh, factor, ow, factor, *px.shape[2:]).sum(axis=(1, 3))
    n = cnt.reshape(oh, factor, ow, factor).sum(axis=(1, 3))
    n = n.reshape(n.shape + (1,) * (s.ndim - 2))
    return ((s + n // 2) // n).astype(np.uint8)
