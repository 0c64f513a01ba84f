"""The libjpeg pixel model's scaled decode (b2j_batch_set_scale) in numpy: libjpeg-turbo's decode with scale_denom 2, 4
or 8 (Pillow's draft()) from a baseline file's dequantised coefficients -- jidctred.c's reduced IDCTs at the DCT size
jdmaster.c chooses per component, jdsample.c's upsampling (no fancy filter at 1/8), jdcolor.c's colour.

Test tooling, built on tests/libjpeg_model.py (the full-size model, scale 1). tests/test_scaled_model.py checks it against
Pillow and libjpeg-turbo's C code; the GPU tests of the scaled decode compare the kernels with it.
"""
import numpy as np

from libjpeg_model import CONST_BITS, PASS1_BITS, _descale, decode_rgb, idct_islow, layout, upsample, ycc_to_rgb


def _range_limit(y):
    """range_limit[y & RANGE_MASK]: wraps, does not clamp (as in idct_islow)."""
    m = (y + 128) & 1023
    return np.where(m < 256, m, np.where(m < 640, 255, 0)).astype(np.uint8)


def _wrap32(w):
    """The pass-1 results are stored in jidctred.c's int workspace: 32 bits."""
    return ((w + (1 << 31)) & 0xFFFFFFFF) - (1 << 31)


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


def dct_size(h, v, hmax, vmax, min_size):
    """jdmaster.c: a component's DCT size, doubled from min_size = 8 / scale while both factors still divide evenly."""
    ss = min_size
    while ss < 8 and (hmax * min_size) % (h * ss * 2) == 0 and (vmax * min_size) % (v * ss * 2) == 0:
        ss *= 2
    return ss


def decode_rgb_scaled(coef, width, height, sampling, mcu_count_w, mcu_count_h, scale):
    """Dequantised coefficients -> RGB uint8 [ceil(height/scale), ceil(width/scale), 3]; scale 1 is decode_rgb."""
    if scale == 1:
        return decode_rgb(coef, width, height, sampling, mcu_count_w, mcu_count_h)
    samp = layout(sampling)
    hmax, vmax = max(h for h, _ in samp), max(v for _, v in samp)
    mins = 8 // scale
    ow, oh = -(-width // scale), -(-height // scale)
    coef = np.asarray(coef).reshape(mcu_count_h, mcu_count_w, sum(h * v for h, v in samp), 64)
    first, comps = 0, []
    for h, v in samp:
        ss = dct_size(h, v, hmax, vmax, mins)
        px = IDCT_BY_SIZE[ss](coef[:, :, first:first + h * v].reshape(-1, 64)).reshape(mcu_count_h, mcu_count_w, v, h, ss, ss)
        plane = px.transpose(0, 2, 4, 1, 3, 5).reshape(mcu_count_h * v * ss, mcu_count_w * h * ss)
        first += h * v
        dw, dh = -(-width * h * ss // (hmax * 8)), -(-height * v * ss // (vmax * 8))
        rh, rv = hmax * mins // (h * ss), vmax * mins // (v * ss)
        if mins > 1:
            comps.append(upsample(plane, rh, rv, dw, dh, ow, oh))
        else:   # jdsample.c: no fancy filter when the smallest DCT size is 1
            s = plane[:dh, :dw].astype(np.int32)
            comps.append(s[(np.arange(oh) // rv)[:, None], (np.arange(ow) // rh)[None, :]])
    if len(comps) == 1:
        g = comps[0].astype(np.uint8)
        return np.stack([g, g, g], axis=-1)
    return ycc_to_rgb(*comps)


def decode_oracle_scaled(oracle, data, gate, scale):
    """The model's RGB pixels of one file at 1/scale, from the oracle's coefficients (non-strict: the intended decode)."""
    oracle.set_strict(False)
    try:
        rc, img, coef, _ = oracle.decode(data, gate=gate, want_pixels=False)
    finally:
        oracle.set_strict(True)
    assert rc == 0, rc
    return decode_rgb_scaled(coef, img.width, img.height, list(img.sampling), img.mcu_count_w, img.mcu_count_h, scale)
