"""The libjpeg pixel model (B2J_PIXELS_LIBJPEG) in numpy: what libjpeg-turbo's C code computes from a baseline file's
dequantised coefficients with its default decompression settings (jidctint.c ISLOW IDCT, jdsample.c "fancy" chroma
upsampling, jdcolor.c fixed-point YCbCr -> RGB).

Test tooling. It is fed the oracle's coefficients (int32 [blk_count, 64], natural order, dequantised, MCU-interleaved) and
is the reference the GPU tests compare the kernels with. tests/test_libjpeg_model.py checks it against Pillow.
"""
import numpy as np

CONST_BITS, PASS1_BITS = 13, 2
# FIX(x) = round(x * 2^13) of the constants jidctint.c names
F0298, F0390, F0541, F0765, F0899, F1175 = 2446, 3196, 4433, 6270, 7373, 9633
F1501, F1847, F1961, F2053, F2562, F3072 = 12299, 15137, 16069, 16819, 20995, 25172


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


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
    ws = _pass([x[:, k, :] for k in range(8)], CONST_BITS - PASS1_BITS)          # columns: out[k] = row k
    ws = [((w + (1 << 31)) & 0xFFFFFFFF) - (1 << 31) for w in ws]
    ws = np.stack(ws, axis=1)                                                     # [n, row, col]
    y = np.stack(_pass([ws[:, :, k] for k in range(8)], CONST_BITS + PASS1_BITS + 3), axis=2)
    m = (y + 128) & 1023                                                          # range_limit[y & RANGE_MASK]
    return np.where(m < 256, m, np.where(m < 640, 255, 0)).astype(np.uint8)


def layout(sampling):
    """Sampling bytes (h << 4 | v, as in SOF0; 0 for absent components) -> [(h, v)] of the components present."""
    return [(s >> 4, s & 15) for s in sampling if s]


def component_planes(coef, sampling, mcu_count_w, mcu_count_h):
    """IDCT of every block, assembled into one MCU-padded sample plane per component (uint8 [rows, cols])."""
    samp = layout(sampling)
    nblk = [h * v for h, v in samp]
    tot = sum(nblk)
    px = idct_islow(coef).reshape(mcu_count_h, mcu_count_w, tot, 8, 8)
    planes, first = [], 0
    for (h, v), n in zip(samp, nblk):
        b = px[:, :, first:first + n].reshape(mcu_count_h, mcu_count_w, v, h, 8, 8)
        planes.append(b.transpose(0, 2, 4, 1, 3, 5).reshape(mcu_count_h * v * 8, mcu_count_w * h * 8))
        first += n
    return planes


def _clamp_idx(i, n):
    return np.clip(i, 0, n - 1)


def upsample(plane, rh, rv, dw, dh, width, height):
    """One component's samples (the dw x dh top-left part of its plane) -> width x height, jdsample.c's choice of method."""
    s = plane[:dh, :dw].astype(np.int32)
    xs = np.arange(width)
    ys = np.arange(height)
    if (rh, rv) == (1, 1):
        return s[:height, :width]
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


def decode_rgb(coef, width, height, sampling, mcu_count_w, mcu_count_h):
    """Dequantised coefficients -> RGB uint8 [height, width, 3] in the libjpeg model (gray: R = G = B = Y)."""
    samp = layout(sampling)
    planes = component_planes(coef, sampling, mcu_count_w, mcu_count_h)
    hmax, vmax = max(h for h, _ in samp), max(v for _, v in samp)
    comps = []
    for (h, v), p in zip(samp, planes):
        dw, dh = -(-width * h // hmax), -(-height * v // vmax)
        comps.append(upsample(p, hmax // h, vmax // v, dw, dh, width, height))
    if len(comps) == 1:
        g = comps[0].astype(np.uint8)
        return np.stack([g, g, g], axis=-1)
    return ycc_to_rgb(*comps)


def decode_oracle(oracle, data, gate):
    """The model's RGB pixels of one file, from the oracle's coefficients (non-strict: the intended decode)."""
    oracle.set_strict(False)
    try:
        rc, img, coef, _ = oracle.decode(data, gate=gate, want_pixels=False)
    finally:
        oracle.set_strict(True)
    assert rc == 0, rc
    return decode_rgb(coef, img.width, img.height, list(img.sampling), img.mcu_count_w, img.mcu_count_h)


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
