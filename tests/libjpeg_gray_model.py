"""The libjpeg pixel model's grayscale output (B2J_OUT_GRAY8) in numpy: libjpeg's out_color_space = JCS_GRAYSCALE, which
outputs the luma component's samples as they are, with no chroma upsampling and no colour conversion; at scale_denom 2,
4 and 8 the reduced luma IDCT's samples. It is the luma plane decode_rgb of tests/libjpeg_model.py computes before colour
conversion, built from the same IDCTs and the same DCT-size rule.

Test tooling, fed the oracle's coefficients like tests/libjpeg_model.py. tests/test_gray_model.py checks it against
Pillow's draft("L"), OpenCV, torchvision and libjpeg-turbo's C code; the GPU tests of GRAY8 compare the kernel with it.
"""
import numpy as np

from libjpeg_model import IDCT_BY_SIZE, dct_size, layout


def decode_gray(coef, width, height, sampling, mcu_count_w, mcu_count_h, scale=1):
    """Dequantised coefficients -> uint8 [ceil(height/scale), ceil(width/scale)]: the luma component's samples. The luma
    has the largest sampling factors, so its DCT size is 8 / scale and its samples are the output size."""
    samp = layout(sampling)
    h, v = samp[0]
    hmax, vmax = max(a for a, _ in samp), max(b for _, b in samp)
    ss = dct_size(h, v, hmax, vmax, 8 // scale)
    assert (h, v, ss) == (hmax, vmax, 8 // scale), (samp, scale)
    coef = np.asarray(coef).reshape(mcu_count_h, mcu_count_w, sum(a * b for a, b in samp), 64)
    px = IDCT_BY_SIZE[ss](coef[:, :, :h * v].reshape(-1, 64)).reshape(mcu_count_h, mcu_count_w, v, h, ss, ss)
    plane = px.transpose(0, 2, 4, 1, 3, 5).reshape(mcu_count_h * v * ss, mcu_count_w * h * ss)   # MCU-padded
    return np.ascontiguousarray(plane[:-(-height // scale), :-(-width // scale)])


def oracle_coefs(oracle, data, gate):
    """The oracle's header and coefficients of one file (non-strict: the intended decode)."""
    oracle.set_strict(False)
    try:
        rc, img, coef, _ = oracle.decode(data, gate=gate, want_pixels=False)
    finally:
        oracle.set_strict(True)
    assert rc == 0, rc
    return img, coef


def decode_oracle_gray(oracle, data, gate, scale=1):
    """The model's grayscale pixels of one file at 1/scale, from the oracle's coefficients."""
    img, coef = oracle_coefs(oracle, data, gate)
    return decode_gray(coef, img.width, img.height, list(img.sampling), img.mcu_count_w, img.mcu_count_h, scale)
