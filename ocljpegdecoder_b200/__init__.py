"""ocljpegdecoder_b200 -- B200-native baseline-JPEG decode path (ctypes view of the C ABI).

The product is the shared library ``lib/libb2j.so`` (hand-written CUDA for sm_100a behind the
extern "C" interface of ``include/b2j.h``). This module only binds it for the Python tests and
for bench.py; it contains no decode logic and no fallback: if the library is missing, importing
fails, and if no B200 is visible, ``Decoder()`` raises.
"""
from .api import (  # noqa: F401
    B2JError, BatchInfo, Decoder, Batch, Idct, ImageDesc, StageTimes, HostOpts, HostArgs, PinnedBuffer, parse_header, parse_orientation, crop_frame, read_files, host_free, decode_host_multi, library_path, load_library,
    GATE_REFERENCE, GATE_EXTENDED, PARSE_ROBUST, GATE_GRAY, OUT_BGRA, OUT_RGB24, OUT_RGB_PLANAR, OUT_GRAY8, PIXELS_REFERENCE, PIXELS_LIBJPEG,
    EXPORTED_SYMBOLS,
)
