"""ctypes bindings of include/b2j.h (one Python method per C entry point)."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

GATE_REFERENCE = 0
GATE_EXTENDED = 1
PARSE_ROBUST = 2     # OR-able: skip COM / late APPn / unknown segments, big-endian 16-bit DQT
GATE_GRAY = 4        # OR-able: one-component (grayscale) frames
OUT_BGRA, OUT_RGB24, OUT_RGB_PLANAR, OUT_GRAY8 = 0, 1, 2, 3
PIXELS_REFERENCE = 0   # the reference's pixels (default)
PIXELS_LIBJPEG = 1     # libjpeg-turbo's default decode: ISLOW IDCT, fancy chroma upsampling, fixed-point colour (Pillow's pixels)

B2J_OK = 0
B2J_E_NODEVICE = -7

# every symbol include/b2j.h declares (tests check that the built library exports all of them)
EXPORTED_SYMBOLS = [
    "b2j_abi_version", "b2j_strerror", "b2j_last_error", "b2j_parse_header", "b2j_device_count",
    "b2j_create", "b2j_destroy", "b2j_batch_create", "b2j_batch_destroy", "b2j_batch_get_info",
    "b2j_batch_upload", "b2j_batch_set_output_format", "b2j_batch_set_pixel_model", "b2j_batch_set_scale", "b2j_batch_decode", "b2j_batch_decode_timed", "b2j_batch_decode_steps", "b2j_batch_sync", "b2j_batch_status", "b2j_batch_sync_stats",
    "b2j_batch_pixels_device", "b2j_batch_coefs_device", "b2j_batch_read_pixels", "b2j_batch_read_all_pixels",
    "b2j_batch_read_coefs", "b2j_decode_host", "b2j_decode_host_ex", "b2j_decode_host_multi", "b2j_host_alloc", "b2j_host_free",
    "b2j_read_files", "b2j_idct_create", "b2j_idct_blk_count", "b2j_idct_upload", "b2j_idct_run", "b2j_idct_read_pixels", "b2j_idct_read_coefs",
    "b2j_idct_destroy", "b2j_batch_downscale", "b2j_batch_downscaled_device", "b2j_batch_read_downscaled",
]


class B2JError(RuntimeError):
    def __init__(self, code, where, detail=""):
        self.code = code
        super().__init__("%s failed: %d%s" % (where, code, (" (" + detail + ")") if detail else ""))


class ImageDesc(ctypes.Structure):
    """b2j_image_desc"""
    _fields_ = [
        ("width", ctypes.c_int32), ("height", ctypes.c_int32),
        ("sampling", ctypes.c_uint8 * 3), ("quant_id", ctypes.c_uint8 * 3), ("huff_id", ctypes.c_uint8 * 3),
        ("color_space", ctypes.c_uint8),
        ("quant_present", ctypes.c_uint8 * 4), ("huff_present", ctypes.c_uint8 * 8),
        ("restart_interval", ctypes.c_int32),
        ("mcu_width", ctypes.c_int32), ("mcu_height", ctypes.c_int32),
        ("mcu_count_w", ctypes.c_int32), ("mcu_count_h", ctypes.c_int32), ("mcu_count", ctypes.c_int32),
        ("blks_per_mcu", ctypes.c_int32 * 3), ("tot_blks_per_mcu", ctypes.c_int32), ("blk_count", ctypes.c_int32),
        ("scan_offset", ctypes.c_uint64), ("scan_size", ctypes.c_uint64),
        ("quant", (ctypes.c_uint16 * 64) * 4),
        ("huff_counts", (ctypes.c_uint8 * 16) * 8),
        ("huff_symbols", (ctypes.c_uint8 * 256) * 8),
    ]


class BatchInfo(ctypes.Structure):
    """b2j_batch_info"""
    _fields_ = [
        ("n_images", ctypes.c_int32), ("kernel_launches", ctypes.c_int32),
        ("total_pixels", ctypes.c_int64), ("total_blocks", ctypes.c_int64), ("scan_bytes", ctypes.c_int64),
        ("coef_plane_bytes", ctypes.c_int64), ("pixel_bytes", ctypes.c_int64), ("algorithmic_bytes", ctypes.c_int64),
        ("device_bytes", ctypes.c_int64), ("h2d_bytes", ctypes.c_int64),
    ]


class HostOpts(ctypes.Structure):
    """b2j_host_opts"""
    _fields_ = [("gate", ctypes.c_int32), ("out_format", ctypes.c_int32), ("n_threads", ctypes.c_int32), ("group", ctypes.c_int32),
                ("group_mb", ctypes.c_int32), ("pixel_model", ctypes.c_int32), ("scale", ctypes.c_int32), ("reserved", ctypes.c_int32 * 1)]


class StageTimes(ctypes.Structure):
    """b2j_stage_times"""
    _fields_ = [("prepass_ms", ctypes.c_float), ("huffman_ms", ctypes.c_float), ("idct_ms", ctypes.c_float),
                ("total_ms", ctypes.c_float)]


def library_path():
    return os.environ.get("B2J_LIBRARY") or os.path.join(_HERE, "lib", "libb2j.so")


_LIB = None


def load_library():
    """Loads lib/libb2j.so. There is no fallback: a missing library is an error."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.isfile(path):
        raise ImportError("%s not built; run `make` or __graft_entry__.build() (there is no CPU fallback)" % path)
    L = ctypes.CDLL(path)
    vp, ci = ctypes.c_void_p, ctypes.c_int
    L.b2j_abi_version.restype = ci
    L.b2j_strerror.restype = ctypes.c_char_p
    L.b2j_strerror.argtypes = [ci]
    L.b2j_last_error.restype = ctypes.c_char_p
    L.b2j_parse_header.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ci, ctypes.POINTER(ImageDesc)]
    L.b2j_device_count.restype = ci
    L.b2j_create.argtypes = [ci, ctypes.POINTER(vp)]
    L.b2j_destroy.argtypes = [vp]
    L.b2j_destroy.restype = None
    L.b2j_batch_create.argtypes = [vp, ci, ctypes.POINTER(ImageDesc), ctypes.POINTER(ctypes.c_char_p),
                                   ctypes.POINTER(ctypes.c_size_t), ctypes.POINTER(vp)]
    L.b2j_batch_destroy.argtypes = [vp]
    L.b2j_batch_destroy.restype = None
    L.b2j_batch_get_info.argtypes = [vp, ctypes.POINTER(BatchInfo)]
    L.b2j_batch_upload.argtypes = [vp, vp]
    L.b2j_batch_set_output_format.argtypes = [vp, ci]
    L.b2j_batch_set_pixel_model.argtypes = [vp, ci]
    L.b2j_batch_set_scale.argtypes = [vp, ci]
    L.b2j_batch_decode.argtypes = [vp, vp]
    L.b2j_batch_decode_timed.argtypes = [vp, vp, ctypes.POINTER(StageTimes)]
    L.b2j_batch_decode_steps.argtypes = [vp, vp, ci, ctypes.POINTER(StageTimes), ctypes.POINTER(ctypes.c_float)]
    L.b2j_batch_sync.argtypes = [vp, vp]
    L.b2j_batch_status.argtypes = [vp, vp, vp]
    L.b2j_batch_sync_stats.argtypes = [vp, vp, vp]
    L.b2j_batch_pixels_device.argtypes = [vp, ci, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_size_t)]
    L.b2j_batch_coefs_device.argtypes = [vp, ci, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_size_t)]
    L.b2j_batch_read_pixels.argtypes = [vp, vp, ci, vp]
    L.b2j_batch_read_all_pixels.argtypes = [vp, vp, ctypes.POINTER(vp)]
    L.b2j_batch_read_coefs.argtypes = [vp, vp, ci, vp]
    L.b2j_decode_host.argtypes = [vp, ci, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_size_t), ci,
                                  ctypes.POINTER(vp), vp]
    L.b2j_decode_host_ex.argtypes = [vp, ci, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_size_t), ctypes.POINTER(HostOpts),
                                     ctypes.POINTER(vp), vp]
    L.b2j_decode_host_multi.argtypes = [ctypes.POINTER(vp), ci, ci, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_size_t),
                                        ctypes.POINTER(HostOpts), ctypes.POINTER(vp), vp]
    L.b2j_host_alloc.argtypes = [ctypes.POINTER(vp), ctypes.c_size_t]
    L.b2j_host_free.argtypes = [vp]
    L.b2j_host_free.restype = None
    L.b2j_read_files.argtypes = [ci, ctypes.POINTER(ctypes.c_char_p), ci, ctypes.POINTER(vp), ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_size_t)]
    L.b2j_batch_downscale.argtypes = [vp, vp, ci]
    L.b2j_batch_downscaled_device.argtypes = [vp, ci, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_size_t), ctypes.POINTER(ci), ctypes.POINTER(ci)]
    L.b2j_batch_read_downscaled.argtypes = [vp, vp, ci, vp]
    L.b2j_idct_create.argtypes = [vp, ci, ci, ci, ci, ctypes.POINTER(vp)]
    L.b2j_idct_blk_count.argtypes = [vp]
    L.b2j_idct_upload.argtypes = [vp, vp, ci, ci]
    L.b2j_idct_run.argtypes = [vp]
    L.b2j_idct_read_pixels.argtypes = [vp, vp]
    L.b2j_idct_read_coefs.argtypes = [vp, vp]
    L.b2j_idct_destroy.argtypes = [vp]
    L.b2j_idct_destroy.restype = None
    _LIB = L
    return L


def _check(rc, where):
    if rc != B2J_OK:
        L = load_library()
        raise B2JError(rc, where, (L.b2j_strerror(rc) or b"").decode() + "; " + (L.b2j_last_error() or b"").decode())


def parse_header(data, gate=GATE_EXTENDED):
    """b2j_parse_header: returns (rc, ImageDesc). rc != 0 means the file is refused."""
    L = load_library()
    d = ImageDesc()
    rc = L.b2j_parse_header(data, len(data), gate, ctypes.byref(d))
    return rc, d


def _out_shape(d, fmt, scale=1):
    """Shape of an image's pixels in output format fmt, at 1/scale of its size (ceil(W/scale) x ceil(H/scale))."""
    w, h = -(-d.width // scale), -(-d.height // scale)
    if fmt == OUT_GRAY8:
        return (h, w)
    return (h, w, 4) if fmt == OUT_BGRA else ((h, w, 3) if fmt == OUT_RGB24 else (3, h, w))


def _host_call_args(files, outs, gate, fmt, scale=1):
    """Argument arrays of the b2j_decode_host* calls; allocates the outputs when none are given."""
    n = len(files)
    if outs is None:
        outs = []
        for f in files:
            rc, d = parse_header(f, gate)
            outs.append(np.zeros(_out_shape(d, fmt, scale or 1), np.uint8) if rc == 0 else np.zeros((0, 0, 4), np.uint8))
    ptrs = [f if isinstance(f, int) else ctypes.cast(ctypes.c_char_p(f), ctypes.c_void_p).value for f in files]
    fp = ctypes.cast((ctypes.c_void_p * n)(*ptrs), ctypes.POINTER(ctypes.c_char_p))
    return outs, fp, (ctypes.c_void_p * n)(*[o if isinstance(o, int) else o.ctypes.data for o in outs])


class HostArgs:
    """The argument arrays of a b2j_decode_host* call, marshalled once (8192 small files cost tens of milliseconds of
    ctypes work per call otherwise): files / lens / outs as for Decoder.decode_host_ex."""

    def __init__(self, files, lens=None, outs=None, gate=GATE_EXTENDED, out_format=OUT_BGRA, n_threads=0, group=0, group_mb=0,
                 pixel_model=PIXELS_REFERENCE, scale=1):
        self.n = len(files)
        self.files = files                      # keeps the bytes objects alive
        lens = lens if lens is not None else [len(f) for f in files]
        self.outs, self.fp, self.op = _host_call_args(files, outs, gate, out_format, scale)
        self.ln = (ctypes.c_size_t * self.n)(*lens)
        self.opts = HostOpts(gate=gate, out_format=out_format, n_threads=n_threads, group=group, group_mb=group_mb, pixel_model=pixel_model,
                             scale=scale)
        self.status = np.zeros(self.n, np.int32)


class PinnedBuffer:
    """b2j_host_alloc / b2j_host_free: page-locked host memory, viewed as a numpy uint8 array."""

    def __init__(self, nbytes):
        self.lib = load_library()
        self._p = ctypes.c_void_p()
        _check(self.lib.b2j_host_alloc(ctypes.byref(self._p), nbytes), "b2j_host_alloc")
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array(ctypes.cast(self._p, ctypes.POINTER(ctypes.c_uint8)), shape=(max(nbytes, 1),))[:nbytes]

    @property
    def address(self):
        return self._p.value

    def close(self):
        if self._p:
            self.array = None
            self.lib.b2j_host_free(self._p)
            self._p = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def read_files(paths, n_threads=0):
    """b2j_read_files: whole files into one pinned arena. Returns (arena address -- pass to host_free() --, [address], [length])."""
    L = load_library()
    n = len(paths)
    pp = (ctypes.c_char_p * n)(*[os.fsencode(p) for p in paths])
    arena = ctypes.c_void_p()
    fl = (ctypes.c_void_p * n)()
    ln = (ctypes.c_size_t * n)()
    rc = L.b2j_read_files(n, pp, n_threads, ctypes.byref(arena), fl, ln)
    return rc, arena.value, [fl[i] for i in range(n)], [ln[i] for i in range(n)]


def host_free(address):
    load_library().b2j_host_free(ctypes.c_void_p(address))


def decode_host_multi(decoders, files, lens=None, outs=None, gate=GATE_EXTENDED, out_format=OUT_BGRA, n_threads=0, group=0,
                      pixel_model=PIXELS_REFERENCE, scale=1):
    """b2j_decode_host_multi over the given Decoder objects (one per GPU). files: bytes objects or addresses (then `lens`)."""
    L = load_library()
    n = len(files)
    lens = lens if lens is not None else [len(f) for f in files]
    outs, fp, op = _host_call_args(files, outs, gate, out_format, scale)
    ln = (ctypes.c_size_t * n)(*lens)
    opts = HostOpts(gate=gate, out_format=out_format, n_threads=n_threads, group=group, pixel_model=pixel_model, scale=scale)
    cx = (ctypes.c_void_p * len(decoders))(*[d._h.value for d in decoders])
    status = np.zeros(n, np.int32)
    _check(L.b2j_decode_host_multi(cx, len(decoders), n, fp, ln, ctypes.byref(opts), op, status.ctypes.data), "b2j_decode_host_multi")
    return outs, status


class Decoder:
    """b2j_ctx: one per GPU."""

    def __init__(self, device=0):
        self.lib = load_library()
        self._h = ctypes.c_void_p()
        _check(self.lib.b2j_create(device, ctypes.byref(self._h)), "b2j_create")
        self.device = device

    def close(self):
        if self._h:
            self.lib.b2j_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def batch(self, files, gate=GATE_EXTENDED):
        """Parse + b2j_batch_create for a list of bytes objects (all must pass the gate)."""
        descs = (ImageDesc * len(files))()
        for i, f in enumerate(files):
            rc = self.lib.b2j_parse_header(f, len(f), gate, ctypes.byref(descs[i]))
            _check(rc, "b2j_parse_header[%d]" % i)
        return Batch(self, files, descs)

    def decode_host(self, files, outs=None, gate=GATE_EXTENDED):
        """b2j_decode_host: host bytes in, host BGRA arrays out. Returns (outs, status)."""
        n = len(files)
        if outs is None:
            outs = []
            for f in files:
                rc, d = parse_header(f, gate)
                outs.append(np.zeros((d.height, d.width, 4), np.uint8) if rc == 0 else np.zeros((0, 0, 4), np.uint8))
        fp = (ctypes.c_char_p * n)(*files)
        ln = (ctypes.c_size_t * n)(*[len(f) for f in files])
        op = (ctypes.c_void_p * n)(*[o.ctypes.data for o in outs])
        status = np.zeros(n, np.int32)
        _check(self.lib.b2j_decode_host(self._h, n, fp, ln, gate, op, status.ctypes.data), "b2j_decode_host")
        return outs, status


    def decode_host_args(self, args):
        """b2j_decode_host_ex with arguments marshalled beforehand (HostArgs). Returns (outs, status)."""
        _check(self.lib.b2j_decode_host_ex(self._h, args.n, args.fp, args.ln, ctypes.byref(args.opts), args.op, args.status.ctypes.data),
               "b2j_decode_host_ex")
        return args.outs, args.status

    def decode_host_ex(self, files, lens=None, outs=None, gate=GATE_EXTENDED, out_format=OUT_BGRA, n_threads=0, group=0,
                       pixel_model=PIXELS_REFERENCE, scale=1):
        """b2j_decode_host_ex: like decode_host with an output layout (OUT_GRAY8 with PIXELS_LIBJPEG only), a pixel model,
        a scale (1, 2, 4 or 8: the libjpeg model's scaled decode) and host threads. files: bytes objects or addresses (then
        `lens`); outs: numpy arrays or addresses."""
        n = len(files)
        lens = lens if lens is not None else [len(f) for f in files]
        outs, fp, op = _host_call_args(files, outs, gate, out_format, scale)
        ln = (ctypes.c_size_t * n)(*lens)
        opts = HostOpts(gate=gate, out_format=out_format, n_threads=n_threads, group=group, pixel_model=pixel_model, scale=scale)
        status = np.zeros(n, np.int32)
        _check(self.lib.b2j_decode_host_ex(self._h, n, fp, ln, ctypes.byref(opts), op, status.ctypes.data), "b2j_decode_host_ex")
        return outs, status


class Idct:
    """b2j_idct: the secondary boundary -- dequantised int32 coefficients in, BGRA pixels out (the clidct_* functions)."""

    def __init__(self, dec, width, height, luma_h, luma_v):
        self.dec, self.lib = dec, dec.lib
        self.width, self.height = width, height
        self._h = ctypes.c_void_p()
        _check(self.lib.b2j_idct_create(dec._h, width, height, luma_h, luma_v, ctypes.byref(self._h)), "b2j_idct_create")
        self.blk_count = self.lib.b2j_idct_blk_count(self._h)

    def upload(self, coefs, offset=0):
        coefs = np.ascontiguousarray(coefs, np.int32)
        _check(self.lib.b2j_idct_upload(self._h, coefs.ctypes.data, offset, coefs.shape[0]), "b2j_idct_upload")

    def run(self):
        _check(self.lib.b2j_idct_run(self._h), "b2j_idct_run")

    def pixels(self):
        out = np.zeros((self.height, self.width, 4), np.uint8)
        _check(self.lib.b2j_idct_read_pixels(self._h, out.ctypes.data), "b2j_idct_read_pixels")
        return out

    def coefs(self):
        out = np.zeros((self.blk_count, 64), np.int32)
        _check(self.lib.b2j_idct_read_coefs(self._h, out.ctypes.data), "b2j_idct_read_coefs")
        return out

    def close(self):
        if self._h:
            self.lib.b2j_idct_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Batch:
    """b2j_batch: a set of images resident on one GPU."""

    def __init__(self, dec, files, descs):
        self.dec = dec
        self.lib = dec.lib
        self.files = list(files)   # keep the bytes alive
        self.descs = descs
        self.n = len(files)
        fp = (ctypes.c_char_p * self.n)(*self.files)
        ln = (ctypes.c_size_t * self.n)(*[len(f) for f in self.files])
        self._h = ctypes.c_void_p()
        _check(self.lib.b2j_batch_create(dec._h, self.n, descs, fp, ln, ctypes.byref(self._h)), "b2j_batch_create")

    def close(self):
        if self._h:
            self.lib.b2j_batch_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        inf = BatchInfo()
        _check(self.lib.b2j_batch_get_info(self._h, ctypes.byref(inf)), "b2j_batch_get_info")
        return inf

    def upload(self, stream=None):
        _check(self.lib.b2j_batch_upload(self._h, stream), "b2j_batch_upload")

    def decode(self, stream=None):
        _check(self.lib.b2j_batch_decode(self._h, stream), "b2j_batch_decode")

    def decode_timed(self, stream=None):
        t = StageTimes()
        _check(self.lib.b2j_batch_decode_timed(self._h, stream, ctypes.byref(t)), "b2j_batch_decode_timed")
        return t

    def decode_steps(self, steps, stream=None):
        """`steps` decodes back to back; returns (per-step StageTimes array, total ms)."""
        per = (StageTimes * steps)()
        total = ctypes.c_float()
        _check(self.lib.b2j_batch_decode_steps(self._h, stream, steps, per, ctypes.byref(total)), "b2j_batch_decode_steps")
        return per, total.value

    def sync(self, stream=None):
        _check(self.lib.b2j_batch_sync(self._h, stream), "b2j_batch_sync")

    def status(self, stream=None):
        st = np.zeros(self.n, np.int32)
        _check(self.lib.b2j_batch_status(self._h, stream, st.ctypes.data), "b2j_batch_status")
        return st

    def sync_stats(self, stream=None):
        out = np.zeros(8, np.uint32)
        _check(self.lib.b2j_batch_sync_stats(self._h, stream, out.ctypes.data), "b2j_batch_sync_stats")
        return out

    def set_output_format(self, fmt):
        """OUT_BGRA (reference layout, default), OUT_RGB24 (H,W,3), OUT_RGB_PLANAR (3,H,W) or OUT_GRAY8 (H,W: libjpeg's
        grayscale output, the luma samples; decodes need PIXELS_LIBJPEG) for the decodes that follow."""
        _check(self.lib.b2j_batch_set_output_format(self._h, fmt), "b2j_batch_set_output_format")
        self.out_format = fmt

    def set_pixel_model(self, model):
        """PIXELS_REFERENCE (the reference's pixels, default) or PIXELS_LIBJPEG (libjpeg-turbo's, what Pillow decodes) for
        the decodes that follow; combines with every output format and with downscale()."""
        _check(self.lib.b2j_batch_set_pixel_model(self._h, model), "b2j_batch_set_pixel_model")
        self.pixel_model = model

    def set_scale(self, denom):
        """1 (default), 2, 4 or 8: the decodes that follow give ceil(W/denom) x ceil(H/denom) pixels, libjpeg-turbo's scaled
        decode (Pillow's draft()). Needs PIXELS_LIBJPEG when decoding; downscale() is refused while denom != 1."""
        _check(self.lib.b2j_batch_set_scale(self._h, denom), "b2j_batch_set_scale")
        self.scale = denom

    def pixel_shape(self, i):
        """Shape of image i's pixels in the batch's output format and scale."""
        return _out_shape(self.descs[i], getattr(self, "out_format", OUT_BGRA), getattr(self, "scale", 1))

    def pixels(self, i, stream=None):
        out = np.zeros(self.pixel_shape(i), np.uint8)
        _check(self.lib.b2j_batch_read_pixels(self._h, stream, i, out.ctypes.data), "b2j_batch_read_pixels")
        return out

    def read_all_pixels(self, outs=None, stream=None):
        """Every image's pixels into outs (arrays or addresses; allocated at pixel_shape() when None). Returns outs."""
        if outs is None:
            outs = [np.zeros(self.pixel_shape(i), np.uint8) for i in range(self.n)]
        op = (ctypes.c_void_p * self.n)(*[o if isinstance(o, int) else o.ctypes.data for o in outs])
        _check(self.lib.b2j_batch_read_all_pixels(self._h, stream, op), "b2j_batch_read_all_pixels")
        return outs

    def coefs(self, i, stream=None):
        """The reference's coefficient tap: int32 [blk_count, 64], natural order, dequantised."""
        d = self.descs[i]
        out = np.zeros((d.blk_count, 64), np.int32)
        _check(self.lib.b2j_batch_read_coefs(self._h, stream, i, out.ctypes.data), "b2j_batch_read_coefs")
        return out

    def downscale(self, factor, stream=None):
        """b2j_batch_downscale: box-filter reduction (factor 2, 4 or 8) of the decoded pixels, in the batch's output format."""
        _check(self.lib.b2j_batch_downscale(self._h, stream, factor), "b2j_batch_downscale")
        self.small_factor = factor

    def downscaled(self, i, stream=None):
        out = np.zeros(_out_shape(self.descs[i], getattr(self, "out_format", OUT_BGRA), self.small_factor), np.uint8)
        _check(self.lib.b2j_batch_read_downscaled(self._h, stream, i, out.ctypes.data), "b2j_batch_read_downscaled")
        return out

    def pixels_device(self, i):
        p, n = ctypes.c_void_p(), ctypes.c_size_t()
        _check(self.lib.b2j_batch_pixels_device(self._h, i, ctypes.byref(p), ctypes.byref(n)), "b2j_batch_pixels_device")
        return p.value, n.value
