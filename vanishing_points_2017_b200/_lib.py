"""ctypes binding of libvpk.so (include/vpk.h).  No CPU fallback: if the
library or a CUDA device is missing, calls fail loudly."""
import collections
import ctypes as C
import os
import sys
import threading

import numpy as np

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libvpk.so")

VPK_MAX_VP = 64
VPK_GRID = 20
VPK_CNN_SIZE = 500
SPHERE_VOTES, SPHERE_CURVES = 0, 1
EM_OK, EM_NO_INITIAL_VPS, EM_NO_VPS_LEFT, EM_CAPACITY = 0, 1, 2, 3

# every symbol include/vpk.h declares (tests check the .so exports each one)
SYMBOLS = [
    "vpk_create", "vpk_destroy", "vpk_abi_version", "vpk_last_error", "vpk_synchronize", "vpk_launch_count", "vpk_mark", "vpk_mark_elapsed",
    "vpk_profile_enable", "vpk_profile_reset", "vpk_profile_read", "vpk_lines_from_segments", "vpk_sphere_map",
    "vpk_cnn_load", "vpk_cnn_forward", "vpk_cnn_debug_fetch", "vpk_debug_gemm", "vpk_em_default_config", "vpk_em", "vpk_em_distribution", "vpk_em_debug_fetch", "vpk_em_stats", "vpk_em_phase_cycles", "vpk_pipeline_upload", "vpk_pipeline_run",
    "vpk_pipeline_fetch", "vpk_pipeline_host", "vpk_pipeline_stage_ms", "vpk_horizon", "vpk_pipeline_horizon",
    "vpk_segments_from_lsd", "vpk_pipeline_upload_lsd",
    "vpk_lsd_default_config", "vpk_lsd", "vpk_lsd_fetch", "vpk_pipeline_upload_images",
    "vpk_prepared_size", "vpk_prepare_images", "vpk_pipeline_upload_photos",
    "vpk_jpeg_info", "vpk_decode_jpegs", "vpk_pipeline_upload_jpegs", "vpk_jpeg_stats",
    "vpk_png_info", "vpk_decode_pngs", "vpk_pipeline_upload_pngs",
    "vpk_file_info", "vpk_decode_files", "vpk_prepare_files", "vpk_pipeline_upload_files",
    "vpk_pipeline_upload_device", "vpk_pipeline_upload_images_device", "vpk_pipeline_upload_photos_device",
    "vpk_pipeline_fetch_device", "vpk_pipeline_horizon_device",
]
PIX_U8, PIX_F64 = 0, 1
# vpk.h VPK_JPEG_*: support codes of vpk_jpeg_info and the decode status
JPEG_REASONS = ["ok", "progressive", "arithmetic", "precision", "color", "layout", "malformed", "lossless", "corrupt"]
JPEG_OK, JPEG_CORRUPT = 0, 8
# vpk.h VPK_PNG_*: support codes of vpk_png_info and the decode status
PNG_REASONS = ["ok", "not png", "depth", "malformed", "corrupt"]
PNG_OK, PNG_CORRUPT = 0, 4
# vpk.h VPK_FILE_*: formats of vpk_file_info; VPK_PGM_*: support codes of a PGM file
FILE_UNKNOWN, FILE_JPEG, FILE_PNG, FILE_PGM = 0, 1, 2, 3
FILE_FORMATS = ["unknown", "jpeg", "png", "pgm"]
PGM_REASONS = ["ok", "ascii", "bitmap", "pam", "ppm", "maxval", "depth", "malformed"]
PGM_OK = 0


class VpkError(RuntimeError):
    pass


class EmConfig(C.Structure):
    """vpk_em_config: kwargs of vp_localisation.expectation_maximisation
    (reference vp_localisation.py:168-172)."""
    _fields_ = [("num_iter", C.c_int32), ("num_init_vp", C.c_int32), ("split_merge_freq", C.c_int32),
                ("num_min_lines", C.c_int32), ("do_merge", C.c_int32), ("do_split", C.c_int32),
                ("do_iterations", C.c_int32), ("use_weights", C.c_int32), ("wbias", C.c_double),
                ("merge_thresh", C.c_double), ("outlier_thresh", C.c_double), ("final_convergence", C.c_double),
                ("s_thresh", C.c_double)]


class LsdConfig(C.Structure):
    """vpk_lsd_config: the parameters of lsd.detect_line_segments (lsdpython/lsd.pyx:17-18)."""
    _fields_ = [("scale", C.c_double), ("sigma_scale", C.c_double), ("quant", C.c_double), ("ang_th", C.c_double),
                ("log_eps", C.c_double), ("density_th", C.c_double), ("n_bins", C.c_int32)]


class EmResult(C.Structure):
    _fields_ = [("status", C.c_void_p), ("n_vp", C.c_void_p), ("iterations", C.c_void_p), ("vp", C.c_void_p),
                ("sigma", C.c_void_p), ("counts", C.c_void_p), ("counts_weighted", C.c_void_p),
                ("vp_assoc", C.c_void_p), ("decision_metric", C.c_void_p)]


_lib = None
_lock = threading.Lock()


def load():
    """dlopen libvpk.so (no GPU needed for loading)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise VpkError("libvpk.so is not built (%s); run `python -m vanishing_points_2017_b200.build` "
                           "or __graft_entry__.build(). There is no CPU fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        lib.vpk_last_error.restype = C.c_char_p
        lib.vpk_launch_count.restype = C.c_int64
        lib.vpk_launch_count.argtypes = [C.c_void_p]
        lib.vpk_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        lib.vpk_destroy.argtypes = [C.c_void_p]
        lib.vpk_synchronize.argtypes = [C.c_void_p]
        lib.vpk_mark.argtypes = [C.c_void_p, C.c_int32]
        lib.vpk_mark_elapsed.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]
        lib.vpk_profile_enable.argtypes = [C.c_void_p, C.c_int]
        lib.vpk_profile_reset.argtypes = [C.c_void_p]
        lib.vpk_profile_read.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_lines_from_segments.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        lib.vpk_sphere_map.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                       C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_cnn_load.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_cnn_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        lib.vpk_cnn_debug_fetch.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
        lib.vpk_debug_gemm.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
        lib.vpk_em_default_config.argtypes = [C.POINTER(EmConfig)]
        lib.vpk_em_default_config.restype = None
        lib.vpk_em.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                               C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(EmConfig), C.POINTER(EmResult)]
        lib.vpk_em_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        lib.vpk_em_distribution.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_em_debug_fetch.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
        lib.vpk_em_phase_cycles.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        lib.vpk_pipeline_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]
        lib.vpk_pipeline_run.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.POINTER(EmConfig)]
        lib.vpk_pipeline_fetch.argtypes = [C.c_void_p, C.POINTER(EmResult), C.c_void_p, C.c_void_p]
        lib.vpk_pipeline_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_double, C.POINTER(EmConfig), C.POINTER(EmResult), C.c_void_p,
                                          C.c_void_p]
        lib.vpk_pipeline_stage_ms.argtypes = [C.c_void_p, C.c_void_p]
        lib.vpk_horizon.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.c_double,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_segments_from_lsd.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                              C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_pipeline_upload_lsd.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]
        lib.vpk_pipeline_horizon.argtypes = [C.c_void_p, C.c_int32, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_lsd_default_config.argtypes = [C.POINTER(LsdConfig)]
        lib.vpk_lsd_default_config.restype = None
        lib.vpk_lsd.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                C.POINTER(LsdConfig), C.c_void_p]
        lib.vpk_lsd_fetch.argtypes = [C.c_void_p, C.c_void_p]
        lib.vpk_pipeline_upload_images.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_int32, C.POINTER(LsdConfig), C.c_void_p]
        lib.vpk_prepared_size.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
        lib.vpk_prepare_images.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                           C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_pipeline_upload_photos.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                                   C.c_int32, C.POINTER(LsdConfig), C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_jpeg_info.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_decode_jpegs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        lib.vpk_pipeline_upload_jpegs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(LsdConfig),
                                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_jpeg_stats.argtypes = [C.c_void_p, C.c_void_p]
        lib.vpk_png_info.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_decode_pngs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        lib.vpk_pipeline_upload_pngs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(LsdConfig),
                                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_file_info.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_decode_files.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        lib.vpk_prepare_files.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                          C.c_void_p]
        lib.vpk_pipeline_upload_files.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(LsdConfig),
                                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_pipeline_upload_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p]
        lib.vpk_pipeline_upload_images_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                                          C.c_int32, C.POINTER(LsdConfig), C.c_void_p, C.c_void_p]
        lib.vpk_pipeline_upload_photos_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                          C.c_int32, C.c_int32, C.POINTER(LsdConfig), C.c_void_p, C.c_void_p,
                                                          C.c_void_p, C.c_void_p]
        lib.vpk_pipeline_fetch_device.argtypes = [C.c_void_p, C.POINTER(EmResult), C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_pipeline_horizon_device.argtypes = [C.c_void_p, C.c_int32, C.c_double, C.c_double, C.c_void_p, C.c_void_p,
                                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.vpk_abi_version.argtypes = []
        lib.vpk_last_error.argtypes = []
        _lib = lib
        return lib


def check(status, what):
    if status != 0:
        msg = load().vpk_last_error().decode("utf-8", "replace")
        raise VpkError("%s failed (status %d): %s" % (what, status, msg))


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    """One vpk_ctx per process and device (reference: caffe.set_device,
    evaluation.py:20-21)."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        check(self.lib.vpk_create(int(device), C.byref(h)), "vpk_create")
        self.h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "h", None):
            self.lib.vpk_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        check(self.lib.vpk_synchronize(self.h), "vpk_synchronize")

    def mark(self, slot=0):
        """Device timestamp `slot` on this context's stream."""
        check(self.lib.vpk_mark(self.h, int(slot)), "vpk_mark")

    def elapsed_ms(self, slot_from, other, slot_to):
        """Device time from this context's mark `slot_from` to `other`'s mark `slot_to` (same device)."""
        ms = C.c_float()
        check(self.lib.vpk_mark_elapsed(self.h, int(slot_from), other.h, int(slot_to), C.byref(ms)), "vpk_mark_elapsed")
        return float(ms.value)

    def launch_count(self):
        return int(self.lib.vpk_launch_count(self.h))

    def profile_enable(self, on=True):
        check(self.lib.vpk_profile_enable(self.h, 1 if on else 0), "vpk_profile_enable")

    def profile_reset(self):
        check(self.lib.vpk_profile_reset(self.h), "vpk_profile_reset")

    def em_stats(self, reset=False):
        out = (C.c_uint64 * 6)()
        check(self.lib.vpk_em_stats(self.h, out, 1 if reset else 0), "vpk_em_stats")
        return {"wmat_bytes": int(out[0]), "wmat_flops": int(out[1]), "wmat_products": int(out[2]),
                "supersteps": int(out[3]), "post_bytes": int(out[4]), "estep_bytes": int(out[5])}

    def em_phase_cycles(self, reset=False):
        out = (C.c_uint64 * 8)()
        check(self.lib.vpk_em_phase_cycles(self.h, out, 1 if reset else 0), "vpk_em_phase_cycles")
        names = ["estep", "sync_e", "wmat", "sync_w", "mstep_sums", "post", "sync_mirror"]
        return {n: int(out[i]) for i, n in enumerate(names)}

    def profile_read(self):
        cap = 64
        names = (C.c_char_p * cap)()
        ms = (C.c_double * cap)()
        n_l = (C.c_int64 * cap)()
        n = self.lib.vpk_profile_read(self.h, cap, names, ms, n_l)
        if n < 0:
            check(1, "vpk_profile_read")
        return {names[i].decode(): {"ms": ms[i], "launches": int(n_l[i])} for i in range(min(n, cap))}


_default = {}


def default_context(device=0):
    ctx = _default.get(device)
    if ctx is None or ctx.h is None:
        ctx = Context(device)
        _default[device] = ctx
    return ctx


def em_config(**kw):
    cfg = EmConfig()
    load().vpk_em_default_config(C.byref(cfg))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise TypeError("unknown EM option %r" % k)
        setattr(cfg, k, v)
    return cfg


def lsd_config(**kw):
    cfg = LsdConfig()
    load().vpk_lsd_default_config(C.byref(cfg))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise TypeError("unknown LSD option %r" % k)
        setattr(cfg, k, v)
    return cfg


def as_f64(a, cols):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if a.ndim != 2 or a.shape[1] != cols:
        raise ValueError("expected an (N,%d) array, got %r" % (cols, a.shape))
    return a


def as_offsets(offsets):
    o = np.ascontiguousarray(offsets, dtype=np.int32)
    if o.ndim != 1 or o.size < 1 or o[0] != 0 or np.any(np.diff(o) < 0):
        raise ValueError("offsets must be a non-decreasing int array starting at 0")
    return o


# ---- arrays in CUDA memory (__cuda_array_interface__), row N9 ----
U8, F64, I32, I64 = "|u1", "<f8", "<i4", "<i8"
_TYPESTR_ALIASES = {"<u1": U8, "=u1": U8, ">u1": U8, "=f8": F64, "=i4": I32, "=i8": I64}

CudaArray = collections.namedtuple("CudaArray", "ptr shape strides typestr stream")
CudaArray.__doc__ = """An array in CUDA memory: data pointer, shape, strides in BYTES (always given), typestr (U8, F64, I32 or
I64 for their aliases) and the stream its producer exported (__cuda_array_interface__ v3; None: none to order after)."""


def is_cuda_array(obj):
    return hasattr(obj, "__cuda_array_interface__")


def cuda_array(obj, typestrs=(U8, F64), ndims=(2, 3), channels=(1, 3)):
    """The __cuda_array_interface__ (v2 or v3) of `obj` as a CudaArray; strides None (C-contiguous) are filled in.
    ValueError for a typestr not in `typestrs`, a rank not in `ndims`, a 3-D array whose last extent is not in
    `channels`, a mask, a negative stride or a stride that is not a whole number of elements.  Imports nothing."""
    cai = obj.__cuda_array_interface__
    version = int(cai.get("version", 0))
    if version < 2:
        raise ValueError("__cuda_array_interface__ version %d; 2 or later is read" % version)
    if cai.get("mask") is not None:
        raise ValueError("masked CUDA arrays are not taken")
    typestr = _TYPESTR_ALIASES.get(cai["typestr"], cai["typestr"])
    if typestr not in typestrs:
        raise ValueError("CUDA array of type %r; expected %s" % (cai["typestr"], " or ".join(typestrs)))
    shape = tuple(int(s) for s in cai["shape"])
    if len(shape) not in ndims:
        raise ValueError("CUDA array of shape %r; expected %s dimensions" % (shape, " or ".join(str(n) for n in ndims)))
    if len(shape) == 3 and channels is not None and shape[2] not in channels:
        raise ValueError("CUDA array of shape %r: %d channels, expected %s" % (shape, shape[2], " or ".join(str(c) for c in channels)))
    itemsize = int(typestr[2:])
    strides = cai.get("strides")
    if strides is None:
        strides, step = [], itemsize
        for s in reversed(shape):
            strides.insert(0, step)
            step *= s
    strides = tuple(int(s) for s in strides)
    if len(strides) != len(shape):
        raise ValueError("CUDA array: %d strides for %d dimensions" % (len(strides), len(shape)))
    if any(s < 0 for s in strides):
        raise ValueError("CUDA array with negative strides %r; make it contiguous first" % (strides,))
    if any(s % itemsize for s in strides):
        raise ValueError("CUDA array strides %r are not whole elements of %d bytes" % (strides, itemsize))
    stream = cai.get("stream") if version >= 3 else None
    return CudaArray(int(cai["data"][0] or 0), shape, strides, typestr, None if stream is None else int(stream))


def _handle(stream):
    """cudaStream_t of a stream object (torch .cuda_stream, cupy .ptr) or an int handle."""
    for attr in ("cuda_stream", "ptr"):
        if hasattr(stream, attr):
            return int(getattr(stream, attr))
    return int(stream)


def torch_stream(handle, device):
    import torch
    if handle in (0, 1):
        return torch.cuda.default_stream(device)
    return torch.cuda.ExternalStream(handle, device=device)


def call_stream(stream, device, arrays=()):
    """The cudaStream_t a device call is ordered on: `stream` (a stream object or handle; 0 the legacy default stream), or
    if None PyTorch's current stream of `device` when torch is imported, else 0.  Work queued on a CAI v3 stream that
    an input exports and that differs from it is ordered before it with an event."""
    if stream is not None:
        h = _handle(stream)
    elif "torch" in sys.modules:
        h = int(sys.modules["torch"].cuda.current_stream(device).cuda_stream)
    else:
        h = 0
    legacy = lambda s: 0 if s in (0, 1) else s      # noqa: E731  (CAI v3 writes the legacy default stream as 1)
    others = {legacy(a.stream) for a in arrays if a.stream is not None} - {legacy(h)}
    if others:
        import torch
        target = torch_stream(h, device)
        for s in sorted(others):
            ev = torch.cuda.Event()
            ev.record(torch_stream(s, device))
            target.wait_event(ev)
    return h
