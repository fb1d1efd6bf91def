"""ctypes binding of libvpk.so (include/vpk.h).  No CPU fallback: if the
library or a CUDA device is missing, calls fail loudly."""
import ctypes as C
import os
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
]
PIX_U8, PIX_F64 = 0, 1
# vpk.h VPK_JPEG_*: support codes of vpk_jpeg_info and the decode status
JPEG_REASONS = ["ok", "progressive", "arithmetic", "precision", "color", "layout", "malformed", "lossless", "corrupt"]
JPEG_OK, JPEG_CORRUPT = 0, 8
# vpk.h VPK_PNG_*: support codes of vpk_png_info and the decode status
PNG_REASONS = ["ok", "not png", "depth", "malformed", "corrupt"]
PNG_OK, PNG_CORRUPT = 0, 4


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
