"""Drop-in for lsdpython's `lsd` module (reference evaluation.py:236): the LSD 1.6 line segment detector on the
device through the C ABI (`vpk_lsd`, row N4).  No CPU fallback."""
import ctypes as C

import numpy as np

from . import _lib


def pack_images(images):
    """List of 2-D gray images -> (flat pixels, dtype code, pixel offsets, widths, heights).  All uint8 stay uint8
    (8x less host-to-device traffic); anything else is converted to float64, the reference's dtype."""
    imgs = [np.asarray(im) for im in images]
    for im in imgs:
        if im.ndim != 2:
            raise ValueError("LSD takes 2-D grayscale images, got shape %r" % (im.shape,))
    u8 = all(im.dtype == np.uint8 for im in imgs)
    dt = np.uint8 if u8 else np.float64
    flat = np.ascontiguousarray(np.concatenate([im.astype(dt, copy=False).reshape(-1) for im in imgs]) if imgs
                                else np.zeros(0, dt))
    off = np.concatenate([[0], np.cumsum([im.size for im in imgs])]).astype(np.int64)
    w = np.array([im.shape[1] for im in imgs], np.int32)
    h = np.array([im.shape[0] for im in imgs], np.int32)
    return flat, (_lib.PIX_U8 if u8 else _lib.PIX_F64), off, w, h


def detect_line_segments_batch(images, scale=0.8, sigma_scale=0.6, quant=2.0, ang_th=22.5, log_eps=0.0, density_th=0.7,
                               n_bins=1024, ctx=None):
    """detect_line_segments for a list of images of any sizes, in one device call; returns a list of (N_b, 7)
    float64 arrays."""
    ctx = ctx or _lib.default_context()
    if len(images) == 0:
        return []
    flat, dt, off, w, h = pack_images(images)
    cfg = _lib.lsd_config(scale=scale, sigma_scale=sigma_scale, quant=quant, ang_th=ang_th, log_eps=log_eps,
                          density_th=density_th, n_bins=n_bins)
    counts = np.empty(len(images), np.int32)
    _lib.check(ctx.lib.vpk_lsd(ctx.h, _lib.ptr(flat), dt, _lib.ptr(off), _lib.ptr(w), _lib.ptr(h), len(images),
                               C.byref(cfg), _lib.ptr(counts)), "vpk_lsd")
    rows = np.empty((int(counts.sum()), 7), np.float64)
    _lib.check(ctx.lib.vpk_lsd_fetch(ctx.h, _lib.ptr(rows)), "vpk_lsd_fetch")
    ro = np.concatenate([[0], np.cumsum(counts)])
    return [rows[ro[b]:ro[b + 1]] for b in range(len(images))]


def detect_line_segments(image, scale=0.8, sigma_scale=0.6, quant=2.0, ang_th=22.5, log_eps=0.0, density_th=0.7,
                         n_bins=1024):
    """lsd.detect_line_segments (lsdpython/lsd.pyx:17-18): image (H, W) gray values -> (N, 7) float64 rows
    x1, y1, x2, y2, width, p, -log10(NFA) in pixels."""
    return detect_line_segments_batch([image], scale, sigma_scale, quant, ang_th, log_eps, density_th, n_bins)[0]
