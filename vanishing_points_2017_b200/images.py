"""Photo preparation in front of LSD on the device (`vpk_prepare_images`, row N5): the head of the reference's
evaluation.create_data_pickles (evaluation.py:139-154), i.e. `convert ... -resize TxT` (example.py:37: 640;
benchmark.py:59-60: 800 for ECD / HLW; OpenCV 4.13's INTER_AREA rule stands in for ImageMagick), the 8-bit RGB read
back, and skimage.color.rgb2gray.  Photos go over PCIe as uint8 RGB; the float64 gray planes are built on the device.
DESIGN.md section 4.7.  No CPU fallback."""
import ctypes as C

import numpy as np

from . import _lib


def _target(target_size):
    return 0 if target_size is None else max(int(target_size), 0)


def prepared_size(w, h, target_size):
    """(W', H') of a w x h photo: s = target_size / max(w, h); if s < 1, W' = max(1, rint(w s)) and
    H' = max(1, rint(h s)), else (w, h).  target_size None or <= 0: no resize.  Needs no GPU."""
    W, H = C.c_int32(), C.c_int32()
    _lib.check(_lib.load().vpk_prepared_size(int(w), int(h), _target(target_size), C.byref(W), C.byref(H)), "vpk_prepared_size")
    return int(W.value), int(H.value)


def pack_photos(photos):
    """List of (H, W, 3) uint8 RGB arrays -> (flat bytes, byte offsets (B+1) int64, widths, heights int32).  Anything
    else raises ValueError (2-D gray images go to lsd.detect_line_segments / Pipeline.upload_images)."""
    if isinstance(photos, np.ndarray) or not hasattr(photos, "__len__"):
        raise ValueError("photos must be a list of (H, W, 3) uint8 arrays")
    ims = [np.asarray(p) for p in photos]
    for im in ims:
        if im.ndim != 3 or im.shape[2] != 3 or im.dtype != np.uint8 or im.shape[0] < 1 or im.shape[1] < 1:
            raise ValueError("photos must be (H, W, 3) uint8 RGB arrays, got %s %r" % (im.dtype, im.shape))
    flat = np.ascontiguousarray(np.concatenate([im.reshape(-1) for im in ims]) if ims else np.zeros(0, np.uint8))
    off = np.concatenate([[0], np.cumsum([im.size for im in ims])]).astype(np.int64)
    w = np.array([im.shape[1] for im in ims], np.int32)
    h = np.array([im.shape[0] for im in ims], np.int32)
    return flat, off, w, h


def prepare_images(photos, target_size=None, ctx=None):
    """The reference's datum['image'] for a list of (H, W, 3) uint8 RGB photos of any sizes, in one device call:
    each photo resized to prepared_size(W, H, target_size) and converted to gray.  Returns a list of float64
    (H', W') arrays in [0, 1]."""
    flat, off, w, h = pack_photos(photos)
    if len(w) == 0:
        return []
    ctx = ctx or _lib.default_context()
    t = _target(target_size)
    sizes = [prepared_size(a, b, t) for a, b in zip(w, h)]
    n = sum(W * H for W, H in sizes)
    out = np.empty(n, np.float64)
    ow = np.empty(len(w), np.int32)
    oh = np.empty(len(w), np.int32)
    _lib.check(ctx.lib.vpk_prepare_images(ctx.h, _lib.ptr(flat), _lib.ptr(off), _lib.ptr(w), _lib.ptr(h), len(w), t,
                                          _lib.ptr(ow), _lib.ptr(oh), _lib.ptr(out)), "vpk_prepare_images")
    res, pos = [], 0
    for W, H in zip(ow, oh):
        res.append(out[pos:pos + int(W) * int(H)].reshape(int(H), int(W)))
        pos += int(W) * int(H)
    return res
