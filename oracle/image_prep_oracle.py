"""Photo preparation in front of LSD (reference evaluation.py:139-154, example.py:37, benchmark.py:59-60), restated in
float64 numpy: `convert ... -resize TxT` (stood in for by OpenCV 4.13's `cv2.resize(..., INTER_AREA)`, SURVEY
section 8(c)), read back as 8-bit RGB, then `skimage.color.rgb2gray` (skimage 0.12).

The summation order is part of the specification (DESIGN.md section 4.7): every tap loop runs over tap indices in
increasing source order and is vectorised across pixels only, every step is one correctly rounded float64
operation (no einsum, no BLAS), so csrc/image_prep.cu is held to bit equality with this file.
"""
import math

import numpy as np

INV255 = 1.0 / 255          # skimage's img_as_float: image * (1. / imax), not image / imax
GRAY = (0.2125, 0.7154, 0.0721)


def prepared_size(w, h, target_size):
    """(W', H') of a w x h photo: s = target / max(w, h) in float64; resize only if s < 1, then
    W' = max(1, rint(w s)), H' = max(1, rint(h s)) (rint: half to even, like Python's round).  target_size None
    or <= 0: no resize.  Enlarging is out of scope."""
    w, h = int(w), int(h)
    if target_size is None or int(target_size) <= 0:
        return w, h
    s = float(int(target_size)) / float(max(w, h))
    if not s < 1.0:
        return w, h
    return max(1, int(round(w * s))), max(1, int(round(h * s)))


def area_taps(ssize, dsize):
    """computeResizeAreaTab (OpenCV imgproc/resize.cpp) in float64: (index (dsize, K), weight (dsize, K)), output d's
    taps in increasing source index, padded behind with (0, 0.0) to the longest tap list (adding +0.0 to the
    non-negative partial sums changes no bit)."""
    scale = 1.0 / (dsize / ssize)
    taps = []
    for d in range(dsize):
        fs1 = d * scale
        fs2 = fs1 + scale
        cw = min(scale, ssize - fs1)
        s1, s2 = math.ceil(fs1), math.floor(fs2)
        s2 = min(s2, ssize - 1)
        s1 = min(s1, s2)
        t = []
        if s1 - fs1 > 1e-3:
            t.append((s1 - 1, (s1 - fs1) / cw))
        t += [(s, 1.0 / cw) for s in range(s1, s2)]
        if fs2 - s2 > 1e-3:
            t.append((s2, min(min(fs2 - s2, 1.0), cw) / cw))
        taps.append(t)
    K = max(len(t) for t in taps)
    idx = np.zeros((dsize, K), np.int64)
    wt = np.zeros((dsize, K), np.float64)
    for d, t in enumerate(taps):
        for k, (s, a) in enumerate(t):
            idx[d, k], wt[d, k] = s, a
    return idx, wt


def _round_mean(total, area, half_up):
    """total / area rounded to the nearest integer, ties up (half_up) or to even; exact integer arithmetic."""
    q, r = np.divmod(total, area)
    up = (2 * r > area) | ((2 * r == area) & (half_up | (q % 2 == 1)))
    return q + up


def resize_area(img, W, H):
    """cv2.resize(img, (W, H), interpolation=INTER_AREA) for an (h, w, 3) uint8 image, W <= w and H <= h, restated
    in float64 (cv2 itself accumulates in float32).  Integer factors (OpenCV's is_area_fast): the exact integer mean
    of each kx x ky block, ties half up for 2 x 2 (OpenCV's vectorised path) and half to even otherwise.  Generic
    factors: the x pass, then the y pass, each a sum of weight * value over the taps in increasing source index,
    rint, clamp to 0..255."""
    img = np.asarray(img)
    h, w = img.shape[:2]
    if (W, H) == (w, h):
        return img.copy()
    if w % W == 0 and h % H == 0:
        kx, ky = w // W, h // H
        total = img.astype(np.int64).reshape(H, ky, W, kx, 3).sum(axis=(1, 3))
        return _round_mean(total, kx * ky, kx == 2 and ky == 2).astype(np.uint8)
    ix, ax = area_taps(w, W)
    iy, ay = area_taps(h, H)
    f = img.astype(np.float64)
    t = np.zeros((h, W, 3))
    for k in range(ix.shape[1]):
        t = t + ax[None, :, k, None] * f[:, ix[:, k], :]
    o = np.zeros((H, W, 3))
    for k in range(iy.shape[1]):
        o = o + ay[:, k, None, None] * t[iy[:, k], :, :]
    return np.clip(np.rint(o), 0.0, 255.0).astype(np.uint8)


def rgb2gray(rgb):
    """skimage 0.12 color.rgb2gray of an (H, W, 3) uint8 image: img_as_float (x * (1./255)), then
    g = 0.2125 r, g += 0.7154 g, g += 0.0721 b, each a single float64 operation (the order skimage's BLAS dot uses is
    unpinned)."""
    f = np.asarray(rgb).astype(np.float64) * INV255
    g = GRAY[0] * f[:, :, 0]
    g = g + GRAY[1] * f[:, :, 1]
    g = g + GRAY[2] * f[:, :, 2]
    return g


def prepare(img, target_size=None):
    """The reference's datum['image'] (evaluation.py:139-154) for an (h, w, 3) uint8 photo: float64 gray in [0, 1] of
    the photo resized to prepared_size(w, h, target_size)."""
    h, w = img.shape[:2]
    W, H = prepared_size(w, h, target_size)
    return rgb2gray(resize_area(img, W, H))
