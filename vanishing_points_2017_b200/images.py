"""Mixed batches of JPEG, PNG and PGM files, colour or gray (`vpk_decode_files` / `vpk_prepare_files`, row N8), PNG decoding (`vpk_decode_pngs`, row N7), JPEG decoding (`vpk_decode_jpegs`, row N6) and photo preparation in front of LSD on the device (`vpk_prepare_images`, row N5): the head of the reference's
evaluation.create_data_pickles (evaluation.py:139-154), i.e. `convert ... -resize TxT` (example.py:37: 640;
benchmark.py:59-60: 800 for ECD / HLW; OpenCV 4.13's INTER_AREA rule stands in for ImageMagick), the 8-bit RGB read
back, and skimage.color.rgb2gray.  Photos go over PCIe as uint8 RGB; the float64 gray planes are built on the device.
DESIGN.md sections 4.7 to 4.10.  No CPU fallback."""
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


def pack_jpegs(blobs, kind="JPEG"):
    """List of JPEG (or `kind`) files (bytes, or 1-D uint8 arrays of the file contents) -> (flat bytes, byte offsets
    (B+1) int64).  Anything else raises ValueError."""
    if isinstance(blobs, (bytes, bytearray, np.ndarray)) or not hasattr(blobs, "__len__"):
        raise ValueError("blobs must be a list of %s files (bytes or 1-D uint8 arrays)" % kind)
    parts = []
    for b in blobs:
        if isinstance(b, (bytes, bytearray, memoryview)):
            a = np.frombuffer(bytes(b), np.uint8)
        else:
            a = np.asarray(b)
            if a.ndim != 1 or a.dtype != np.uint8:
                raise ValueError("a %s file must be bytes or a 1-D uint8 array, got %s %r" % (kind, a.dtype, a.shape))
        parts.append(a)
    flat = np.ascontiguousarray(np.concatenate(parts) if parts else np.zeros(0, np.uint8))
    off = np.concatenate([[0], np.cumsum([p.size for p in parts])]).astype(np.int64)
    return flat, off


def jpeg_info(blobs):
    """Reads each file's markers up to the scan (never the entropy-coded data); needs no GPU.  Returns a list of
    (width, height, components, support) with support 0 for a file the decoder takes, else the reason it is refused
    (vpk.h VPK_JPEG_*, named in _lib.JPEG_REASONS)."""
    flat, off = pack_jpegs(blobs)
    B = len(off) - 1
    if B == 0:
        return []
    w, h, c, s = (np.zeros(B, np.int32) for _ in range(4))
    _lib.check(_lib.load().vpk_jpeg_info(_lib.ptr(flat), _lib.ptr(off), B, _lib.ptr(w), _lib.ptr(h), _lib.ptr(c), _lib.ptr(s)),
               "vpk_jpeg_info")
    return [(int(a), int(b), int(d), int(e)) for a, b, d, e in zip(w, h, c, s)]


def decode_jpegs(blobs, ctx=None):
    """Decodes baseline JPEG files on the device, bit for bit with libjpeg-turbo's default decode (EXIF orientation
    ignored).  Returns (arrays, status): (H, W, 3) uint8 RGB arrays, (H, W) for 1-component files, and an int32 status
    per file (0, or _lib.JPEG_CORRUPT for inconsistent entropy-coded data, whose pixels are unspecified).  A refused
    file raises VpkError naming its index and reason."""
    flat, off = pack_jpegs(blobs)
    B = len(off) - 1
    if B == 0:
        return [], np.zeros(0, np.int32)
    info = jpeg_info(blobs)
    for k, (w, h, c, s) in enumerate(info):
        if s != 0:
            raise _lib.VpkError("decode_jpegs: file %d is not supported: %s" % (k, _lib.JPEG_REASONS[s]))
    ctx = ctx or _lib.default_context()
    out = np.empty(max(sum(w * h * c for w, h, c, _ in info), 1), np.uint8)
    status = np.empty(B, np.int32)
    _lib.check(ctx.lib.vpk_decode_jpegs(ctx.h, _lib.ptr(flat), _lib.ptr(off), B, _lib.ptr(out), _lib.ptr(status)), "vpk_decode_jpegs")
    res, pos = [], 0
    for w, h, c, _ in info:
        n = w * h * c
        res.append(out[pos:pos + n].reshape((h, w, 3) if c == 3 else (h, w)))
        pos += n
    return res, status


def jpeg_stats(ctx=None):
    """Decoder statistics of the context's last decode: subsequences, re-decoded subsequences and the most rounds
    inside one CTA (both counted only while profiling is enabled), extra launches across CTAs."""
    ctx = ctx or _lib.default_context()
    out = np.zeros(4, np.int64)
    _lib.check(ctx.lib.vpk_jpeg_stats(ctx.h, _lib.ptr(out)), "vpk_jpeg_stats")
    return {"subsequences": int(out[0]), "redecoded": int(out[1]), "max_rounds": int(out[2]), "global_rounds": int(out[3])}


def png_info(blobs):
    """Walks each file's chunks (headers, IHDR and PLTE; never the image data); needs no GPU.  Returns a list of
    (width, height, colour type, support) with support 0 for a file the decoder takes, else the reason it is refused
    (vpk.h VPK_PNG_*, named in _lib.PNG_REASONS)."""
    flat, off = pack_jpegs(blobs, "PNG")
    B = len(off) - 1
    if B == 0:
        return []
    w, h, t, s = (np.zeros(B, np.int32) for _ in range(4))
    _lib.check(_lib.load().vpk_png_info(_lib.ptr(flat), _lib.ptr(off), B, _lib.ptr(w), _lib.ptr(h), _lib.ptr(t), _lib.ptr(s)),
               "vpk_png_info")
    return [(int(a), int(b), int(c), int(d)) for a, b, c, d in zip(w, h, t, s)]


def decode_pngs(blobs, ctx=None):
    """Decodes 8-bit and lower PNG files on the device, bit for bit with libpng (alpha dropped, no colour management).
    Returns (arrays, status): (H, W, 3) uint8 RGB arrays for colour types 2, 3 and 6, (H, W) gray for types 0 and 4,
    and an int32 status per file (0, or _lib.PNG_CORRUPT for a damaged stream, whose pixels are unspecified).  A
    refused file raises VpkError naming its index and reason."""
    flat, off = pack_jpegs(blobs, "PNG")
    B = len(off) - 1
    if B == 0:
        return [], np.zeros(0, np.int32)
    info = png_info(blobs)
    for k, (w, h, t, s) in enumerate(info):
        if s != 0:
            raise _lib.VpkError("decode_pngs: file %d is not supported: %s" % (k, _lib.PNG_REASONS[s]))
    ctx = ctx or _lib.default_context()
    nc = [1 if t in (0, 4) else 3 for _, _, t, _ in info]
    out = np.empty(max(sum(w * h * c for (w, h, _, _), c in zip(info, nc)), 1), np.uint8)
    status = np.empty(B, np.int32)
    _lib.check(ctx.lib.vpk_decode_pngs(ctx.h, _lib.ptr(flat), _lib.ptr(off), B, _lib.ptr(out), _lib.ptr(status)), "vpk_decode_pngs")
    res, pos = [], 0
    for (w, h, _, _), c in zip(info, nc):
        n = w * h * c
        res.append(out[pos:pos + n].reshape((h, w, 3) if c == 3 else (h, w)))
        pos += n
    return res, status


def file_info(blobs):
    """Sniffs each file (JPEG, PNG or netpbm by its leading bytes) and reads its header; needs no GPU.  Returns a list
    of (format, width, height, channels, support): format a _lib.FILE_* code (named in _lib.FILE_FORMATS), channels 3
    for RGB and 1 for gray, support 0 for a file decode_files takes, else the format's own reason code
    (_lib.JPEG_REASONS, _lib.PNG_REASONS, _lib.PGM_REASONS; 1 for an unknown format)."""
    flat, off = pack_jpegs(blobs, "image")
    B = len(off) - 1
    if B == 0:
        return []
    f, w, h, c, s = (np.zeros(B, np.int32) for _ in range(5))
    _lib.check(_lib.load().vpk_file_info(_lib.ptr(flat), _lib.ptr(off), B, _lib.ptr(f), _lib.ptr(w), _lib.ptr(h), _lib.ptr(c),
                                         _lib.ptr(s)), "vpk_file_info")
    return [(int(a), int(b), int(d), int(e), int(g)) for a, b, d, e, g in zip(f, w, h, c, s)]


def _split(buf, shapes):
    res, pos = [], 0
    for shape in shapes:
        n = int(np.prod(shape))
        res.append(buf[pos:pos + n].reshape(shape))
        pos += n
    return res


def decode_files(blobs, ctx=None):
    """Decodes a mixed batch of JPEG, PNG and binary PGM files on the device, each format by its decoder, in one call.
    Returns (arrays, status): (H, W, 3) uint8 RGB arrays, (H, W) for gray files, and an int32 status per file (the
    format's own code: 0, _lib.JPEG_CORRUPT or _lib.PNG_CORRUPT).  A refused or unknown file raises VpkError naming its
    index, format and reason (file_info tells them beforehand)."""
    flat, off = pack_jpegs(blobs, "image")
    B = len(off) - 1
    if B == 0:
        return [], np.zeros(0, np.int32)
    ctx = ctx or _lib.default_context()
    info = file_info(blobs)
    shapes = [(h, w, 3) if c == 3 else (h, w) for _, w, h, c, _ in info]
    out = np.empty(max(sum(int(np.prod(s)) for s in shapes), 1), np.uint8)
    status = np.empty(B, np.int32)
    _lib.check(ctx.lib.vpk_decode_files(ctx.h, _lib.ptr(flat), _lib.ptr(off), B, _lib.ptr(out), _lib.ptr(status)), "vpk_decode_files")
    return _split(out, shapes), status


def prepare_files(blobs, target_size=None, ctx=None):
    """The reference's datum['image'] of each file of a mixed batch (decode_files, then the preparation of
    prepare_images), in one device call: float64 (H', W') planes in [0, 1] for colour files (rgb2gray), uint8 (H', W')
    planes for gray files (skimage 0.12's rgb2gray returns a 2-D input unchanged), which is what
    evaluation.reference_data(images=...) stores.  Refused files as decode_files."""
    flat, off = pack_jpegs(blobs, "image")
    B = len(off) - 1
    if B == 0:
        return []
    ctx = ctx or _lib.default_context()
    t = _target(target_size)
    info = file_info(blobs)
    n = sum(int(np.prod(prepared_size(w, h, t))) if s == 0 and w > 0 and h > 0 else 0 for _, w, h, _, s in info)
    out = np.empty(max(n, 1), np.float64)
    ow = np.empty(B, np.int32)
    oh = np.empty(B, np.int32)
    _lib.check(ctx.lib.vpk_prepare_files(ctx.h, _lib.ptr(flat), _lib.ptr(off), B, t, _lib.ptr(ow), _lib.ptr(oh), _lib.ptr(out)),
               "vpk_prepare_files")
    planes = _split(out, [(int(H), int(W)) for W, H in zip(ow, oh)])
    return [p if c == 3 else p.astype(np.uint8) for p, (_, _, _, c, _) in zip(planes, info)]
