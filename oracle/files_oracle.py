"""Mixed batches of dataset files (row N8): the reference's evaluation.get_data_list lists *.jpg, *.png and *.pgm into
one dataset, and evaluation.create_data_pickles prepares each file (evaluation.py:139-154, DESIGN.md section 4.10).

- `resize_area` is image_prep_oracle.resize_area for a 2-D uint8 (gray) image, with the same summation order.
- `prepare_file(blob, target)` returns the reference's datum['image'] and the plane detect_lsd_lines gives LSD. A
  colour file gives rgb2gray's float64 plane, which LSD sees times 255. For a gray file (one decoded channel: a
  1-component JPEG, PNG colour type 0 or 4, a PGM), skimage 0.12's rgb2gray returns the 2-D input unchanged, so
  datum['image'] is the resized uint8 plane. detect_lsd_lines multiplies it by 255 only if its maximum is at most 1.
- The PGM reference decode is cv2 (IMREAD_UNCHANGED), cross-checked against PIL. `write_pgm` is a hand-written
  writer. `pgm_corpus()` holds the files the library takes (comments, odd whitespace, 1 x N and N x 1, extra
  trailing data), `pgm_refused()` the ones it refuses, with the reason.
"""
import io

import cv2
import numpy as np
from PIL import Image

from . import image_prep_oracle as P
from . import jpeg_oracle as J
from . import png_oracle as G

UNKNOWN, JPEG, PNG, PGM = 0, 1, 2, 3
PGM_OK, PGM_ASCII, PGM_BITMAP, PGM_PAM, PGM_PPM, PGM_MAXVAL, PGM_DEPTH, PGM_MALFORMED = range(8)


def resize_area(img, W, H):
    """cv2.resize(img, (W, H), interpolation=INTER_AREA) for an (h, w) uint8 image, W <= w and H <= h: the rules of
    image_prep_oracle.resize_area on one channel."""
    img = np.asarray(img)
    h, w = img.shape
    if (W, H) == (w, h):
        return img.copy()
    if w % W == 0 and h % H == 0:
        kx, ky = w // W, h // H
        total = img.astype(np.int64).reshape(H, ky, W, kx).sum(axis=(1, 3))
        return P._round_mean(total, kx * ky, kx == 2 and ky == 2).astype(np.uint8)
    ix, ax = P.area_taps(w, W)
    iy, ay = P.area_taps(h, H)
    f = img.astype(np.float64)
    t = np.zeros((h, W))
    for k in range(ix.shape[1]):
        t = t + ax[None, :, k] * f[:, ix[:, k]]
    o = np.zeros((H, W))
    for k in range(iy.shape[1]):
        o = o + ay[:, k, None] * t[iy[:, k], :]
    return np.clip(np.rint(o), 0.0, 255.0).astype(np.uint8)


def sniff(blob):
    b = bytes(blob[:8])
    if b[:3] == b"\xff\xd8\xff":
        return JPEG
    if b[:8] == G.SIG:
        return PNG
    if len(b) >= 2 and b[:1] == b"P" and b[1:2] in b"1234567":
        return PGM
    return UNKNOWN


def decode_pgm(blob):
    return cv2.imdecode(np.frombuffer(bytes(blob), np.uint8), cv2.IMREAD_UNCHANGED)


def decode_pgm_pil(blob):
    return np.asarray(Image.open(io.BytesIO(bytes(blob))))


def decode(blob):
    """the reference decode of any file: (H, W, 3) uint8 RGB, or (H, W) uint8 for a gray file"""
    return {JPEG: J.decode, PNG: G.decode, PGM: decode_pgm}[sniff(blob)](blob)


def prepare_file(blob, target_size=None):
    """(datum['image'], LSD's input plane) of one file: float64 rgb2gray and it times 255 for a colour file; the
    resized uint8 plane and its float64 values, times 255 if they are all at most 1, for a gray file."""
    img = decode(blob)
    if img.ndim == 3:
        g = P.prepare(img, target_size)
        return g, g * 255
    W, H = P.prepared_size(img.shape[1], img.shape[0], target_size)
    g = resize_area(img, W, H)
    lsd = g.astype(np.float64)                  # evaluation.detect_lsd_lines
    if lsd.max() <= 1:
        lsd *= 255
    return g, lsd


def write_pgm(img, magic=b"P5", sep=(b"\n", b" ", b"\n", b"\n"), maxval=255, comments=(), extra=b"", payload=None):
    """A netpbm file: magic, sep[0], width, sep[1], height, sep[2], maxval, sep[3] (the one byte before the payload),
    then the payload (the image's bytes unless given) and `extra`.  comments: (position, text) pairs, each '#text\\n'
    inserted after the whitespace that follows the magic (0), the width (1) or the height (2)."""
    img = np.asarray(img, np.uint8)
    h, w = img.shape
    parts = [magic, sep[0], b"", b"%d" % w, sep[1], b"", b"%d" % h, sep[2], b"", b"%d" % maxval, sep[3]]
    for pos, text in comments:
        parts[2 + 3 * pos] += b"#" + text + b"\n"
    return b"".join(parts) + (img.tobytes() if payload is None else payload) + extra


def gray_image(seed, w, h):
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    base = 128 + 70 * np.sin(xx / 17.0 + seed) * np.cos(yy / 11.0)
    return np.clip(np.round(base + rs.normal(0, 25, (h, w))), 0, 255).astype(np.uint8)


def pgm_corpus():
    """(name, file, image) triples of PGM files the library takes; seeded"""
    out = []
    for k, (w, h) in enumerate([(1, 1), (1, 57), (61, 1), (2, 3), (40, 30), (257, 191), (640, 480), (1001, 667)]):
        img = gray_image(k, w, h)
        out.append(("plain_%dx%d" % (w, h), write_pgm(img), img))
    img = gray_image(20, 123, 77)
    out += [("comments", write_pgm(img, comments=[(0, b" made by hand"), (1, b""), (2, b"two\tcomments"), (2, b"#")]), img),
            ("spaces", write_pgm(img, sep=(b"  \t", b"\t\t", b"\r\n ", b" ")), img),
            ("tab_before_payload", write_pgm(img, sep=(b" ", b" ", b" ", b"\t")), img),
            ("cr_before_payload", write_pgm(img, sep=(b"\n", b"\n", b"\n", b"\r")), img),
            ("extra_data", write_pgm(img, extra=b"\x00\xffextra bytes after the payload"), img),
            ("payload_starts_with_space", write_pgm(np.full((5, 7), 32, np.uint8)), np.full((5, 7), 32, np.uint8)),
            ("black", write_pgm(np.zeros((31, 45), np.uint8)), np.zeros((31, 45), np.uint8)),
            ("white", write_pgm(np.full((29, 33), 255, np.uint8)), np.full((29, 33), 255, np.uint8))]
    return out


def pgm_refused():
    """(name, file, reason) triples of netpbm files the library refuses"""
    img = gray_image(30, 20, 10)
    ascii_payload = b" ".join(b"%d" % v for v in img.reshape(-1))
    rgb = np.dstack([img] * 3)
    return [("ascii_p2", write_pgm(img, magic=b"P2", payload=ascii_payload), PGM_ASCII),
            ("bitmap_p1", write_pgm(img, magic=b"P1", payload=b"0 1 " * 100), PGM_BITMAP),
            ("bitmap_p4", b"P4\n20 10\n" + bytes(30), PGM_BITMAP),
            ("pam_p7", b"P7\nWIDTH 20\nHEIGHT 10\nDEPTH 1\nMAXVAL 255\nTUPLTYPE GRAYSCALE\nENDHDR\n" + img.tobytes(), PGM_PAM),
            ("ppm_p6", b"P6\n20 10\n255\n" + rgb.tobytes(), PGM_PPM),
            ("maxval_100", write_pgm(img // 3, maxval=100), PGM_MAXVAL),
            ("maxval_65535", write_pgm(img, maxval=65535, payload=np.repeat(img.reshape(-1), 2).tobytes()), PGM_DEPTH),
            ("truncated", write_pgm(img)[:-1], PGM_MALFORMED),
            ("no_payload_byte", b"P5\n20 10\n255", PGM_MALFORMED),
            ("zero_width", write_pgm(np.zeros((10, 0), np.uint8)), PGM_MALFORMED),
            ("no_height", b"P5\n20\n", PGM_MALFORMED),
            ("garbage_size", b"P5\n20 x10\n255\n" + img.tobytes(), PGM_MALFORMED)]
