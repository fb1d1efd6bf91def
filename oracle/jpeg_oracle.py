"""Row N6 oracle: the reference decode of baseline JPEG files and a seeded corpus of them.

The reference decode is libjpeg-turbo 3.1's default (islow IDCT, fancy upsampling, jdcolor.c's tables) through
cv2.imdecode with IMREAD_COLOR | IMREAD_IGNORE_ORIENTATION, converted to RGB (IMREAD_GRAYSCALE for 1-component
files); PIL, which links its own libjpeg-turbo and never rotates, decodes the same bytes for a cross-check.  Whether
the reference's ImageMagick linked libjpeg-turbo or IJG libjpeg 9 is not pinned (DESIGN.md section 2).

corpus() encodes seeded photos with cv2 and PIL: every sampling layout, qualities 50 / 75 / 90 / 100, optimised
Huffman tables, restart intervals, custom quantisation tables, COM / APPn markers, EXIF orientation 6, sizes from
1 x 1 to 6000 x 4000, and content that stresses the decoder (noise: long codes and dense streams; saturated
primaries: the range limit; constant images: EOB-only streams).  refused() builds files the decoder must refuse."""
import io

import cv2
import numpy as np
from PIL import Image

# support codes (include/vpk.h VPK_JPEG_*)
OK, PROGRESSIVE, ARITHMETIC, PRECISION, COLOR, LAYOUT, MALFORMED, LOSSLESS, CORRUPT = range(9)
SAMPLING = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "411": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411,
            "440": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440}


def components(blob):
    """number of components of the frame, from PIL's mode"""
    return {"L": 1, "RGB": 3, "CMYK": 4}[Image.open(io.BytesIO(bytes(blob))).mode]


def decode(blob):
    """the reference decode: (H, W, 3) uint8 RGB, or (H, W) uint8 for a 1-component file"""
    buf = np.frombuffer(bytes(blob), np.uint8)
    if components(blob) == 1:
        return cv2.imdecode(buf, cv2.IMREAD_GRAYSCALE)
    return np.ascontiguousarray(cv2.imdecode(buf, cv2.IMREAD_COLOR | cv2.IMREAD_IGNORE_ORIENTATION)[:, :, ::-1])


def decode_pil(blob):
    return np.asarray(Image.open(io.BytesIO(bytes(blob))))


def noise(seed, w, h):
    return np.random.RandomState(seed).randint(0, 256, (h, w, 3)).astype(np.uint8)


def primaries(seed, w, h):
    """saturated red / green / blue / white / black stripes with noise on top: IDCT outputs beyond 0..255"""
    rs = np.random.RandomState(seed)
    cols = np.array([[255, 0, 0], [0, 255, 0], [0, 0, 255], [255, 255, 255], [0, 0, 0]], np.uint8)
    idx = (np.arange(w)[None, :] // 3 + np.arange(h)[:, None] // 5) % 5
    img = cols[idx].astype(np.int32) + rs.randint(-2, 3, (h, w, 3))
    return np.clip(img, 0, 255).astype(np.uint8)


def constant(seed, w, h):
    return np.full((h, w, 3), np.random.RandomState(seed).randint(0, 256, 3), np.uint8)


def photo(seed, w, h, texture=0.0):
    """synth.render_photo, optionally with uniform noise texture of amplitude `texture` (more bits per pixel,
    nearer real photos)"""
    from vanishing_points_2017_b200 import synth
    img = synth.render_photo(seed, 150, w, h).astype(np.int32)
    if texture:
        img += np.random.RandomState(seed + 1).randint(-int(texture), int(texture) + 1, img.shape)
    return np.clip(img, 0, 255).astype(np.uint8)


def encode_cv2(rgb, quality=90, sampling="420", optimize=False, restart=0, progressive=False):
    if rgb.ndim == 2:
        params = [cv2.IMWRITE_JPEG_QUALITY, quality]
        img = rgb
    else:
        params = [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sampling]]
        img = np.ascontiguousarray(rgb[:, :, ::-1])
    params += [cv2.IMWRITE_JPEG_OPTIMIZE, int(optimize), cv2.IMWRITE_JPEG_RST_INTERVAL, int(restart),
               cv2.IMWRITE_JPEG_PROGRESSIVE, int(progressive)]
    ok, buf = cv2.imencode(".jpg", img, params)
    assert ok
    return buf.tobytes()


def encode_pil(rgb, quality=90, subsampling=2, **kw):
    im = Image.fromarray(rgb)
    out = io.BytesIO()
    im.save(out, format="JPEG", quality=quality, subsampling=subsampling, **kw)
    return out.getvalue()


def with_app(blob, marker=0xE5, payload=b"vpk test segment"):
    """an extra APPn segment right after SOI"""
    n = len(payload) + 2
    return blob[:2] + bytes([0xFF, marker, n >> 8, n & 255]) + payload + blob[2:]


def exif_orientation_6():
    ex = Image.Exif()
    ex[0x0112] = 6
    return ex.tobytes()


def corpus(large=True):
    """[(name, blob)] of supported files; `large` adds the 2000 x 1333 and larger photos"""
    out = []
    sizes = [(1, 1), (2, 2), (3, 5), (7, 9), (17, 33), (33, 17), (5000, 3), (1200, 800), (800, 1200)]
    if large:
        sizes += [(2000, 1333), (6000, 4000)]
    for i, (w, h) in enumerate(sizes):
        img = photo(10 + i, w, h, texture=6) if w * h >= 64 * 64 else noise(10 + i, w, h)
        out.append(("cv2_420_q90_%dx%d" % (w, h), encode_cv2(img, 90, "420")))
    # every sampling layout at every quality on odd sizes (edge replication of the fancy upsamplers)
    for s in ("444", "422", "420", "411", "440"):
        for q in (50, 75, 90, 100):
            img = photo(100 + q, 75, 53, texture=10)
            out.append(("cv2_%s_q%d_75x53" % (s, q), encode_cv2(img, q, s)))
        out.append(("cv2_%s_q90_3x5" % s, encode_cv2(noise(3, 3, 5), 90, s)))
        out.append(("cv2_%s_q90_17x33" % s, encode_cv2(noise(4, 17, 33), 90, s)))
        out.append(("cv2_%s_noise_q100_opt_131x97" % s, encode_cv2(noise(5, 131, 97), 100, s, optimize=True)))
        out.append(("cv2_%s_primaries_q100_123x77" % s, encode_cv2(primaries(6, 123, 77), 100, s)))
        out.append(("cv2_%s_restart1_q90_67x45" % s, encode_cv2(photo(7, 67, 45, texture=8), 90, s, restart=1)))
        out.append(("cv2_%s_restart7_opt_q75_301x211" % s, encode_cv2(photo(8, 301, 211, texture=8), 75, s, optimize=True, restart=7)))
    out.append(("cv2_gray_q90_301x211", encode_cv2(photo(9, 301, 211, texture=8)[:, :, 1], 90)))
    out.append(("cv2_gray_noise_q100_restart7_97x61", encode_cv2(noise(10, 97, 61)[:, :, 0], 100, restart=7)))
    out.append(("cv2_gray_1x1", encode_cv2(noise(11, 1, 1)[:, :, 0], 90)))
    out.append(("cv2_constant_q90_640x480", encode_cv2(constant(12, 640, 480), 90, "420")))
    out.append(("cv2_constant_q50_444_33x17", encode_cv2(constant(13, 33, 17), 50, "444")))
    out.append(("cv2_noise_q100_444_640x480", encode_cv2(noise(14, 640, 480), 100, "444")))
    out.append(("cv2_primaries_q90_420_640x480", encode_cv2(primaries(15, 640, 480), 90, "420")))
    # PIL: its own tables and markers
    img = photo(20, 257, 191, texture=8)
    out.append(("pil_420_q90_257x191", encode_pil(img, 90, 2)))
    out.append(("pil_422_q75_257x191", encode_pil(img, 75, 1)))
    out.append(("pil_444_q100_opt_257x191", encode_pil(img, 100, 0, optimize=True)))
    qt = [[int(1 + (i * 7 + 3) % 40) for i in range(64)], [int(2 + (i * 5 + 1) % 60) for i in range(64)]]
    out.append(("pil_custom_qtables_257x191", encode_pil(img, subsampling=2, qtables=qt)))
    out.append(("pil_comment_app_257x191", with_app(encode_pil(img, 90, 2, comment=b"a comment"))))
    out.append(("pil_exif_orientation6_257x191", encode_pil(img, 90, 2, exif=exif_orientation_6())))
    out.append(("pil_gray_q90_257x191", encode_pil(img[:, :, 0], 90, 0)))
    return out


def _find_marker(blob, code):
    """byte offset of the first marker `code` in the header (segment walk from SOI)"""
    p = 2
    while p + 4 <= len(blob):
        m = blob[p + 1]
        if m == code:
            return p
        p += 2 + (blob[p + 2] << 8 | blob[p + 3])
    raise ValueError("marker %02x not found" % code)


def refused():
    """[(name, blob, reason)] of files the decoder refuses before any device work"""
    img = photo(30, 97, 65, texture=8)
    base = encode_cv2(img, 90, "420")
    out = [("progressive_cv2", encode_cv2(img, 90, "420", progressive=True), PROGRESSIVE),
           ("progressive_pil", encode_pil(img, 90, 2, progressive=True), PROGRESSIVE)]
    cm = io.BytesIO()
    Image.fromarray(img).convert("CMYK").save(cm, format="JPEG", quality=90)
    out.append(("cmyk_pil", cm.getvalue(), COLOR))
    sof = _find_marker(base, 0xC0)
    b = bytearray(base); b[sof + 1] = 0xC9
    out.append(("sof_arithmetic", bytes(b), ARITHMETIC))
    b = bytearray(base); b[sof + 4] = 12
    out.append(("sof_12bit", bytes(b), PRECISION))
    b = bytearray(base); b[sof + 1] = 0xC3
    out.append(("sof_lossless", bytes(b), LOSSLESS))
    sos = _find_marker(base, 0xDA)
    for k in (0, 1, 3, 11, sof + 5, sof + 12, sos, sos + 6):
        out.append(("truncated_header_%d" % k, base[:k], MALFORMED))
    dht = _find_marker(base, 0xC4)
    b = bytearray(base); b[dht + 5 + 15] = 200           # 16-bit code count of the first table: beyond its segment
    out.append(("dht_counts_overrun", bytes(b), MALFORMED))
    b = bytearray(base); b[0] = 0x00
    out.append(("no_soi", bytes(b), MALFORMED))
    out.append(("garbage", bytes(np.random.RandomState(1).randint(0, 256, 500).astype(np.uint8)), MALFORMED))
    return out


def corrupted(blob, seed):
    """[(name, blob)]: the file truncated in its entropy-coded data, with bits flipped there, and with garbage
    appended before EOI"""
    rs = np.random.RandomState(seed)
    sos = _find_marker(blob, 0xDA)
    data0 = sos + 2 + (blob[sos + 2] << 8 | blob[sos + 3])
    out = [("truncated", blob[:data0 + (len(blob) - data0) // 2])]
    b = bytearray(blob)
    for _ in range(8):
        i = rs.randint(data0, len(blob) - 2)
        b[i] ^= 1 << rs.randint(0, 8)
    out.append(("bitflip", bytes(b)))
    out.append(("garbage_appended", blob[:-2] + bytes(rs.randint(0, 255, 64).astype(np.uint8)) + blob[-2:]))
    return out
