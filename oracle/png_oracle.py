"""Row N7 oracle: the reference decode of 8-bit and lower PNG files and a seeded corpus of them.

The reference decode is libpng through cv2.imdecode with IMREAD_COLOR | IMREAD_IGNORE_ORIENTATION, converted to RGB,
for colour types 2, 3 and 6, and IMREAD_GRAYSCALE for the gray types 0 and 4.  PIL decodes the same bytes for a
cross-check (its own inflate and unfiltering; alpha dropped by .convert("RGB") / .convert("L")).  PNG is lossless and
fully specified, so a third reference exists for the files written here: the array they were written from (expand()).

corpus() builds files with a hand-written writer (struct + zlib + crc32) that controls every colour type and bit
depth, the filter of every row, the zlib level, strategy and window, how the stream is split over IDAT chunks,
ancillary chunks, Adam7 and palettes with tRNS and out-of-range indices; with cv2.imencode at every compression level
and strategy; and with PIL's optimize=True.  The content comes from oracle.jpeg_oracle's renderers.  refused() builds
files the decoder refuses before any device work, corrupted() damaged files it must flag VPK_PNG_CORRUPT."""
import io
import struct
import zlib

import cv2
import numpy as np
from PIL import Image

from oracle.jpeg_oracle import constant, noise, photo, primaries  # noqa: F401  (the shared renderers)

# support codes (include/vpk.h VPK_PNG_*)
OK, NOT_PNG, DEPTH, MALFORMED, CORRUPT = range(5)
SIG = b"\x89PNG\r\n\x1a\n"
CHANNELS = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}
# Adam7 passes: (x0, y0, dx, dy)
ADAM7 = [(0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)]


def color_type(blob):
    return bytes(blob)[25]


def decode(blob):
    """the reference decode: (H, W, 3) uint8 RGB for colour types 2, 3, 6; (H, W) uint8 for the gray types 0, 4;
    None where libpng fails"""
    buf = np.frombuffer(bytes(blob), np.uint8)
    if color_type(blob) in (0, 4):
        return cv2.imdecode(buf, cv2.IMREAD_GRAYSCALE)
    im = cv2.imdecode(buf, cv2.IMREAD_COLOR | cv2.IMREAD_IGNORE_ORIENTATION)
    return None if im is None else np.ascontiguousarray(im[:, :, ::-1])


def decode_pil(blob):
    im = Image.open(io.BytesIO(bytes(blob)))
    return np.asarray(im.convert("L") if color_type(blob) in (0, 4) else im.convert("RGB"))


def expand(src, ctype, depth, palette=None):
    """what a file written from `src` must decode to (the decoder's output convention)"""
    if ctype == 0:
        return (src.astype(np.int32) * (255 // ((1 << depth) - 1))).astype(np.uint8)
    if ctype == 3:
        pal = np.zeros((256, 3), np.uint8)
        pal[:len(palette)] = palette
        return pal[src]
    if ctype == 4:
        return src[:, :, 0].copy()
    return src[:, :, :3].copy()


# ---- the hand-written writer ------------------------------------------------------------------------------------

def chunk(ctype, data, crc=None):
    c = zlib.crc32(ctype + data) if crc is None else crc
    return struct.pack(">I", len(data)) + ctype + data + struct.pack(">I", c & 0xFFFFFFFF)


def pack_rows(src, ctype, depth):
    """(h, rowbytes) uint8 raw scanlines of a (h, w[, c]) sample array"""
    h, w = src.shape[:2]
    s = src.reshape(h, w * CHANNELS[ctype]).astype(np.uint8)
    if depth == 8:
        return s
    per = 8 // depth
    n = s.shape[1]
    pad = (-n) % per
    s = np.pad(s, ((0, 0), (0, pad))).reshape(h, -1, per).astype(np.uint16)
    out = np.zeros(s.shape[:2], np.uint16)
    for k in range(per):
        out |= s[:, :, k] << (8 - depth * (k + 1))
    return out.astype(np.uint8)


def paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def filter_rows(raw, bpp, filters):
    """filtered scanlines (filter byte first) of raw rows; filters: one int per row (0..4; other values are
    written as they are, unfiltered)"""
    h, n = raw.shape
    out = np.zeros((h, n + 1), np.uint8)
    r = raw.astype(np.int32)
    for y in range(h):
        f = int(filters[y])
        cur = r[y]
        up = r[y - 1] if y else np.zeros(n, np.int32)
        left = np.concatenate([np.zeros(bpp, np.int32), cur[:-bpp]]) if n else cur
        ul = np.concatenate([np.zeros(bpp, np.int32), up[:-bpp]]) if n else up
        pred = {1: left, 2: up, 3: (left + up) // 2, 4: paeth(left, up, ul)}.get(f, 0)
        out[y, 0] = f
        out[y, 1:] = (cur - pred) & 255
    return out


def filtered_stream(src, ctype, depth, interlace=0, filters="mixed", seed=0):
    """the concatenated filtered scanlines of the image (all Adam7 passes in order)"""
    bpp = max(1, CHANNELS[ctype] * depth // 8)
    rs = np.random.RandomState(seed)
    parts = []
    subs = [src] if not interlace else [src[y0::dy, x0::dx] for x0, y0, dx, dy in ADAM7]
    for sub in subs:
        if sub.shape[0] == 0 or sub.shape[1] == 0:
            continue
        raw = pack_rows(sub, ctype, depth)
        if filters == "mixed":
            f = rs.randint(0, 5, raw.shape[0])
        elif isinstance(filters, int):
            f = np.full(raw.shape[0], filters)
        else:
            f = np.asarray(filters)[:raw.shape[0]]
        parts.append(filter_rows(raw, bpp, f).reshape(-1))
    return np.concatenate(parts).tobytes() if parts else b""


def compress(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, wbits=15):
    c = zlib.compressobj(level, zlib.DEFLATED, wbits, 9, strategy)
    return c.compress(data) + c.flush()


def ihdr(w, h, depth, ctype, interlace=0):
    return chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, ctype, 0, 0, interlace))


def assemble(w, h, depth, ctype, z, interlace=0, palette=None, trns=None, idat_size=None, empty_idat=False,
             ancillary=False):
    """a PNG file around the zlib stream z"""
    out = [SIG, ihdr(w, h, depth, ctype, interlace)]
    if ancillary:
        out += [chunk(b"gAMA", struct.pack(">I", 45455)), chunk(b"tEXt", b"Comment\x00vpk test")]
    if palette is not None:
        out.append(chunk(b"PLTE", np.asarray(palette, np.uint8).tobytes()))
    if trns is not None:
        out.append(chunk(b"tRNS", bytes(trns)))
    if ancillary:
        out.append(chunk(b"pHYs", struct.pack(">IIB", 2835, 2835, 1)))
    step = len(z) if not idat_size else idat_size
    pieces = [z[i:i + step] for i in range(0, len(z), max(step, 1))] or [b""]
    for k, p in enumerate(pieces):
        if empty_idat and k % 2 == 1:
            out.append(chunk(b"IDAT", b""))
        out.append(chunk(b"IDAT", p))
    if empty_idat:
        out.append(chunk(b"IDAT", b""))
    if ancillary:
        out.append(chunk(b"tEXt", b"Author\x00after the image data"))
    out.append(chunk(b"IEND", b""))
    return b"".join(out)


def write(src, ctype, depth, palette=None, trns=None, interlace=0, filters="mixed", level=6,
          strategy=zlib.Z_DEFAULT_STRATEGY, wbits=15, idat_size=None, empty_idat=False, ancillary=False, seed=0, extra=b""):
    """a PNG file of the sample array `src` ((h, w) for types 0 and 3, (h, w, c) otherwise); `extra`: bytes
    compressed after the last row"""
    h, w = src.shape[:2]
    z = compress(filtered_stream(src, ctype, depth, interlace, filters, seed) + extra, level, strategy, wbits)
    return assemble(w, h, depth, ctype, z, interlace, palette, trns, idat_size, empty_idat, ancillary)


def samples(seed, w, h, ctype, depth):
    """a sample array with photo content, scaled to the bit depth"""
    rgb = photo(seed, w, h, texture=6) if w * h >= 256 else noise(seed, w, h)
    if ctype == 0:
        return rgb[:, :, 1] >> (8 - depth)
    if ctype == 3:
        return (rgb[:, :, 0] >> (8 - depth)).astype(np.uint8)
    if ctype == 4:
        return np.dstack([rgb[:, :, 1], rgb[:, :, 2]])
    if ctype == 6:
        return np.dstack([rgb, rgb[:, :, :1] ^ 0x5A])
    return rgb


def palette_of(seed, n):
    return np.random.RandomState(seed).randint(0, 256, (n, 3)).astype(np.uint8)


def encode_cv2(rgb, compression=3, strategy=cv2.IMWRITE_PNG_STRATEGY_DEFAULT):
    img = rgb if rgb.ndim == 2 else np.ascontiguousarray(rgb[:, :, ::-1])
    ok, buf = cv2.imencode(".png", img, [cv2.IMWRITE_PNG_COMPRESSION, compression, cv2.IMWRITE_PNG_STRATEGY, strategy])
    assert ok
    return buf.tobytes()


def encode_pil(img, **kw):
    """img: an array or a PIL image"""
    out = io.BytesIO()
    (img if isinstance(img, Image.Image) else Image.fromarray(img)).save(out, format="PNG", **kw)
    return out.getvalue()


def written():
    """[(name, blob, expected)]: the hand-written files and the arrays they must decode to"""
    out = []

    def add(name, src, ctype, depth, palette=None, **kw):
        out.append((name, write(src, ctype, depth, palette=palette, **kw), expand(src, ctype, depth, palette)))
    # every colour type and bit depth, each filter forced on every row and mixed, non-interlaced and Adam7
    for ctype, depths in ((0, (1, 2, 4, 8)), (2, (8,)), (3, (1, 2, 4, 8)), (4, (8,)), (6, (8,))):
        for depth in depths:
            for il in (0, 1):
                for f in (0, 1, 2, 3, 4, "mixed"):
                    w, h = (37, 23) if f != "mixed" else (61, 45)
                    src = samples(7 * ctype + depth + il, w, h, ctype, depth)
                    pal = palette_of(ctype + depth, 1 << depth) if ctype == 3 else None
                    add("w_t%d_d%d_i%d_f%s_%dx%d" % (ctype, depth, il, f, w, h), src, ctype, depth, pal, interlace=il,
                        filters=f, seed=depth)
    # zlib levels and strategies, window bits 9..15
    src = samples(3, 97, 71, 2, 8)
    for level in (0, 1, 6, 9):
        add("w_rgb_level%d" % level, src, 2, 8, level=level)
    for name, s in (("filtered", zlib.Z_FILTERED), ("huffman_only", zlib.Z_HUFFMAN_ONLY), ("rle", zlib.Z_RLE),
                    ("fixed", zlib.Z_FIXED)):
        add("w_rgb_strategy_%s" % name, src, 2, 8, strategy=s)
    for wb in range(9, 16):
        add("w_rgb_wbits%d" % wb, samples(4, 211, 97, 2, 8), 2, 8, wbits=wb, level=9)
    # IDAT splits
    src = samples(5, 120, 80, 6, 8)
    for size in (1, 7, 8192):
        add("w_rgba_idat%d" % size, src, 6, 8, idat_size=size)
    add("w_rgba_idat_empty_chunks", src, 6, 8, idat_size=300, empty_idat=True)
    add("w_rgba_ancillary", src, 6, 8, ancillary=True, idat_size=1000)
    # Adam7 at tiny and odd sizes (empty passes), odd widths at low bit depths
    for w, h in ((1, 1), (2, 1), (1, 2), (3, 5), (7, 9), (9, 7), (33, 17), (301, 203)):
        add("w_rgb_adam7_%dx%d" % (w, h), samples(w * 31 + h, w, h, 2, 8), 2, 8, interlace=1)
        add("w_gray1_adam7_%dx%d" % (w, h), samples(w * 17 + h, w, h, 0, 1), 0, 1, interlace=1)
    for w in (1, 3, 5, 7, 9, 13, 15, 17):
        for depth in (1, 2, 4):
            add("w_gray%d_w%d" % (depth, w), samples(w + depth, w, 11, 0, depth), 0, depth)
            add("w_pal%d_w%d_i1" % (depth, w), samples(w + depth + 1, w, 11, 3, depth), 3, depth,
                palette_of(w, 1 << depth), interlace=1)
    # palette with tRNS, short palettes (indices beyond PLTE decode to black)
    src = samples(6, 64, 48, 3, 8)
    add("w_pal8_trns", src, 3, 8, palette_of(9, 256), trns=bytes(range(0, 256, 3)))
    add("w_pal8_short_palette", src, 3, 8, palette_of(10, 100))
    add("w_pal4_short_palette_i1", samples(8, 45, 31, 3, 4), 3, 4, palette_of(11, 5), interlace=1)
    add("w_pal2_one_entry", samples(12, 19, 13, 3, 2), 3, 2, palette_of(12, 1))
    return out


def corpus(large=True):
    """[(name, blob)] of supported files; `large` adds the 2000 x 1333 and larger photos"""
    out = [(n, b) for n, b, _ in written()]
    img = photo(20, 131, 97, texture=8)
    for c in range(10):
        out.append(("cv2_rgb_c%d" % c, encode_cv2(img, c)))
    for name, s in (("filtered", cv2.IMWRITE_PNG_STRATEGY_FILTERED), ("huffman_only", cv2.IMWRITE_PNG_STRATEGY_HUFFMAN_ONLY),
                    ("rle", cv2.IMWRITE_PNG_STRATEGY_RLE), ("fixed", cv2.IMWRITE_PNG_STRATEGY_FIXED)):
        out.append(("cv2_rgb_strategy_%s" % name, encode_cv2(img, 6, s)))
    out.append(("cv2_gray", encode_cv2(img[:, :, 1])))
    out.append(("cv2_noise_640x480", encode_cv2(noise(21, 640, 480))))
    out.append(("cv2_primaries_640x480", encode_cv2(primaries(22, 640, 480))))
    out.append(("cv2_constant_640x480", encode_cv2(constant(23, 640, 480))))
    out.append(("cv2_constant_1x1", encode_cv2(constant(24, 1, 1))))
    out.append(("cv2_photo_5000x3", encode_cv2(photo(25, 5000, 3))))
    out.append(("pil_rgb_optimize", encode_pil(img, optimize=True)))
    out.append(("pil_rgba_optimize", encode_pil(np.dstack([img, img[:, :, :1]]), optimize=True)))
    out.append(("pil_gray_optimize", encode_pil(img[:, :, 0], optimize=True)))
    out.append(("pil_palette_optimize", encode_pil(Image.fromarray(img).quantize(37), optimize=True)))
    sizes = [(1200, 800), (800, 1200)] + ([(2000, 1333), (6000, 4000)] if large else [])
    for i, (w, h) in enumerate(sizes):
        out.append(("cv2_photo_%dx%d" % (w, h), encode_cv2(photo(30 + i, w, h, texture=6))))
    return out


def _chunks(blob):
    """[(offset, type, length)] of every chunk"""
    p, out = 8, []
    while p + 8 <= len(blob):
        n = struct.unpack(">I", blob[p:p + 4])[0]
        out.append((p, blob[p + 4:p + 8], n))
        p += 12 + n
    return out


def _zstream(blob):
    return b"".join(blob[p + 8:p + 8 + n] for p, t, n in _chunks(blob) if t == b"IDAT")


def _rebuild(blob, z, idat_size=None):
    """the file with its IDAT run replaced by the zlib stream z"""
    cs = _chunks(blob)
    first = next(p for p, t, _ in cs if t == b"IDAT")
    last = max(p + 12 + n for p, t, n in cs if t == b"IDAT")
    step = idat_size or max(len(z), 1)
    idats = b"".join(chunk(b"IDAT", z[i:i + step]) for i in range(0, max(len(z), 1), step))
    return blob[:first] + idats + blob[last:]


def _base():
    src = samples(40, 53, 37, 2, 8)
    return src, write(src, 2, 8)


def _zhdr(cmf, flg):
    """a zlib header with a valid check field"""
    return bytes([cmf, flg + (31 - (cmf * 256 + flg) % 31) % 31])


def refused():
    """[(name, blob, reason)] of files the decoder refuses before any device work"""
    src, base = _base()
    cs = _chunks(base)
    ip = next(p for p, t, _ in cs if t == b"IDAT")
    out = [("jpeg", bytes.fromhex("ffd8ffe000104a464946") + bytes(64), NOT_PNG), ("empty", b"", NOT_PNG),
           ("bad_signature", b"\x89PNG\r\n\x1a\x0a"[:7] + b"\x00" + base[8:], NOT_PNG)]
    out.append(("depth16_rgb", assemble(53, 37, 16, 2, compress(b"\x00" * (37 * (1 + 53 * 6)))), DEPTH))
    out.append(("depth16_gray", assemble(5, 3, 16, 0, compress(b"\x00" * (3 * 11))), DEPTH))
    for k in (8, 20, 33, ip + 4, len(base) - 20):
        out.append(("truncated_%d" % k, base[:k], MALFORMED))
    for name, (w, h, d, t, il) in (("zero_width", (0, 3, 8, 2, 0)), ("depth3", (3, 3, 3, 0, 0)), ("rgb_depth4", (3, 3, 4, 2, 0)),
                                   ("type5", (3, 3, 8, 5, 0)), ("interlace2", (3, 3, 8, 2, 2)), ("huge_width", (1 << 31, 3, 8, 2, 0))):
        out.append(("ihdr_" + name, SIG + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, d, t, 0, 0, il)) + base[33:], MALFORMED))
    b = bytearray(base); b[29] ^= 1                                 # IHDR CRC
    out.append(("ihdr_crc", bytes(b), MALFORMED))
    out.append(("no_ihdr_first", SIG + chunk(b"tEXt", b"a\x00b") + base[8:], MALFORMED))
    out.append(("no_idat", base[:ip] + chunk(b"IEND", b""), MALFORMED))
    out.append(("no_iend", base[:-12], MALFORMED))
    out.append(("unknown_critical", base[:ip] + chunk(b"ABCD", b"xyz") + base[ip:], MALFORMED))
    z = _zstream(base)
    split = _rebuild(base, z, 300)
    q = [p for p, t, _ in _chunks(split) if t == b"IDAT"][1]
    out.append(("idat_not_consecutive", split[:q] + chunk(b"tEXt", b"a\x00b") + split[q:], MALFORMED))
    out.append(("zlib_bad_method", _rebuild(base, _zhdr(0x79, 0) + z[2:]), MALFORMED))
    out.append(("zlib_fdict", _rebuild(base, _zhdr(0x78, 0x20) + z[2:]), MALFORMED))
    out.append(("zlib_window_64k", _rebuild(base, _zhdr(0x88, 0) + z[2:]), MALFORMED))
    out.append(("zlib_bad_check", _rebuild(base, bytes([0x78, 0x9D]) + z[2:]), MALFORMED))
    pal = samples(41, 20, 10, 3, 8)
    out.append(("palette_missing", write(pal, 3, 8), MALFORMED))
    pb = write(pal, 3, 8, palette_of(1, 256))
    pp = next(p for p, t, _ in _chunks(pb) if t == b"PLTE")
    b = bytearray(pb); b[pp + 8] ^= 0x40                           # PLTE payload, CRC left as it was
    out.append(("plte_crc", bytes(b), MALFORMED))
    out.append(("plte_after_idat", SIG + ihdr(20, 10, 8, 3) + chunk(b"IDAT", compress(filtered_stream(pal, 3, 8))) +
                chunk(b"PLTE", palette_of(1, 256).tobytes()) + chunk(b"IEND", b""), MALFORMED))
    out.append(("plte_length", SIG + ihdr(20, 10, 8, 3) + chunk(b"PLTE", bytes(10)) +
                chunk(b"IDAT", compress(filtered_stream(pal, 3, 8))) + chunk(b"IEND", b""), MALFORMED))
    out.append(("garbage", SIG + bytes(np.random.RandomState(1).randint(0, 256, 300).astype(np.uint8)), MALFORMED))
    return out


def _deflate_bits(bits):
    """bytes of an LSB-first bit list"""
    out = bytearray((len(bits) + 7) // 8)
    for i, b in enumerate(bits):
        out[i >> 3] |= b << (i & 7)
    return bytes(out)


def _raw_deflate(data):
    """a raw deflate stream of data in non-final blocks (a sync flush), without the zlib header and check"""
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    return c.compress(data) + c.flush(zlib.Z_SYNC_FLUSH)


def _tail(seed):
    return bytes(np.random.RandomState(seed % 1000).randint(0, 256, 777).astype(np.uint8))


def _with_stream(base, raw_deflate, adler):
    return _rebuild(base, b"\x78\x9c" + raw_deflate + struct.pack(">I", adler & 0xFFFFFFFF))


def corrupted(blob=None):
    """[(name, blob)]: files that pass the chunk walk and must decode with status VPK_PNG_CORRUPT"""
    if blob is None:
        blob = _base()[1]
    cs = _chunks(blob)
    z = _zstream(blob)
    ihdr_b = blob[16:29]
    w, h, depth, ctype, il = struct.unpack(">IIBBxxB", ihdr_b)
    out = []
    ip, _, n = next(c for c in cs if c[1] == b"IDAT")
    b = bytearray(blob); b[ip + 8 + n // 2] ^= 0x10                # IDAT payload, CRC left as it was
    out.append(("idat_payload", bytes(b)))
    b = bytearray(blob); b[ip + 8 + n] ^= 0x01                     # IDAT CRC field, payload intact
    out.append(("idat_crc", bytes(b)))
    out.append(("adler", _rebuild(blob, z[:-4] + bytes(x ^ 0xFF for x in z[-4:]))))
    out.append(("truncated_stream", _rebuild(blob, z[:len(z) // 2])))
    raw = zlib.decompress(z)
    short = compress(raw[:len(raw) // 2])
    out.append(("stream_ends_early", _rebuild(blob, short)))
    bad = bytearray(raw); bad[0] = 5                                # filter byte of the first row
    out.append(("filter_byte_5", _rebuild(blob, compress(bytes(bad)))))
    bad = bytearray(raw); bad[len(raw) - len(raw) // h] = 200       # filter byte of the last row
    out.append(("filter_byte_200_last_row", _rebuild(blob, compress(bytes(bad)))))
    ad = zlib.adler32(raw)
    # block type 3
    out.append(("block_type_3", _with_stream(blob, _deflate_bits([1, 1, 1]) + bytes(16), ad)))
    # stored block with NLEN != ~LEN
    out.append(("stored_nlen", _with_stream(blob, bytes([1, 5, 0, 0, 0]) + bytes(5), ad)))
    # dynamic block with an over-subscribed code-length code (four lengths of 1)
    bits = [1, 0, 1] + [0] * 5 + [0] * 5 + [0] * 4 + [1, 0, 0] * 4
    out.append(("oversubscribed_codelens", _with_stream(blob, _deflate_bits(bits) + bytes(32), ad)))
    # dynamic block with an incomplete code-length code (one length of 2)
    bits = [1, 0, 1] + [0] * 5 + [0] * 5 + [0] * 4 + [0, 1, 0] + [0, 0, 0] * 3
    out.append(("incomplete_codelens", _with_stream(blob, _deflate_bits(bits) + bytes(32), ad)))
    # fixed block: literal 0 then a match of length 3 at distance 2 (before the start of the output)
    lit0 = [0, 0, 1, 1, 0, 0, 0, 0]                                 # code 00110000 (literal 0), MSB first
    len3 = [0, 0, 0, 0, 0, 0, 1]                                    # code 0000001 (length symbol 257)
    dist2 = [0, 0, 0, 0, 1]                                         # distance code 1: distance 2
    out.append(("distance_too_far", _with_stream(blob, _deflate_bits([1, 1, 0] + lit0 + len3 + dist2 + [0] * 7) + bytes(8), ad)))
    # damage right after the rows, before any byte past the last row: zlib meets it in the call that writes the
    # last row, and running out of IDAT data is an error wherever it happens
    rows = _raw_deflate(raw)
    out.append(("after_rows_block_type_3", _with_stream(blob, rows + _deflate_bits([1, 1, 1]) + bytes(4), ad)))
    out.append(("after_rows_stored_nlen", _with_stream(blob, rows + bytes([1, 5, 0, 0, 0]) + bytes(5), ad)))
    out.append(("after_rows_no_final_block", _rebuild(blob, b"\x78\x9c" + rows)))
    out.append(("adler_cut", _rebuild(blob, z[:-2])))
    tail = _tail(len(raw))
    out.append(("extra_data_truncated", _rebuild(blob, compress(raw + tail)[:-30])))
    out.append(("extra_data_no_final_block", _rebuild(blob, b"\x78\x9c" + _raw_deflate(raw + tail))))
    return out


def extra_data(seed=50):
    """[(name, blob, expected)]: files libpng only warns about and decodes: data compressed after the last row (with
    a bad Adler-32 or an invalid block after it too: zlib's errors past the last row are warnings), and a PLTE chunk
    with a bad length or CRC in an RGB file"""
    out = []
    for ctype, depth, il in ((2, 8, 0), (3, 4, 1), (0, 1, 0)):
        src = samples(seed + ctype, 29, 17, ctype, depth)
        pal = palette_of(seed, 1 << depth) if ctype == 3 else None
        tail = bytes(np.random.RandomState(seed).randint(0, 256, 777).astype(np.uint8))
        out.append(("extra_t%d_d%d_i%d" % (ctype, depth, il),
                    write(src, ctype, depth, palette=pal, interlace=il, extra=tail), expand(src, ctype, depth, pal)))
    src, base = _base()
    raw = zlib.decompress(_zstream(base))
    tail = _tail(seed)
    ze = compress(raw + tail)
    out.append(("extra_bad_adler", _rebuild(base, ze[:-4] + bytes(x ^ 0xFF for x in ze[-4:])), src))
    out.append(("extra_then_block_type_3", _with_stream(base, _raw_deflate(raw + tail) + _deflate_bits([1, 1, 1]) + bytes(4),
                                                        zlib.adler32(raw + tail)), src))
    pl = write(src, 2, 8, palette=palette_of(1, 10))
    pp = next(p for p, t, _ in _chunks(pl) if t == b"PLTE")
    b = bytearray(pl); b[pp + 8] ^= 0x40
    out.append(("rgb_plte_crc", bytes(b), src))
    out.append(("rgb_plte_length", SIG + ihdr(src.shape[1], src.shape[0], 8, 2) + chunk(b"PLTE", bytes(10)) +
                chunk(b"IDAT", _zstream(base)) + chunk(b"IEND", b""), src))
    return out
