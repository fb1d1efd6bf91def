// Row N7: the sequential core of PNG decoding, compiled for the device (csrc/png.cu) and for the host
// (tests/hostsim/png_hostsim.cpp).  The target is libpng's decode of 8-bit and lower files, bit for bit (DESIGN.md
// section 4.9): zlib's inflate with its verdicts on damaged streams, the five PNG predictors, Adam7 and the bit-depth
// and palette expansion.  Integer code throughout.
//
//   parse        host only: the chunk walk (chunk headers, IHDR and PLTE; never the IDAT payloads) -> Header, or a refusal
//   crc_*        CRC-32 of a byte range and zlib's crc32_combine (the GF(2) shift), for the IDAT chunks
//   Reader       the bit buffer over a file's IDAT payloads, read in place through the chunk list
//   huff_*       canonical Huffman tables: zlib's inflate_table checks, sorted symbols, a 9-bit lookup table
//   next_event   the inflate state machine up to its next event: 32 staged literals, a match, new tables, the end
//   unfilter     the five predictors
//   adam7_*      the Adam7 pass geometry (empty passes of tiny images included)
//   expand       bit depth, palette and alpha of one output pixel
#pragma once
#include <stdint.h>
#include <string.h>
#include <vector>

#if defined(__CUDACC__)
#define PHD __host__ __device__ __forceinline__
#else
#define PHD inline
#endif

#if defined(VPK_PNG_CHECKS) && defined(__CUDA_ARCH__)
#include <assert.h>
#define PNG_CHECK(c) assert(c)
#else
#define PNG_CHECK(c) ((void)0)
#endif

namespace vpk {
namespace png {

// support / status codes: the VPK_PNG_* values of include/vpk.h
enum { OK = 0, NOT_PNG = 1, DEPTH = 2, MALFORMED = 3, CORRUPT = 4 };

static constexpr int kFast = 9;                 // bits of the direct lookup table
static constexpr int kMaxLit = 288, kMaxDist = 32, kStage = 32;
static constexpr uint32_t kAdlerMod = 65521;

// ---- CRC-32 (PNG chunks) --------------------------------------------------------------------------------------
PHD uint32_t crc_entry(uint32_t n) {
    uint32_t c = n;
    for (int k = 0; k < 8; ++k) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
    return c;
}
// CRC-32 of n bytes (tab: the 256 crc_entry values)
PHD uint32_t crc_bytes(const uint32_t* tab, const uint8_t* p, int64_t n) {
    uint32_t c = 0xFFFFFFFFu;
    for (int64_t i = 0; i < n; ++i) c = tab[(c ^ p[i]) & 255] ^ (c >> 8);
    return ~c;
}
// a * b modulo the CRC polynomial (zlib's multmodp, reflected)
PHD uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}
// x^(8 n) modulo the polynomial: the shift of a CRC over n zero bytes
PHD uint32_t x8nmodp(int64_t n) {
    uint32_t p = 1u << 31, sq = 1u << 23;       // x^0, x^8
    while (n) {
        if (n & 1) p = multmodp(sq, p);
        sq = multmodp(sq, sq);
        n >>= 1;
    }
    return p;
}
// zlib's crc32_combine: the CRC of A || B from crc(A), crc(B) and |B|
PHD uint32_t crc_combine(uint32_t ca, uint32_t cb, int64_t nb) { return multmodp(x8nmodp(nb), ca) ^ cb; }

// ---- geometry ------------------------------------------------------------------------------------------------
PHD int channels(int ctype) { return ctype == 2 ? 3 : ctype == 4 ? 2 : ctype == 6 ? 4 : 1; }
PHD int out_channels(int ctype) { return (ctype == 0 || ctype == 4) ? 1 : 3; }
PHD int64_t row_bytes(int64_t w, int bitspp) { return (w * bitspp + 7) >> 3; }
// Adam7 pass p (0..6): first column / row and steps, packed 4 bits per pass
PHD int a7_x0(int p) { return (0x0102040 >> (4 * p)) & 15; }
PHD int a7_y0(int p) { return (0x1020400 >> (4 * p)) & 15; }
PHD int a7_dx(int p) { return (0x1224488 >> (4 * p)) & 15; }
PHD int a7_dy(int p) { return (0x2244888 >> (4 * p)) & 15; }
// columns / rows of pass p of a w x h image (0 for an empty pass)
PHD int64_t a7_size(int64_t n, int o, int d) { return n > o ? (n - o + d - 1) / d : 0; }
// the pass a pixel of an interlaced image belongs to
PHD int adam7_pass_of(int x, int y) {
    if ((y & 7) == 0 && (x & 7) == 0) return 0;
    if ((y & 7) == 0 && (x & 7) == 4) return 1;
    if ((y & 7) == 4 && (x & 3) == 0) return 2;
    if ((y & 3) == 0 && (x & 3) == 2) return 3;
    if ((y & 3) == 2 && (x & 1) == 0) return 4;
    if ((y & 1) == 0) return 5;
    return 6;
}

// per-file geometry (host-built, read by the kernels)
struct Geom {
    int32_t w, h, depth, ctype, bitspp, bpp, npass, npal;   // bpp: bytes per complete pixel (>= 1) for the predictors
    int32_t pw[7], ph[7];           // pixels of each pass (one pass, the image, if not interlaced)
    int64_t rb[7];                  // row bytes of each pass (without the filter byte)
    int64_t poff[7];                // offset of each pass's first filtered scanline in the file's scanline buffer
    int64_t raw;                    // filtered scanline bytes of the image (inflate's output)
    int64_t scan;                   // offset of the file's scanline buffer in the call's buffer
    int64_t pix;                    // offset of the decoded photo (h x w x out_channels)
    int32_t interlace, nidat, idat0, pad_;     // IDAT chunks: [idat0, idat0 + nidat) of the call's chunk list
};

PHD void make_passes(Geom& g) {
    g.raw = 0;
    for (int p = 0; p < 7; ++p) { g.pw[p] = g.ph[p] = 0; g.rb[p] = 0; g.poff[p] = 0; }
    g.npass = g.interlace ? 7 : 1;
    for (int p = 0; p < g.npass; ++p) {
        g.pw[p] = g.interlace ? (int32_t)a7_size(g.w, a7_x0(p), a7_dx(p)) : g.w;
        g.ph[p] = g.interlace ? (int32_t)a7_size(g.h, a7_y0(p), a7_dy(p)) : g.h;
        g.rb[p] = row_bytes(g.pw[p], g.bitspp);
        g.poff[p] = g.raw;
        if (g.pw[p] && g.ph[p]) g.raw += (1 + g.rb[p]) * g.ph[p];
    }
}

// ---- host: the chunk walk ------------------------------------------------------------------------------------
struct Header {
    int support = NOT_PNG;
    int w = 0, h = 0, depth = 0, ctype = 0, interlace = 0, npal = 0;
    uint8_t pal[768];
    std::vector<int64_t> idat;      // per IDAT chunk: offset of its payload, its length
};

inline uint32_t be32(const uint8_t* p) { return (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | p[3]; }

inline const uint32_t* host_crc_table() {
    static uint32_t t[256];
    static bool init = false;
    if (!init) { for (int i = 0; i < 256; ++i) t[i] = crc_entry(i); init = true; }
    return t;
}

// the zlib header: deflate, a window of at most 32 K, a valid check, no preset dictionary
inline bool zlib_header_ok(int cmf, int flg) {
    return (cmf & 15) == 8 && (cmf >> 4) <= 7 && ((cmf << 8) | flg) % 31 == 0 && !(flg & 0x20);
}

// Walks the chunks of one file; reads IHDR, PLTE and the first two payload bytes of the IDAT run (the zlib header).
inline int parse(const uint8_t* d, int64_t n, Header& hd) {
    hd = Header();
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
    if (n < 8 || memcmp(d, sig, 8) != 0) return hd.support = NOT_PNG;
    hd.support = MALFORMED;
    int64_t p = 8;
    bool have_ihdr = false, have_plte = false, idat_done = false, in_idat = false;
    const uint32_t* tab = host_crc_table();
    for (;;) {
        if (p + 12 > n) return MALFORMED;                       // truncated: no IEND
        const uint32_t len = be32(d + p);
        const uint8_t* t = d + p + 4;
        if (len > 0x7FFFFFFFu || p + 12 + (int64_t)len > n) return MALFORMED;
        for (int k = 0; k < 4; ++k)
            if (!((t[k] >= 'A' && t[k] <= 'Z') || (t[k] >= 'a' && t[k] <= 'z'))) return MALFORMED;
        const bool is_idat = !memcmp(t, "IDAT", 4);
        if (!have_ihdr && memcmp(t, "IHDR", 4)) return MALFORMED;
        if (in_idat && !is_idat) { in_idat = false; idat_done = true; }
        if (!memcmp(t, "IHDR", 4)) {
            if (have_ihdr || len != 13 || crc_bytes(tab, t, 17) != be32(t + 17)) return MALFORMED;
            const uint8_t* q = t + 4;
            const uint32_t w = be32(q), h = be32(q + 4);
            const int depth = q[8], ct = q[9];
            if (w == 0 || h == 0 || w > 0x7FFFFFFFu || h > 0x7FFFFFFFu || q[10] || q[11] || q[12] > 1) return MALFORMED;
            const bool okd = (ct == 0 && (depth == 1 || depth == 2 || depth == 4 || depth == 8 || depth == 16)) ||
                             ((ct == 2 || ct == 4 || ct == 6) && (depth == 8 || depth == 16)) ||
                             (ct == 3 && (depth == 1 || depth == 2 || depth == 4 || depth == 8));
            if (!okd) return MALFORMED;
            hd.w = (int)w; hd.h = (int)h; hd.depth = depth; hd.ctype = ct; hd.interlace = q[12];
            have_ihdr = true;
        } else if (!memcmp(t, "PLTE", 4)) {
            if (have_plte || !hd.idat.empty()) return MALFORMED;
            if (hd.ctype == 3) {                                // elsewhere libpng ignores a bad PLTE; so does this decoder
                if (len == 0 || len > 768 || len % 3 || crc_bytes(tab, t, 4 + len) != be32(t + 4 + len)) return MALFORMED;
                hd.npal = (int)(len / 3);
                memcpy(hd.pal, t + 4, len);
            }
            have_plte = true;
        } else if (is_idat) {
            if (idat_done) return MALFORMED;                    // IDAT chunks must be consecutive
            if (hd.ctype == 3 && !have_plte) return MALFORMED;
            hd.idat.push_back(p + 8);
            hd.idat.push_back(len);
            in_idat = true;
        } else if (!memcmp(t, "IEND", 4)) {
            break;
        } else if (!(t[0] & 0x20)) {
            return MALFORMED;                                   // an unknown critical chunk
        }
        p += 12 + len;
    }
    if (hd.idat.empty()) return MALFORMED;
    int zh[2], k = 0;
    for (size_t c = 0; c < hd.idat.size() && k < 2; c += 2)
        for (int64_t i = 0; i < hd.idat[c + 1] && k < 2; ++i) zh[k++] = d[hd.idat[c] + i];
    if (k < 2 || !zlib_header_ok(zh[0], zh[1])) return MALFORMED;
    if (hd.ctype != 3) hd.npal = 0;
    return hd.support = hd.depth == 16 ? DEPTH : OK;
}

inline void make_geom(const Header& hd, Geom& g) {
    memset(&g, 0, sizeof(g));
    g.w = hd.w; g.h = hd.h; g.depth = hd.depth; g.ctype = hd.ctype; g.interlace = hd.interlace; g.npal = hd.npal;
    g.bitspp = channels(hd.ctype) * hd.depth;
    g.bpp = g.bitspp >= 8 ? g.bitspp / 8 : 1;
    g.nidat = (int32_t)(hd.idat.size() / 2);
    make_passes(g);
}

// ---- the bit buffer over the IDAT payloads ---------------------------------------------------------------------
struct Reader {
    const uint8_t* f;               // the file
    const int64_t* idat;            // (payload offset, length) per chunk
    int32_t n, ci;                  // chunks, current chunk
    int64_t pos;                    // next byte in the current chunk
    uint64_t buf;
    int32_t cnt, pad;               // bits in buf; zero bytes fed past the end of the stream

    PHD int next_byte() {
        while (ci < n && pos >= idat[2 * ci + 1]) { ++ci; pos = 0; }
        if (ci >= n) { ++pad; return 0; }
        return f[idat[2 * ci] + pos++];
    }
    PHD void fill() { while (cnt <= 56) { buf |= (uint64_t)next_byte() << cnt; cnt += 8; } }
    PHD uint32_t bits(int k) const { return (uint32_t)(buf & ((1ull << k) - 1)); }
    PHD void drop(int k) { buf >>= k; cnt -= k; }
    PHD bool over() const { return cnt < 8 * pad; }      // a bit past the end of the stream was consumed
};

PHD void reader_init(Reader& r, const uint8_t* f, const int64_t* idat, int n) {
    r.f = f; r.idat = idat; r.n = n; r.ci = 0; r.pos = 0; r.buf = 0; r.cnt = 0; r.pad = 0;
    r.fill();
    r.drop(16);                     // the zlib header (checked on the host)
}

// ---- canonical Huffman tables ---------------------------------------------------------------------------------
enum { CODES = 0, LENS = 1, DISTS = 2 };

struct Huff {
    uint16_t count[16];             // codes of each length
    uint16_t sym[kMaxLit];          // symbols sorted by (length, value)
    uint16_t fast[1 << kFast];      // next kFast bits -> (length << 9) | symbol; 0: longer or invalid
};

// zlib's inflate_table verdict on a set of code lengths: 0 usable, -1 over-subscribed or incomplete (an incomplete
// set is allowed for a literal / length or distance code of a single code of length 1)
PHD int huff_check(const uint16_t* count, int type) {
    int max = 15;
    while (max >= 1 && count[max] == 0) --max;
    if (max == 0) return type == CODES ? -1 : 0;   // no codes: the first use of the code fails (CODES: never usable)
    int left = 1;
    for (int l = 1; l <= 15; ++l) {
        left <<= 1;
        left -= count[l];
        if (left < 0) return -1;
    }
    if (left > 0 && (type == CODES || max != 1)) return -1;
    return 0;
}

// puff.c's canonical decode of the code in the low bits of `v` (LSB first); -1 if no code matches within `maxlen`
PHD int huff_slow(const Huff& t, uint32_t v, int maxlen, int& used) {
    int code = 0, first = 0, index = 0;
    for (int l = 1; l <= maxlen; ++l) {
        code |= (v >> (l - 1)) & 1;
        const int c = t.count[l];
        if (code - first < c) { used = l; return t.sym[index + code - first]; }
        index += c;
        first += c;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}

PHD uint16_t fast_entry(const Huff& t, int e) {
    int used = 0;
    const int s = huff_slow(t, (uint32_t)e, kFast, used);
    return s < 0 ? 0 : (uint16_t)(used << 9 | s);
}

PHD int huff_decode(const Huff& t, uint32_t v, int& used) {
    const uint16_t f = t.fast[v & ((1u << kFast) - 1)];
    if (f) { used = f >> 9; return f & 511; }
    return huff_slow(t, v, 15, used);
}

// the sequential build (host tables, and lane 0's code-length code): counts, zlib's checks, sorted symbols, and
// with `fast` the lookup table; returns 0 or -1
PHD int huff_build(const uint8_t* lens, int n, int type, Huff& t, bool fast) {
    for (int l = 0; l < 16; ++l) t.count[l] = 0;
    for (int s = 0; s < n; ++s) t.count[lens[s]]++;
    t.count[0] = 0;
    if (huff_check(t.count, type)) return -1;
    uint16_t offs[16];
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + t.count[l];
    for (int s = 0; s < n; ++s)
        if (lens[s]) t.sym[offs[lens[s]]++] = (uint16_t)s;
    if (fast)
        for (int e = 0; e < (1 << kFast); ++e) t.fast[e] = fast_entry(t, e);
    return 0;
}

// ---- inflate up to the next event ------------------------------------------------------------------------------
enum { M_HEADER = 0, M_STORED = 1, M_CODES = 2, M_CHECK = 3, M_DONE = 4 };
enum { EV_FLUSH = 0, EV_MATCH = 1, EV_TABLES = 2, EV_END = 3, EV_ERROR = 4 };

struct Inflate {
    int32_t mode, last;
    uint32_t stored_left;
    int32_t nlen, ndist;            // EV_TABLES: literal / length and distance code lengths in lens[0..nlen + ndist)
    int32_t mlen, mdist;            // EV_MATCH
    uint32_t adler;                 // EV_END: the stream's Adler-32
    int32_t nstage;                 // staged literals
};

PHD void inflate_init(Inflate& s) { s.mode = M_HEADER; s.last = 0; s.stored_left = 0; s.nstage = 0; s.nlen = s.ndist = 0; }

// one literal / length symbol and its match: 0 literal (len = byte), 1 match, 2 end of block, -1 invalid
PHD int lz_step(const Huff& lit, const Huff& dist, Reader& r, int& len, int& d) {
    r.fill();
    int used = 0;
    const int s = huff_decode(lit, r.bits(15), used);
    if (s < 0) return -1;
    r.drop(used);
    if (s < 256) { len = s; return 0; }
    if (s == 256) return 2;
    if (s > 285) return -1;
    int base, extra;
    if (s < 265) { base = s - 254; extra = 0; }
    else if (s == 285) { base = 258; extra = 0; }
    else { const int i = s - 261; extra = i >> 2; base = ((4 + (i & 3)) << extra) + 3; }
    len = base + (int)r.bits(extra);
    r.drop(extra);
    const int ds = huff_decode(dist, r.bits(15), used);
    if (ds < 0 || ds > 29) return -1;
    r.drop(used);
    if (ds < 4) { base = ds + 1; extra = 0; }
    else { extra = (ds >> 1) - 1; base = ((2 + (ds & 1)) << extra) + 1; }
    d = base + (int)r.bits(extra);
    r.drop(extra);
    return 1;
}

// Runs the decoder until an event: EV_FLUSH (kStage literals staged), EV_MATCH (mlen, mdist; literals may be staged
// before it), EV_TABLES (a block's code lengths in lens; cl: scratch for the code-length code), EV_END (the stream
// ended; staged literals remain to flush; adler read), EV_ERROR.  pos: bytes output so far, for the distance check.
PHD int next_event(Inflate& s, Reader& r, const Huff& lit, const Huff& dist, Huff& cl, uint8_t* stage, uint8_t* lens, int64_t pos) {
    for (;;) {
        if (r.over()) return EV_ERROR;
        if (s.mode == M_HEADER) {
            r.fill();
            s.last = (int)r.bits(1);
            const int type = (int)(r.bits(3) >> 1);
            r.drop(3);
            if (type == 0) {
                r.drop(r.cnt & 7);
                r.fill();
                const uint32_t len = r.bits(16), nlen = (uint32_t)(r.buf >> 16) & 0xFFFF;
                r.drop(32);
                if (len != (~nlen & 0xFFFF)) return EV_ERROR;
                s.stored_left = len;
                s.mode = M_STORED;
                continue;
            }
            if (type == 3) return EV_ERROR;
            s.mode = M_CODES;
            if (type == 1) {
                for (int i = 0; i < 288; ++i) lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
                for (int i = 0; i < 32; ++i) lens[288 + i] = 5;
                s.nlen = 288; s.ndist = 32;
                return EV_TABLES;
            }
            // dynamic: the code-length code, then the lengths of both codes
            const int nlen = (int)r.bits(5) + 257, ndist = (int)(r.bits(10) >> 5) + 1, ncode = (int)(r.bits(14) >> 10) + 4;
            r.drop(14);
            if (nlen > 286 || ndist > 30) return EV_ERROR;
            const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
            uint8_t cll[19];
            for (int i = 0; i < 19; ++i) cll[i] = 0;
            for (int i = 0; i < ncode; ++i) {
                r.fill();
                cll[order[i]] = (uint8_t)r.bits(3);
                r.drop(3);
            }
            if (huff_build(cll, 19, CODES, cl, false)) return EV_ERROR;
            int have = 0;
            while (have < nlen + ndist) {
                r.fill();
                int used = 0;
                const int sym = huff_slow(cl, r.bits(15), 7, used);
                if (sym < 0) return EV_ERROR;
                r.drop(used);
                if (sym < 16) { lens[have++] = (uint8_t)sym; continue; }
                int rep, val = 0;
                if (sym == 16) {
                    if (have == 0) return EV_ERROR;
                    val = lens[have - 1];
                    rep = 3 + (int)r.bits(2); r.drop(2);
                } else if (sym == 17) { rep = 3 + (int)r.bits(3); r.drop(3); }
                else { rep = 11 + (int)r.bits(7); r.drop(7); }
                if (have + rep > nlen + ndist) return EV_ERROR;
                while (rep--) lens[have++] = (uint8_t)val;
            }
            if (r.over()) return EV_ERROR;
            if (lens[256] == 0) return EV_ERROR;                  // no end-of-block code
            s.nlen = nlen; s.ndist = ndist;
            return EV_TABLES;
        }
        if (s.mode == M_STORED) {
            while (s.stored_left) {
                r.fill();
                stage[s.nstage++] = (uint8_t)r.bits(8);
                r.drop(8);
                --s.stored_left;
                if (s.nstage == kStage) { if (r.over()) return EV_ERROR; return EV_FLUSH; }
            }
            s.mode = s.last ? M_CHECK : M_HEADER;
            continue;
        }
        if (s.mode == M_CODES) {
            for (;;) {
                int len = 0, d = 0;
                const int k = lz_step(lit, dist, r, len, d);
                if (k < 0 || r.over()) return EV_ERROR;
                if (k == 0) {
                    stage[s.nstage++] = (uint8_t)len;
                    if (s.nstage == kStage) return EV_FLUSH;
                    continue;
                }
                if (k == 2) { s.mode = s.last ? M_CHECK : M_HEADER; break; }
                if ((int64_t)d > pos + s.nstage) return EV_ERROR;         // before the start of the output
                s.mlen = len; s.mdist = d;
                return EV_MATCH;
            }
            continue;
        }
        if (s.mode == M_CHECK) {
            r.drop(r.cnt & 7);
            r.fill();
            const uint32_t a = (uint32_t)r.bits(32);
            r.drop(32);
            if (r.over()) return EV_ERROR;
            s.adler = (a >> 24) | ((a >> 8) & 0xFF00) | ((a << 8) & 0xFF0000) | (a << 24);
            s.mode = M_DONE;
            return EV_END;
        }
        return EV_ERROR;
    }
}

// the match copy rule: byte k of a match of distance d at output position p comes from p - d + (k mod d), which
// is always before p, so every byte of a match can be copied independently (the periodic copy when d < length)
PHD int64_t match_src(int64_t p, int d, int k) { return p - d + (k % d); }

// Adler-32 of n more bytes from the per-segment sums s1 = sum x_i and s2 = sum (n - i) x_i
PHD void adler_add(uint32_t& a, uint32_t& b, uint32_t n, uint32_t s1, uint32_t s2) {
    b = (uint32_t)((b + (uint64_t)n * a + s2) % kAdlerMod);
    a = (a + s1) % kAdlerMod;
}

// ---- the predictors -------------------------------------------------------------------------------------------
PHD uint8_t unfilter(int f, uint8_t x, int a, int b, int c) {
    switch (f) {
        case 1: return (uint8_t)(x + a);
        case 2: return (uint8_t)(x + b);
        case 3: return (uint8_t)(x + ((a + b) >> 1));
        case 4: {
            const int p = a + b - c;
            const int pa = p > a ? p - a : a - p, pb = p > b ? p - b : b - p, pc = p > c ? p - c : c - p;
            return (uint8_t)(x + ((pa <= pb && pa <= pc) ? a : pb <= pc ? b : c));
        }
        default: return x;
    }
}

// ---- expansion ------------------------------------------------------------------------------------------------
// output pixel (x, y): where its samples are in the unfiltered scanlines (buf: the file's buffer), then gray
// (types 0, 4) or RGB (types 2, 3, 6); alpha dropped, an index beyond the palette black
PHD void expand(const Geom& g, const uint8_t* buf, const uint8_t* pal, int x, int y, uint8_t* out) {
    int p = 0, px = x, py = y;
    if (g.interlace) {
        p = adam7_pass_of(x, y);
        px = (x - a7_x0(p)) / a7_dx(p);
        py = (y - a7_y0(p)) / a7_dy(p);
    }
    const uint8_t* row = buf + g.poff[p] + (int64_t)py * (1 + g.rb[p]) + 1;
    if (g.depth < 8) {
        const int64_t bit = (int64_t)px * g.depth;
        const int v = (row[bit >> 3] >> (8 - g.depth - (int)(bit & 7))) & ((1 << g.depth) - 1);
        if (g.ctype == 0) { out[0] = (uint8_t)(v * (255 / ((1 << g.depth) - 1))); return; }
        if (v < g.npal) { out[0] = pal[3 * v]; out[1] = pal[3 * v + 1]; out[2] = pal[3 * v + 2]; }
        else { out[0] = out[1] = out[2] = 0; }
        return;
    }
    const int nc = channels(g.ctype);
    const uint8_t* s = row + (int64_t)px * nc;
    switch (g.ctype) {
        case 0: case 4: out[0] = s[0]; return;
        case 3:
            if (s[0] < g.npal) { out[0] = pal[3 * s[0]]; out[1] = pal[3 * s[0] + 1]; out[2] = pal[3 * s[0] + 2]; }
            else { out[0] = out[1] = out[2] = 0; }
            return;
        default: out[0] = s[0]; out[1] = s[1]; out[2] = s[2]; return;
    }
}

}  // namespace png
}  // namespace vpk
