// Row N6: the sequential core of baseline JPEG decoding, compiled for the device (csrc/jpeg.cu) and for the host
// (tests/hostsim/jpeg_hostsim.cpp).  The target is libjpeg-turbo 3.1's default decode, bit for bit (DESIGN.md
// section 4.8): jdhuff.c's Huffman decoding, jidctint.c's jpeg_idct_islow, the upsampling jdsample.c's
// jinit_upsampler selects with do_fancy_upsampling (fancy h2v1 / h1v2 / h2v2, plain replication otherwise) and
// jdcolor.c's ycc_rgb_convert.  Integer arithmetic throughout; the IDCT wraps in 32 bits instead of overflowing.
//
//   parse        host only: the marker segments up to SOS (never the entropy-coded data) -> Header, or a refusal
//   byte_kind    unstuffing rule of one entropy-coded byte from its neighbours (data / dropped / RSTn / end)
//   step         one Huffman symbol from a decoder state (bit position, block of the MCU cycle, coefficient k)
//   walk         the symbols that start in [st.pos, end): the transition of one subsequence, counting blocks
//   write_sub    the same, writing the coefficients and DC differences of the blocks that start there
//   idct_islow   dequantisation + islow IDCT + range limit of one 8 x 8 block
//   pixel        upsampling + colour conversion of one output pixel
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define JHD __host__ __device__ __forceinline__
#else
#define JHD inline
#endif

#if defined(VPK_JPEG_CHECKS) && defined(__CUDA_ARCH__)
#include <assert.h>
#define JPEG_CHECK(c) assert(c)
#else
#define JPEG_CHECK(c) ((void)0)
#endif

namespace vpk {
namespace jpeg {

// support / status codes: the VPK_JPEG_* values of include/vpk.h
enum {
    OK = 0, PROGRESSIVE = 1, ARITHMETIC = 2, PRECISION = 3, COLOR = 4, LAYOUT = 5, MALFORMED = 6, LOSSLESS = 7,
    CORRUPT = 8
};

static constexpr int kMaxComp = 3, kMaxBlocks = 10, kFastBits = 9;

// Huffman table in decoding form: codes of up to 9 bits by direct lookup on the next 9 bits ((length << 8) |
// symbol, 0: longer or invalid), longer codes by length (maxcode / valoff as in jdhuff.c's d_derived_tbl)
struct HuffTab {
    uint16_t fast[1 << kFastBits];
    int32_t maxcode[18];
    int32_t valoff[18];
    uint8_t val[256];
};

#if defined(__CUDACC__)
static __constant__ uint8_t kNaturalDev[64] = {
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
#endif
static const uint8_t kNaturalHost[64] = {
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

JHD int natural(int k) {
#if defined(__CUDA_ARCH__)
    return kNaturalDev[k];
#else
    return kNaturalHost[k];
#endif
}

// ---- per-photo geometry (host-built, read by the kernels) ------------------------------------------------------
struct Geom {
    int32_t w, h, nc, bpm;          // size, components, blocks per MCU (1 for a gray, non-interleaved scan)
    int32_t hmax, vmax, mcux;       // MCUs per row (blocks per row for gray)
    int32_t restart;                // MCUs per restart interval (0: the whole scan is one interval)
    int32_t ch[kMaxComp], cv[kMaxComp];         // sampling factors (1 for gray)
    int32_t bw[kMaxComp], bh[kMaxComp];         // block grid of each component (whole MCUs)
    int32_t dw[kMaxComp], dh[kMaxComp];         // downsampled_width / _height
    int32_t qt[kMaxComp];                        // quantisation table of each component
    int8_t slot_comp[kMaxBlocks], slot_dx[kMaxBlocks], slot_dy[kMaxBlocks], slot_dc[kMaxBlocks], slot_ac[kMaxBlocks];
    int64_t coef[kMaxComp];         // first block of each component grid in the coefficient array
    int64_t dc[kMaxComp];           // first entry of each component's DC array (decoding order)
    int64_t plane[kMaxComp];        // byte offset of each component's sample plane (bw * 8 x bh * 8)
    int64_t pix;                    // byte offset of the decoded photo (h x w x nc)
    int64_t mcus;                   // MCUs of the scan
    int32_t ival0, nival;           // first restart interval (global index), intervals of the scan
};

// ---- host: marker parser -------------------------------------------------------------------------------------
struct Header {
    int support = MALFORMED;
    int w = 0, h = 0, nc = 0, restart = 0;
    int hmax = 1, vmax = 1;
    int id[4] = {0, 0, 0, 0}, hs[4] = {0, 0, 0, 0}, vs[4] = {0, 0, 0, 0}, tq[4] = {0, 0, 0, 0};
    int scan_comp[4] = {0, 0, 0, 0}, td[4] = {0, 0, 0, 0}, ta[4] = {0, 0, 0, 0};     // in scan order
    int16_t q[4][64];               // natural order, as ISLOW_MULT_TYPE (short)
    HuffTab tab[8];                 // DC 0..3, AC 4..7
    int64_t ecs = 0;                // byte offset of the entropy-coded data
};

inline int build_huff(const uint8_t* counts, const uint8_t* vals, bool dc, HuffTab& t) {
    memset(&t, 0, sizeof(t));
    int n = 0;
    for (int l = 1; l <= 16; ++l) n += counts[l];
    if (n > 256) return MALFORMED;
    for (int i = 0; i < n; ++i) {
        if (dc && vals[i] > 15) return MALFORMED;           // jdhuff.c: DC symbols above 15 are a bad table
        t.val[i] = vals[i];
    }
    int32_t code = 0, p = 0;
    for (int l = 1; l <= 16; ++l) {
        t.valoff[l] = p - code;
        for (int i = 0; i < counts[l]; ++i, ++p, ++code) {
            if (l <= kFastBits) {
                const int span = 1 << (kFastBits - l);
                for (int x = 0; x < span; ++x) t.fast[(code << (kFastBits - l)) + x] = (uint16_t)(l << 8 | vals[p]);
            }
        }
        t.maxcode[l] = counts[l] ? code - 1 : -1;
        if (code > (1 << l)) return MALFORMED;             // jdhuff.c: code >= 1 << si after the length
        code <<= 1;
    }
    t.maxcode[17] = 0x7fffffff;
    return OK;
}

// Parses SOI .. SOS.  Returns the support code (OK or a refusal) and fills h; reads only inside d[0, n).
inline int parse(const uint8_t* d, int64_t n, Header& h) {
    h = Header();
    uint8_t counts[8][17], vals[8][256];
    bool have_q[4] = {false, false, false, false}, have_t[8] = {false, false, false, false, false, false, false, false};
    bool sof = false, jfif = false, adobe = false;
    int adobe_transform = -1;
    int64_t p = 2;
    if (n < 4 || d[0] != 0xFF || d[1] != 0xD8) return h.support = MALFORMED;
    for (;;) {
        if (p >= n || d[p] != 0xFF) return h.support = MALFORMED;
        while (p < n && d[p] == 0xFF) ++p;                  // fill bytes
        if (p >= n) return h.support = MALFORMED;
        const int m = d[p++];
        if (m == 0x01 || (m >= 0xD0 && m <= 0xD7)) continue;        // standalone markers
        if (m == 0xD8 || m == 0xD9 || m == 0x00) return h.support = MALFORMED;
        if (p + 2 > n) return h.support = MALFORMED;
        const int len = d[p] << 8 | d[p + 1];
        if (len < 2 || p + len > n) return h.support = MALFORMED;
        const uint8_t* s = d + p + 2;
        const int L = len - 2;
        p += len;
        if (m == 0xC2) return h.support = PROGRESSIVE;
        if (m == 0xC3 || m == 0xC5 || m == 0xC6 || m == 0xC7 || m == 0xDE || m == 0xDF) return h.support = LOSSLESS;
        if ((m >= 0xC9 && m <= 0xCB) || (m >= 0xCD && m <= 0xCF) || m == 0xCC) return h.support = ARITHMETIC;
        if (m == 0xC0 || m == 0xC1) {
            if (sof || L < 6) return h.support = MALFORMED;
            sof = true;
            if (s[0] != 8) return h.support = PRECISION;
            h.h = s[1] << 8 | s[2];
            h.w = s[3] << 8 | s[4];
            h.nc = s[5];
            if (L != 6 + 3 * h.nc || h.nc == 0) return h.support = MALFORMED;
            if (h.nc == 4) return h.support = COLOR;
            if (h.nc != 1 && h.nc != 3) return h.support = LAYOUT;
            if (h.w == 0) return h.support = MALFORMED;
            if (h.h == 0) return h.support = LAYOUT;                // height from a DNL marker
            for (int c = 0; c < h.nc; ++c) {
                h.id[c] = s[6 + 3 * c];
                h.hs[c] = s[7 + 3 * c] >> 4;
                h.vs[c] = s[7 + 3 * c] & 15;
                h.tq[c] = s[8 + 3 * c];
                if (h.hs[c] < 1 || h.hs[c] > 4 || h.vs[c] < 1 || h.vs[c] > 4 || h.tq[c] > 3) return h.support = MALFORMED;
                for (int e = 0; e < c; ++e)
                    if (h.id[e] == h.id[c]) return h.support = MALFORMED;
            }
        } else if (m == 0xC4) {
            int o = 0;
            while (o < L) {
                if (o + 17 > L) return h.support = MALFORMED;
                const int tc = s[o] >> 4, th = s[o] & 15;
                if (tc > 1 || th > 3) return h.support = MALFORMED;
                const int k = tc * 4 + th;
                int tot = 0;
                counts[k][0] = 0;
                for (int l = 1; l <= 16; ++l) { counts[k][l] = s[o + l]; tot += s[o + l]; }
                if (tot > 256 || o + 17 + tot > L) return h.support = MALFORMED;
                memcpy(vals[k], s + o + 17, tot);
                have_t[k] = true;
                o += 17 + tot;
            }
        } else if (m == 0xDB) {
            int o = 0;
            while (o < L) {
                const int pq = s[o] >> 4, tq = s[o] & 15;
                if (pq > 1 || tq > 3 || o + 1 + 64 * (pq + 1) > L) return h.support = MALFORMED;
                for (int k = 0; k < 64; ++k) {
                    const int v = pq ? (s[o + 1 + 2 * k] << 8 | s[o + 2 + 2 * k]) : s[o + 1 + k];
                    h.q[tq][kNaturalHost[k]] = (int16_t)(uint16_t)v;
                }
                have_q[tq] = true;
                o += 1 + 64 * (pq + 1);
            }
        } else if (m == 0xDD) {
            if (L != 2) return h.support = MALFORMED;
            h.restart = s[0] << 8 | s[1];
        } else if (m == 0xE0) {
            if (L >= 5 && s[0] == 'J' && s[1] == 'F' && s[2] == 'I' && s[3] == 'F' && s[4] == 0) jfif = true;
        } else if (m == 0xEE) {
            if (L >= 12 && s[0] == 'A' && s[1] == 'd' && s[2] == 'o' && s[3] == 'b' && s[4] == 'e') { adobe = true; adobe_transform = s[11]; }
        } else if (m == 0xDC) {
            return h.support = MALFORMED;                   // DNL before the scan
        } else if (m == 0xDA) {
            if (!sof || L < 1) return h.support = MALFORMED;
            const int ns = s[0];
            if (L != 4 + 2 * ns) return h.support = MALFORMED;
            if (ns != h.nc) return h.support = LAYOUT;      // a scan without every component: a multi-scan file
            bool seen[4] = {false, false, false, false};
            for (int i = 0; i < ns; ++i) {
                int c = -1;
                for (int e = 0; e < h.nc; ++e)
                    if (h.id[e] == s[1 + 2 * i]) c = e;
                if (c < 0 || seen[c]) return h.support = MALFORMED;
                seen[c] = true;
                h.scan_comp[i] = c;
                h.td[i] = s[2 + 2 * i] >> 4;
                h.ta[i] = s[2 + 2 * i] & 15;
                if (h.td[i] > 3 || h.ta[i] > 3) return h.support = MALFORMED;
            }
            if (s[1 + 2 * ns] != 0 || s[2 + 2 * ns] != 63 || s[3 + 2 * ns] != 0) return h.support = MALFORMED;
            // colour space as jdapimin.c's default_decompress_parms decides it
            if (h.nc == 3) {
                if (!jfif && adobe && adobe_transform == 0) return h.support = COLOR;
                if (!jfif && !adobe && h.id[0] == 82 && h.id[1] == 71 && h.id[2] == 66) return h.support = COLOR;
            }
            for (int c = 0; c < h.nc; ++c)
                if (!have_q[h.tq[c]]) return h.support = MALFORMED;
            for (int i = 0; i < ns; ++i) {
                if (!have_t[h.td[i]] || !have_t[4 + h.ta[i]]) return h.support = MALFORMED;
                if (build_huff(counts[h.td[i]], vals[h.td[i]], true, h.tab[h.td[i]]) != OK) return h.support = MALFORMED;
                if (build_huff(counts[4 + h.ta[i]], vals[4 + h.ta[i]], false, h.tab[4 + h.ta[i]]) != OK) return h.support = MALFORMED;
            }
            if (h.nc == 1) {
                h.hs[0] = h.vs[0] = 1;                       // a non-interleaved scan: one block per MCU
            } else {
                for (int c = 0; c < 3; ++c) { h.hmax = h.hmax > h.hs[c] ? h.hmax : h.hs[c]; h.vmax = h.vmax > h.vs[c] ? h.vmax : h.vs[c]; }
                int bpm = 0;
                for (int c = 0; c < 3; ++c) {
                    if (h.hmax % h.hs[c] || h.vmax % h.vs[c]) return h.support = LAYOUT;
                    bpm += h.hs[c] * h.vs[c];
                }
                if (bpm > kMaxBlocks) return h.support = MALFORMED;
            }
            h.ecs = p;
            return h.support = OK;
        }
        // APPn, COM and anything else with a length: skipped
    }
}

// geometry of a supported header; coef / dc / plane / pix bases and the first interval are the caller's
inline void make_geom(const Header& h, Geom& g) {
    memset(&g, 0, sizeof(g));
    g.w = h.w; g.h = h.h; g.nc = h.nc; g.restart = h.restart;
    g.hmax = h.hmax; g.vmax = h.vmax;
    const int mw = 8 * h.hmax, mh = 8 * h.vmax;
    g.mcux = (h.w + mw - 1) / mw;
    const int mcuy = (h.h + mh - 1) / mh;
    g.mcus = (int64_t)g.mcux * mcuy;
    g.bpm = 0;
    for (int i = 0; i < h.nc; ++i) {
        const int c = h.scan_comp[i];
        for (int dy = 0; dy < h.vs[c]; ++dy)
            for (int dx = 0; dx < h.hs[c]; ++dx) {
                g.slot_comp[g.bpm] = (int8_t)c; g.slot_dx[g.bpm] = (int8_t)dx; g.slot_dy[g.bpm] = (int8_t)dy;
                g.slot_dc[g.bpm] = (int8_t)h.td[i]; g.slot_ac[g.bpm] = (int8_t)h.ta[i];
                ++g.bpm;
            }
    }
    for (int c = 0; c < h.nc; ++c) {
        g.ch[c] = h.hs[c]; g.cv[c] = h.vs[c]; g.qt[c] = h.tq[c];
        g.bw[c] = g.mcux * h.hs[c]; g.bh[c] = mcuy * h.vs[c];
        g.dw[c] = (int)(((int64_t)h.w * h.hs[c] + h.hmax - 1) / h.hmax);
        g.dh[c] = (int)(((int64_t)h.h * h.vs[c] + h.vmax - 1) / h.vmax);
    }
    g.nival = h.restart ? (int32_t)((g.mcus + h.restart - 1) / h.restart) : 1;
}

// blocks, DC entries and plane bytes one photo needs
inline int64_t geom_blocks(const Geom& g) { int64_t n = 0; for (int c = 0; c < g.nc; ++c) n += (int64_t)g.bw[c] * g.bh[c]; return n; }
inline int64_t geom_plane_bytes(const Geom& g) { return 64 * geom_blocks(g); }

// lays out component arrays from the given bases (blocks, DC entries, bytes)
inline void geom_place(Geom& g, int64_t coef0, int64_t plane0, int64_t pix0, int32_t ival0) {
    for (int c = 0; c < g.nc; ++c) {
        g.coef[c] = coef0; g.dc[c] = coef0; g.plane[c] = plane0;
        coef0 += (int64_t)g.bw[c] * g.bh[c];
        plane0 += 64 * (int64_t)g.bw[c] * g.bh[c];
    }
    g.pix = pix0;
    g.ival0 = ival0;
}

// MCUs of interval r of the scan
JHD int64_t ival_mcus(const Geom& g, int64_t r) {
    if (!g.restart) return g.mcus;
    const int64_t a = r * g.restart, b = a + g.restart < g.mcus ? a + g.restart : g.mcus;
    return b - a;
}

// ---- entropy-coded data ----------------------------------------------------------------------------------------
enum { BYTE_DROP = 0, BYTE_DATA = 1, BYTE_RST = 2, BYTE_END = 3 };

// jdmarker.c / jdhuff.c's reading of one byte of the entropy-coded segment given its neighbours (-1: none).
// FF 00 is a data FF (the 00 is dropped); FF before FF or a marker code is a fill byte; a marker code after FF
// is RSTn (interval boundary) or ends the data.
JHD int byte_kind(int prev, int cur, int next) {
    if (prev == 0xFF && cur != 0xFF) {
        if (cur == 0x00) return BYTE_DROP;
        return (cur >= 0xD0 && cur <= 0xD7) ? BYTE_RST : BYTE_END;
    }
    if (cur == 0xFF) return next == 0x00 ? BYTE_DATA : BYTE_DROP;
    return BYTE_DATA;
}

// one restart interval: its bytes (unstuffed) in 32-bit words, first byte in the high bits after bswap.  The words
// past nbits hold 0xFF bytes, and reads past the last word return ones.
struct Stream {
    const uint32_t* w;
    uint32_t nwords, nbits;
};

JHD uint32_t bswap32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, 0, 0x0123);
#else
    return __builtin_bswap32(x);
#endif
}

JHD uint32_t word_at(const Stream& s, uint32_t i) { return i < s.nwords ? bswap32(s.w[i]) : 0xFFFFFFFFu; }

JHD uint32_t peek32(const Stream& s, uint32_t pos) {
    const uint32_t i = pos >> 5, o = pos & 31;
    const uint32_t a = word_at(s, i);
    return o ? (a << o) | (word_at(s, i + 1) >> (32 - o)) : a;
}

// decoder state at a symbol boundary: bit position in the interval, block of the MCU cycle and coefficient k
// (0: the DC symbol is next)
struct State {
    uint32_t pos, bk;               // bk = block << 8 | k
};
JHD bool same(const State& a, const State& b) { return a.pos == b.pos && a.bk == b.bk; }

// the symbol of the code at the head of `bits`; -1 (length 16) if no code matches
JHD int huff(const HuffTab& t, uint32_t bits, int& len) {
    const uint32_t f = t.fast[bits >> (32 - kFastBits)];
    if (f) { len = (int)(f >> 8); return (int)(f & 255); }
    for (int l = kFastBits + 1; l <= 16; ++l) {
        const int32_t c = (int32_t)(bits >> (32 - l));
        if (c <= t.maxcode[l]) { len = l; return t.val[(c + t.valoff[l]) & 255]; }
    }
    len = 16;
    return -1;
}

// HUFF_EXTEND
JHD int extend(uint32_t r, int s) { return r < (1u << (s - 1)) ? (int)r - (1 << s) + 1 : (int)r; }

// One symbol from st: the DC difference (k == 0) or one AC run / size, with its magnitude bits.  coef (the block's
// 64 coefficients, natural order) and dcdiff may be NULL.  Returns 1 if the data is inconsistent here (no such
// code, a size or run out of range); the state still advances deterministically (an unknown code takes 16 bits and
// ends the block), so decoding from any state always makes progress.
JHD int step(const Stream& s, const HuffTab* tabs, const Geom& g, State& st, int16_t* coef, int32_t* dcdiff) {
    const uint32_t blk = st.bk >> 8;
    uint32_t k = st.bk & 255;
    const uint32_t bits = peek32(s, st.pos);
    int len, err = 0;
    if (k == 0) {
        int sym = huff(tabs[g.slot_dc[blk]], bits, len);
        if (sym < 0 || sym > 11) { err = 1; sym = 0; }
        const int v = sym ? extend(peek32(s, st.pos + len) >> (32 - sym), sym) : 0;
        st.pos += len + sym;
        if (dcdiff) *dcdiff = v;
        st.bk = blk << 8 | 1;
        return err;
    }
    const int sym = huff(tabs[4 + g.slot_ac[blk]], bits, len);
    if (sym < 0) {
        err = 1; k = 64; st.pos += len;
    } else {
        const int r = sym >> 4, sz = sym & 15;
        if (sz) {
            k += r;
            if (k > 63 || sz > 10) {
                err = 1; k = 64;
            } else {
                if (coef) coef[natural((int)k)] = (int16_t)extend(peek32(s, st.pos + len) >> (32 - sz), sz);
                ++k;
            }
            st.pos += len + sz;
        } else {
            k = r == 15 ? k + 16 : 64;                      // ZRL, or EOB
            st.pos += len;
        }
    }
    st.bk = k >= 64 ? ((blk + 1) % (uint32_t)g.bpm) << 8 : (blk << 8 | k);
    return err;
}

// The transition of one subsequence: decodes every symbol that starts before `end` (a block begun earlier is
// continued, a block begun here may run past `end`'s symbol boundary only in the next call).  Returns the number
// of blocks whose DC symbol starts here.
JHD int32_t walk(const Stream& s, const HuffTab* tabs, const Geom& g, State& st, uint32_t end) {
    int32_t n = 0;
    while (st.pos < end) {
        n += (st.bk & 255) == 0;
        step(s, tabs, g, st, nullptr, nullptr);
    }
    return n;
}

// where block `slot` of MCU `mcu` goes: component, coefficient block index and DC entry index
JHD int place(const Geom& g, int64_t mcu, int slot, int64_t* coef, int64_t* dc) {
    const int c = g.slot_comp[slot];
    const int64_t my = mcu / g.mcux, mx = mcu - my * g.mcux;
    const int64_t bx = mx * g.ch[c] + g.slot_dx[slot], by = my * g.cv[c] + g.slot_dy[slot];
    *coef = g.coef[c] + by * g.bw[c] + bx;
    *dc = g.dc[c] + mcu * (g.ch[c] * g.cv[c]) + g.slot_dy[slot] * g.ch[c] + g.slot_dx[slot];
    return c;
}

// The decode of one subsequence from its true start state st: the rest of a block begun in the previous one is
// skipped (its starter writes it), then every block that starts before `end` is decoded to its end.  Block m
// (interval-local, from the scan of the walk counts) of the `expected` ones writes its coefficients into coef and
// its DC difference and segment key into dcd / keys; blocks past `expected` (the padding bits) are not written.
// The block that ends the interval stores its end position in *last_end.  Returns 1 if a written block is
// inconsistent.
JHD int write_sub(const Stream& s, const HuffTab* tabs, const Geom& g, State st, uint32_t end, int64_t m, int64_t expected,
                  int64_t mcu0, int32_t key, int16_t* coef, int32_t* dcd, int32_t* keys, uint32_t* last_end, int64_t n_coef,
                  int64_t n_dc) {
    int err = 0;
    while ((st.bk & 255) != 0) step(s, tabs, g, st, nullptr, nullptr);
    while (st.pos < end) {
        const bool real = m < expected;
        int16_t* cb = nullptr;
        int32_t* dp = nullptr;
        if (real) {
            const int64_t mcu = mcu0 + m / g.bpm;
            int64_t ci, di;
            const int c = place(g, mcu, (int)(m % g.bpm), &ci, &di);
            JPEG_CHECK(ci >= 0 && ci < n_coef && di >= 0 && di < n_dc);
            (void)n_coef; (void)n_dc;
            cb = coef + ci * 64;
            dp = dcd + di;
            keys[di] = key * kMaxComp + c;
            err |= (int)((st.bk >> 8) != (uint32_t)(m % g.bpm));
        }
        do {
            const int e = step(s, tabs, g, st, cb, dp);
            if (real) err |= e;
        } while ((st.bk & 255) != 0);
        if (real && st.pos > s.nbits) err = 1;          // the block ran past the data
        if (m == expected - 1) *last_end = st.pos;
        ++m;
    }
    return err;
}

// ---- IDCT (jidctint.c, jpeg_idct_islow) -------------------------------------------------------------------------
// The range-limit table of jdmaster.c's prepare_range_limit_table, indexed by (x & 1023) with x = sample - 128
JHD int range_limit(uint32_t x) {
    const int i = (int)(x & 1023);
    return i < 128 ? i + 128 : i < 512 ? 255 : i < 896 ? 0 : i - 896;
}

// wrapping 32-bit arithmetic (what the 32-bit SIMD lanes of libjpeg-turbo compute; no overflow for valid data)
typedef uint32_t W;
JHD int32_t descale(W x, int n) { return (int32_t)(x + (1u << (n - 1))) >> n; }

// coef: 64 coefficients, natural order (coef[0] the DC value); q: quantisation table, natural order
JHD void idct_islow(const int16_t* coef, const int16_t* q, uint8_t* out, int64_t stride) {
    const W F0298 = 2446, F0390 = 3196, F0541 = 4433, F0765 = 6270, F0899 = 7373, F1175 = 9633, F1501 = 12299,
            F1847 = 15137, F1961 = 16069, F2053 = 16819, F2562 = 20995, F3072 = 25172;
    int32_t ws[64];
    for (int c = 0; c < 8; ++c) {
        W in[8];
        for (int r = 0; r < 8; ++r) in[r] = (W)((int32_t)coef[8 * r + c] * (int32_t)q[8 * r + c]);
        if (!(in[1] | in[2] | in[3] | in[4] | in[5] | in[6] | in[7])) {
            const int32_t dc = (int32_t)(in[0] << 2);
            for (int r = 0; r < 8; ++r) ws[8 * r + c] = dc;
            continue;
        }
        W z1 = (in[2] + in[6]) * F0541;
        W tmp2 = z1 - in[6] * F1847;
        W tmp3 = z1 + in[2] * F0765;
        W tmp0 = (in[0] + in[4]) << 13;
        W tmp1 = (in[0] - in[4]) << 13;
        const W t10 = tmp0 + tmp3, t13 = tmp0 - tmp3, t11 = tmp1 + tmp2, t12 = tmp1 - tmp2;
        tmp0 = in[7]; tmp1 = in[5]; tmp2 = in[3]; tmp3 = in[1];
        z1 = tmp0 + tmp3;
        W z2 = tmp1 + tmp2, z3 = tmp0 + tmp2, z4 = tmp1 + tmp3;
        const W z5 = (z3 + z4) * F1175;
        tmp0 *= F0298; tmp1 *= F2053; tmp2 *= F3072; tmp3 *= F1501;
        z1 *= (W)0 - F0899; z2 *= (W)0 - F2562; z3 *= (W)0 - F1961; z4 *= (W)0 - F0390;
        z3 += z5; z4 += z5;
        tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
        ws[8 * 0 + c] = descale(t10 + tmp3, 11);
        ws[8 * 7 + c] = descale(t10 - tmp3, 11);
        ws[8 * 1 + c] = descale(t11 + tmp2, 11);
        ws[8 * 6 + c] = descale(t11 - tmp2, 11);
        ws[8 * 2 + c] = descale(t12 + tmp1, 11);
        ws[8 * 5 + c] = descale(t12 - tmp1, 11);
        ws[8 * 3 + c] = descale(t13 + tmp0, 11);
        ws[8 * 4 + c] = descale(t13 - tmp0, 11);
    }
    for (int r = 0; r < 8; ++r) {
        const int32_t* w = ws + 8 * r;
        uint8_t* o = out + r * stride;
        if (!(w[1] | w[2] | w[3] | w[4] | w[5] | w[6] | w[7])) {
            const uint8_t v = (uint8_t)range_limit((W)descale((W)w[0], 5));
            for (int c = 0; c < 8; ++c) o[c] = v;
            continue;
        }
        W z2 = (W)w[2], z3 = (W)w[6];
        W z1 = (z2 + z3) * F0541;
        W tmp2 = z1 - z3 * F1847;
        W tmp3 = z1 + z2 * F0765;
        W tmp0 = ((W)w[0] + (W)w[4]) << 13;
        W tmp1 = ((W)w[0] - (W)w[4]) << 13;
        const W t10 = tmp0 + tmp3, t13 = tmp0 - tmp3, t11 = tmp1 + tmp2, t12 = tmp1 - tmp2;
        tmp0 = (W)w[7]; tmp1 = (W)w[5]; tmp2 = (W)w[3]; tmp3 = (W)w[1];
        z1 = tmp0 + tmp3; z2 = tmp1 + tmp2; z3 = tmp0 + tmp2;
        W z4 = tmp1 + tmp3;
        const W z5 = (z3 + z4) * F1175;
        tmp0 *= F0298; tmp1 *= F2053; tmp2 *= F3072; tmp3 *= F1501;
        z1 *= (W)0 - F0899; z2 *= (W)0 - F2562; z3 *= (W)0 - F1961; z4 *= (W)0 - F0390;
        z3 += z5; z4 += z5;
        tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
        o[0] = (uint8_t)range_limit((W)descale(t10 + tmp3, 18));
        o[7] = (uint8_t)range_limit((W)descale(t10 - tmp3, 18));
        o[1] = (uint8_t)range_limit((W)descale(t11 + tmp2, 18));
        o[6] = (uint8_t)range_limit((W)descale(t11 - tmp2, 18));
        o[2] = (uint8_t)range_limit((W)descale(t12 + tmp1, 18));
        o[5] = (uint8_t)range_limit((W)descale(t12 - tmp1, 18));
        o[3] = (uint8_t)range_limit((W)descale(t13 + tmp0, 18));
        o[4] = (uint8_t)range_limit((W)descale(t13 - tmp0, 18));
    }
}

// ---- upsampling (jdsample.c) and colour conversion (jdcolor.c) ---------------------------------------------------
// sample of component c at output pixel (x, y); p: the component's plane, row stride bw[c] * 8
JHD int upsample(const Geom& g, int c, const uint8_t* p, int x, int y) {
    const int64_t st = (int64_t)g.bw[c] * 8;
    const int hx = g.hmax / g.ch[c], vy = g.vmax / g.cv[c], dw = g.dw[c], dh = g.dh[c];
    if (hx == 1 && vy == 1) return p[y * st + x];
    if (hx == 1 && vy == 2) {                                   // h1v2_fancy_upsample
        const int r = y >> 1, odd = y & 1;
        const int r2 = odd ? (r + 1 < dh ? r + 1 : dh - 1) : (r > 0 ? r - 1 : 0);
        return (3 * p[r * st + x] + p[r2 * st + x] + (odd ? 2 : 1)) >> 2;
    }
    if (hx == 2 && vy == 1 && dw > 2) {                         // h2v1_fancy_upsample
        const int i = x >> 1;
        const uint8_t* row = p + y * st;
        if (!(x & 1)) return i == 0 ? row[0] : (3 * row[i] + row[i - 1] + 1) >> 2;
        return i == dw - 1 ? row[i] : (3 * row[i] + row[i + 1] + 2) >> 2;
    }
    if (hx == 2 && vy == 2 && dw > 2) {                         // h2v2_fancy_upsample
        const int r = y >> 1, odd = y & 1, i = x >> 1;
        const int r2 = odd ? (r + 1 < dh ? r + 1 : dh - 1) : (r > 0 ? r - 1 : 0);
        const uint8_t* a = p + r * st;
        const uint8_t* b = p + r2 * st;
        const int cs = 3 * a[i] + b[i];
        if (!(x & 1)) return i == 0 ? (cs * 4 + 8) >> 4 : (3 * cs + 3 * a[i - 1] + b[i - 1] + 8) >> 4;
        return i == dw - 1 ? (cs * 4 + 7) >> 4 : (3 * cs + 3 * a[i + 1] + b[i + 1] + 7) >> 4;
    }
    return p[(int64_t)(y / vy) * st + x / hx];                  // h2v1 / h2v2 / int_upsample: replication
}

JHD int clamp255(int v) { return v < 0 ? 0 : v > 255 ? 255 : v; }

// ycc_rgb_convert with build_ycc_rgb_table's entries (SCALEBITS 16)
JHD void ycc_rgb(int y, int cb, int cr, uint8_t* out) {
    const int32_t x_cb = cb - 128, x_cr = cr - 128;
    const int32_t ONE_HALF = 1 << 15;
    const int32_t cr_r = (91881 * x_cr + ONE_HALF) >> 16;           // FIX(1.40200)
    const int32_t cb_b = (116130 * x_cb + ONE_HALF) >> 16;          // FIX(1.77200)
    const int32_t g = (-46802 * x_cr + (-22554 * x_cb + ONE_HALF)) >> 16;   // FIX(0.71414), FIX(0.34414)
    out[0] = (uint8_t)clamp255(y + cr_r);
    out[1] = (uint8_t)clamp255(y + g);
    out[2] = (uint8_t)clamp255(y + cb_b);
}

// output pixel (x, y) of a photo whose planes start at `planes` (g.plane[] relative to it): nc bytes at out
JHD void pixel(const Geom& g, const uint8_t* planes, int x, int y, uint8_t* out) {
    const int Y = upsample(g, 0, planes + g.plane[0], x, y);
    if (g.nc == 1) { out[0] = (uint8_t)Y; return; }
    ycc_rgb(Y, upsample(g, 1, planes + g.plane[1], x, y), upsample(g, 2, planes + g.plane[2], x, y), out);
}

}  // namespace jpeg
}  // namespace vpk
