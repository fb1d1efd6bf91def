// Row N6: baseline JPEG decoding on the device, in front of photo preparation (reference evaluation.py:142-143,
// `convert`'s read of the dataset's JPEG files).  Bit for bit with libjpeg-turbo 3.1's default decode; the
// sequential pieces are csrc/jpeg_core.cuh, shared with the host build the CPU tests run.  DESIGN.md section 4.8.
//
//   host         jpeg::parse of every file's markers up to SOS (never the entropy-coded data), refusals first
//   jpeg_scan_end, jpeg_flags, (CUB scan), jpeg_bounds
//                every entropy-coded byte classified from its neighbours (jpeg::byte_kind); the data ends at the
//                first marker that is not RSTn; one 64-bit exclusive scan gives each kept byte its offset and each
//                byte its restart interval; the interval starts go back to the host (one small copy)
//   jpeg_compact each interval unstuffed into its own word-aligned bitstream
//   jpeg_sync    self-synchronising Huffman decoding (Weissenberger & Schmidt, ICPP 2018): every interval cut into
//                subsequences of L bits, one thread each, a CTA holding consecutive subsequences of one photo with its
//                tables in shared memory.  Each thread decodes its subsequence from a guessed state (block 0, k = 0)
//                and records the state at the first symbol boundary past its end.  Then, in rounds, every thread whose
//                predecessor's record changed re-decodes from that record; a thread whose new record equals the old
//                one has synchronised.  Rounds run inside the CTA to a fixpoint, then launches repeat across CTAs
//                until no CTA's incoming state changes.  The first subsequence of an interval knows its state, so
//                the fixpoint is the true decode; the worst case is sequential, never wrong.
//   (CUB scan)   blocks per subsequence -> each subsequence's first block in its interval
//   jpeg_write   the final pass from the true states: int16 coefficients in natural order, DC differences with a
//                segment key (interval, component); inconsistent data marks the photo VPK_JPEG_CORRUPT
//   jpeg_ival_check  every interval must end its last block within the final byte of its data
//   (CUB scan by key)  DC differences -> DC values, reset at every interval for every component
//   jpeg_idct    dequantisation + islow IDCT of every block into per-component planes padded to whole MCUs
//   jpeg_color   upsampling + colour conversion of every output pixel, interleaved RGB (or gray) at the photo's offset
//
// VPK_DEFINES=VPK_JPEG_CHECKS asserts every index into the bitstreams, the block arrays and the planes.
// VPK_JPEG_SUBSEQ_BITS=n (n >= 32) overrides the subsequence length (a test switch: small ones force many rounds).
#include <algorithm>
#include <cstdlib>
#include <cub/device/device_scan.cuh>
#include "vpk_internal.cuh"
#include "jpeg_core.cuh"

namespace vpk {

using jpeg::Geom;
using jpeg::HuffTab;
using jpeg::State;

static_assert(jpeg::OK == VPK_JPEG_OK && jpeg::PROGRESSIVE == VPK_JPEG_PROGRESSIVE && jpeg::ARITHMETIC == VPK_JPEG_ARITHMETIC &&
              jpeg::PRECISION == VPK_JPEG_PRECISION && jpeg::COLOR == VPK_JPEG_COLOR && jpeg::LAYOUT == VPK_JPEG_LAYOUT &&
              jpeg::MALFORMED == VPK_JPEG_MALFORMED && jpeg::LOSSLESS == VPK_JPEG_LOSSLESS && jpeg::CORRUPT == VPK_JPEG_CORRUPT,
              "jpeg_core.cuh and vpk.h disagree on the VPK_JPEG_* codes");

static constexpr int kThreads = 256;
static constexpr int kChunkBytes = 4096;        // entropy-coded bytes per CTA of the byte kernels
static constexpr int kCta = 128;                // subsequences per CTA of the decode kernels
static constexpr int kSubseqBits = 1024;        // default subsequence length
static constexpr int kPixTile = 256;            // output pixels per CTA of jpeg_color
static constexpr uint64_t kKeptMask = (1ull << 40) - 1;

struct IvalDev {
    int64_t word_off;       // first word of the interval's bitstream
    int64_t kept0;          // its first kept byte in the photo's unstuffed data
    int64_t mcu0, expected; // first MCU, blocks
    uint32_t nwords, nbits;
    int32_t img, first_sub;
};

struct JpegState {
    DBuf data, meta, end, flags, scan, ival_start, ivals, words, subs, ctas, rec, cnt, cscan, tail[2], used_in, changed,
        last_end, coef, dcd, keys, dcs, planes, pix, status, stats, cub_tmp;
    HBuf h_ival_start, h_flag;
    std::vector<jpeg::Header> hs;   // the files of the last jpeg_plan
    int64_t last_stats[4] = {0, 0, 0, 0};
};

void jpeg_free(vpk_ctx* ctx) {
    if (!ctx->jpeg) return;
    JpegState* s = ctx->jpeg;
    for (DBuf* b : {&s->data, &s->meta, &s->end, &s->flags, &s->scan, &s->ival_start, &s->ivals, &s->words, &s->subs, &s->ctas,
                    &s->rec, &s->cnt, &s->cscan, &s->tail[0], &s->tail[1], &s->used_in, &s->changed, &s->last_end, &s->coef,
                    &s->dcd, &s->keys, &s->dcs, &s->planes, &s->pix, &s->status, &s->stats, &s->cub_tmp})
        b->release();
    s->h_ival_start.release(); s->h_flag.release();
    delete s;
    ctx->jpeg = nullptr;
}

// per-photo arrays of one call on the device (all in JpegState::meta)
struct Meta {
    const Geom* g;
    const HuffTab* tabs;        // 8 per photo: DC 0..3, AC 4..7
    const int16_t* quant;       // 4 x 64 per photo, natural order
    const int64_t* src;         // byte offset of each photo's entropy-coded data in `data`
    const int64_t* ecs_off;     // B+1: its first byte in the flag / scan arrays
    const int32_t* chunk_off;   // B+1: first CTA of the byte kernels
    const int64_t* blk_off;     // B+1: first block
    const int32_t* tile_off;    // B+1: first CTA of jpeg_color
};

template <typename T>
__device__ __forceinline__ int find_image(const T* off, int B, T i) {
    int lo = 0, hi = B - 1;
    while (lo < hi) {                               // last photo with off[b] <= i
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__device__ __forceinline__ int kind_at(const uint8_t* e, int64_t i, int64_t len) {
    return jpeg::byte_kind(i ? e[i - 1] : -1, e[i], i + 1 < len ? e[i + 1] : -1);
}

// end[b] (preset to the photo's byte count) := the first marker that is not RSTn
__global__ void __launch_bounds__(kThreads) jpeg_scan_end(const uint8_t* __restrict__ data, Meta m, int B, unsigned long long* end) {
    const int b = find_image(m.chunk_off, B, (int32_t)blockIdx.x);
    const int64_t len = m.ecs_off[b + 1] - m.ecs_off[b];
    const uint8_t* e = data + m.src[b];
    const int64_t i0 = (int64_t)(blockIdx.x - m.chunk_off[b]) * kChunkBytes;
    for (int64_t i = i0 + threadIdx.x; i < len && i < i0 + kChunkBytes; i += blockDim.x)
        if (i > 0 && e[i - 1] == 0xFF && kind_at(e, i, len) == jpeg::BYTE_END) atomicMin(end + b, (unsigned long long)i);
}

// flags: kept data byte in bits 0..39, RSTn in bits 40..63 (one exclusive scan counts both)
__global__ void __launch_bounds__(kThreads) jpeg_flags(const uint8_t* __restrict__ data, Meta m, int B, const unsigned long long* __restrict__ end,
                                                       uint64_t* __restrict__ flags) {
    const int b = find_image(m.chunk_off, B, (int32_t)blockIdx.x);
    const int64_t len = m.ecs_off[b + 1] - m.ecs_off[b], stop = (int64_t)end[b];
    const uint8_t* e = data + m.src[b];
    const int64_t i0 = (int64_t)(blockIdx.x - m.chunk_off[b]) * kChunkBytes;
    for (int64_t i = i0 + threadIdx.x; i < len && i < i0 + kChunkBytes; i += blockDim.x) {
        const int k = i < stop ? kind_at(e, i, len) : jpeg::BYTE_DROP;
        flags[m.ecs_off[b] + i] = (uint64_t)(k == jpeg::BYTE_DATA) | ((uint64_t)(k == jpeg::BYTE_RST) << 40);
    }
}

// interval starts (kept bytes) from the RSTn positions, RSTn numbering and counts checked; ival_start[n_ival + b]
// receives photo b's kept bytes
__global__ void __launch_bounds__(kThreads) jpeg_bounds(const uint8_t* __restrict__ data, Meta m, int B, const unsigned long long* __restrict__ end,
                                                        const uint64_t* __restrict__ scan, int64_t* __restrict__ ival_start,
                                                        int32_t* __restrict__ status, int64_t n_ival) {
    const int b = find_image(m.chunk_off, B, (int32_t)blockIdx.x);
    const int64_t len = m.ecs_off[b + 1] - m.ecs_off[b], stop = (int64_t)end[b];
    const uint8_t* e = data + m.src[b];
    const Geom& g = m.g[b];
    const uint64_t base = scan[m.ecs_off[b]];
    const int64_t i0 = (int64_t)(blockIdx.x - m.chunk_off[b]) * kChunkBytes;
    if (blockIdx.x == (unsigned)m.chunk_off[b] && threadIdx.x == 0) {
        const uint64_t tot = scan[m.ecs_off[b] + stop] - base;
        if ((int64_t)(tot >> 40) + 1 != g.nival) atomicOr(status + b, 1 << jpeg::CORRUPT);
        JPEG_CHECK(g.ival0 < n_ival);
        ival_start[g.ival0] = 0;
        ival_start[n_ival + b] = (int64_t)(tot & kKeptMask);
    }
    for (int64_t i = i0 + threadIdx.x; i < stop && i < i0 + kChunkBytes; i += blockDim.x) {
        if (kind_at(e, i, len) != jpeg::BYTE_RST) continue;
        const uint64_t rel = scan[m.ecs_off[b] + i] - base;
        const int64_t q = (int64_t)(rel >> 40);
        if (e[i] != 0xD0 + (q & 7) || q + 1 >= g.nival) { atomicOr(status + b, 1 << jpeg::CORRUPT); continue; }
        JPEG_CHECK(g.ival0 + q + 1 < n_ival);
        ival_start[g.ival0 + q + 1] = (int64_t)(rel & kKeptMask);
    }
}

// each kept byte into its interval's bitstream
__global__ void __launch_bounds__(kThreads) jpeg_compact(const uint8_t* __restrict__ data, Meta m, int B, const unsigned long long* __restrict__ end,
                                                         const uint64_t* __restrict__ scan, const IvalDev* __restrict__ iv,
                                                         uint8_t* __restrict__ words, int64_t n_word_bytes) {
    const int b = find_image(m.chunk_off, B, (int32_t)blockIdx.x);
    const int64_t len = m.ecs_off[b + 1] - m.ecs_off[b], stop = (int64_t)end[b];
    const uint8_t* e = data + m.src[b];
    const Geom& g = m.g[b];
    const uint64_t base = scan[m.ecs_off[b]];
    const int64_t i0 = (int64_t)(blockIdx.x - m.chunk_off[b]) * kChunkBytes;
    for (int64_t i = i0 + threadIdx.x; i < stop && i < i0 + kChunkBytes; i += blockDim.x) {
        const uint64_t f = (scan[m.ecs_off[b] + i + 1] - scan[m.ecs_off[b] + i]) & kKeptMask;
        if (!f) continue;
        const uint64_t rel = scan[m.ecs_off[b] + i] - base;
        const int64_t q = (int64_t)(rel >> 40);
        if (q >= g.nival) continue;                     // past a surplus RSTn: the photo is already CORRUPT
        const IvalDev& v = iv[g.ival0 + q];
        const int64_t p = (int64_t)(rel & kKeptMask) - v.kept0;
        if (p < 0 || p >= (int64_t)v.nbits / 8) continue;
        JPEG_CHECK(v.word_off * 4 + p < n_word_bytes);
        words[v.word_off * 4 + p] = e[i];
    }
}

struct Subs {
    const int32_t* ival;        // interval of each subsequence
    const uint32_t* begin;      // its first bit in the interval
    const int32_t* cta_sub0;    // first subsequence of each CTA
    const int32_t* cta_n;       // subsequences of each CTA
    const int32_t* cta_img;     // photo of each CTA
};

__device__ __forceinline__ void load_tables(const Meta& m, int b, HuffTab* tabs, Geom* g) {
    const int4* src = reinterpret_cast<const int4*>(m.tabs + 8 * (int64_t)b);
    int4* dst = reinterpret_cast<int4*>(tabs);
    for (int i = threadIdx.x; i < (int)(8 * sizeof(HuffTab) / 16); i += blockDim.x) dst[i] = src[i];
    const int* gs = reinterpret_cast<const int*>(m.g + b);
    int* gd = reinterpret_cast<int*>(g);
    for (int i = threadIdx.x; i < (int)(sizeof(Geom) / 4); i += blockDim.x) gd[i] = gs[i];
}

__device__ __forceinline__ jpeg::Stream stream_of(const IvalDev& v, const uint32_t* words, int64_t n_words) {
    JPEG_CHECK(v.word_off + v.nwords <= n_words);
    (void)n_words;
    return jpeg::Stream{words + v.word_off, v.nwords, v.nbits};
}

// first = 1: every subsequence from its guess, then rounds to the CTA's fixpoint; first = 0: only CTAs whose
// incoming state (the previous CTA's last record, tail_in) differs from the one they used re-decode, from it.
// tail_out receives every CTA's last record; *changed is set if any CTA re-decoded.
__global__ void __launch_bounds__(kCta) jpeg_sync(Meta m, Subs sb, const IvalDev* __restrict__ iv, const uint32_t* __restrict__ words,
                                                  int64_t n_words, int L, int first, const State* __restrict__ tail_in,
                                                  State* __restrict__ tail_out, State* __restrict__ used_in, State* __restrict__ rec,
                                                  int32_t* __restrict__ cnt, int* __restrict__ changed, unsigned long long* stats) {
    __shared__ __align__(16) HuffTab tabs[8];
    __shared__ __align__(16) Geom g;
    __shared__ State sh[kCta];
    __shared__ uint8_t chg[kCta];
    const int cta = blockIdx.x, t = threadIdx.x;
    const int j0 = sb.cta_sub0[cta], n = sb.cta_n[cta], b = sb.cta_img[cta];
    State in{0, 0};
    if (!first) {
        const bool own = sb.begin[j0] == 0 || (tail_in[cta - 1].pos == used_in[cta].pos && tail_in[cta - 1].bk == used_in[cta].bk);
        if (own) {
            if (t == 0) tail_out[cta] = tail_in[cta];
            return;
        }
        in = tail_in[cta - 1];
    }
    load_tables(m, b, tabs, &g);
    const int j = j0 + t;
    const bool active = t < n;
    jpeg::Stream s{nullptr, 0, 0};
    uint32_t end = 0, begin = 0;
    if (active) {
        const IvalDev& v = iv[sb.ival[j]];
        s = stream_of(v, words, n_words);
        begin = sb.begin[j];
        end = min(v.nbits, begin + (uint32_t)L);
    }
    __syncthreads();
    int32_t my_cnt = 0;
    bool did = false;
    unsigned long long redecodes = 0;
    if (first) {
        if (active) {
            State st{begin, 0};
            my_cnt = jpeg::walk(s, tabs, g, st, end);
            sh[t] = st;
            did = true;
        }
        chg[t] = active;
        if (t == 0) used_in[cta] = State{begin, 0};
    } else {
        if (active) sh[t] = rec[j];
        bool ch = false;
        if (t == 0) {
            State st = in;
            my_cnt = jpeg::walk(s, tabs, g, st, end);
            ch = !jpeg::same(st, sh[0]);
            sh[0] = st;
            did = true;
            ++redecodes;
            used_in[cta] = in;
            *changed = 1;
        }
        chg[t] = ch;
    }
    int rounds = 0;
    for (;;) {
        __syncthreads();
        const bool work = active && t > 0 && chg[t - 1] && begin != 0;
        State st = work ? sh[t - 1] : State{0, 0};
        __syncthreads();
        bool ch = false;
        if (work) {
            my_cnt = jpeg::walk(s, tabs, g, st, end);
            ch = !jpeg::same(st, sh[t]);
            sh[t] = st;
            did = true;
            ++redecodes;
        }
        chg[t] = ch;
        if (!__syncthreads_or(ch)) break;
        ++rounds;
    }
    if (active) {
        rec[j] = sh[t];
        if (did) cnt[j] = my_cnt;
    }
    if (t == 0) tail_out[cta] = sh[n - 1];
    if (stats) {
        if (redecodes) atomicAdd(stats, redecodes);
        if (t == 0) atomicMax(stats + 1, (unsigned long long)rounds);
    }
}

// the final pass from the true start states
__global__ void __launch_bounds__(kCta) jpeg_write(Meta m, Subs sb, const IvalDev* __restrict__ iv, const uint32_t* __restrict__ words,
                                                   int64_t n_words, int L, const State* __restrict__ rec, const int32_t* __restrict__ cscan,
                                                   int16_t* __restrict__ coef, int32_t* __restrict__ dcd, int32_t* __restrict__ keys,
                                                   uint32_t* __restrict__ last_end, int32_t* __restrict__ status, int64_t n_blk) {
    __shared__ __align__(16) HuffTab tabs[8];
    __shared__ __align__(16) Geom g;
    const int cta = blockIdx.x, t = threadIdx.x;
    const int j0 = sb.cta_sub0[cta], n = sb.cta_n[cta], b = sb.cta_img[cta];
    load_tables(m, b, tabs, &g);
    __syncthreads();
    if (t >= n) return;
    const int j = j0 + t;
    const int32_t r = sb.ival[j];
    const IvalDev& v = iv[r];
    const jpeg::Stream s = stream_of(v, words, n_words);
    const uint32_t begin = sb.begin[j], end = min(v.nbits, begin + (uint32_t)L);
    const State st = begin == 0 ? State{0, 0} : rec[j - 1];
    const int64_t m0 = (int64_t)cscan[j] - cscan[v.first_sub];
    const int err = jpeg::write_sub(s, tabs, g, st, end, m0, v.expected, v.mcu0, r, coef, dcd, keys, last_end + r, n_blk, n_blk);
    if (err) atomicOr(status + b, 1 << jpeg::CORRUPT);
}

__global__ void jpeg_ival_check(const IvalDev* __restrict__ iv, int64_t n_ival, const uint32_t* __restrict__ last_end, int32_t* __restrict__ status) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_ival) return;
    const uint32_t e = last_end[r], nb = iv[r].nbits;
    if (e > nb || nb - e >= 8) atomicOr(status + iv[r].img, 1 << jpeg::CORRUPT);
}

__global__ void __launch_bounds__(kThreads) jpeg_idct(Meta m, int B, int64_t n_blk, const int16_t* __restrict__ coef, const int32_t* __restrict__ dcs,
                                                      uint8_t* __restrict__ planes, int64_t n_plane) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_blk) return;
    const int b = find_image(m.blk_off, B, i);
    const Geom& g = m.g[b];
    int c = 0;
    while (c + 1 < g.nc && i >= g.coef[c + 1]) ++c;
    const int64_t l = i - g.coef[c];
    const int by = (int)(l / g.bw[c]), bx = (int)(l - (int64_t)by * g.bw[c]);
    const int my = by / g.cv[c], mx = bx / g.ch[c];
    const int64_t di = g.dc[c] + ((int64_t)my * g.mcux + mx) * (g.ch[c] * g.cv[c]) + (by - my * g.cv[c]) * g.ch[c] + (bx - mx * g.ch[c]);
    JPEG_CHECK(di >= g.coef[c] && di < g.coef[c] + (int64_t)g.bw[c] * g.bh[c]);
    int16_t blk[64];
    const int4* src = reinterpret_cast<const int4*>(coef + i * 64);
#pragma unroll
    for (int k = 0; k < 8; ++k) reinterpret_cast<int4*>(blk)[k] = src[k];
    blk[0] = (int16_t)dcs[di];
    const int64_t st = (int64_t)g.bw[c] * 8;
    const int64_t o = g.plane[c] + (int64_t)by * 8 * st + bx * 8;
    JPEG_CHECK(o >= 0 && o + 7 * st + 8 <= n_plane);
    (void)n_plane;
    jpeg::idct_islow(blk, m.quant + ((int64_t)b * 4 + g.qt[c]) * 64, planes + o, st);
}

__global__ void __launch_bounds__(kPixTile) jpeg_color(Meta m, int B, const uint8_t* __restrict__ planes, uint8_t* __restrict__ out, int64_t n_out) {
    const int b = find_image(m.tile_off, B, (int32_t)blockIdx.x);
    const Geom& g = m.g[b];
    const int64_t p = (int64_t)(blockIdx.x - m.tile_off[b]) * kPixTile + threadIdx.x;
    if (p >= (int64_t)g.w * g.h) return;
    const int y = (int)(p / g.w), x = (int)(p - (int64_t)y * g.w);
    JPEG_CHECK(g.pix + (p + 1) * g.nc <= n_out);
    (void)n_out;
    jpeg::pixel(g, planes, x, y, out + g.pix + p * g.nc);
}

// ---- host ---------------------------------------------------------------------------------------------------------

int jpeg_parse(const uint8_t* data, const int64_t* byte_offsets, int32_t B, const char* who, std::vector<jpeg::Header>& hs) {
    if (!byte_offsets || B <= 0) { set_error("%s: bad argument", who); return VPK_ERR_ARG; }
    for (int b = 0; b < B; ++b)
        if (byte_offsets[b + 1] < byte_offsets[b] || byte_offsets[b] < 0) { set_error("%s: byte_offsets must be non-decreasing from >= 0", who); return VPK_ERR_ARG; }
    if (!data && byte_offsets[B] > byte_offsets[0]) { set_error("%s: data is NULL", who); return VPK_ERR_ARG; }
    hs.resize(B);
    for (int b = 0; b < B; ++b) jpeg::parse(data + byte_offsets[b], byte_offsets[b + 1] - byte_offsets[b], hs[b]);
    return VPK_OK;
}

static const char* reason_name(int r) {
    switch (r) {
        case VPK_JPEG_PROGRESSIVE: return "progressive";
        case VPK_JPEG_ARITHMETIC: return "arithmetic coding";
        case VPK_JPEG_PRECISION: return "not 8-bit precision";
        case VPK_JPEG_COLOR: return "colour space (CMYK, YCCK or RGB)";
        case VPK_JPEG_LAYOUT: return "layout (components, sampling or scans)";
        case VPK_JPEG_MALFORMED: return "malformed markers";
        case VPK_JPEG_LOSSLESS: return "lossless or hierarchical";
        default: return "unknown";
    }
}

int jpeg_require(const std::vector<jpeg::Header>& hs, bool rgb_only, const char* who) {
    for (size_t b = 0; b < hs.size(); ++b) {
        if (hs[b].support != jpeg::OK) {
            set_error("%s: photo %zu is not supported: reason %d (%s)", who, b, hs[b].support, reason_name(hs[b].support));
            return VPK_ERR_ARG;
        }
        if (rgb_only && hs[b].nc != 3) {
            set_error("%s: photo %zu has 1 component (gray); gray photos cannot be prepared", who, b);
            return VPK_ERR_ARG;
        }
    }
    return VPK_OK;
}

static int subseq_bits() {
    const char* e = getenv("VPK_JPEG_SUBSEQ_BITS");
    if (!e || !*e) return kSubseqBits;
    const int v = atoi(e);
    return v >= 32 ? v : kSubseqBits;
}

// packs host arrays into one device upload; returns the byte offset of each
struct Packer {
    std::vector<char> buf;
    template <typename T> size_t add(const T* p, size_t n) {
        const size_t o = (buf.size() + 15) & ~(size_t)15;
        buf.resize(o + n * sizeof(T));
        if (n) memcpy(buf.data() + o, p, n * sizeof(T));
        return o;
    }
};

int jpeg_plan(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t B, bool rgb_only, const char* who,
              std::vector<int32_t>& widths, std::vector<int32_t>& heights, std::vector<int32_t>& components) {
    if (!ctx->jpeg) ctx->jpeg = new JpegState();
    std::vector<jpeg::Header>& hs = ctx->jpeg->hs;
    VPK_TRY(jpeg_parse(data, byte_offsets, B, who, hs));
    VPK_TRY(jpeg_require(hs, rgb_only, who));
    widths.resize(B); heights.resize(B); components.resize(B);
    for (int b = 0; b < B; ++b) { widths[b] = hs[b].w; heights[b] = hs[b].h; components[b] = hs[b].nc; }
    return VPK_OK;
}

int jpeg_decode(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, const int64_t* pix_off, uint8_t* d_out, int32_t* status_out) {
    VPK_CUDA(cudaSetDevice(ctx->device));
    JpegState* s = ctx->jpeg;
    const std::vector<jpeg::Header>& hs = s->hs;
    const int B = (int)hs.size();
    cudaStream_t st = ctx->stream;
    const int L = subseq_bits();
    // geometry and layout on the host
    std::vector<Geom> geo(B);
    std::vector<HuffTab> tabs((size_t)B * 8);
    std::vector<int16_t> quant((size_t)B * 4 * 64);
    std::vector<int64_t> src(B), ecs_off(B + 1, 0), blk_off(B + 1, 0), plane_off(B + 1, 0);
    std::vector<int32_t> chunk_off(B + 1, 0), tile_off(B + 1, 0), ival_base(B + 1, 0);
    for (int b = 0; b < B; ++b) {
        const jpeg::Header& h = hs[b];
        Geom& g = geo[b];
        jpeg::make_geom(h, g);
        jpeg::geom_place(g, blk_off[b], plane_off[b], pix_off[b], ival_base[b]);
        blk_off[b + 1] = blk_off[b] + jpeg::geom_blocks(g);
        plane_off[b + 1] = plane_off[b] + jpeg::geom_plane_bytes(g);
        if ((int64_t)ival_base[b] + g.nival > INT32_MAX) { set_error("jpeg: more than 2^31 restart intervals in one call; split the batch"); return VPK_ERR_ARG; }
        ival_base[b + 1] = ival_base[b] + g.nival;
        memcpy(&tabs[(size_t)b * 8], h.tab, sizeof(h.tab));
        memcpy(&quant[(size_t)b * 256], h.q, sizeof(h.q));
        src[b] = byte_offsets[b] + h.ecs;
        const int64_t len = byte_offsets[b + 1] - src[b];
        ecs_off[b + 1] = ecs_off[b] + len;
        const int64_t nch = std::max<int64_t>(1, (len + kChunkBytes - 1) / kChunkBytes);
        const int64_t ntile = ((int64_t)g.w * g.h + kPixTile - 1) / kPixTile;
        if (chunk_off[b] + nch > INT32_MAX || tile_off[b] + ntile > INT32_MAX) { set_error("jpeg: batch too large for one call; split it"); return VPK_ERR_ARG; }
        chunk_off[b + 1] = chunk_off[b] + (int32_t)nch;
        tile_off[b + 1] = tile_off[b] + (int32_t)ntile;
    }
    const int64_t N = ecs_off[B], NI = ival_base[B], NB = blk_off[B];
    if (N >= INT32_MAX || NB > INT32_MAX || NI > INT32_MAX / jpeg::kMaxComp) { set_error("jpeg: batch too large for one call; split it"); return VPK_ERR_ARG; }
    Packer pk;
    const size_t o_g = pk.add(geo.data(), B), o_t = pk.add(tabs.data(), tabs.size()), o_q = pk.add(quant.data(), quant.size()),
                 o_src = pk.add(src.data(), B), o_ecs = pk.add(ecs_off.data(), B + 1), o_ch = pk.add(chunk_off.data(), B + 1),
                 o_blk = pk.add(blk_off.data(), B + 1), o_tile = pk.add(tile_off.data(), B + 1);
    VPK_TRY(s->meta.ensure(pk.buf.size()));
    char* mb = s->meta.as<char>();
    Meta m{reinterpret_cast<const Geom*>(mb + o_g), reinterpret_cast<const HuffTab*>(mb + o_t), reinterpret_cast<const int16_t*>(mb + o_q),
           reinterpret_cast<const int64_t*>(mb + o_src), reinterpret_cast<const int64_t*>(mb + o_ecs), reinterpret_cast<const int32_t*>(mb + o_ch),
           reinterpret_cast<const int64_t*>(mb + o_blk), reinterpret_cast<const int32_t*>(mb + o_tile)};
    const int64_t n_data = byte_offsets[B];
    VPK_TRY(s->data.ensure((size_t)std::max<int64_t>(n_data, 1)));
    VPK_TRY(s->end.ensure((size_t)B * 8));
    VPK_TRY(s->flags.ensure((size_t)(N + 1) * 8));
    VPK_TRY(s->scan.ensure((size_t)(N + 1) * 8));
    VPK_TRY(s->ival_start.ensure((size_t)(NI + B) * 8));
    VPK_TRY(s->status.ensure((size_t)B * 4));
    VPK_TRY(s->h_ival_start.ensure((size_t)(NI + B) * 8));
    VPK_TRY(s->h_flag.ensure(sizeof(int)));
    std::vector<unsigned long long> end0(B);
    for (int b = 0; b < B; ++b) end0[b] = (unsigned long long)(ecs_off[b + 1] - ecs_off[b]);
    VPK_CUDA(cudaMemcpyAsync(s->meta.p, pk.buf.data(), pk.buf.size(), cudaMemcpyHostToDevice, st));
    if (n_data) VPK_CUDA(cudaMemcpyAsync(s->data.p, data, (size_t)n_data, cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemcpyAsync(s->end.p, end0.data(), (size_t)B * 8, cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemsetAsync(s->status.p, 0, (size_t)B * 4, st));
    VPK_CUDA(cudaMemsetAsync(s->ival_start.p, 0xFF, (size_t)NI * 8, st));
    VPK_CUDA(cudaMemsetAsync(s->flags.as<uint64_t>() + N, 0, 8, st));
    const uint8_t* d_data = s->data.as<uint8_t>();
    unsigned long long* d_end = s->end.as<unsigned long long>();
    int32_t* d_status = s->status.as<int32_t>();
    const int nchunks = chunk_off[B];
    {
        KernelScope ks(ctx, "jpeg_scan_end");
        jpeg_scan_end<<<nchunks, kThreads, 0, st>>>(d_data, m, B, d_end);
        VPK_TRY(check_launch("jpeg_scan_end"));
    }
    {
        KernelScope ks(ctx, "jpeg_flags");
        jpeg_flags<<<nchunks, kThreads, 0, st>>>(d_data, m, B, d_end, s->flags.as<uint64_t>());
        VPK_TRY(check_launch("jpeg_flags"));
    }
    // CUB temporary storage for the three scans of this call
    size_t t1 = 0, t2 = 0, t3 = 0;
    VPK_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, t1, s->flags.as<uint64_t>(), s->scan.as<uint64_t>(), (int)(N + 1), st));
    {
        KernelScope ks(ctx, "jpeg_scan_bytes");
        VPK_TRY(s->cub_tmp.ensure(t1));
        VPK_CUDA(cub::DeviceScan::ExclusiveSum(s->cub_tmp.p, t1, s->flags.as<uint64_t>(), s->scan.as<uint64_t>(), (int)(N + 1), st));
    }
    {
        KernelScope ks(ctx, "jpeg_bounds");
        jpeg_bounds<<<nchunks, kThreads, 0, st>>>(d_data, m, B, d_end, s->scan.as<uint64_t>(), s->ival_start.as<int64_t>(), d_status, NI);
        VPK_TRY(check_launch("jpeg_bounds"));
    }
    // interval starts and kept totals back to the host: the subsequence layout depends on them
    int64_t* h_start = s->h_ival_start.as<int64_t>();
    const int64_t* h_tot = h_start + NI;
    VPK_CUDA(cudaMemcpyAsync(h_start, s->ival_start.p, (size_t)(NI + B) * 8, cudaMemcpyDeviceToHost, st));
    VPK_CUDA(cudaStreamSynchronize(st));
    // intervals, words, subsequences, CTAs
    std::vector<IvalDev> iv(NI);
    std::vector<int32_t> sub_ival, cta_sub0, cta_n, cta_img;
    std::vector<uint32_t> sub_begin;
    int64_t n_words = 0;
    for (int b = 0; b < B; ++b) {
        const Geom& g = geo[b];
        const int64_t sub_first = (int64_t)sub_ival.size();
        for (int r = 0; r < g.nival; ++r) {
            const int64_t k = g.ival0 + r;
            int64_t a = h_start[k] < 0 ? (int64_t)h_tot[b] : h_start[k];
            int64_t e = (int64_t)h_tot[b];
            if (r + 1 < g.nival && h_start[k + 1] >= 0) e = h_start[k + 1];
            a = std::min(a, (int64_t)h_tot[b]);
            e = std::max(a, std::min(e, (int64_t)h_tot[b]));
            if (e - a > (int64_t)(UINT32_MAX / 8)) { set_error("jpeg: photo %d: a restart interval of more than 512 MB", b); return VPK_ERR_ARG; }
            IvalDev& v = iv[k];
            v.word_off = n_words; v.kept0 = a;
            v.nbits = (uint32_t)((e - a) * 8);
            v.nwords = (uint32_t)((e - a + 3) / 4);
            v.img = b;
            v.mcu0 = g.restart ? (int64_t)r * g.restart : 0;
            v.expected = jpeg::ival_mcus(g, r) * g.bpm;
            v.first_sub = (int32_t)sub_ival.size();
            n_words += v.nwords;
            const uint32_t ns = std::max<uint32_t>(1, (uint32_t)(((uint64_t)v.nbits + L - 1) / L));
            for (uint32_t q = 0; q < ns; ++q) { sub_ival.push_back((int32_t)k); sub_begin.push_back(q * (uint32_t)L); }
        }
        const int64_t nsub = (int64_t)sub_ival.size() - sub_first;
        for (int64_t c = 0; c < nsub; c += kCta) {
            cta_sub0.push_back((int32_t)(sub_first + c));
            cta_n.push_back((int32_t)std::min<int64_t>(kCta, nsub - c));
            cta_img.push_back(b);
        }
        if ((int64_t)sub_ival.size() > INT32_MAX / 2) { set_error("jpeg: too many subsequences in one call; split the batch"); return VPK_ERR_ARG; }
    }
    const int64_t S = (int64_t)sub_ival.size();
    const int ncta = (int)cta_sub0.size();
    Packer ps;
    const size_t o_si = ps.add(sub_ival.data(), S), o_sb = ps.add(sub_begin.data(), S), o_c0 = ps.add(cta_sub0.data(), ncta),
                 o_cn = ps.add(cta_n.data(), ncta), o_ci = ps.add(cta_img.data(), ncta);
    VPK_TRY(s->subs.ensure(ps.buf.size()));
    VPK_TRY(s->ivals.ensure((size_t)NI * sizeof(IvalDev)));
    VPK_TRY(s->words.ensure((size_t)std::max<int64_t>(n_words, 1) * 4));
    VPK_TRY(s->rec.ensure((size_t)S * sizeof(State)));
    VPK_TRY(s->cnt.ensure((size_t)(S + 1) * 4));
    VPK_TRY(s->cscan.ensure((size_t)(S + 1) * 4));
    VPK_TRY(s->tail[0].ensure((size_t)ncta * sizeof(State)));
    VPK_TRY(s->tail[1].ensure((size_t)ncta * sizeof(State)));
    VPK_TRY(s->used_in.ensure((size_t)ncta * sizeof(State)));
    VPK_TRY(s->changed.ensure(sizeof(int)));
    VPK_TRY(s->last_end.ensure((size_t)NI * 4));
    VPK_TRY(s->coef.ensure((size_t)NB * 128));
    VPK_TRY(s->dcd.ensure((size_t)NB * 4));
    VPK_TRY(s->keys.ensure((size_t)NB * 4));
    VPK_TRY(s->dcs.ensure((size_t)NB * 4));
    VPK_TRY(s->planes.ensure((size_t)plane_off[B]));
    VPK_TRY(s->stats.ensure(2 * sizeof(unsigned long long)));
    char* sbp = s->subs.as<char>();
    Subs sb{reinterpret_cast<const int32_t*>(sbp + o_si), reinterpret_cast<const uint32_t*>(sbp + o_sb), reinterpret_cast<const int32_t*>(sbp + o_c0),
            reinterpret_cast<const int32_t*>(sbp + o_cn), reinterpret_cast<const int32_t*>(sbp + o_ci)};
    VPK_CUDA(cudaMemcpyAsync(s->subs.p, ps.buf.data(), ps.buf.size(), cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemcpyAsync(s->ivals.p, iv.data(), (size_t)NI * sizeof(IvalDev), cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemsetAsync(s->words.p, 0xFF, (size_t)std::max<int64_t>(n_words, 1) * 4, st));
    VPK_CUDA(cudaMemsetAsync(s->stats.p, 0, 2 * sizeof(unsigned long long), st));
    const IvalDev* d_iv = s->ivals.as<IvalDev>();
    const uint32_t* d_words = s->words.as<uint32_t>();
    {
        KernelScope ks(ctx, "jpeg_compact");
        jpeg_compact<<<nchunks, kThreads, 0, st>>>(d_data, m, B, d_end, s->scan.as<uint64_t>(), d_iv, s->words.as<uint8_t>(), n_words * 4);
        VPK_TRY(check_launch("jpeg_compact"));
    }
    unsigned long long* d_stats = ctx->profiling ? s->stats.as<unsigned long long>() : nullptr;
    {
        KernelScope ks(ctx, "jpeg_sync");
        jpeg_sync<<<ncta, kCta, 0, st>>>(m, sb, d_iv, d_words, n_words, L, 1, nullptr, s->tail[0].as<State>(), s->used_in.as<State>(),
                                         s->rec.as<State>(), s->cnt.as<int32_t>(), s->changed.as<int>(), d_stats);
        VPK_TRY(check_launch("jpeg_sync"));
    }
    int cur = 0;
    int64_t global_rounds = 0;
    int* h_changed = reinterpret_cast<int*>(s->h_flag.p);
    for (;;) {
        VPK_CUDA(cudaMemsetAsync(s->changed.p, 0, sizeof(int), st));
        {
            KernelScope ks(ctx, "jpeg_sync");
            jpeg_sync<<<ncta, kCta, 0, st>>>(m, sb, d_iv, d_words, n_words, L, 0, s->tail[cur].as<State>(), s->tail[cur ^ 1].as<State>(),
                                             s->used_in.as<State>(), s->rec.as<State>(), s->cnt.as<int32_t>(), s->changed.as<int>(), d_stats);
            VPK_TRY(check_launch("jpeg_sync"));
        }
        cur ^= 1;
        VPK_CUDA(cudaMemcpyAsync(h_changed, s->changed.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        VPK_CUDA(cudaStreamSynchronize(st));
        if (!*h_changed) break;
        ++global_rounds;
    }
    // first block of every subsequence within its interval
    VPK_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, t2, s->cnt.as<int32_t>(), s->cscan.as<int32_t>(), (int)S, st));
    VPK_CUDA(cub::DeviceScan::InclusiveSumByKey(nullptr, t3, s->keys.as<int32_t>(), s->dcd.as<int32_t>(), s->dcs.as<int32_t>(), (int)NB,
                                                cub::Equality(), st));
    VPK_TRY(s->cub_tmp.ensure(std::max(t2, t3)));
    {
        KernelScope ks(ctx, "jpeg_scan_blocks");
        VPK_CUDA(cub::DeviceScan::ExclusiveSum(s->cub_tmp.p, t2, s->cnt.as<int32_t>(), s->cscan.as<int32_t>(), (int)S, st));
    }
    VPK_CUDA(cudaMemsetAsync(s->coef.p, 0, (size_t)NB * 128, st));
    VPK_CUDA(cudaMemsetAsync(s->dcd.p, 0, (size_t)NB * 4, st));
    VPK_CUDA(cudaMemsetAsync(s->keys.p, 0xFF, (size_t)NB * 4, st));
    VPK_CUDA(cudaMemsetAsync(s->last_end.p, 0xFF, (size_t)NI * 4, st));
    {
        KernelScope ks(ctx, "jpeg_write");
        jpeg_write<<<ncta, kCta, 0, st>>>(m, sb, d_iv, d_words, n_words, L, s->rec.as<State>(), s->cscan.as<int32_t>(), s->coef.as<int16_t>(),
                                          s->dcd.as<int32_t>(), s->keys.as<int32_t>(), s->last_end.as<uint32_t>(), d_status, NB);
        VPK_TRY(check_launch("jpeg_write"));
    }
    {
        KernelScope ks(ctx, "jpeg_ival_check");
        jpeg_ival_check<<<(unsigned)((NI + kThreads - 1) / kThreads), kThreads, 0, st>>>(d_iv, NI, s->last_end.as<uint32_t>(), d_status);
        VPK_TRY(check_launch("jpeg_ival_check"));
    }
    {
        KernelScope ks(ctx, "jpeg_scan_dc");
        VPK_CUDA(cub::DeviceScan::InclusiveSumByKey(s->cub_tmp.p, t3, s->keys.as<int32_t>(), s->dcd.as<int32_t>(), s->dcs.as<int32_t>(), (int)NB,
                                                    cub::Equality(), st));
    }
    {
        KernelScope ks(ctx, "jpeg_idct");
        jpeg_idct<<<(unsigned)((NB + kThreads - 1) / kThreads), kThreads, 0, st>>>(m, B, NB, s->coef.as<int16_t>(), s->dcs.as<int32_t>(),
                                                                                    s->planes.as<uint8_t>(), plane_off[B]);
        VPK_TRY(check_launch("jpeg_idct"));
    }
    {
        KernelScope ks(ctx, "jpeg_color");
        jpeg_color<<<tile_off[B], kPixTile, 0, st>>>(m, B, s->planes.as<uint8_t>(), d_out, pix_off[B]);
        VPK_TRY(check_launch("jpeg_color"));
    }
    std::vector<int32_t> stat(B);
    VPK_CUDA(cudaMemcpyAsync(stat.data(), d_status, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    unsigned long long hs2[2] = {0, 0};
    VPK_CUDA(cudaMemcpyAsync(hs2, s->stats.p, sizeof(hs2), cudaMemcpyDeviceToHost, st));
    VPK_CUDA(cudaStreamSynchronize(st));
    for (int b = 0; b < B; ++b) status_out[b] = stat[b] ? jpeg::CORRUPT : jpeg::OK;
    s->last_stats[0] = S; s->last_stats[1] = (int64_t)hs2[0]; s->last_stats[2] = (int64_t)hs2[1]; s->last_stats[3] = global_rounds;
    return VPK_OK;
}

}  // namespace vpk

using namespace vpk;

extern "C" {

int vpk_jpeg_info(const uint8_t* data, const int64_t* byte_offsets, int32_t n, int32_t* widths, int32_t* heights, int32_t* components,
                  int32_t* support) {
    std::vector<jpeg::Header> hs;
    VPK_TRY(jpeg_parse(data, byte_offsets, n, "vpk_jpeg_info", hs));
    for (int b = 0; b < n; ++b) {
        if (widths) widths[b] = hs[b].w;
        if (heights) heights[b] = hs[b].h;
        if (components) components[b] = hs[b].nc;
        if (support) support[b] = hs[b].support;
    }
    return VPK_OK;
}

int vpk_decode_jpegs(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t n, uint8_t* pixels_out, int32_t* status_out) {
    if (!ctx || !pixels_out || !status_out) { set_error("vpk_decode_jpegs: bad argument"); return VPK_ERR_ARG; }
    std::vector<int32_t> w, h, nc;
    VPK_TRY(jpeg_plan(ctx, data, byte_offsets, n, false, "vpk_decode_jpegs", w, h, nc));
    std::vector<int64_t> pix_off(n + 1, 0);
    for (int b = 0; b < n; ++b) pix_off[b + 1] = pix_off[b] + (int64_t)w[b] * h[b] * nc[b];
    VPK_CUDA(cudaSetDevice(ctx->device));
    VPK_TRY(ctx->jpeg->pix.ensure((size_t)std::max<int64_t>(pix_off[n], 1)));
    VPK_TRY(jpeg_decode(ctx, data, byte_offsets, pix_off.data(), ctx->jpeg->pix.as<uint8_t>(), status_out));
    VPK_CUDA(cudaMemcpyAsync(pixels_out, ctx->jpeg->pix.p, (size_t)pix_off[n], cudaMemcpyDeviceToHost, ctx->stream));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    return VPK_OK;
}

int vpk_jpeg_stats(vpk_ctx* ctx, int64_t* out) {
    if (!ctx || !out) { set_error("vpk_jpeg_stats: bad argument"); return VPK_ERR_ARG; }
    if (!ctx->jpeg) { set_error("vpk_jpeg_stats: no decode ran on this context"); return VPK_ERR_STATE; }
    for (int i = 0; i < 4; ++i) out[i] = ctx->jpeg->last_stats[i];
    return VPK_OK;
}

}  // extern "C"
