// Row N7: PNG decoding on the device, in front of photo preparation (reference evaluation.py:142-143: the dataset's
// PNG files, and the 8-bit PNG every photo is written to and read back from).  Bit for bit with libpng's decode of
// 8-bit and lower files; the sequential pieces are csrc/png_core.cuh, shared with the host build the CPU tests run.
// DESIGN.md section 4.9.
//
//   host          png::parse of every file's chunks (headers, IHDR and PLTE; never the IDAT payloads), refusals first
//   png_crc       CRC-32 of every IDAT chunk in slices of at most kSlice bytes, one thread each
//   png_crc_combine  each chunk's slices combined with zlib's crc32_combine (GF(2) shift); a mismatch is CORRUPT
//   png_inflate   one warp per file: lane 0 keeps the bit buffer (reading the IDAT payloads in place through the
//                 chunk list) and decodes symbols; the warp builds each block's tables in its shared memory (code
//                 lengths counted with ballots, canonical codes by a warp scan), flushes literals 32 at a time, copies
//                 every match with all lanes (byte k from p - d + k mod d: the periodic copy is parallel too) and
//                 accumulates the Adler-32 as it writes.  Output: the file's filtered scanlines, never past their size
//   png_unfilter  one warp per file or Adam7 pass: bands of 32 rows as a wavefront, lane j on row r0 + j one chunk of
//                 kCol bytes behind lane j - 1 (Sub, Avg and Paeth are serial along a row)
//   png_expand    one thread per output pixel: bit depth, palette, alpha dropped, Adam7 scatter, interleaved RGB (or
//                 gray) at the photo's offset
//
// VPK_DEFINES=VPK_PNG_CHECKS asserts every index into the files, tables, scanline buffers and outputs.
#include <algorithm>
#include "vpk_internal.cuh"
#include "png_core.cuh"

namespace vpk {

using png::Geom;
using png::Huff;

static_assert(png::OK == VPK_PNG_OK && png::NOT_PNG == VPK_PNG_NOT_PNG && png::DEPTH == VPK_PNG_DEPTH &&
              png::MALFORMED == VPK_PNG_MALFORMED && png::CORRUPT == VPK_PNG_CORRUPT,
              "png_core.cuh and vpk.h disagree on the VPK_PNG_* codes");

static constexpr int kThreads = 256;
static constexpr int kSlice = 4096;         // bytes per thread of png_crc
static constexpr int kWarps = 4;            // files (png_inflate) or passes (png_unfilter) per CTA
static constexpr int kCol = 16;             // bytes per wavefront step of png_unfilter
static constexpr int kPixTile = 256;        // output pixels per CTA of png_expand
static constexpr unsigned kFull = 0xFFFFFFFFu;

struct Slice { int64_t off; int32_t len, chunk; };
struct CrcChunk { int64_t crc_at; int32_t img, s0, ns, pad_; };
struct Unit { int32_t img, pass; };

struct PngState {
    DBuf data, meta, scan, pix, status, slice_crc;
    std::vector<png::Header> hs;    // the files of the last png_plan
};

void png_free(vpk_ctx* ctx) {
    if (!ctx->png) return;
    PngState* s = ctx->png;
    for (DBuf* b : {&s->data, &s->meta, &s->scan, &s->pix, &s->status, &s->slice_crc}) b->release();
    delete s;
    ctx->png = nullptr;
}

template <typename T>
__device__ __forceinline__ int find_image(const T* off, int B, T i) {
    int lo = 0, hi = B - 1;
    while (lo < hi) {                               // last file with off[b] <= i
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(kThreads) png_crc(const uint8_t* __restrict__ data, int64_t n_data, const Slice* __restrict__ sl, int n,
                                                    uint32_t* __restrict__ out) {
    __shared__ uint32_t tab[256];
    tab[threadIdx.x] = png::crc_entry(threadIdx.x);
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    PNG_CHECK(sl[i].off >= 0 && sl[i].off + sl[i].len <= n_data);
    (void)n_data;
    out[i] = png::crc_bytes(tab, data + sl[i].off, sl[i].len);
}

__global__ void __launch_bounds__(kThreads) png_crc_combine(const uint8_t* __restrict__ data, const Slice* __restrict__ sl,
                                                            const CrcChunk* __restrict__ ch, int n, const uint32_t* __restrict__ crc,
                                                            int32_t* __restrict__ status) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const CrcChunk c = ch[i];
    const uint32_t shift = png::x8nmodp(kSlice);   // every slice but a chunk's last is kSlice bytes long
    uint32_t v = crc[c.s0];
    for (int s = c.s0 + 1; s < c.s0 + c.ns; ++s)
        v = (sl[s].len == kSlice ? png::multmodp(shift, v) : png::multmodp(png::x8nmodp(sl[s].len), v)) ^ crc[s];
    const uint8_t* p = data + c.crc_at;
    const uint32_t want = (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | p[3];
    if (v != want) atomicOr(status + c.img, 1);
}

struct WarpSmem {
    Huff lit, dist, cl;
    uint16_t base[16];
    uint8_t lens[png::kMaxLit + png::kMaxDist];
    uint8_t stage[png::kStage];
};

// the block's table from its code lengths, by the whole warp; 0, or -1 for a set zlib refuses
__device__ int build_warp(const uint8_t* lens, int n, int type, Huff& t, uint16_t* base, int lane) {
    uint32_t cnt = 0;                               // lane l (1..15): codes of length l
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int l = c0 + lane < n ? lens[c0 + lane] : 0;
        for (int q = 1; q < 16; ++q) {
            const unsigned m = __ballot_sync(kFull, l == q);
            if (lane == q) cnt += __popc(m);
        }
    }
    if (lane < 16) t.count[lane] = (uint16_t)cnt;
    uint32_t inc = cnt;                             // the first sorted index of each length: an exclusive warp scan
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(kFull, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane < 16) base[lane] = (uint16_t)(inc - cnt);
    __syncwarp();
    int bad = lane == 0 ? png::huff_check(t.count, type) : 0;
    bad = __shfl_sync(kFull, bad, 0);
    if (bad) return -1;
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int s = c0 + lane;
        const int l = s < n ? lens[s] : 0;
        const unsigned m = __match_any_sync(kFull, l);
        const int rank = __popc(m & ((1u << lane) - 1));
        if (l) {
            PNG_CHECK(base[l] + rank < png::kMaxLit);
            t.sym[base[l] + rank] = (uint16_t)s;
        }
        __syncwarp();
        if (l && rank == 0) base[l] += (uint16_t)__popc(m);
        __syncwarp();
    }
    for (int e = lane; e < (1 << png::kFast); e += 32) t.fast[e] = png::fast_entry(t, e);
    __syncwarp();
    return 0;
}

// Adler-32 sums of a segment of n bytes, lane-strided: s1 = sum x_k, s2 = sum (n - k) x_k
__device__ __forceinline__ void adler_warp(uint32_t& a, uint32_t& b, uint32_t n, uint32_t s1, uint32_t s2) {
    s1 = __reduce_add_sync(kFull, s1);
    s2 = __reduce_add_sync(kFull, s2);
    png::adler_add(a, b, n, s1, s2);
}

__global__ void __launch_bounds__(kWarps * 32) png_inflate(const uint8_t* __restrict__ data, const Geom* __restrict__ geo,
                                                           const int64_t* __restrict__ idat, int B, uint8_t* __restrict__ scan,
                                                           int64_t n_scan, int32_t* __restrict__ status) {
    __shared__ WarpSmem sm[kWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * kWarps + warp;
    if (b >= B) return;
    WarpSmem& w = sm[warp];
    const Geom& g = geo[b];
    uint8_t* out = scan + g.scan;
    const int64_t total = g.raw;
    PNG_CHECK(g.scan >= 0 && g.scan + total <= n_scan);
    (void)n_scan;
    png::Reader r;
    png::Inflate s;
    if (lane == 0) { png::reader_init(r, data, idat + 2 * (int64_t)g.idat0, g.nidat); png::inflate_init(s); }
    int64_t pos = 0;
    uint32_t a = 1, bs = 0;
    int err = 0;
    for (;;) {
        int ev = 0, nst = 0, ml = 0, md = 0, nl = 0, nd = 0;
        uint32_t ad = 0;
        if (lane == 0) {
            ev = png::next_event(s, r, w.lit, w.dist, w.cl, w.stage, w.lens, pos);
            nst = s.nstage; s.nstage = 0;
            ml = s.mlen; md = s.mdist; nl = s.nlen; nd = s.ndist; ad = s.adler;
        }
        ev = __shfl_sync(kFull, ev, 0); nst = __shfl_sync(kFull, nst, 0);
        __syncwarp();
        // Past the last row (pos > total) nothing is stored and no check is summed, but the stream is still decoded:
        // libpng's verdicts there are zlib's errors and the Adler-32 as warnings only, running out of IDAT data as
        // an error.  Up to the last row every error counts, whatever follows.
        if (nst) {                                  // staged literals
            if (pos <= total) {
                const uint32_t v = lane < nst ? w.stage[lane] : 0;
                if (lane < nst && pos + lane < total) out[pos + lane] = (uint8_t)v;
                adler_warp(a, bs, nst, v, lane < nst ? (nst - lane) * v : 0);
            }
            pos += nst;
            __syncwarp();
        }
        if (ev == png::EV_MATCH) {
            ml = __shfl_sync(kFull, ml, 0); md = __shfl_sync(kFull, md, 0);
            if (pos <= total) {
                uint32_t s1 = 0, s2 = 0;
                for (int k = lane; k < ml; k += 32) {
                    const int64_t src = png::match_src(pos, md, k);
                    PNG_CHECK(src >= 0 && src < pos && src < total);
                    const uint32_t v = out[src];
                    if (pos + k < total) out[pos + k] = (uint8_t)v;
                    s1 += v; s2 += (uint32_t)(ml - k) * v;
                }
                adler_warp(a, bs, ml, s1, s2);
            }
            pos += ml;
            __syncwarp();
        } else if (ev == png::EV_TABLES) {
            nl = __shfl_sync(kFull, nl, 0); nd = __shfl_sync(kFull, nd, 0);
            if (build_warp(w.lens, nl, png::LENS, w.lit, w.base, lane) || build_warp(w.lens + nl, nd, png::DISTS, w.dist, w.base, lane)) {
                err = pos <= total;
                break;
            }
        } else if (ev == png::EV_END) {
            ad = __shfl_sync(kFull, ad, 0);
            err = pos < total || (pos == total && ad != (bs << 16 | a));
            break;
        } else if (ev == png::EV_ERROR) {
            const int trunc = __shfl_sync(kFull, lane == 0 ? (int)r.over() : 0, 0);
            err = trunc || pos <= total;
            break;
        }
    }
    if (lane == 0 && err) atomicOr(status + b, 1);
}

__global__ void __launch_bounds__(kWarps * 32) png_unfilter(const Geom* __restrict__ geo, const Unit* __restrict__ units, int n_units,
                                                            uint8_t* __restrict__ scan, int64_t n_scan, int32_t* __restrict__ status) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int u = blockIdx.x * kWarps + warp;
    if (u >= n_units) return;
    const Geom& g = geo[units[u].img];
    const int p = units[u].pass;
    const int64_t rows = g.ph[p], rb = g.rb[p], stride = rb + 1;
    const int bpp = g.bpp;
    uint8_t* base = scan + g.scan + g.poff[p];
    PNG_CHECK(g.scan + g.poff[p] + rows * stride <= n_scan);
    (void)n_scan;
    const int64_t nch = (rb + kCol - 1) / kCol;
    for (int64_t r0 = 0; r0 < rows; r0 += 32) {
        const int64_t r = r0 + lane;
        const bool active = r < rows;
        uint8_t* row = base + r * stride + 1;
        const uint8_t* prev = row - stride;
        int f = active ? row[-1] : 0;
        if (f > 4) { atomicOr(status + units[u].img, 1); f = 0; }
        const int64_t steps = nch + std::min<int64_t>(32, rows - r0) - 1;
        for (int64_t t = 0; t < steps; ++t) {
            const int64_t c = t - lane;
            if (active && f && c >= 0 && c < nch) {
                const int64_t x1 = std::min(rb, (c + 1) * kCol);
                for (int64_t x = c * kCol; x < x1; ++x) {
                    const int a = x >= bpp ? row[x - bpp] : 0;
                    const int up = r ? prev[x] : 0;
                    const int ul = (r && x >= bpp) ? prev[x - bpp] : 0;
                    row[x] = png::unfilter(f, row[x], a, up, ul);
                }
            }
            __syncwarp();
        }
    }
}

__global__ void __launch_bounds__(kPixTile) png_expand(const Geom* __restrict__ geo, const int32_t* __restrict__ tile_off, int B,
                                                       const uint8_t* __restrict__ pal, const uint8_t* __restrict__ scan,
                                                       uint8_t* __restrict__ out, int64_t n_out) {
    const int b = find_image(tile_off, B, (int32_t)blockIdx.x);
    const Geom& g = geo[b];
    const int64_t p = (int64_t)(blockIdx.x - tile_off[b]) * kPixTile + threadIdx.x;
    if (p >= (int64_t)g.w * g.h) return;
    const int y = (int)(p / g.w), x = (int)(p - (int64_t)y * g.w);
    const int nc = png::out_channels(g.ctype);
    PNG_CHECK(g.pix + (p + 1) * nc <= n_out);
    (void)n_out;
    png::expand(g, scan + g.scan, pal + 768 * (int64_t)b, x, y, out + g.pix + p * nc);
}

// ---- host ---------------------------------------------------------------------------------------------------------

int png_parse(const uint8_t* data, const int64_t* byte_offsets, int32_t B, const char* who, std::vector<png::Header>& hs) {
    if (!byte_offsets || B <= 0) { set_error("%s: bad argument", who); return VPK_ERR_ARG; }
    for (int b = 0; b < B; ++b)
        if (byte_offsets[b + 1] < byte_offsets[b] || byte_offsets[b] < 0) { set_error("%s: byte_offsets must be non-decreasing from >= 0", who); return VPK_ERR_ARG; }
    if (!data && byte_offsets[B] > byte_offsets[0]) { set_error("%s: data is NULL", who); return VPK_ERR_ARG; }
    hs.resize(B);
    for (int b = 0; b < B; ++b) hs[b].support = png::parse(data + byte_offsets[b], byte_offsets[b + 1] - byte_offsets[b], hs[b]);
    return VPK_OK;
}

static const char* reason_name(int r) {
    switch (r) {
        case VPK_PNG_NOT_PNG: return "not a PNG file";
        case VPK_PNG_DEPTH: return "16-bit samples";
        case VPK_PNG_MALFORMED: return "malformed chunks or zlib header";
        default: return "unknown";
    }
}

int png_plan(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t B, bool rgb_only, const char* who,
             std::vector<int32_t>& widths, std::vector<int32_t>& heights, std::vector<int32_t>& components) {
    if (!ctx->png) ctx->png = new PngState();
    std::vector<png::Header>& hs = ctx->png->hs;
    VPK_TRY(png_parse(data, byte_offsets, B, who, hs));
    for (int b = 0; b < B; ++b) {
        if (hs[b].support != png::OK) {
            set_error("%s: photo %d is not supported: reason %d (%s)", who, b, hs[b].support, reason_name(hs[b].support));
            return VPK_ERR_ARG;
        }
        if (rgb_only && png::out_channels(hs[b].ctype) != 3) {
            set_error("%s: photo %d is gray (colour type %d); gray photos cannot be prepared", who, b, hs[b].ctype);
            return VPK_ERR_ARG;
        }
    }
    widths.resize(B); heights.resize(B); components.resize(B);
    for (int b = 0; b < B; ++b) { widths[b] = hs[b].w; heights[b] = hs[b].h; components[b] = png::out_channels(hs[b].ctype); }
    return VPK_OK;
}

// packs host arrays into one device upload; returns the byte offset of each
struct PngPacker {
    std::vector<char> buf;
    template <typename T> size_t add(const T* p, size_t n) {
        const size_t o = (buf.size() + 15) & ~(size_t)15;
        buf.resize(o + n * sizeof(T));
        if (n) memcpy(buf.data() + o, p, n * sizeof(T));
        return o;
    }
};

int png_decode(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, const int64_t* pix_off, uint8_t* d_out, int32_t* status_out) {
    VPK_CUDA(cudaSetDevice(ctx->device));
    PngState* s = ctx->png;
    const std::vector<png::Header>& hs = s->hs;
    const int B = (int)hs.size();
    cudaStream_t st = ctx->stream;
    std::vector<Geom> geo(B);
    std::vector<int64_t> idat;
    std::vector<uint8_t> pal((size_t)B * 768, 0);
    std::vector<Slice> slices;
    std::vector<CrcChunk> chunks;
    std::vector<Unit> units;
    std::vector<int32_t> tile_off(B + 1, 0);
    int64_t n_scan = 0;
    for (int b = 0; b < B; ++b) {
        const png::Header& h = hs[b];
        Geom& g = geo[b];
        png::make_geom(h, g);
        g.scan = n_scan;
        g.pix = pix_off[b];
        g.idat0 = (int32_t)(idat.size() / 2);
        n_scan += g.raw;
        memcpy(&pal[(size_t)b * 768], h.pal, (size_t)h.npal * 3);
        for (size_t c = 0; c < h.idat.size(); c += 2) {
            const int64_t off = byte_offsets[b] + h.idat[c], len = h.idat[c + 1];
            idat.push_back(off);
            idat.push_back(len);
            CrcChunk k{off + len, b, (int32_t)slices.size(), 0, 0};
            for (int64_t q = 0; q < len + 4; q += kSlice)            // the CRC covers the chunk type and the payload
                slices.push_back(Slice{off - 4 + q, (int32_t)std::min<int64_t>(kSlice, len + 4 - q), (int32_t)chunks.size()});
            k.ns = (int32_t)slices.size() - k.s0;
            chunks.push_back(k);
        }
        for (int p = 0; p < g.npass; ++p)
            if (g.pw[p] && g.ph[p]) units.push_back(Unit{b, p});
        const int64_t ntile = ((int64_t)g.w * g.h + kPixTile - 1) / kPixTile;
        if (tile_off[b] + ntile > INT32_MAX || slices.size() > (size_t)INT32_MAX / 2) { set_error("png: batch too large for one call; split it"); return VPK_ERR_ARG; }
        tile_off[b + 1] = tile_off[b] + (int32_t)ntile;
    }
    const int n_sl = (int)slices.size(), n_ch = (int)chunks.size(), n_u = (int)units.size();
    PngPacker pk;
    const size_t o_g = pk.add(geo.data(), B), o_i = pk.add(idat.data(), idat.size()), o_p = pk.add(pal.data(), pal.size()),
                 o_s = pk.add(slices.data(), slices.size()), o_c = pk.add(chunks.data(), chunks.size()), o_u = pk.add(units.data(), units.size()),
                 o_t = pk.add(tile_off.data(), B + 1);
    VPK_TRY(s->meta.ensure(pk.buf.size()));
    VPK_TRY(s->data.ensure((size_t)std::max<int64_t>(byte_offsets[B], 1)));
    VPK_TRY(s->scan.ensure((size_t)std::max<int64_t>(n_scan, 1)));
    VPK_TRY(s->status.ensure((size_t)B * 4));
    VPK_TRY(s->slice_crc.ensure((size_t)std::max(n_sl, 1) * 4));
    char* mb = s->meta.as<char>();
    const Geom* d_geo = reinterpret_cast<const Geom*>(mb + o_g);
    const int64_t* d_idat = reinterpret_cast<const int64_t*>(mb + o_i);
    const uint8_t* d_pal = reinterpret_cast<const uint8_t*>(mb + o_p);
    const Slice* d_sl = reinterpret_cast<const Slice*>(mb + o_s);
    const CrcChunk* d_ch = reinterpret_cast<const CrcChunk*>(mb + o_c);
    const Unit* d_u = reinterpret_cast<const Unit*>(mb + o_u);
    const int32_t* d_tile = reinterpret_cast<const int32_t*>(mb + o_t);
    const uint8_t* d_data = s->data.as<uint8_t>();
    int32_t* d_status = s->status.as<int32_t>();
    uint8_t* d_scan = s->scan.as<uint8_t>();
    VPK_CUDA(cudaMemcpyAsync(s->meta.p, pk.buf.data(), pk.buf.size(), cudaMemcpyHostToDevice, st));
    if (byte_offsets[B]) VPK_CUDA(cudaMemcpyAsync(s->data.p, data, (size_t)byte_offsets[B], cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemsetAsync(s->status.p, 0, (size_t)B * 4, st));
    // a damaged stream leaves part of its buffer unwritten: zeros, so that its pixels are deterministic
    if (n_scan) VPK_CUDA(cudaMemsetAsync(d_scan, 0, (size_t)n_scan, st));
    if (n_sl) {
        {
            KernelScope ks(ctx, "png_crc");
            png_crc<<<(n_sl + kThreads - 1) / kThreads, kThreads, 0, st>>>(d_data, byte_offsets[B], d_sl, n_sl, s->slice_crc.as<uint32_t>());
            VPK_TRY(check_launch("png_crc"));
        }
        {
            KernelScope ks(ctx, "png_crc_combine");
            png_crc_combine<<<(n_ch + kThreads - 1) / kThreads, kThreads, 0, st>>>(d_data, d_sl, d_ch, n_ch, s->slice_crc.as<uint32_t>(), d_status);
            VPK_TRY(check_launch("png_crc_combine"));
        }
    }
    {
        KernelScope ks(ctx, "png_inflate");
        png_inflate<<<(B + kWarps - 1) / kWarps, kWarps * 32, 0, st>>>(d_data, d_geo, d_idat, B, d_scan, n_scan, d_status);
        VPK_TRY(check_launch("png_inflate"));
    }
    if (n_u) {
        KernelScope ks(ctx, "png_unfilter");
        png_unfilter<<<(n_u + kWarps - 1) / kWarps, kWarps * 32, 0, st>>>(d_geo, d_u, n_u, d_scan, n_scan, d_status);
        VPK_TRY(check_launch("png_unfilter"));
    }
    {
        KernelScope ks(ctx, "png_expand");
        png_expand<<<tile_off[B], kPixTile, 0, st>>>(d_geo, d_tile, B, d_pal, d_scan, d_out, pix_off[B]);
        VPK_TRY(check_launch("png_expand"));
    }
    std::vector<int32_t> stat(B);
    VPK_CUDA(cudaMemcpyAsync(stat.data(), d_status, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    VPK_CUDA(cudaStreamSynchronize(st));
    for (int b = 0; b < B; ++b) status_out[b] = stat[b] ? png::CORRUPT : png::OK;
    return VPK_OK;
}

}  // namespace vpk

using namespace vpk;

extern "C" {

int vpk_png_info(const uint8_t* data, const int64_t* byte_offsets, int32_t n, int32_t* widths, int32_t* heights, int32_t* color_types,
                 int32_t* support) {
    std::vector<png::Header> hs;
    VPK_TRY(png_parse(data, byte_offsets, n, "vpk_png_info", hs));
    for (int b = 0; b < n; ++b) {
        if (widths) widths[b] = hs[b].w;
        if (heights) heights[b] = hs[b].h;
        if (color_types) color_types[b] = hs[b].ctype;
        if (support) support[b] = hs[b].support;
    }
    return VPK_OK;
}

int vpk_decode_pngs(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t n, uint8_t* pixels_out, int32_t* status_out) {
    if (!ctx || !pixels_out || !status_out) { set_error("vpk_decode_pngs: bad argument"); return VPK_ERR_ARG; }
    std::vector<int32_t> w, h, nc;
    VPK_TRY(png_plan(ctx, data, byte_offsets, n, false, "vpk_decode_pngs", w, h, nc));
    std::vector<int64_t> pix_off(n + 1, 0);
    for (int b = 0; b < n; ++b) pix_off[b + 1] = pix_off[b] + (int64_t)w[b] * h[b] * nc[b];
    VPK_CUDA(cudaSetDevice(ctx->device));
    VPK_TRY(ctx->png->pix.ensure((size_t)std::max<int64_t>(pix_off[n], 1)));
    VPK_TRY(png_decode(ctx, data, byte_offsets, pix_off.data(), ctx->png->pix.as<uint8_t>(), status_out));
    VPK_CUDA(cudaMemcpyAsync(pixels_out, ctx->png->pix.p, (size_t)pix_off[n], cudaMemcpyDeviceToHost, ctx->stream));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    return VPK_OK;
}

}  // extern "C"
