// TEST INFRASTRUCTURE ONLY.  Host build of the PNG decoder from the same source the CUDA kernels use
// (vanishing_points_2017_b200/csrc/png_core.cuh), so that the decode can be checked against zlib and libpng on a box
// without a GPU.  The IDAT CRCs are combined from slices as png_crc / png_crc_combine do (with small slices, so that
// every chunk of more than a few bytes is combined).  Inflate runs the core's event loop; each event is applied
//   mode 0   sequentially, byte after byte
//   mode 1   as the warp of png_inflate does: literals by lane, every match byte k of every lane from
//            match_src (lanes visited in reverse order, so that no copy may rely on another of the same step), the
//            Adler-32 from the lanes' partial sums
// Unfiltering and expansion use the core's predictors and expand().  Never linked into libvpk.so.
#include <algorithm>
#include <vector>
#include "../../vanishing_points_2017_b200/csrc/png_core.cuh"

using namespace vpk::png;

static constexpr int kSlice = 61;

// dims: width, height, colour type, filtered bytes, output channels.  Returns the support code, CORRUPT / OK after
// decoding, or -1 if raw_cap or cap is too small.
extern "C" int hostsim_png(const uint8_t* d, int64_t n, int mode, uint8_t* raw_out, int64_t raw_cap, uint8_t* out, int64_t cap,
                           int64_t* dims) {
    Header hd;
    const int sup = parse(d, n, hd);
    dims[0] = hd.w; dims[1] = hd.h; dims[2] = hd.ctype;
    if (sup != OK) return sup;
    Geom g;
    make_geom(hd, g);
    dims[3] = g.raw; dims[4] = out_channels(g.ctype);
    if (g.raw > raw_cap || (int64_t)g.w * g.h * dims[4] > cap) return -1;
    int corrupt = 0;
    const uint32_t* tab = host_crc_table();
    for (size_t c = 0; c < hd.idat.size(); c += 2) {
        const int64_t off = hd.idat[c], len = hd.idat[c + 1];
        uint32_t v = crc_bytes(tab, d + off - 4, std::min<int64_t>(kSlice, len + 4));
        for (int64_t q = kSlice; q < len + 4; q += kSlice) {
            const int64_t m = std::min<int64_t>(kSlice, len + 4 - q);
            v = crc_combine(v, crc_bytes(tab, d + off - 4 + q, m), m);
        }
        if (v != be32(d + off + len)) corrupt = 1;
    }
    std::vector<uint8_t> buf((size_t)std::max<int64_t>(g.raw, 1), 0);
    const int64_t total = g.raw;
    Reader r;
    Inflate s;
    reader_init(r, d, hd.idat.data(), (int)hd.idat.size() / 2);
    inflate_init(s);
    Huff lit, dist, cl;
    uint8_t stage[kStage], lens[kMaxLit + kMaxDist];
    int64_t pos = 0;
    uint32_t a = 1, b = 0;
    int err = 0;
    auto emit = [&](const uint8_t* src, int cnt, bool is_match, int dd) {
        // src: literals; or a match of cnt bytes at distance dd
        if (mode == 0) {
            for (int k = 0; k < cnt; ++k) {
                const int64_t si = pos + k - dd;     // at or past total only for bytes that are not stored
                const uint8_t v = is_match ? (si < total ? buf[si] : 0) : src[k];
                if (pos + k < total) buf[pos + k] = v;
                a = (a + v) % kAdlerMod;
                b = (b + a) % kAdlerMod;
            }
        } else {
            uint32_t s1 = 0, s2 = 0;
            for (int lane = 31; lane >= 0; --lane)
                for (int k = lane; k < cnt; k += 32) {
                    const uint8_t v = is_match ? buf[match_src(pos, dd, k)] : src[k];
                    if (is_match && match_src(pos, dd, k) >= pos) return false;
                    if (pos + k < total) buf[pos + k] = v;
                    s1 += v;
                    s2 += (uint32_t)(cnt - k) * v;
                }
            adler_add(a, b, cnt, s1, s2);
        }
        pos += cnt;
        return true;
    };
    // past the last row: decoded, not stored; zlib's errors and the Adler-32 are libpng's warnings there, running
    // out of IDAT data an error (png_inflate's rule)
    for (;;) {
        const int ev = next_event(s, r, lit, dist, cl, stage, lens, pos);
        const int nst = s.nstage;
        s.nstage = 0;
        if (nst) {
            if (pos <= total) emit(stage, nst, false, 0);
            else pos += nst;
        }
        if (ev == EV_MATCH) {
            if (pos <= total) {
                if (!emit(nullptr, s.mlen, true, s.mdist)) { err = 1; break; }
            } else {
                pos += s.mlen;
            }
        } else if (ev == EV_TABLES) {
            if (huff_build(lens, s.nlen, LENS, lit, true) || huff_build(lens + s.nlen, s.ndist, DISTS, dist, true)) { err = pos <= total; break; }
        } else if (ev == EV_END) {
            err = pos < total || (pos == total && s.adler != (b << 16 | a));
            break;
        } else if (ev == EV_ERROR) {
            err = r.over() || pos <= total;
            break;
        }
    }
    corrupt |= err;
    if (raw_out) memcpy(raw_out, buf.data(), (size_t)total);
    // unfilter pass by pass, row after row
    for (int p = 0; p < g.npass; ++p) {
        if (!g.pw[p] || !g.ph[p]) continue;
        const int64_t stride = g.rb[p] + 1;
        for (int64_t y = 0; y < g.ph[p]; ++y) {
            uint8_t* row = buf.data() + g.poff[p] + y * stride + 1;
            const uint8_t* prev = row - stride;
            int f = row[-1];
            if (f > 4) { corrupt = 1; f = 0; }
            for (int64_t x = 0; x < g.rb[p]; ++x)
                row[x] = unfilter(f, row[x], x >= g.bpp ? row[x - g.bpp] : 0, y ? prev[x] : 0, (y && x >= g.bpp) ? prev[x - g.bpp] : 0);
        }
    }
    const int nc = out_channels(g.ctype);
    uint8_t pal[768] = {0};
    memcpy(pal, hd.pal, (size_t)hd.npal * 3);
    for (int y = 0; y < g.h; ++y)
        for (int x = 0; x < g.w; ++x) expand(g, buf.data(), pal, x, y, out + ((int64_t)y * g.w + x) * nc);
    return corrupt ? CORRUPT : OK;
}
