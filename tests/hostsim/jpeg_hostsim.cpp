// TEST INFRASTRUCTURE ONLY.  Host build of the JPEG decoder from the same source the CUDA kernels use
// (vanishing_points_2017_b200/csrc/jpeg_core.cuh), so that the decode can be checked against libjpeg-turbo on a box
// without a GPU.  Two ways through the entropy-coded data:
//   L == 0   sequential: each restart interval decoded from its start in one pass
//   L > 0    the device's algorithm: subsequences of L bits, decoded from a guessed state, synchronised in rounds
//            inside CTAs of kCta subsequences and then across CTAs, block counts scanned, a final write pass
// Unstuffing, the DC scan per (interval, component), the IDCT and the upsampling follow the kernels' definitions.
// Never linked into libvpk.so, never imported by the package.
#include <algorithm>
#include <vector>
#include "../../vanishing_points_2017_b200/csrc/jpeg_core.cuh"

using namespace vpk::jpeg;

static constexpr int kCta = 128;        // subsequences per CTA, as csrc/jpeg.cu

struct Ival {
    std::vector<uint32_t> words;
    uint32_t nbits;
};

// stats[0] subsequences, [1] re-decoded subsequences, [2] longest chain of re-decodes, [3] global rounds
extern "C" int hostsim_jpeg(const uint8_t* data, int64_t n, int L, uint8_t* out, int64_t cap, int* dims, int64_t* stats) {
    Header hd;
    const int sup = parse(data, n, hd);
    dims[0] = hd.w; dims[1] = hd.h; dims[2] = hd.nc;
    if (sup != OK) return sup;
    Geom g;
    make_geom(hd, g);
    geom_place(g, 0, 0, 0, 0);
    if ((int64_t)g.w * g.h * g.nc > cap) return -1;
    int corrupt = 0;
    // unstuff and split at RSTn (jpeg.cu: jpeg_scan_end, jpeg_flags, jpeg_compact)
    const uint8_t* e = data + hd.ecs;
    const int64_t len = n - hd.ecs;
    int64_t end = len;
    for (int64_t i = 0; i < len && end == len; ++i)
        if (byte_kind(i ? e[i - 1] : -1, e[i], i + 1 < len ? e[i + 1] : -1) == BYTE_END) end = i;
    std::vector<std::vector<uint8_t>> bytes(g.nival);
    int64_t q = 0;
    for (int64_t i = 0; i < end; ++i) {
        const int k = byte_kind(i ? e[i - 1] : -1, e[i], i + 1 < len ? e[i + 1] : -1);
        if (k == BYTE_RST) {
            if (e[i] != 0xD0 + (q & 7)) corrupt = 1;
            ++q;
            if (q >= g.nival) corrupt = 1;
        } else if (k == BYTE_DATA && q < g.nival) {
            bytes[q].push_back(e[i]);
        }
    }
    if (q + 1 != g.nival) corrupt = 1;
    std::vector<Ival> iv(g.nival);
    for (int r = 0; r < g.nival; ++r) {
        iv[r].nbits = (uint32_t)(bytes[r].size() * 8);
        iv[r].words.assign((bytes[r].size() + 3) / 4, 0xFFFFFFFFu);
        if (!bytes[r].empty()) memcpy(iv[r].words.data(), bytes[r].data(), bytes[r].size());
    }
    const int64_t nblk = geom_blocks(g);
    std::vector<int16_t> coef((size_t)nblk * 64, 0);
    std::vector<int32_t> dcd((size_t)nblk, 0), keys((size_t)nblk, -1);
    std::vector<uint32_t> last_end(g.nival, 0xFFFFFFFFu);
    const HuffTab* tabs = hd.tab;
    // subsequences of each interval; L == 0: one per interval
    std::vector<int32_t> sub_ival;
    std::vector<uint32_t> sub_begin, sub_end;
    for (int r = 0; r < g.nival; ++r) {
        const uint32_t nb = iv[r].nbits;
        const uint32_t step_bits = L > 0 ? (uint32_t)L : std::max(nb, 1u);
        const uint32_t ns = std::max(1u, (nb + step_bits - 1) / step_bits);
        for (uint32_t j = 0; j < ns; ++j) {
            sub_ival.push_back(r);
            sub_begin.push_back(j * step_bits);
            sub_end.push_back(std::min(nb, (j + 1) * step_bits));
        }
    }
    const int64_t S = (int64_t)sub_ival.size();
    auto stream = [&](int64_t j) { const Ival& v = iv[sub_ival[j]]; return Stream{v.words.data(), (uint32_t)v.words.size(), v.nbits}; };
    auto first_of_ival = [&](int64_t j) { return j == 0 || sub_ival[j - 1] != sub_ival[j]; };
    auto start_guess = [&](int64_t j) { return State{sub_begin[j], 0u}; };
    std::vector<State> rec(S);
    std::vector<int32_t> cnt(S);
    int64_t redecodes = 0, chain = 0, rounds = 0;
    // phase 1 and the rounds inside each CTA (jpeg.cu: jpeg_sync, first launch), then rounds across CTAs (its later launches)
    const int64_t ncta = (S + kCta - 1) / kCta;
    auto cta_fixpoint = [&](int64_t c, bool first_launch, State in) {
        const int64_t j0 = c * kCta, j1 = std::min(S, j0 + kCta);
        std::vector<char> dirty(j1 - j0, 0);
        if (first_launch) {
            for (int64_t j = j0; j < j1; ++j) {
                State st = start_guess(j);
                cnt[j] = walk(stream(j), tabs, g, st, sub_end[j]);
                rec[j] = st;
            }
            for (int64_t j = j0 + 1; j < j1; ++j) dirty[j - j0] = !first_of_ival(j);
        } else {
            State st = in;
            cnt[j0] = walk(stream(j0), tabs, g, st, sub_end[j0]);
            const bool ch = !same(st, rec[j0]);
            rec[j0] = st;
            ++redecodes;
            if (j0 + 1 < j1) dirty[1] = ch && !first_of_ival(j0 + 1);
        }
        int64_t r = 0;
        while (std::any_of(dirty.begin(), dirty.end(), [](char d) { return d != 0; })) {
            ++r;
            std::vector<State> snap(rec.begin() + j0, rec.begin() + j1);
            std::vector<char> next(j1 - j0, 0);
            for (int64_t j = j0; j < j1; ++j) {
                if (!dirty[j - j0]) continue;
                State st = snap[j - 1 - j0];
                cnt[j] = walk(stream(j), tabs, g, st, sub_end[j]);
                ++redecodes;
                const bool ch = !same(st, rec[j]);
                rec[j] = st;
                if (ch && j + 1 < j1 && !first_of_ival(j + 1)) next[j + 1 - j0] = 1;
            }
            dirty.swap(next);
        }
        chain = std::max(chain, r);
    };
    for (int64_t c = 0; c < ncta; ++c) cta_fixpoint(c, true, State{0, 0});
    std::vector<State> used_in(ncta);
    for (int64_t c = 0; c < ncta; ++c) used_in[c] = start_guess(c * kCta);
    for (;;) {
        std::vector<State> tail(ncta);
        for (int64_t c = 0; c < ncta; ++c) tail[c] = rec[std::min(S, (c + 1) * kCta) - 1];
        bool any = false;
        for (int64_t c = 1; c < ncta; ++c) {
            const int64_t j0 = c * kCta;
            if (first_of_ival(j0) || same(tail[c - 1], used_in[c])) continue;
            used_in[c] = tail[c - 1];
            cta_fixpoint(c, false, tail[c - 1]);
            any = true;
        }
        if (!any) break;
        ++rounds;
    }
    // block counts -> exclusive scan -> write pass (jpeg_write)
    std::vector<int64_t> scan(S + 1, 0);
    for (int64_t j = 0; j < S; ++j) scan[j + 1] = scan[j] + cnt[j];
    int64_t ival_first = 0;
    for (int64_t j = 0; j < S; ++j) {
        if (first_of_ival(j)) ival_first = j;
        const int r = sub_ival[j];
        const State st = first_of_ival(j) ? start_guess(j) : rec[j - 1];
        const int64_t mcu0 = g.restart ? (int64_t)r * g.restart : 0;
        corrupt |= write_sub(stream(j), tabs, g, st, sub_end[j], scan[j] - scan[ival_first], ival_mcus(g, r) * g.bpm, mcu0,
                             g.ival0 + r, coef.data(), dcd.data(), keys.data(), &last_end[r], nblk, nblk);
    }
    for (int r = 0; r < g.nival; ++r)
        if (last_end[r] > iv[r].nbits || iv[r].nbits - last_end[r] >= 8) corrupt = 1;
    // DC: inclusive sum over runs of equal keys (cub::DeviceScan::InclusiveSumByKey), wrapping like the device
    uint32_t acc = 0;
    for (int64_t i = 0; i < nblk; ++i) {
        acc = (i > 0 && keys[i] == keys[i - 1]) ? acc + (uint32_t)dcd[i] : (uint32_t)dcd[i];
        dcd[i] = (int32_t)acc;
    }
    // IDCT of every block into the planes (jpeg_idct), then upsampling and colour (jpeg_color)
    std::vector<uint8_t> planes((size_t)geom_plane_bytes(g));
    for (int c = 0; c < g.nc; ++c)
        for (int by = 0; by < g.bh[c]; ++by)
            for (int bx = 0; bx < g.bw[c]; ++bx) {
                const int64_t b = g.coef[c] + (int64_t)by * g.bw[c] + bx;
                const int64_t my = by / g.cv[c], mx = bx / g.ch[c];
                const int64_t di = g.dc[c] + (my * g.mcux + mx) * (g.ch[c] * g.cv[c]) + (by % g.cv[c]) * g.ch[c] + bx % g.ch[c];
                int16_t blk[64];
                memcpy(blk, &coef[(size_t)b * 64], sizeof(blk));
                blk[0] = (int16_t)dcd[di];
                const int64_t st = (int64_t)g.bw[c] * 8;
                idct_islow(blk, hd.q[g.qt[c]], planes.data() + g.plane[c] + (int64_t)by * 8 * st + bx * 8, st);
            }
    for (int y = 0; y < g.h; ++y)
        for (int x = 0; x < g.w; ++x) pixel(g, planes.data(), x, y, out + ((int64_t)y * g.w + x) * g.nc);
    if (stats) { stats[0] = S; stats[1] = redecodes; stats[2] = chain; stats[3] = rounds; }
    return corrupt ? CORRUPT : OK;
}
