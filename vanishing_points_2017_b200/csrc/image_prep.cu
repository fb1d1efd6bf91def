// Row N5: photo preparation in front of LSD (reference evaluation.py:139-154): `convert ... -resize TxT` (stood in
// for by OpenCV 4.13's cv2.resize(..., INTER_AREA), SURVEY section 8(c)), the 8-bit RGB read back, and
// skimage 0.12's rgb2gray, for a ragged batch of uint8 RGB photos in one launch.  Restated from
// oracle/image_prep_oracle.py and held to bit equality with it (DESIGN.md section 4.7):
//
//   image_prep   one CTA per TW x TH output tile of one image: the tile's source rectangle of RGB bytes is staged
//                in shared memory once, the x pass (every source row of the rectangle x TW columns x 3 channels,
//                float64) and then the y pass run there, each output channel is rounded to uint8, converted to gray
//                and the tile is written as float64.  Per image, one of three paths:
//                  identity   (no resize)     gray of the source pixels, straight from global memory
//                  integer    (w/W', h/H' integers: OpenCV's is_area_fast) exact integer mean of each block, ties
//                             half up for 2 x 2 (OpenCV's vectorised path), half to even otherwise
//                  generic    computeResizeAreaTab's partial / full / partial taps in float64, rint, clamp
//
// Gray photos (one channel: row N8, section 4.10) take the same paths on one channel and write the uint8 values
// themselves (skimage 0.12's rgb2gray returns a 2-D input unchanged); for LSD's input, prep_gray_scale then applies
// detect_lsd_lines' "* 255 if max <= 1" per gray image from a flag the tiles set.
// Tile extents adapt to the largest factor of the batch so the source rectangle fits in shared memory.  Every
// floating-point operation is a single correctly rounded __d*_rn operation (no FMA contraction, no libm), every sum
// runs in increasing source index.  A VPK_DEFINES=VPK_PREP_CHECKS build asserts every shared- and global-memory index.
#include <algorithm>
#include <cmath>
#include "vpk_internal.cuh"

#if defined(VPK_PREP_CHECKS)
#include <assert.h>
#define PREP_CHECK(c) assert(c)
#else
#define PREP_CHECK(c) ((void)0)
#endif

namespace vpk {

static constexpr int kPrepThreads = 256;
static constexpr int kTileW = 32, kTileH = 16;           // largest tile; both shrink for large factors
static constexpr size_t kPrepSmemBudget = 64 * 1024;     // preferred shared memory per CTA (three CTAs per SM)

enum { PREP_IDENTITY = 0, PREP_AREA = 1, PREP_INTEGER = 2 };

struct PrepState {
    DBuf rgb, meta, out, big;
};

void prep_free(vpk_ctx* ctx) {
    if (!ctx->prep) return;
    ctx->prep->rgb.release(); ctx->prep->meta.release(); ctx->prep->out.release(); ctx->prep->big.release();
    delete ctx->prep;
    ctx->prep = nullptr;
}

// per-image geometry on the device
struct PrepImage {
    int64_t src, dst;       // byte offset of the photo, pixel offset of its output plane
    double sx, sy;          // computeResizeAreaTab's scale per axis: 1 / (W' / w), 1 / (H' / h)
    int32_t w, h, W, H;
    int32_t mode, kx, ky;   // PREP_*; block size of the integer path
    int32_t tiles_x;
    int32_t ch;             // channels of the photo: 3 (RGB) or 1 (gray)
};

// the taps of one output column (row): lead partial tap, nfull full taps, trail partial tap, consecutive source
// indices from `first`
struct Taps {
    int32_t first, nfull, lead, trail;
    double wl, wf, wt;
};

__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }

// computeResizeAreaTab (OpenCV imgproc/resize.cpp) for output d, in float64; integer path: k full taps of weight 1
__device__ Taps make_taps(int d, int ssize, double scale, int mode, int k) {
    Taps q;
    if (mode == PREP_INTEGER) {
        q.first = d * k; q.nfull = k; q.lead = 0; q.trail = 0;
        q.wl = 0.0; q.wf = 1.0; q.wt = 0.0;
        return q;
    }
    const double fs1 = mul((double)d, scale);
    const double fs2 = add(fs1, scale);
    const double cw = fmin(scale, sub((double)ssize, fs1));
    int s1 = (int)ceil(fs1), s2 = (int)floor(fs2);
    s2 = min(s2, ssize - 1);
    s1 = min(s1, s2);
    const double lead = sub((double)s1, fs1), trail = sub(fs2, (double)s2);
    q.lead = lead > 1e-3;
    q.trail = trail > 1e-3;
    q.wl = q.lead ? __ddiv_rn(lead, cw) : 0.0;
    q.wf = __ddiv_rn(1.0, cw);
    q.wt = q.trail ? __ddiv_rn(fmin(fmin(trail, 1.0), cw), cw) : 0.0;
    q.first = q.lead ? s1 - 1 : s1;
    q.nfull = s2 - s1;
    return q;
}

__device__ __forceinline__ int last_tap(const Taps& q) { return q.first + q.lead + q.nfull + q.trail - 1; }

// sum of weight * value over the taps, in increasing source index; v[k * stride] is the value of source first + k
template <typename T>
__device__ __forceinline__ double tap_sum(const Taps& q, const T* v, int stride) {
    double s = 0.0;
    int k = 0;
    if (q.lead) { s = add(s, mul(q.wl, (double)v[0])); k = 1; }
    for (const int e = k + q.nfull; k < e; ++k) s = add(s, mul(q.wf, (double)v[k * stride]));
    if (q.trail) s = add(s, mul(q.wt, (double)v[k * stride]));
    return s;
}

// rgb2gray of skimage 0.12: img_as_float (x * (1./255)), then 0.2125 r + 0.7154 g + 0.0721 b left to right;
// times out_scale (255 for LSD's input: detect_lsd_lines' "* 255 if max <= 1", evaluation.py:229-231)
__device__ __forceinline__ double gray(int r, int g, int b, double out_scale) {
    constexpr double inv = 1.0 / 255;
    double y = mul(0.2125, mul((double)r, inv));
    y = add(y, mul(0.7154, mul((double)g, inv)));
    y = add(y, mul(0.0721, mul((double)b, inv)));
    return mul(y, out_scale);
}

// generic path: rint and clamp; integer path: the exact integer mean of the block (the sum is an exact integer)
__device__ __forceinline__ int to_u8(double s, const PrepImage& g) {
    if (g.mode == PREP_AREA) return min(max(__double2int_rn(s), 0), 255);
    const long long tot = (long long)s, area = (long long)g.kx * g.ky;
    const long long q = tot / area, r = tot - q * area;
    const bool half_up = g.kx == 2 && g.ky == 2;
    return (int)(q + (2 * r > area || (2 * r == area && (half_up || (q & 1)))));
}

// One tile of one image with C channels (3: RGB, 1: gray).  RGB: rgb2gray of the uint8 result, times out_scale.  Gray:
// the uint8 values themselves; if `big` is set, big[b] becomes 1 when some value of image b exceeds 1.
template <int C>
__device__ __forceinline__ void prep_tile(const PrepImage& g, int b, int x0, int y0, int TW, int TH, int nx_max, int ny_max,
                                          double out_scale, const uint8_t* __restrict__ src, double* __restrict__ dst,
                                          int32_t* __restrict__ big, unsigned char* smem, int64_t n_src, int64_t n_out) {
    const int nc = min(TW, g.W - x0), nr = min(TH, g.H - y0);
    PREP_CHECK(nc > 0 && nr > 0);
    bool over = false;                              // gray: some value of this tile exceeds 1
    if (g.mode == PREP_IDENTITY) {
        for (int i = threadIdx.x; i < nc * nr; i += blockDim.x) {
            const int x = x0 + i % nc, y = y0 + i / nc;
            const int64_t p = ((int64_t)y * g.w + x) * C;
            PREP_CHECK(g.src + p + C - 1 < n_src && g.dst + (int64_t)y * g.W + x < n_out);
            if (C == 3) {
                dst[(int64_t)y * g.W + x] = gray(src[p], src[p + 1], src[p + 2], out_scale);
            } else {
                dst[(int64_t)y * g.W + x] = (double)src[p];
                over |= src[p] > 1;
            }
        }
    } else {
        Taps* tx = reinterpret_cast<Taps*>(smem);
        Taps* ty = tx + TW;
        double* T = reinterpret_cast<double*>(ty + TH);                               // ny_max x TW x C
        uint8_t* S = reinterpret_cast<uint8_t*>(T + (size_t)ny_max * TW * C);         // ny_max x nx_max x C
        if (threadIdx.x < nc) tx[threadIdx.x] = make_taps(x0 + threadIdx.x, g.w, g.sx, g.mode, g.kx);
        else if (threadIdx.x >= TW && threadIdx.x < TW + nr) ty[threadIdx.x - TW] = make_taps(y0 + threadIdx.x - TW, g.h, g.sy, g.mode, g.ky);
        __syncthreads();
        const int xa = tx[0].first, ya = ty[0].first;
        const int nx = last_tap(tx[nc - 1]) - xa + 1, ny = last_tap(ty[nr - 1]) - ya + 1;
        PREP_CHECK(xa >= 0 && ya >= 0 && xa + nx <= g.w && ya + ny <= g.h && nx <= nx_max && ny <= ny_max);
        // stage the source rectangle (row by row, contiguous bytes)
        const int rowb = nx * C;
        for (int i = threadIdx.x; i < ny * rowb; i += blockDim.x) {
            const int r = i / rowb, c = i - r * rowb;
            const int64_t p = ((int64_t)(ya + r) * g.w + xa) * C + c;
            PREP_CHECK(g.src + p < n_src && i < ny_max * nx_max * C);
            S[i] = src[p];
        }
        __syncthreads();
        // x pass: T[r][j][c] for every staged row r and output column j
        for (int i = threadIdx.x; i < ny * nc * C; i += blockDim.x) {
            const int c = i % C, j = (i / C) % nc, r = i / (C * nc);
            const Taps& q = tx[j];
            PREP_CHECK(q.first >= xa && last_tap(q) < xa + nx && (r * TW + j) * C + c < ny_max * TW * C);
            T[(r * TW + j) * C + c] = tap_sum(q, S + r * rowb + (q.first - xa) * C + c, C);
        }
        __syncthreads();
        // y pass, uint8, then gray (RGB) or the value itself (gray)
        for (int i = threadIdx.x; i < nr * nc; i += blockDim.x) {
            const int j = i % nc, r = i / nc;
            const Taps& q = ty[r];
            PREP_CHECK(q.first >= ya && last_tap(q) < ya + ny);
            const double* col = T + ((q.first - ya) * TW + j) * C;
            const int64_t o = (int64_t)(y0 + r) * g.W + x0 + j;
            if (C == 3) {
                const int v0 = to_u8(tap_sum(q, col, TW * 3), g);
                const int v1 = to_u8(tap_sum(q, col + 1, TW * 3), g);
                const int v2 = to_u8(tap_sum(q, col + 2, TW * 3), g);
                PREP_CHECK(g.dst + o < n_out && v0 >= 0 && v0 <= 255 && v1 >= 0 && v1 <= 255 && v2 >= 0 && v2 <= 255);
                dst[o] = gray(v0, v1, v2, out_scale);
            } else {
                const int v = to_u8(tap_sum(q, col, TW), g);
                PREP_CHECK(g.dst + o < n_out && v >= 0 && v <= 255);
                dst[o] = (double)v;
                over |= v > 1;
            }
        }
    }
    if (C == 1 && big) {                            // uniform per CTA: every thread reaches the barrier
        if (__syncthreads_or(over) && threadIdx.x == 0) big[b] = 1;
    }
}

__global__ void __launch_bounds__(kPrepThreads) image_prep(const uint8_t* __restrict__ rgb, const PrepImage* __restrict__ im,
                                                           const int32_t* __restrict__ tile_off, int B, int TW, int TH, int nx_max,
                                                           int ny_max, double out_scale, double* __restrict__ out,
                                                           int32_t* __restrict__ big, int64_t n_src, int64_t n_out) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int t = blockIdx.x;
    int lo = 0, hi = B - 1;
    while (lo < hi) {                               // last image with tile_off[b] <= t
        const int mid = (lo + hi + 1) >> 1;
        if (tile_off[mid] <= t) lo = mid; else hi = mid - 1;
    }
    const PrepImage g = im[lo];
    const int tl = t - tile_off[lo];
    const int x0 = (tl % g.tiles_x) * TW, y0 = (tl / g.tiles_x) * TH;
    if (g.ch == 3) prep_tile<3>(g, lo, x0, y0, TW, TH, nx_max, ny_max, out_scale, rgb + g.src, out + g.dst, big, smem, n_src, n_out);
    else prep_tile<1>(g, lo, x0, y0, TW, TH, nx_max, ny_max, out_scale, rgb + g.src, out + g.dst, big, smem, n_src, n_out);
}

// detect_lsd_lines' "* 255 if max <= 1" for the gray images: the plane of gray image gray_idx[k] is multiplied by
// `scale` unless the preparation kernel flagged a value above 1 in it
__global__ void __launch_bounds__(kPrepThreads) prep_gray_scale(const PrepImage* __restrict__ im, const int32_t* __restrict__ gray_idx,
                                                                int n_gray, const int32_t* __restrict__ big, double scale,
                                                                double* __restrict__ out, int64_t n_out) {
    for (int k = blockIdx.y; k < n_gray; k += gridDim.y) {
        const int b = gray_idx[k];
        if (big[b]) continue;
        const PrepImage& g = im[b];
        const int64_t n = (int64_t)g.W * g.H;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
            PREP_CHECK(g.ch == 1 && g.dst + i < n_out);
            out[g.dst + i] = mul(out[g.dst + i], scale);
        }
    }
    (void)n_out;
}

static void prepared_size(int w, int h, int target, int* W, int* H) {
    *W = w; *H = h;
    if (target <= 0) return;
    const double s = (double)target / (double)std::max(w, h);
    if (!(s < 1.0)) return;
    *W = std::max(1, (int)nearbyint(w * s));        // rint: half to even, like Python's round
    *H = std::max(1, (int)nearbyint(h * s));
}

int prep_plan(const int64_t* byte_offsets, const int32_t* widths, const int32_t* heights, const int32_t* channels, int32_t B,
              int32_t target_size, const char* who, PrepPlan& p) {
    if (!byte_offsets || !widths || !heights || B <= 0) { set_error("%s: bad argument", who); return VPK_ERR_ARG; }
    if (byte_offsets[0] != 0) { set_error("%s: byte_offsets[0] must be 0", who); return VPK_ERR_ARG; }
    p.B = B;
    p.w.assign(widths, widths + B); p.h.assign(heights, heights + B);
    if (channels) p.c.assign(channels, channels + B); else p.c.assign(B, 3);
    p.W.resize(B); p.H.resize(B);
    p.src_off.assign(byte_offsets, byte_offsets + B + 1);
    p.pix_off.assign(B + 1, 0);
    for (int b = 0; b < B; ++b) {
        const int w = widths[b], h = heights[b], c = p.c[b];
        if (c != 1 && c != 3) { set_error("%s: photo %d: %d channels (1 or 3)", who, b, c); return VPK_ERR_ARG; }
        if (w <= 0 || h <= 0 || byte_offsets[b + 1] - byte_offsets[b] != c * (int64_t)w * h) {
            if (channels) set_error("%s: photo %d: byte_offsets[b+1] - byte_offsets[b] must be channels[b] * widths[b] * heights[b] > 0", who, b);
            else set_error("%s: photo %d: byte_offsets[b+1] - byte_offsets[b] must be 3 * widths[b] * heights[b] > 0", who, b);
            return VPK_ERR_ARG;
        }
        prepared_size(w, h, target_size, &p.W[b], &p.H[b]);
        p.pix_off[b + 1] = p.pix_off[b] + (int64_t)p.W[b] * p.H[b];
    }
    return VPK_OK;
}

int prep_input(vpk_ctx* ctx, const PrepPlan& p, uint8_t** d_rgb) {
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->prep) ctx->prep = new PrepState();
    VPK_TRY(ctx->prep->rgb.ensure((size_t)std::max<int64_t>(p.src_off[p.B], 1)));
    *d_rgb = ctx->prep->rgb.as<uint8_t>();
    return VPK_OK;
}

int prep_output(vpk_ctx* ctx, int64_t n_out, double** d_out) {
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->prep) ctx->prep = new PrepState();
    VPK_TRY(ctx->prep->out.ensure((size_t)std::max<int64_t>(n_out, 1) * sizeof(double)));
    *d_out = ctx->prep->out.as<double>();
    return VPK_OK;
}

// shared memory of a TW x TH tile whose source rectangle spans at most fx, fy source pixels per output pixel
static size_t tile_smem(int TW, int TH, double fx, double fy, int C, int* nx, int* ny) {
    *nx = (int)ceil(TW * fx) + 3;
    *ny = (int)ceil(TH * fy) + 3;
    return (size_t)(TW + TH) * sizeof(Taps) + (size_t)*ny * TW * C * sizeof(double) + (((size_t)*nx * *ny * C + 15) & ~(size_t)15);
}

int prep_run(vpk_ctx* ctx, const PrepPlan& p, double out_scale, double* d_out) {
    const int B = p.B;
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->prep) ctx->prep = new PrepState();
    PrepState* s = ctx->prep;
    cudaStream_t st = ctx->stream;
    std::vector<PrepImage> im(B);
    std::vector<int32_t> gray_idx;
    double fx = 1.0, fy = 1.0;
    int C = 1;                                      // the most channels of a resized photo: sizes the staging
    for (int b = 0; b < B; ++b) {
        PrepImage& g = im[b];
        g.src = p.src_off[b]; g.dst = p.pix_off[b];
        g.w = p.w[b]; g.h = p.h[b]; g.W = p.W[b]; g.H = p.H[b];
        g.ch = p.c[b];
        g.sx = 1.0 / ((double)g.W / g.w);
        g.sy = 1.0 / ((double)g.H / g.h);
        g.kx = g.w / g.W; g.ky = g.h / g.H;
        g.mode = g.W == g.w && g.H == g.h ? PREP_IDENTITY : g.w % g.W == 0 && g.h % g.H == 0 ? PREP_INTEGER : PREP_AREA;
        if (g.mode != PREP_IDENTITY) { fx = std::max(fx, g.sx); fy = std::max(fy, g.sy); C = std::max(C, g.ch); }
        if (g.ch == 1) gray_idx.push_back(b);
    }
    // the largest tile whose source rectangle fits the budget: halve the height first, then the width
    int TW = kTileW, TH = kTileH, nx = 0, ny = 0;
    size_t smem = tile_smem(TW, TH, fx, fy, C, &nx, &ny);
    while (smem > kPrepSmemBudget && (TH > 1 || TW > 1)) {
        if (TH > 1) TH >>= 1; else TW >>= 1;
        smem = tile_smem(TW, TH, fx, fy, C, &nx, &ny);
    }
    int smem_max = 0;
    VPK_CUDA(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
    if (smem > (size_t)smem_max) {
        set_error("image_prep: downscale factor %.1f x %.1f too large: the source of one output pixel needs %zu bytes of "
                  "shared memory (at most %d)", fx, fy, smem, smem_max);
        return VPK_ERR_ARG;
    }
    std::vector<int32_t> tile_off(B + 1, 0);
    for (int b = 0; b < B; ++b) {
        im[b].tiles_x = (im[b].W + TW - 1) / TW;
        const int64_t n = (int64_t)im[b].tiles_x * ((im[b].H + TH - 1) / TH);
        if (tile_off[b] + n > INT32_MAX) { set_error("image_prep: more than 2^31 tiles in one call; split the batch"); return VPK_ERR_ARG; }
        tile_off[b + 1] = tile_off[b] + (int32_t)n;
    }
    const int64_t n_src = p.src_off[B], n_out = p.pix_off[B];
    const int n_gray = (int)gray_idx.size();
    // gray planes of LSD's input (out_scale != 1) follow detect_lsd_lines' rule: each image's "some value > 1" flag
    const bool rule = n_gray > 0 && out_scale != 1.0;
    const size_t im_bytes = (size_t)B * sizeof(PrepImage), tile_bytes = (size_t)(B + 1) * sizeof(int32_t);
    VPK_TRY(s->meta.ensure(im_bytes + tile_bytes + (size_t)n_gray * sizeof(int32_t)));
    VPK_CUDA(cudaMemcpyAsync(s->meta.p, im.data(), im_bytes, cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemcpyAsync(s->meta.as<char>() + im_bytes, tile_off.data(), tile_bytes, cudaMemcpyHostToDevice, st));
    int32_t* d_big = nullptr;
    const int32_t* d_gray = reinterpret_cast<const int32_t*>(s->meta.as<char>() + im_bytes + tile_bytes);
    if (rule) {
        VPK_CUDA(cudaMemcpyAsync(s->meta.as<char>() + im_bytes + tile_bytes, gray_idx.data(), (size_t)n_gray * sizeof(int32_t),
                                 cudaMemcpyHostToDevice, st));
        VPK_TRY(s->big.ensure((size_t)B * sizeof(int32_t)));
        d_big = s->big.as<int32_t>();
        VPK_CUDA(cudaMemsetAsync(d_big, 0, (size_t)B * sizeof(int32_t), st));
    }
    if (smem > 48 * 1024) VPK_CUDA(cudaFuncSetAttribute(image_prep, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    {
        KernelScope ks(ctx, "image_prep");
        image_prep<<<tile_off[B], kPrepThreads, smem, st>>>(s->rgb.as<uint8_t>(), s->meta.as<PrepImage>(),
                                                            reinterpret_cast<const int32_t*>(s->meta.as<char>() + im_bytes), B, TW, TH,
                                                            nx, ny, out_scale, d_out, d_big, n_src, n_out);
        VPK_TRY(check_launch("image_prep"));
    }
    if (rule) {
        int64_t most = 1;
        for (int b : gray_idx) most = std::max<int64_t>(most, (int64_t)p.W[b] * p.H[b]);
        const dim3 grid((unsigned)std::min<int64_t>((most + kPrepThreads - 1) / kPrepThreads, 64), (unsigned)std::min(n_gray, 65535));
        KernelScope ks(ctx, "prep_gray_scale");
        prep_gray_scale<<<grid, kPrepThreads, 0, st>>>(s->meta.as<PrepImage>(), d_gray, n_gray, d_big, out_scale, d_out, n_out);
        VPK_TRY(check_launch("prep_gray_scale"));
    }
    return VPK_OK;
}

}  // namespace vpk

using namespace vpk;

extern "C" {

int vpk_prepared_size(int32_t w, int32_t h, int32_t target_size, int32_t* out_w, int32_t* out_h) {
    if (w <= 0 || h <= 0 || !out_w || !out_h) { set_error("vpk_prepared_size: sides must be > 0 and the outputs non-NULL"); return VPK_ERR_ARG; }
    int W, H;
    prepared_size(w, h, target_size, &W, &H);
    *out_w = W; *out_h = H;
    return VPK_OK;
}

int vpk_prepare_images(vpk_ctx* ctx, const uint8_t* rgb, const int64_t* byte_offsets, const int32_t* widths, const int32_t* heights,
                       int32_t n_images, int32_t target_size, int32_t* out_widths, int32_t* out_heights, double* gray_out) {
    if (!ctx || !out_widths || !out_heights) { set_error("vpk_prepare_images: bad argument"); return VPK_ERR_ARG; }
    PrepPlan p;
    VPK_TRY(prep_plan(byte_offsets, widths, heights, nullptr, n_images, target_size, "vpk_prepare_images", p));
    if (!rgb) { set_error("vpk_prepare_images: rgb is NULL"); return VPK_ERR_ARG; }
    if (!gray_out) { set_error("vpk_prepare_images: gray_out is NULL"); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->prep) ctx->prep = new PrepState();
    const int64_t n_out = p.pix_off[n_images];
    VPK_TRY(ctx->prep->out.ensure((size_t)n_out * sizeof(double)));
    uint8_t* d_rgb = nullptr;
    VPK_TRY(prep_input(ctx, p, &d_rgb));
    VPK_CUDA(cudaMemcpyAsync(d_rgb, rgb, (size_t)p.src_off[n_images], cudaMemcpyHostToDevice, ctx->stream));
    VPK_TRY(prep_run(ctx, p, 1.0, ctx->prep->out.as<double>()));
    VPK_CUDA(cudaMemcpyAsync(gray_out, ctx->prep->out.p, (size_t)n_out * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    memcpy(out_widths, p.W.data(), (size_t)n_images * sizeof(int32_t));
    memcpy(out_heights, p.H.data(), (size_t)n_images * sizeof(int32_t));
    return VPK_OK;
}

}  // extern "C"
