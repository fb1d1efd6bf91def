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
    DBuf rgb, meta, out;
};

void prep_free(vpk_ctx* ctx) {
    if (!ctx->prep) return;
    ctx->prep->rgb.release(); ctx->prep->meta.release(); ctx->prep->out.release();
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

__global__ void __launch_bounds__(kPrepThreads) image_prep(const uint8_t* __restrict__ rgb, const PrepImage* __restrict__ im,
                                                           const int32_t* __restrict__ tile_off, int B, int TW, int TH, int nx_max,
                                                           int ny_max, double out_scale, double* __restrict__ out, int64_t n_src,
                                                           int64_t n_out) {
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
    const int nc = min(TW, g.W - x0), nr = min(TH, g.H - y0);
    PREP_CHECK(nc > 0 && nr > 0);
    const uint8_t* src = rgb + g.src;
    double* dst = out + g.dst;
    if (g.mode == PREP_IDENTITY) {
        for (int i = threadIdx.x; i < nc * nr; i += blockDim.x) {
            const int x = x0 + i % nc, y = y0 + i / nc;
            const int64_t p = ((int64_t)y * g.w + x) * 3;
            PREP_CHECK(g.src + p + 2 < n_src && g.dst + (int64_t)y * g.W + x < n_out);
            dst[(int64_t)y * g.W + x] = gray(src[p], src[p + 1], src[p + 2], out_scale);
        }
        return;
    }
    Taps* tx = reinterpret_cast<Taps*>(smem);
    Taps* ty = tx + TW;
    double* T = reinterpret_cast<double*>(ty + TH);                               // ny_max x TW x 3
    uint8_t* S = reinterpret_cast<uint8_t*>(T + (size_t)ny_max * TW * 3);         // ny_max x nx_max x 3
    if (threadIdx.x < nc) tx[threadIdx.x] = make_taps(x0 + threadIdx.x, g.w, g.sx, g.mode, g.kx);
    else if (threadIdx.x >= TW && threadIdx.x < TW + nr) ty[threadIdx.x - TW] = make_taps(y0 + threadIdx.x - TW, g.h, g.sy, g.mode, g.ky);
    __syncthreads();
    const int xa = tx[0].first, ya = ty[0].first;
    const int nx = last_tap(tx[nc - 1]) - xa + 1, ny = last_tap(ty[nr - 1]) - ya + 1;
    PREP_CHECK(xa >= 0 && ya >= 0 && xa + nx <= g.w && ya + ny <= g.h && nx <= nx_max && ny <= ny_max);
    // stage the source rectangle (row by row, contiguous bytes)
    const int rowb = nx * 3;
    for (int i = threadIdx.x; i < ny * rowb; i += blockDim.x) {
        const int r = i / rowb, c = i - r * rowb;
        const int64_t p = ((int64_t)(ya + r) * g.w + xa) * 3 + c;
        PREP_CHECK(g.src + p < n_src && i < ny_max * nx_max * 3);
        S[i] = src[p];
    }
    __syncthreads();
    // x pass: T[r][j][c] for every staged row r and output column j
    for (int i = threadIdx.x; i < ny * nc * 3; i += blockDim.x) {
        const int c = i % 3, j = (i / 3) % nc, r = i / (3 * nc);
        const Taps& q = tx[j];
        PREP_CHECK(q.first >= xa && last_tap(q) < xa + nx && (r * TW + j) * 3 + c < ny_max * TW * 3);
        T[(r * TW + j) * 3 + c] = tap_sum(q, S + r * rowb + (q.first - xa) * 3 + c, 3);
    }
    __syncthreads();
    // y pass, uint8, gray
    for (int i = threadIdx.x; i < nr * nc; i += blockDim.x) {
        const int j = i % nc, r = i / nc;
        const Taps& q = ty[r];
        PREP_CHECK(q.first >= ya && last_tap(q) < ya + ny);
        const double* col = T + ((q.first - ya) * TW + j) * 3;
        const int v0 = to_u8(tap_sum(q, col, TW * 3), g);
        const int v1 = to_u8(tap_sum(q, col + 1, TW * 3), g);
        const int v2 = to_u8(tap_sum(q, col + 2, TW * 3), g);
        const int64_t o = (int64_t)(y0 + r) * g.W + x0 + j;
        PREP_CHECK(g.dst + o < n_out && v0 >= 0 && v0 <= 255 && v1 >= 0 && v1 <= 255 && v2 >= 0 && v2 <= 255);
        dst[o] = gray(v0, v1, v2, out_scale);
    }
}

static void prepared_size(int w, int h, int target, int* W, int* H) {
    *W = w; *H = h;
    if (target <= 0) return;
    const double s = (double)target / (double)std::max(w, h);
    if (!(s < 1.0)) return;
    *W = std::max(1, (int)nearbyint(w * s));        // rint: half to even, like Python's round
    *H = std::max(1, (int)nearbyint(h * s));
}

int prep_plan(const uint8_t* rgb, const int64_t* byte_offsets, const int32_t* widths, const int32_t* heights, int32_t B,
              int32_t target_size, const char* who, PrepPlan& p) {
    if (!byte_offsets || !widths || !heights || B <= 0) { set_error("%s: bad argument", who); return VPK_ERR_ARG; }
    if (byte_offsets[0] != 0) { set_error("%s: byte_offsets[0] must be 0", who); return VPK_ERR_ARG; }
    p.B = B;
    p.w.assign(widths, widths + B); p.h.assign(heights, heights + B);
    p.W.resize(B); p.H.resize(B);
    p.src_off.assign(byte_offsets, byte_offsets + B + 1);
    p.pix_off.assign(B + 1, 0);
    for (int b = 0; b < B; ++b) {
        const int w = widths[b], h = heights[b];
        if (w <= 0 || h <= 0 || byte_offsets[b + 1] - byte_offsets[b] != 3 * (int64_t)w * h) {
            set_error("%s: photo %d: byte_offsets[b+1] - byte_offsets[b] must be 3 * widths[b] * heights[b] > 0", who, b);
            return VPK_ERR_ARG;
        }
        prepared_size(w, h, target_size, &p.W[b], &p.H[b]);
        p.pix_off[b + 1] = p.pix_off[b] + (int64_t)p.W[b] * p.H[b];
    }
    if (!rgb) { set_error("%s: rgb is NULL", who); return VPK_ERR_ARG; }
    return VPK_OK;
}

// shared memory of a TW x TH tile whose source rectangle spans at most fx, fy source pixels per output pixel
static size_t tile_smem(int TW, int TH, double fx, double fy, int* nx, int* ny) {
    *nx = (int)ceil(TW * fx) + 3;
    *ny = (int)ceil(TH * fy) + 3;
    return (size_t)(TW + TH) * sizeof(Taps) + (size_t)*ny * TW * 3 * sizeof(double) + (((size_t)*nx * *ny * 3 + 15) & ~(size_t)15);
}

int prep_run(vpk_ctx* ctx, const PrepPlan& p, const uint8_t* rgb, double out_scale, double* d_out) {
    const int B = p.B;
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->prep) ctx->prep = new PrepState();
    PrepState* s = ctx->prep;
    cudaStream_t st = ctx->stream;
    std::vector<PrepImage> im(B);
    double fx = 1.0, fy = 1.0;
    for (int b = 0; b < B; ++b) {
        PrepImage& g = im[b];
        g.src = p.src_off[b]; g.dst = p.pix_off[b];
        g.w = p.w[b]; g.h = p.h[b]; g.W = p.W[b]; g.H = p.H[b];
        g.sx = 1.0 / ((double)g.W / g.w);
        g.sy = 1.0 / ((double)g.H / g.h);
        g.kx = g.w / g.W; g.ky = g.h / g.H;
        g.mode = g.W == g.w && g.H == g.h ? PREP_IDENTITY : g.w % g.W == 0 && g.h % g.H == 0 ? PREP_INTEGER : PREP_AREA;
        if (g.mode != PREP_IDENTITY) { fx = std::max(fx, g.sx); fy = std::max(fy, g.sy); }
    }
    // the largest tile whose source rectangle fits the budget: halve the height first, then the width
    int TW = kTileW, TH = kTileH, nx = 0, ny = 0;
    size_t smem = tile_smem(TW, TH, fx, fy, &nx, &ny);
    while (smem > kPrepSmemBudget && (TH > 1 || TW > 1)) {
        if (TH > 1) TH >>= 1; else TW >>= 1;
        smem = tile_smem(TW, TH, fx, fy, &nx, &ny);
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
    const size_t im_bytes = (size_t)B * sizeof(PrepImage);
    VPK_TRY(s->meta.ensure(im_bytes + (size_t)(B + 1) * sizeof(int32_t)));
    VPK_TRY(s->rgb.ensure((size_t)n_src));
    VPK_CUDA(cudaMemcpyAsync(s->meta.p, im.data(), im_bytes, cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemcpyAsync(s->meta.as<char>() + im_bytes, tile_off.data(), (size_t)(B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemcpyAsync(s->rgb.p, rgb, (size_t)n_src, cudaMemcpyHostToDevice, st));
    if (smem > 48 * 1024) VPK_CUDA(cudaFuncSetAttribute(image_prep, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    KernelScope ks(ctx, "image_prep");
    image_prep<<<tile_off[B], kPrepThreads, smem, st>>>(s->rgb.as<uint8_t>(), s->meta.as<PrepImage>(),
                                                        reinterpret_cast<const int32_t*>(s->meta.as<char>() + im_bytes), B, TW, TH,
                                                        nx, ny, out_scale, d_out, n_src, n_out);
    return check_launch("image_prep");
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
    VPK_TRY(prep_plan(rgb, byte_offsets, widths, heights, n_images, target_size, "vpk_prepare_images", p));
    if (!gray_out) { set_error("vpk_prepare_images: gray_out is NULL"); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->prep) ctx->prep = new PrepState();
    const int64_t n_out = p.pix_off[n_images];
    VPK_TRY(ctx->prep->out.ensure((size_t)n_out * sizeof(double)));
    VPK_TRY(prep_run(ctx, p, rgb, 1.0, ctx->prep->out.as<double>()));
    VPK_CUDA(cudaMemcpyAsync(gray_out, ctx->prep->out.p, (size_t)n_out * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    memcpy(out_widths, p.W.data(), (size_t)n_images * sizeof(int32_t));
    memcpy(out_heights, p.H.data(), (size_t)n_images * sizeof(int32_t));
    return VPK_OK;
}

}  // extern "C"
