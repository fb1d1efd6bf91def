// Row N4: the LSD line segment detector 1.6 (lsd.detect_line_segments, reference evaluation.py:227-251) for a
// ragged batch of grayscale images of mixed sizes.
//
//   lsd_sample_x / lsd_sample_y   gaussian_sampler, one thread per output pixel, taps summed in order
//   lsd_gradient                  ll_angle's 2x2 gradient, level-line angle / NOTDEF, per-image max gradient
//   lsd_keys + CUB radix sort     the pseudo-ordering: a stable sort of the pixels, enumerated in ll_angle's
//                                 traversal order (x outer, y inner), on (image, descending bin); NOTDEF pixels
//                                 sort behind every seed of their image
//   lsd_region                    one warp per image walks its seeds in order through lsd_core.cuh and appends
//                                 the rows to the image's slab (lsd.c's output order); warps take images from a
//                                 counter, so a batch larger than the resident warps runs in several waves
//   lsd_gather                    slabs -> the flat (sum N, 7) rows
//
// The `used` map is a bitmap in shared memory when the largest image's fits in kSmemBitmapMax; otherwise every
// warp keeps it in a global-memory slot (same code, another pointer).
#include <cub/device/device_radix_sort.cuh>
#include <algorithm>
#include <cstdlib>
#include "vpk_internal.cuh"
#include "lsd_core.cuh"

namespace vpk {

static constexpr int kThreads = 256;
static constexpr int kMaxSlots = 1024;                  // warps of the region kernel (bounds the region scratch)
static constexpr size_t kSmemBitmapMax = 96 * 1024;     // 786432 pixels of the sampled image
static constexpr int kDefaultCap = 2048;                // rows per image slab before an image is re-run with more

struct LsdState {
    int B = 0;
    int64_t sumN = 0;
    DBuf in, aux, smp, ang, mod, maxg, meta, ktab, keys, vals, keys2, vals2, sort_tmp, used, reg, slab, counts, row_off,
        rows, next;
};

void lsd_free(vpk_ctx* ctx) {
    if (!ctx->lsd) return;
    LsdState* s = ctx->lsd;
    for (DBuf* b : {&s->in, &s->aux, &s->smp, &s->ang, &s->mod, &s->maxg, &s->meta, &s->ktab, &s->keys, &s->vals, &s->keys2,
                    &s->vals2, &s->sort_tmp, &s->used, &s->reg, &s->slab, &s->counts, &s->row_off, &s->rows, &s->next})
        b->release();
    delete s;
    ctx->lsd = nullptr;
}

// per-image geometry on the device: offsets (B+1 each) of the input, x-pass, sampled-pixel and seed-item arrays,
// then the input and sampled sizes (B each)
struct Meta {
    const int64_t *in_off, *aux_off, *pix_off, *item_off;
    const int32_t *W, *H, *X, *Y;
};

__device__ __forceinline__ int find_image(const int64_t* off, int B, int64_t i) {
    int lo = 0, hi = B - 1;
    while (lo < hi) {                               // last image with off[b] <= i
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid - 1;
    }
    return lo;
}

template <typename T>
__global__ void lsd_sample_x(const T* __restrict__ in, Meta m, int B, double scale, int h, const double* __restrict__ ktab,
                             double* __restrict__ aux) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= m.aux_off[B]) return;
    const int b = find_image(m.aux_off, B, i);
    const int X = m.X[b], W = m.W[b];
    const int64_t l = i - m.aux_off[b];
    const int x = (int)(l % X), y = (int)(l / X);
    const int xc = lsd::sampler_centre(x, scale), n = 2 * h + 1;
    const T* row = in + m.in_off[b] + (int64_t)y * W;
    double s = 0.0;
    for (int t = 0; t < n; ++t) s = lsd::add(s, lsd::mul((double)row[lsd::mirror(xc - h + t, W)], ktab[(int64_t)x * n + t]));
    aux[i] = s;
}

__global__ void lsd_sample_y(const double* __restrict__ aux, Meta m, int B, double scale, int h, const double* __restrict__ ktab,
                             double* __restrict__ out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= m.pix_off[B]) return;
    const int b = find_image(m.pix_off, B, i);
    const int X = m.X[b], H = m.H[b];
    const int64_t l = i - m.pix_off[b];
    const int x = (int)(l % X), y = (int)(l / X);
    const int yc = lsd::sampler_centre(y, scale), n = 2 * h + 1;
    const double* col = aux + m.aux_off[b] + x;
    double s = 0.0;
    for (int t = 0; t < n; ++t) s = lsd::add(s, lsd::mul(col[(int64_t)lsd::mirror(yc - h + t, H) * X], ktab[(int64_t)y * n + t]));
    out[i] = s;
}

// img: the sampled image (double), or the input itself at scale 1 (then its offsets are in_off == pix_off)
template <typename T>
__global__ void lsd_gradient(const T* __restrict__ img, Meta m, int B, double rho, double* __restrict__ ang, double* __restrict__ mod,
                             unsigned long long* __restrict__ maxg) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= m.pix_off[B]) return;
    const int b = find_image(m.pix_off, B, i);
    const int X = m.X[b], Y = m.Y[b];
    const int64_t l = i - m.pix_off[b];
    const int x = (int)(l % X), y = (int)(l / X);
    if (x == X - 1 || y == Y - 1) { ang[i] = lsd::kNotDef; mod[i] = 0.0; return; }
    const T* p = img + m.pix_off[b] + l;
    double a;
    const double norm = lsd::gradient((double)p[0], (double)p[1], (double)p[X], (double)p[X + 1], rho, &a);
    ang[i] = a;
    mod[i] = norm;
    if (a != lsd::kNotDef) atomicMax(maxg + b, (unsigned long long)__double_as_longlong(norm));   // norm > 0: bits order as values
}

__global__ void lsd_keys(Meta m, int B, int n_bins, const double* __restrict__ ang, const double* __restrict__ mod,
                         const unsigned long long* __restrict__ maxg, unsigned long long* __restrict__ keys, uint32_t* __restrict__ vals) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= m.item_off[B]) return;
    const int b = find_image(m.item_off, B, i);
    const int X = m.X[b], Y = m.Y[b];
    const int64_t t = i - m.item_off[b];
    const int x = (int)(t / (Y - 1)), y = (int)(t % (Y - 1));
    const int a = x + y * X;
    const int64_t p = m.pix_off[b] + a;
    const int k = ang[p] == lsd::kNotDef ? n_bins : n_bins - 1 - lsd::grad_bin(mod[p], n_bins, __longlong_as_double((long long)maxg[b]));
    keys[i] = (unsigned long long)b * (unsigned long long)(n_bins + 1) + (unsigned long long)k;
    vals[i] = (uint32_t)a;
}

struct RegionArgs {
    double scale, ang_th, log_eps, density_th;
    int n_bins, B, cap;
    bool smem_used;
    size_t used_words, reg_slot;    // per warp slot (global bitmap only when !smem_used)
};

__global__ void __launch_bounds__(32) lsd_region(Meta m, RegionArgs r, const double* __restrict__ ang, const double* __restrict__ mod,
                                                 const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                 uint32_t* used_g, uint32_t* reg_g, double* __restrict__ slab, int32_t* __restrict__ counts,
                                                 int* next) {
    extern __shared__ uint32_t used_s[];
    const int lane = threadIdx.x & 31;
    uint32_t* used = r.smem_used ? used_s : used_g + (size_t)blockIdx.x * r.used_words;
    uint32_t* reg = reg_g + (size_t)blockIdx.x * r.reg_slot;
    for (;;) {
        int b = 0;
        if (lane == 0) b = atomicAdd(next, 1);
        b = __shfl_sync(0xffffffffu, b, 0);
        if (b >= r.B) break;
        const int X = m.X[b], Y = m.Y[b];
        const int words = (X * Y + 31) >> 5;
        for (int w = lane; w < words; w += 32) {
            LSD_CHECK(w < (r.smem_used ? words : (int)r.used_words));
            used[w] = 0u;
        }
        __syncwarp();
        lsd::View v{ang + m.pix_off[b], mod + m.pix_off[b], used, reg, X, Y};
        const lsd::Params q = lsd::make_params(r.scale, r.ang_th, r.log_eps, r.density_th, X, Y);
        const unsigned long long notdef = (unsigned long long)b * (unsigned long long)(r.n_bins + 1) + (unsigned long long)r.n_bins;
        int count = 0;
        for (int64_t s = m.item_off[b]; s < m.item_off[b + 1] && keys[s] != notdef; ++s) {
            const int a = (int)vals[s];
            if (lsd::used_get(v, a)) continue;
            double row[7];
            if (!lsd::process_seed(v, a % X, a / X, q, row)) continue;
            if (lane == 0 && count < r.cap) {
                double* dst = slab + ((size_t)b * r.cap + count) * 7;
                LSD_CHECK((size_t)b * r.cap + count < (size_t)r.B * r.cap);
                for (int c = 0; c < 7; ++c) dst[c] = row[c];
            }
            ++count;
        }
        if (lane == 0) counts[b] = count;
        __syncwarp();
    }
}

__global__ void lsd_gather(const double* __restrict__ slab, const int32_t* __restrict__ row_off, int B, int cap, double* __restrict__ rows) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= (int64_t)row_off[B] * 7) return;
    const int64_t rr = i / 7;
    int lo = 0, hi = B - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (row_off[mid] <= rr) lo = mid; else hi = mid - 1;
    }
    rows[i] = slab[((size_t)lo * cap + (rr - row_off[lo])) * 7 + i % 7];
}

static unsigned blocks(int64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

static Meta meta_view(const char* mp, int B) {
    Meta m;
    m.in_off = reinterpret_cast<const int64_t*>(mp);
    m.aux_off = m.in_off + (B + 1); m.pix_off = m.aux_off + (B + 1); m.item_off = m.pix_off + (B + 1);
    m.W = reinterpret_cast<const int32_t*>(m.item_off + (B + 1));
    m.H = m.W + B; m.X = m.H + B; m.Y = m.X + B;
    return m;
}

int lsd_plan(const int64_t* pixel_offsets, const int32_t* widths, const int32_t* heights, int32_t B, int32_t dtype,
             const vpk_lsd_config* cfg_in, int32_t* counts_out, LsdPlan& p) {
    vpk_lsd_config& cfg = p.cfg;
    if (cfg_in) cfg = *cfg_in; else vpk_lsd_default_config(&cfg);
    if (!pixel_offsets || !widths || !heights || B <= 0 || !counts_out) { set_error("vpk_lsd: bad argument"); return VPK_ERR_ARG; }
    if (dtype != VPK_PIX_U8 && dtype != VPK_PIX_F64) { set_error("vpk_lsd: dtype must be VPK_PIX_U8 or VPK_PIX_F64"); return VPK_ERR_ARG; }
    if (!(cfg.scale > 0.0) || !(cfg.sigma_scale > 0.0) || !(cfg.quant >= 0.0) || !(cfg.ang_th > 0.0 && cfg.ang_th < 180.0) ||
        !(cfg.density_th >= 0.0 && cfg.density_th <= 1.0) || cfg.n_bins <= 0 || cfg.n_bins > (1 << 24)) {
        set_error("vpk_lsd: parameter out of range (scale, sigma_scale > 0; quant >= 0; 0 < ang_th < 180; 0 <= density_th <= 1; n_bins >= 1)");
        return VPK_ERR_ARG;
    }
    if (pixel_offsets[0] != 0) { set_error("vpk_lsd: pixel_offsets[0] must be 0"); return VPK_ERR_ARG; }
    p.B = B; p.dtype = dtype;
    // geometry: int64 offsets for in / aux / pix / item, then W, H, X, Y
    p.off64.assign(4 * (size_t)(B + 1), 0);
    p.dims.assign(4 * (size_t)B, 0);
    int64_t *in_off = p.off64.data(), *aux_off = in_off + (B + 1), *pix_off = aux_off + (B + 1), *item_off = pix_off + (B + 1);
    int32_t* dims = p.dims.data();
    p.maxX = 0; p.maxY = 0; p.max_pix = 0;
    for (int b = 0; b < B; ++b) {
        const int W = widths[b], H = heights[b];
        if (W <= 0 || H <= 0 || pixel_offsets[b + 1] - pixel_offsets[b] != (int64_t)W * H) {
            set_error("vpk_lsd: image %d: pixel_offsets[b+1] - pixel_offsets[b] must be widths[b] * heights[b] > 0", b);
            return VPK_ERR_ARG;
        }
        const double xs = ceil(W * cfg.scale), ys = ceil(H * cfg.scale);     // gaussian_sampler's N, M
        if (xs >= 65536.0 || ys >= 65536.0) {
            set_error("vpk_lsd: image %d: sampled size %.0f x %.0f, each side must be below 65536", b, xs, ys);
            return VPK_ERR_ARG;
        }
        const int X = cfg.scale != 1.0 ? (int)xs : W, Y = cfg.scale != 1.0 ? (int)ys : H;
        dims[b] = W; dims[B + b] = H; dims[2 * B + b] = X; dims[3 * B + b] = Y;
        in_off[b + 1] = pixel_offsets[b + 1];
        aux_off[b + 1] = aux_off[b] + (int64_t)X * H;
        pix_off[b + 1] = pix_off[b] + (int64_t)X * Y;
        item_off[b + 1] = item_off[b] + (X > 1 && Y > 1 ? (int64_t)(X - 1) * (Y - 1) : 0);
        p.maxX = std::max(p.maxX, X); p.maxY = std::max(p.maxY, Y);
        p.max_pix = std::max(p.max_pix, (int64_t)X * Y);
    }
    if (item_off[B] > INT32_MAX) { set_error("vpk_lsd: %lld pixels in one call; split the batch below 2^31", (long long)item_off[B]); return VPK_ERR_ARG; }
    return VPK_OK;
}

int lsd_input(vpk_ctx* ctx, const LsdPlan& p, void** d_in) {
    const int B = p.B;
    const int64_t* in_off = p.off64.data();
    const int64_t *aux_off = in_off + (B + 1), *pix_off = aux_off + (B + 1), *item_off = pix_off + (B + 1);
    const int64_t n_in = in_off[B], n_pix = pix_off[B], n_items = item_off[B];
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->lsd) ctx->lsd = new LsdState();
    LsdState* s = ctx->lsd;
    s->B = 0; s->sumN = 0;
    cudaStream_t st = ctx->stream;
    const size_t esz = p.dtype == VPK_PIX_U8 ? 1 : sizeof(double);
    const bool sampled = p.cfg.scale != 1.0;
    VPK_TRY(s->meta.ensure(p.off64.size() * sizeof(int64_t) + p.dims.size() * sizeof(int32_t)));
    VPK_TRY(s->in.ensure((size_t)n_in * esz));
    if (sampled) { VPK_TRY(s->aux.ensure((size_t)aux_off[B] * sizeof(double))); VPK_TRY(s->smp.ensure((size_t)n_pix * sizeof(double))); }
    VPK_TRY(s->ang.ensure((size_t)n_pix * sizeof(double)));
    VPK_TRY(s->mod.ensure((size_t)n_pix * sizeof(double)));
    VPK_TRY(s->maxg.ensure((size_t)B * sizeof(unsigned long long)));
    VPK_TRY(s->keys.ensure((size_t)(n_items + 1) * 8)); VPK_TRY(s->keys2.ensure((size_t)(n_items + 1) * 8));
    VPK_TRY(s->vals.ensure((size_t)(n_items + 1) * 4)); VPK_TRY(s->vals2.ensure((size_t)(n_items + 1) * 4));
    VPK_TRY(s->counts.ensure((size_t)B * sizeof(int32_t)));
    VPK_TRY(s->next.ensure(sizeof(int)));
    char* mp = s->meta.as<char>();
    VPK_CUDA(cudaMemcpyAsync(mp, p.off64.data(), p.off64.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemcpyAsync(mp + p.off64.size() * sizeof(int64_t), p.dims.data(), p.dims.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    *d_in = s->in.p;
    return VPK_OK;
}

int lsd_detect(vpk_ctx* ctx, const LsdPlan& p, int32_t* counts_out, const double** d_rows, std::vector<int32_t>& row_offsets) {
    const int B = p.B;
    const vpk_lsd_config& cfg = p.cfg;
    const int32_t dtype = p.dtype;
    const int64_t* in_off = p.off64.data();
    const int64_t *aux_off = in_off + (B + 1), *pix_off = aux_off + (B + 1), *item_off = pix_off + (B + 1);
    const int64_t n_pix = pix_off[B], n_items = item_off[B];
    const int maxX = p.maxX, maxY = p.maxY;
    const int64_t max_pix = p.max_pix;
    LsdState* s = ctx->lsd;
    cudaStream_t st = ctx->stream;
    const bool sampled = cfg.scale != 1.0;
    const Meta m = meta_view(s->meta.as<char>(), B);
    VPK_CUDA(cudaMemsetAsync(s->maxg.p, 0, (size_t)B * sizeof(unsigned long long), st));

    const double prec = lsd::dv(lsd::mul(lsd::kPi, cfg.ang_th), 180.0);
    const double rho = lsd::dv(cfg.quant, sin(prec));
    double* ang = s->ang.as<double>();
    double* mod = s->mod.as<double>();
    unsigned long long* maxg = s->maxg.as<unsigned long long>();
    if (sampled) {
        const int h = lsd::sampler_half(cfg.scale, cfg.sigma_scale), n = 2 * h + 1;
        const int positions = std::max(maxX, maxY);
        std::vector<double> ktab((size_t)positions * n);
        lsd::sampler_table(cfg.scale, cfg.sigma_scale, positions, ktab.data());
        VPK_TRY(s->ktab.ensure(ktab.size() * sizeof(double)));
        VPK_CUDA(cudaMemcpyAsync(s->ktab.p, ktab.data(), ktab.size() * sizeof(double), cudaMemcpyHostToDevice, st));
        {
            KernelScope ks(ctx, "lsd_sample_x");
            if (dtype == VPK_PIX_U8)
                lsd_sample_x<uint8_t><<<blocks(aux_off[B]), kThreads, 0, st>>>(s->in.as<uint8_t>(), m, B, cfg.scale, h, s->ktab.as<double>(), s->aux.as<double>());
            else
                lsd_sample_x<double><<<blocks(aux_off[B]), kThreads, 0, st>>>(s->in.as<double>(), m, B, cfg.scale, h, s->ktab.as<double>(), s->aux.as<double>());
            VPK_TRY(check_launch("lsd_sample_x"));
        }
        {
            KernelScope ks(ctx, "lsd_sample_y");
            lsd_sample_y<<<blocks(n_pix), kThreads, 0, st>>>(s->aux.as<double>(), m, B, cfg.scale, h, s->ktab.as<double>(), s->smp.as<double>());
            VPK_TRY(check_launch("lsd_sample_y"));
        }
        KernelScope ks(ctx, "lsd_gradient");
        lsd_gradient<double><<<blocks(n_pix), kThreads, 0, st>>>(s->smp.as<double>(), m, B, rho, ang, mod, maxg);
        VPK_TRY(check_launch("lsd_gradient"));
    } else {
        KernelScope ks(ctx, "lsd_gradient");
        if (dtype == VPK_PIX_U8) lsd_gradient<uint8_t><<<blocks(n_pix), kThreads, 0, st>>>(s->in.as<uint8_t>(), m, B, rho, ang, mod, maxg);
        else lsd_gradient<double><<<blocks(n_pix), kThreads, 0, st>>>(s->in.as<double>(), m, B, rho, ang, mod, maxg);
        VPK_TRY(check_launch("lsd_gradient"));
    }
    unsigned long long* keys_out = s->keys2.as<unsigned long long>();
    uint32_t* vals_out = s->vals2.as<uint32_t>();
    if (n_items) {
        {
            KernelScope ks(ctx, "lsd_keys");
            lsd_keys<<<blocks(n_items), kThreads, 0, st>>>(m, B, cfg.n_bins, ang, mod, maxg, s->keys.as<unsigned long long>(), s->vals.as<uint32_t>());
            VPK_TRY(check_launch("lsd_keys"));
        }
        const unsigned long long max_key = (unsigned long long)B * (unsigned long long)(cfg.n_bins + 1);
        int end_bit = 1;
        while (end_bit < 64 && (max_key >> end_bit) != 0) ++end_bit;
        size_t tmp = 0;
        VPK_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, s->keys.as<unsigned long long>(), keys_out, s->vals.as<uint32_t>(), vals_out,
                                                 (int)n_items, 0, end_bit, st));
        VPK_TRY(s->sort_tmp.ensure(tmp));
        KernelScope ks(ctx, "lsd_sort");
        VPK_CUDA(cub::DeviceRadixSort::SortPairs(s->sort_tmp.p, tmp, s->keys.as<unsigned long long>(), keys_out, s->vals.as<uint32_t>(), vals_out,
                                                 (int)n_items, 0, end_bit, st));
    }

    // region stage
    const size_t bitmap_bytes = (size_t)((max_pix + 31) / 32) * 4;
    const bool smem_used = bitmap_bytes <= kSmemBitmapMax;
    const size_t smem = smem_used ? bitmap_bytes : 0;
    if (smem > 48 * 1024) VPK_CUDA(cudaFuncSetAttribute(lsd_region, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    VPK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lsd_region, 32, smem));
    const int slots = std::max(1, std::min({B, std::max(per_sm, 1) * ctx->num_sms, kMaxSlots}));
    RegionArgs ra;
    ra.scale = cfg.scale; ra.ang_th = cfg.ang_th; ra.log_eps = cfg.log_eps; ra.density_th = cfg.density_th;
    ra.n_bins = cfg.n_bins; ra.B = B; ra.smem_used = smem_used;
    ra.used_words = smem_used ? 0 : bitmap_bytes / 4;
    ra.reg_slot = (size_t)max_pix;
    VPK_TRY(s->reg.ensure((size_t)slots * ra.reg_slot * sizeof(uint32_t)));
    if (!smem_used) VPK_TRY(s->used.ensure((size_t)slots * bitmap_bytes));
    static const int cap_env = getenv("VPK_LSD_ROWS_CAP") ? atoi(getenv("VPK_LSD_ROWS_CAP")) : 0;   // tests: force the re-run
    int cap = cap_env > 0 ? cap_env : kDefaultCap;
    std::vector<int32_t> counts(B);
    for (int pass = 0; pass < 2; ++pass) {
        ra.cap = cap;
        VPK_TRY(s->slab.ensure((size_t)B * cap * 7 * sizeof(double)));
        VPK_CUDA(cudaMemsetAsync(s->next.p, 0, sizeof(int), st));
        {
            KernelScope ks(ctx, "lsd_region");
            lsd_region<<<slots, 32, smem, st>>>(m, ra, ang, mod, keys_out, vals_out, s->used.as<uint32_t>(), s->reg.as<uint32_t>(),
                                                s->slab.as<double>(), s->counts.as<int32_t>(), s->next.as<int>());
            VPK_TRY(check_launch("lsd_region"));
        }
        VPK_CUDA(cudaMemcpyAsync(counts.data(), s->counts.p, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        VPK_CUDA(cudaStreamSynchronize(st));
        const int most = *std::max_element(counts.begin(), counts.end());
        if (most <= cap) break;
        cap = most;      // the detector is deterministic: the re-run finds exactly these rows again
    }
    row_offsets.assign(B + 1, 0);
    for (int b = 0; b < B; ++b) {
        if ((int64_t)row_offsets[b] + counts[b] > INT32_MAX) { set_error("vpk_lsd: more than 2^31 segments"); return VPK_ERR_ARG; }
        row_offsets[b + 1] = row_offsets[b] + counts[b];
    }
    const int64_t sumN = row_offsets[B];
    VPK_TRY(s->row_off.ensure((size_t)(B + 1) * sizeof(int32_t)));
    VPK_TRY(s->rows.ensure((size_t)(sumN + 1) * 7 * sizeof(double)));
    VPK_CUDA(cudaMemcpyAsync(s->row_off.p, row_offsets.data(), (size_t)(B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (sumN) {
        KernelScope ks(ctx, "lsd_gather");
        lsd_gather<<<blocks(sumN * 7), kThreads, 0, st>>>(s->slab.as<double>(), s->row_off.as<int32_t>(), B, ra.cap, s->rows.as<double>());
        VPK_TRY(check_launch("lsd_gather"));
    }
    memcpy(counts_out, counts.data(), (size_t)B * sizeof(int32_t));
    s->B = B;
    s->sumN = sumN;
    *d_rows = s->rows.as<double>();
    return VPK_OK;
}

int lsd_dev(vpk_ctx* ctx, const void* images, int32_t dtype, const int64_t* pixel_offsets, const int32_t* widths,
            const int32_t* heights, int32_t B, const vpk_lsd_config* cfg_in, int32_t* counts_out, const double** d_rows,
            std::vector<int32_t>& row_offsets) {
    if (!ctx) { set_error("vpk_lsd: bad argument"); return VPK_ERR_ARG; }
    LsdPlan p;
    VPK_TRY(lsd_plan(pixel_offsets, widths, heights, B, dtype, cfg_in, counts_out, p));
    if (!images) { set_error("vpk_lsd: images is NULL"); return VPK_ERR_ARG; }
    void* d_in = nullptr;
    VPK_TRY(lsd_input(ctx, p, &d_in));
    const int64_t n_in = p.off64[B];
    const size_t esz = dtype == VPK_PIX_U8 ? 1 : sizeof(double);
    if (n_in) VPK_CUDA(cudaMemcpyAsync(d_in, images, (size_t)n_in * esz, cudaMemcpyHostToDevice, ctx->stream));
    return lsd_detect(ctx, p, counts_out, d_rows, row_offsets);
}

}  // namespace vpk

using namespace vpk;

extern "C" {

void vpk_lsd_default_config(vpk_lsd_config* cfg) {
    if (!cfg) return;
    cfg->scale = 0.8; cfg->sigma_scale = 0.6; cfg->quant = 2.0; cfg->ang_th = 22.5;
    cfg->log_eps = 0.0; cfg->density_th = 0.7; cfg->n_bins = 1024;
}

int vpk_lsd(vpk_ctx* ctx, const void* images, int32_t dtype, const int64_t* pixel_offsets, const int32_t* widths,
            const int32_t* heights, int32_t B, const vpk_lsd_config* cfg, int32_t* counts_out) {
    const double* d_rows = nullptr;
    std::vector<int32_t> row_off;
    VPK_TRY(lsd_dev(ctx, images, dtype, pixel_offsets, widths, heights, B, cfg, counts_out, &d_rows, row_off));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    return VPK_OK;
}

int vpk_lsd_fetch(vpk_ctx* ctx, double* rows_out) {
    if (!ctx || !ctx->lsd || ctx->lsd->B <= 0) { set_error("vpk_lsd_fetch: no vpk_lsd result on this context"); return VPK_ERR_STATE; }
    if (ctx->lsd->sumN == 0) return VPK_OK;
    if (!rows_out) { set_error("vpk_lsd_fetch: rows_out is NULL"); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    VPK_CUDA(cudaMemcpyAsync(rows_out, ctx->lsd->rows.p, (size_t)ctx->lsd->sumN * 7 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    return VPK_OK;
}

}  // extern "C"
