// Stage 2: forward pass of cnn/deploy.prototxt (reference evaluation.py:17-38).
//
// data 1x500x500 -> conv1(96,k11,s4)+ReLU -> LRN -> pool -> conv2(256,k5,p2,g2)
// +ReLU -> LRN -> pool -> conv3(384,k3,p1)+ReLU -> conv4(384,k3,p1,g2)+ReLU ->
// conv5(256,k3,p1,g2)+ReLU -> pool -> fc6+ReLU -> fc7+ReLU -> fc8 -> sigmoid.
//
// Every contraction runs on the tcgen05 implicit-GEMM kernel of
// gemm_tcgen05.cuh; activations are bf16 NHWC with the next layer's zero
// padding stored in memory, so a k x k convolution is k*k row-shifted 2-D TMA
// loads of the same tensor.  conv1 (stride 4, one input channel) is first
// turned into a stride-1 3x3 convolution over a 4x4 space-to-depth image.
// Bias + ReLU are fused into the GEMM epilogue; LRN + max-pool are one fused
// elementwise kernel (Caffe semantics: ACROSS_CHANNELS, ceil-mode pooling).
#include <math.h>
#include "vpk_internal.cuh"
#include "gemm_tcgen05.cuh"

namespace vpk {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct CnnState {
    bool loaded = false;
    bool attr2 = false, attr3 = false, attr4 = false;     // dynamic shared-memory opt-in of the two GEMM instantiations: per CONTEXT (device)
    bool attr_p3 = false, attr_p4 = false, attr_p6 = false, attr_p1 = false;      // ... of the persistent instantiations
    bool persistent = true;                                  // the convolutions through the persistent kernel (VPK_GEMM_PERSIST=0: off)
    EncodeTiledFn encode = nullptr;
    // bf16 weight matrices (K-major) and fp32 biases, one per layer conv1..fc8
    DBuf w[8], b[8], mean;
    bool has_mean = false;
    // activations (sized for `cap` images)
    int cap = 0;
    DBuf a1, c1, a2, c2, a3, a4, a5, c5, a6, f6, f7, logits, sig, img, splitk;
    int last_n = 0;                                          // images of the last chunk vpk_cnn_forward ran (0: none, see vpk_cnn_debug_fetch)
};

void cnn_free(vpk_ctx* ctx) {
    if (!ctx->cnn) return;
    CnnState* s = ctx->cnn;
    for (int i = 0; i < 8; ++i) { s->w[i].release(); s->b[i].release(); }
    s->mean.release();
    DBuf* bufs[] = {&s->a1, &s->c1, &s->a2, &s->c2, &s->a3, &s->a4, &s->a5, &s->c5, &s->a6, &s->f6, &s->f7, &s->logits, &s->sig, &s->img, &s->splitk};
    for (DBuf* d : bufs) d->release();
    delete s;
    ctx->cnn = nullptr;
}

// ---------------------------------------------------------------------------
// weight repacking (device side): fp32 Caffe blobs -> bf16 K-major GEMM operands
// ---------------------------------------------------------------------------
enum { PACK_CONV1 = 0, PACK_CONV = 1, PACK_FC6 = 2, PACK_PLAIN = 3 };

// dst[o, k] for o < n_out, k < k_total
__global__ void pack_weights_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int mode, int n_out,
                                    long long k_total, int cin_g, int cpad, int ksz) {
    long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (idx >= (long long)n_out * k_total) return;
    int o = (int)(idx / k_total);
    long long k = idx % k_total;
    float v = 0.f;
    if (mode == PACK_CONV1) {
        // k = khb*64 + kwb*16 + dy*4 + dx  ->  W[o][0][4*khb+dy][4*kwb+dx]   (11x11, zero beyond)
        int khb = (int)(k / 64), r = (int)(k % 64), kwb = r / 16, dy = (r % 16) / 4, dx = r % 4;
        int row = 4 * khb + dy, col = 4 * kwb + dx;
        if (row < 11 && col < 11) v = src[(o * 11 + row) * 11 + col];
    } else if (mode == PACK_CONV) {
        // k = tap*cpad + c  ->  W[o][c][kh][kw]  (c < cin_g, zero for the channel padding)
        int tap = (int)(k / cpad), c = (int)(k % cpad);
        if (c < cin_g) v = src[((long long)o * cin_g + c) * ksz * ksz + tap];
    } else if (mode == PACK_FC6) {
        // ours: k = (y*15+x)*256 + c ; Caffe flattens NCHW: c*225 + y*15 + x
        int pix = (int)(k / 256), c = (int)(k % 256);
        v = src[(long long)o * k_total + (long long)c * 225 + pix];
    } else {
        v = src[(long long)o * k_total + k];
    }
    dst[idx] = __float2bfloat16_rn(v);
}

// ---------------------------------------------------------------------------
// elementwise kernels
// ---------------------------------------------------------------------------
// image - mean -> conv1 operand: row (n, Y, X) of the 125x125 block grid holds the
// 4x4 pixel blocks X..X+3 of block row Y (64 bf16), so the three kernel block rows
// are three row-shifted K blocks of one 2-D tensor.
__global__ void conv1_operand_kernel(const uint8_t* __restrict__ img, const float* __restrict__ mean, int n_images,
                                     __nv_bfloat16* __restrict__ a1) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;      // one thread per (row, 8-value chunk)
    long long rows = (long long)n_images * 15625;
    if (t >= rows * 8) return;
    long long m = t >> 3;
    int q = (int)(t & 7);
    int n = (int)(m / 15625), r = (int)(m % 15625), Y = r / 125, X = r % 125;
    int kwb = q >> 1;
    uint32_t pk[4];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        int dy = (q & 1) * 2 + h;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        if (X + kwb < 125) {
            int py = 4 * Y + dy, px = 4 * (X + kwb);
            const uint8_t* p = img + ((long long)n * 500 + py) * 500 + px;
            uchar4 u = *reinterpret_cast<const uchar4*>(p);
            v[0] = u.x; v[1] = u.y; v[2] = u.z; v[3] = u.w;
            if (mean) {
                const float* mp = mean + py * 500 + px;
                v[0] -= mp[0]; v[1] -= mp[1]; v[2] -= mp[2]; v[3] -= mp[3];
            }
        }
        __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
        pk[2 * h] = *reinterpret_cast<uint32_t*>(&lo);
        pk[2 * h + 1] = *reinterpret_cast<uint32_t*>(&hi);
    }
    *reinterpret_cast<uint4*>(a1 + m * 64 + q * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
}

// Fused LRN (ACROSS_CHANNELS, size 5, alpha 1e-4, beta 0.75, k 1) + 3x3/2 ceil-mode max
// pool (Caffe).  in: NHWC (n,H,W,C) bf16, C % 8 == 0.  out: (n, Ho+2*opad, Wo+2*opad, Cout)
// with channel c stored at (c / cg) * cgp + c % cg  (group padding of the next convolution;
// cg % 8 == 0).
// One thread owns 8 channels of a 2x2 block of output pixels: it walks the 5x5 input
// patch once (16-byte loads + two 4-byte channel-halo loads per pixel), normalises each
// pixel once and folds it into the up to four windows it belongs to.
__device__ __forceinline__ void bf16x8_to_float(const uint4& v, float f[8]) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 t = __bfloat1622float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
}

template <bool kLrn>
__global__ void __launch_bounds__(256) lrn_pool_kernel(const __nv_bfloat16* __restrict__ in, int n_images, int H, int W, int C,
                                                       int Ho, int Wo, int opad, int Cout, int cg, int cgp,
                                                       __nv_bfloat16* __restrict__ out) {
    const int CG = C >> 3, Hb = (Ho + 1) >> 1, Wb = (Wo + 1) >> 1;
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long total = (long long)n_images * Hb * Wb * CG;
    if (t >= total) return;
    const int g = (int)(t % CG);
    long long r = t / CG;
    const int bx = (int)(r % Wb); r /= Wb;
    const int by = (int)(r % Hb);
    const int n = (int)(r / Hb);
    const int c0 = g * 8;
    const int oy0 = by * 2, ox0 = bx * 2;
    const int y0 = oy0 * 2, x0 = ox0 * 2;
    float best[2][2][8];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b)
#pragma unroll
            for (int k = 0; k < 8; ++k) best[a][b][k] = -INFINITY;
#pragma unroll
    for (int dy = 0; dy < 5; ++dy) {
        const int y = y0 + dy;
        // the five loads of a patch row are issued together (no early exits in between), then reduced
        uint4 raw[5];
        bool ok[5];
#pragma unroll
        for (int dx = 0; dx < 5; ++dx) {
            const int x = x0 + dx;
            ok[dx] = y < H && x < W;
            raw[dx] = make_uint4(0u, 0u, 0u, 0u);
            if (ok[dx]) raw[dx] = *reinterpret_cast<const uint4*>(in + (((long long)n * H + y) * W + x) * C + c0);
        }
#pragma unroll
        for (int dx = 0; dx < 5; ++dx) {
            if (!ok[dx]) continue;
            float v[8];
            bf16x8_to_float(raw[dx], v);
            if (kLrn) {
                const __nv_bfloat16* p = in + (((long long)n * H + y) * W + x0 + dx) * C + c0;
                float lo0 = 0.f, lo1 = 0.f, hi0 = 0.f, hi1 = 0.f;
                if (c0 > 0) { float2 q = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p - 2)); lo0 = q.x; lo1 = q.y; }
                if (c0 + 8 < C) { float2 q = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p + 8)); hi0 = q.x; hi1 = q.y; }
                float sq[12];
                sq[0] = lo0 * lo0; sq[1] = lo1 * lo1; sq[10] = hi0 * hi0; sq[11] = hi1 * hi1;
#pragma unroll
                for (int k = 0; k < 8; ++k) sq[2 + k] = v[k] * v[k];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float ss = sq[k] + sq[k + 1] + sq[k + 2] + sq[k + 3] + sq[k + 4];
                    v[k] = v[k] * __powf(1.f + (1e-4f / 5.f) * ss, -0.75f);
                }
            }
            // rows dy 0..2 feed output row 0, rows 2..4 output row 1 (same for columns)
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int b = 0; b < 2; ++b)
                    if (dy >= 2 * a && dy <= 2 * a + 2 && dx >= 2 * b && dx <= 2 * b + 2) {
#pragma unroll
                        for (int k = 0; k < 8; ++k) best[a][b][k] = fmaxf(best[a][b][k], v[k]);
                    }
        }
    }
    const int Hop = Ho + 2 * opad, Wop = Wo + 2 * opad;
    const int co = (c0 / cg) * cgp + (c0 % cg);
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            const int oy = oy0 + a, ox = ox0 + b;
            if (oy < Ho && ox < Wo) {
                uint4 o;
                __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
                for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(best[a][b][2 * i], best[a][b][2 * i + 1]);
                *reinterpret_cast<uint4*>(out + (((long long)n * Hop + oy + opad) * Wop + ox + opad) * Cout + co) = o;
            }
        }
}

__global__ void sigmoid_kernel(const float* __restrict__ x, long long n, float* __restrict__ y) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) y[i] = 1.f / (1.f + __expf(-x[i]));
}

// ---------------------------------------------------------------------------
// GEMM launch
// ---------------------------------------------------------------------------
static int make_map(CnnState* st, CUtensorMap* map, const void* base, uint64_t inner, uint64_t rows, uint64_t pitch_bytes,
                    uint32_t box_rows) {
    cuuint64_t dims[2] = {inner, rows};
    cuuint64_t strides[1] = {pitch_bytes};
    cuuint32_t box[2] = {(cuuint32_t)kBK, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = st->encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d): inner=%llu rows=%llu pitch=%llu box_rows=%u", (int)r,
                  (unsigned long long)inner, (unsigned long long)rows, (unsigned long long)pitch_bytes, box_rows);
        return VPK_ERR_CUDA;
    }
    return VPK_OK;
}

struct GemmCall {
    const char* name;
    const void* A; uint64_t a_inner, a_rows, a_pitch;     // A tensor: inner elements, rows, pitch bytes
    const void* B; uint64_t b_inner, b_rows;              // B tensor (pitch = inner*2)
    int groups;
    GemmParams p;
};

int launch_gemm(vpk_ctx* ctx, const GemmCall& c) {
    CnnState* st = ctx->cnn;
    CUtensorMap ma, mb;
    VPK_TRY(make_map(st, &ma, c.A, c.a_inner, c.a_rows, c.a_pitch, kBM));
    VPK_TRY(make_map(st, &mb, c.B, c.b_inner, c.b_rows, c.b_inner * 2, (uint32_t)c.p.bn));
    const int m_tiles = (c.p.m_total + kBM - 1) / kBM;
    const int n_tiles = (c.p.n_valid + c.p.bn - 1) / c.p.bn;
    const int ksplit = c.p.ksplit > 1 ? c.p.ksplit : 1;
    if (ksplit > 1 && ((ksplit - 1) * ((c.p.k_blocks + ksplit - 1) / ksplit) >= c.p.k_blocks || !c.p.partial)) {
        set_error("%s: bad split-K configuration", c.name);
        return VPK_ERR_ARG;
    }
    const int fold = c.p.fold > 1 ? c.p.fold : 1;
    if (fold > 1 && (!c.p.lrn || ksplit > 1 || n_tiles != 1 || c.groups % fold || fold * c.p.bn > 256 || c.p.n_valid != c.p.bn ||
                     c.p.c_col_group != c.p.bn)) {
        set_error("%s: bad group-folding configuration", c.name);
        return VPK_ERR_ARG;
    }
    if (c.p.lrn && (n_tiles != 1 || ksplit > 1 || c.p.out_f32)) { set_error("%s: the fused LRN needs all channels in one tile", c.name); return VPK_ERR_ARG; }
    dim3 grid(m_tiles, n_tiles, (c.groups / fold) * ksplit);
    const size_t stage = kABytes + (size_t)c.p.bn * kBK * 2;
    KernelScope ks(ctx, c.name);
    if (ksplit == 1 && st->persistent && c.p.lrn && c.p.bn * fold > 128) {
        // conv2 (LRN epilogue over both groups, 256 columns per tile): persistent with ONE accumulator and two CTAs per SM
        // (0.429 -> 0.420 ms).  With two accumulators it needs all 512 columns, i.e. one CTA per SM, and that runs at
        // 0.59 ms -- with 8 or with 16 epilogue warps alike: a single TMA / MMA stream per SM cannot keep the operands coming.
        const int total = m_tiles * n_tiles * (c.groups / fold);
        const int ctas = std::min(total, 2 * ctx->num_sms);
        const size_t smem = 3 * stage + 1024;
        if (!st->attr_p1) { VPK_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_persistent_kernel<3, 8, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * (kABytes + 128 * kBK * 2) + 1024)); st->attr_p1 = true; }
        gemm_bf16_tcgen05_persistent_kernel<3, 8, 1><<<ctas, kGemmThreads, smem, ctx->stream>>>(ma, mb, c.p, m_tiles, n_tiles, total);
        return check_launch(c.name);
    }
    if (ksplit == 1 && st->persistent && (!c.p.lrn || c.p.bn * fold <= 128)) {
        // persistent CTAs with two accumulators in tensor memory (gemm_tcgen05.cuh): two per SM when the accumulators of
        // both fit the 512 columns, else one per SM with a deeper ring.  Measured on the YUD batch: conv1 0.247 -> 0.219,
        // conv3 0.219 -> 0.184, conv4 0.215 -> 0.166, conv5 0.124 -> 0.102 ms.
        int ncols1 = 32;
        while (ncols1 < c.p.bn * fold) ncols1 <<= 1;
        const int total = m_tiles * n_tiles * (c.groups / fold);
        const int per_sm = 2 * ncols1 <= 256 ? 2 : 1;
        const int ctas = std::min(total, per_sm * ctx->num_sms);
        auto launch = [&](auto kern, int stages, int max_stage, int epi_warps, bool& done) -> int {
            const size_t smem = stages * stage + 1024;
            if (!done) { VPK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, stages * max_stage + 1024)); done = true; }
            kern<<<ctas, 64 + 32 * epi_warps, smem, ctx->stream>>>(ma, mb, c.p, m_tiles, n_tiles, total);
            return check_launch(c.name);
        };
        if (per_sm == 2) return launch(gemm_bf16_tcgen05_persistent_kernel<3, 8, 2>, 3, kABytes + 128 * kBK * 2, 8, st->attr_p3);
        if (stage <= 32768) return launch(gemm_bf16_tcgen05_persistent_kernel<6, 8, 2>, 6, 32768, 8, st->attr_p6);
        return launch(gemm_bf16_tcgen05_persistent_kernel<4, 8, 2>, 4, kABytes + 256 * kBK * 2, 8, st->attr_p4);
    }
    if (c.p.bn <= 128 && c.p.k_blocks * fold <= 3) {
        // very short K loops (conv1: 3 blocks): latency bound per CTA, so two stages and three CTAs per SM
        size_t smem = 2 * stage + 1024;
        bool& attr2 = st->attr2;
        if (!attr2) { VPK_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * (kABytes + 128 * kBK * 2) + 1024)); attr2 = true; }
        gemm_bf16_tcgen05_kernel<2><<<grid, kGemmThreads, smem, ctx->stream>>>(ma, mb, c.p);
    } else if (c.p.bn <= 128) {
        size_t smem = 3 * stage + 1024;
        bool& attr3 = st->attr3;
        if (!attr3) { VPK_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * (kABytes + 128 * kBK * 2) + 1024)); attr3 = true; }
        gemm_bf16_tcgen05_kernel<3><<<grid, kGemmThreads, smem, ctx->stream>>>(ma, mb, c.p);
    } else {
        size_t smem = 4 * stage + 1024;
        bool& attr4 = st->attr4;
        if (!attr4) { VPK_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * (kABytes + 256 * kBK * 2) + 1024)); attr4 = true; }
        gemm_bf16_tcgen05_kernel<4><<<grid, kGemmThreads, smem, ctx->stream>>>(ma, mb, c.p);
    }
    return check_launch(c.name);
}

// plain GEMM (m x n x k) with the K range dealt to `ksplit` CTAs per output tile + the finishing pass
static int launch_gemm_splitk(vpk_ctx* ctx, GemmCall c, int ksplit, const char* finish_name) {
    if (ksplit <= 1) return launch_gemm(ctx, c);
    CnnState* s = ctx->cnn;
    const int M = c.p.m_total, N = c.p.n_valid, ld = c.p.ldc;
    const long long stride = (long long)M * ld;
    VPK_TRY(s->splitk.ensure((size_t)ksplit * stride * sizeof(float)));
    c.p.ksplit = ksplit; c.p.partial = s->splitk.as<float>(); c.p.partial_stride = stride;
    VPK_TRY(launch_gemm(ctx, c));
    KernelScope ks(ctx, finish_name);
    const long long t = (long long)M * (N / 4);
    splitk_finish_kernel<<<(unsigned)((t + 255) / 256), 256, 0, ctx->stream>>>(c.p.partial, ksplit, stride, M, N, ld, c.p.bias, c.p.relu,
                                                                             c.p.out_f32, c.p.out);
    return check_launch(finish_name);
}

static GemmParams plain_params(int m, int n, int k, int bn, int ldc, const float* bias, int relu, int out_f32, void* out) {
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.m_total = m; p.k_blocks = k / kBK; p.cblocks = k / kBK; p.taps_x = 1; p.row_pitch = 0;
    p.hp_wp = 1; p.wp = 1; p.h_valid = 1; p.w_valid = 1; p.out_hp_wp = 1; p.out_wp = 1; p.out_pad = 0;
    p.ldc = ldc; p.n_valid = n; p.relu = relu; p.out_f32 = out_f32; p.bn = bn; p.bias = bias; p.out = out;
    return p;
}

static int ensure_driver_entry(CnnState* st) {
    if (st->encode) return VPK_OK;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
        set_error("cuTensorMapEncodeTiled is not available from the driver (%s)", cudaGetErrorString(e));
        return VPK_ERR_CUDA;
    }
    st->encode = reinterpret_cast<EncodeTiledFn>(fn);
    return VPK_OK;
}

// ---------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------
static int ensure_activations(vpk_ctx* ctx, int n) {
    CnnState* s = ctx->cnn;
    if (n <= s->cap) return VPK_OK;
    size_t N = (size_t)n;
    struct { DBuf* d; size_t bytes; bool zero; } plan[] = {
        {&s->a1, N * 15625 * 64 * 2 + 256, false},            // conv1 operand (125x125 rows x 64)
        {&s->c1, N * 123 * 123 * 96 * 2, false},              // conv1 out
        {&s->a2, N * 65 * 65 * 128 * 2, true},                // conv2 in: pad 2, 2 groups x (48 -> 64)
        {&s->c2, N * 61 * 61 * 256 * 2, false},               // conv2 out
        {&s->a3, N * 32 * 32 * 256 * 2, true},                // conv3 in: pad 1
        {&s->a4, N * 32 * 32 * 384 * 2, true},                // conv4 in: pad 1
        {&s->a5, N * 32 * 32 * 384 * 2, true},                // conv5 in: pad 1
        {&s->c5, N * 30 * 30 * 256 * 2, false},               // conv5 out
        {&s->a6, N * 57600 * 2, false},                       // pool5 = fc6 in
        {&s->f6, N * 4096 * 2, false},
        {&s->f7, N * 4096 * 2, false},
        {&s->logits, N * 400 * 4, false},
        {&s->sig, N * 400 * 4, false},
    };
    for (auto& e : plan) {
        VPK_TRY(e.d->ensure(e.bytes));
        if (e.zero) VPK_CUDA(cudaMemsetAsync(e.d->p, 0, e.d->cap, ctx->stream));
    }
    s->cap = n;
    return VPK_OK;
}

int cnn_forward_dev(vpk_ctx* ctx, const uint8_t* d_images, int32_t n, float* d_sigout, float* d_logits) {
    CnnState* s = ctx->cnn;
    if (!s || !s->loaded) { set_error("vpk_cnn_forward: call vpk_cnn_load first"); return VPK_ERR_STATE; }
    if (n <= 0) return VPK_OK;
    s->last_n = 0;                                         // the buffers no longer hold what vpk_cnn_forward left (sigout may go elsewhere)
    VPK_TRY(ensure_activations(ctx, n));
    s->persistent = !(getenv("VPK_GEMM_PERSIST") && atoi(getenv("VPK_GEMM_PERSIST")) == 0);      // A/B switch, default on
    typedef __nv_bfloat16 bf;
    const float* mean = s->has_mean ? s->mean.as<float>() : nullptr;
    {
        KernelScope ks(ctx, "conv1_operand");
        long long t = (long long)n * 15625 * 8;
        conv1_operand_kernel<<<(unsigned)((t + 255) / 256), 256, 0, ctx->stream>>>(d_images, mean, n, s->a1.as<bf>());
        VPK_TRY(check_launch("conv1_operand"));
    }
    GemmCall c;
    // conv1: 3 block rows x 64 (4 blocks x 16) -> 96
    memset(&c, 0, sizeof(c));
    c.name = "gemm_conv1"; c.A = s->a1.p; c.a_inner = 64; c.a_rows = (uint64_t)n * 15625; c.a_pitch = 128;
    c.B = s->w[0].p; c.b_inner = 192; c.b_rows = 96; c.groups = 1;
    c.p.m_total = n * 15625; c.p.k_blocks = 3; c.p.cblocks = 1; c.p.taps_x = 1; c.p.row_pitch = 125;
    c.p.hp_wp = 15625; c.p.wp = 125; c.p.h_valid = 123; c.p.w_valid = 123;
    c.p.out_hp_wp = 123 * 123; c.p.out_wp = 123; c.p.out_pad = 0; c.p.ldc = 96; c.p.n_valid = 96; c.p.relu = 1; c.p.bn = 96;
    c.p.lrn = 1;                                           // norm1 (cnn/deploy.prototxt:34-44) in the epilogue: a thread owns a pixel's 96 channels
    c.p.bias = s->b[0].as<float>(); c.p.out = s->c1.p;
    VPK_TRY(launch_gemm(ctx, c));
    {
        KernelScope ks(ctx, "pool1");                      // pool1 (:45-55): 3x3 / 2 ceil-mode maximum of the normalised map
        long long t = (long long)n * 31 * 31 * 12;
        lrn_pool_kernel<false><<<(unsigned)((t + 255) / 256), 256, 0, ctx->stream>>>(s->c1.as<bf>(), n, 123, 123, 96, 61, 61, 2, 128, 48, 64, s->a2.as<bf>());
        VPK_TRY(check_launch("pool1"));
    }
    // conv2: 5x5 pad 2, 2 groups of 48 (stored as 64) -> 128 each
    memset(&c, 0, sizeof(c));
    c.name = "gemm_conv2"; c.A = s->a2.p; c.a_inner = 128; c.a_rows = (uint64_t)n * 4225; c.a_pitch = 256;
    c.B = s->w[1].p; c.b_inner = 1600; c.b_rows = 256; c.groups = 2;
    c.p.m_total = n * 4225; c.p.k_blocks = 25; c.p.cblocks = 1; c.p.taps_x = 5; c.p.row_pitch = 65; c.p.a_col_group = 64; c.p.b_row_group = 128;
    c.p.hp_wp = 4225; c.p.wp = 65; c.p.h_valid = 61; c.p.w_valid = 61;
    c.p.out_hp_wp = 61 * 61; c.p.out_wp = 61; c.p.out_pad = 0; c.p.ldc = 256; c.p.c_col_group = 128; c.p.n_valid = 128; c.p.relu = 1; c.p.bn = 128;
    c.p.lrn = 1; c.p.fold = 2;        // norm2 (cnn/deploy.prototxt:82-92) in the epilogue: one CTA computes both groups of its
                                      // pixels, so the window of channels 126..129 crosses the group seam inside a thread
    c.p.bias = s->b[1].as<float>(); c.p.out = s->c2.p;
    VPK_TRY(launch_gemm(ctx, c));
    {
        KernelScope ks(ctx, "pool2");     // pool2 (:93-103)
        long long t = (long long)n * 15 * 15 * 32;
        lrn_pool_kernel<false><<<(unsigned)((t + 255) / 256), 256, 0, ctx->stream>>>(s->c2.as<bf>(), n, 61, 61, 256, 30, 30, 1, 256, 256, 256, s->a3.as<bf>());
        VPK_TRY(check_launch("pool2"));
    }
    // conv3: 3x3 pad 1, 256 -> 384, written into conv4's padded input
    memset(&c, 0, sizeof(c));
    c.name = "gemm_conv3"; c.A = s->a3.p; c.a_inner = 256; c.a_rows = (uint64_t)n * 1024; c.a_pitch = 512;
    c.B = s->w[2].p; c.b_inner = 2304; c.b_rows = 384; c.groups = 1;
    c.p.m_total = n * 1024; c.p.k_blocks = 36; c.p.cblocks = 4; c.p.taps_x = 3; c.p.row_pitch = 32;
    c.p.hp_wp = 1024; c.p.wp = 32; c.p.h_valid = 30; c.p.w_valid = 30;
    c.p.out_hp_wp = 1024; c.p.out_wp = 32; c.p.out_pad = 1; c.p.ldc = 384; c.p.n_valid = 384; c.p.relu = 1; c.p.bn = 128;
    c.p.bias = s->b[2].as<float>(); c.p.out = s->a4.p;
    VPK_TRY(launch_gemm(ctx, c));
    // conv4: 3x3 pad 1, 2 groups 192 -> 192, into conv5's padded input
    memset(&c, 0, sizeof(c));
    c.name = "gemm_conv4"; c.A = s->a4.p; c.a_inner = 384; c.a_rows = (uint64_t)n * 1024; c.a_pitch = 768;
    c.B = s->w[3].p; c.b_inner = 1728; c.b_rows = 384; c.groups = 2;
    c.p.m_total = n * 1024; c.p.k_blocks = 27; c.p.cblocks = 3; c.p.taps_x = 3; c.p.row_pitch = 32; c.p.a_col_group = 192; c.p.b_row_group = 192;
    c.p.hp_wp = 1024; c.p.wp = 32; c.p.h_valid = 30; c.p.w_valid = 30;
    c.p.out_hp_wp = 1024; c.p.out_wp = 32; c.p.out_pad = 1; c.p.ldc = 384; c.p.c_col_group = 192; c.p.n_valid = 192; c.p.relu = 1; c.p.bn = 192;
    c.p.bias = s->b[3].as<float>(); c.p.out = s->a5.p;
    VPK_TRY(launch_gemm(ctx, c));
    // conv5: 3x3 pad 1, 2 groups 192 -> 128
    memset(&c, 0, sizeof(c));
    c.name = "gemm_conv5"; c.A = s->a5.p; c.a_inner = 384; c.a_rows = (uint64_t)n * 1024; c.a_pitch = 768;
    c.B = s->w[4].p; c.b_inner = 1728; c.b_rows = 256; c.groups = 2;
    c.p.m_total = n * 1024; c.p.k_blocks = 27; c.p.cblocks = 3; c.p.taps_x = 3; c.p.row_pitch = 32; c.p.a_col_group = 192; c.p.b_row_group = 128;
    c.p.hp_wp = 1024; c.p.wp = 32; c.p.h_valid = 30; c.p.w_valid = 30;
    c.p.out_hp_wp = 900; c.p.out_wp = 30; c.p.out_pad = 0; c.p.ldc = 256; c.p.c_col_group = 128; c.p.n_valid = 128; c.p.relu = 1; c.p.bn = 128;
    c.p.bias = s->b[4].as<float>(); c.p.out = s->c5.p;
    VPK_TRY(launch_gemm(ctx, c));
    {
        KernelScope ks(ctx, "pool5");
        long long t = (long long)n * 8 * 8 * 32;
        lrn_pool_kernel<false><<<(unsigned)((t + 255) / 256), 256, 0, ctx->stream>>>(s->c5.as<bf>(), n, 30, 30, 256, 15, 15, 0, 256, 256, 256, s->a6.as<bf>());
        VPK_TRY(check_launch("pool5"));
    }
    // fc6 / fc7 / fc8
    memset(&c, 0, sizeof(c));
    c.name = "gemm_fc6"; c.A = s->a6.p; c.a_inner = 57600; c.a_rows = n; c.a_pitch = 57600 * 2;
    c.B = s->w[5].p; c.b_inner = 57600; c.b_rows = 4096; c.groups = 1;
    c.p = plain_params(n, 4096, 57600, 256, 4096, s->b[5].as<float>(), 1, 0, s->f6.p);
    VPK_TRY(launch_gemm_splitk(ctx, c, n <= 256 ? 9 : 1, "splitk_fc6"));
    c.name = "gemm_fc7"; c.A = s->f6.p; c.a_inner = 4096; c.a_rows = n; c.a_pitch = 8192;
    c.B = s->w[6].p; c.b_inner = 4096; c.b_rows = 4096;
    c.p = plain_params(n, 4096, 4096, 256, 4096, s->b[6].as<float>(), 1, 0, s->f7.p);
    VPK_TRY(launch_gemm_splitk(ctx, c, n <= 256 ? 8 : 1, "splitk_fc7"));
    float* logits = d_logits ? d_logits : s->logits.as<float>();
    c.name = "gemm_fc8"; c.A = s->f7.p; c.a_inner = 4096; c.a_rows = n; c.a_pitch = 8192;
    c.B = s->w[7].p; c.b_inner = 4096; c.b_rows = 400;
    c.p = plain_params(n, 400, 4096, 80, 400, s->b[7].as<float>(), 0, 1, logits);
    VPK_TRY(launch_gemm_splitk(ctx, c, n <= 256 ? 16 : 1, "splitk_fc8"));
    if (d_sigout) {
        KernelScope ks(ctx, "sigmoid");
        long long t = (long long)n * 400;
        sigmoid_kernel<<<(unsigned)((t + 255) / 256), 256, 0, ctx->stream>>>(logits, t, d_sigout);
        VPK_TRY(check_launch("sigmoid"));
    }
    return VPK_OK;
}

}  // namespace vpk

using namespace vpk;

extern "C" {

int vpk_cnn_load(vpk_ctx* ctx, const float* const* weights, const float* const* biases, const float* mean) {
    if (!ctx || !weights || !biases) { set_error("vpk_cnn_load: bad argument"); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->cnn) ctx->cnn = new CnnState();
    CnnState* s = ctx->cnn;
    VPK_TRY(ensure_driver_entry(s));
    // (n_out, source elements, packed K, mode, cin_g, cpad, ksz)
    struct L { int n_out; long long src; long long k; int mode, cin_g, cpad, ksz; };
    const L layers[8] = {
        {96, 96LL * 121, 192, PACK_CONV1, 1, 0, 11},
        {256, 256LL * 48 * 25, 1600, PACK_CONV, 48, 64, 5},
        {384, 384LL * 256 * 9, 2304, PACK_CONV, 256, 256, 3},
        {384, 384LL * 192 * 9, 1728, PACK_CONV, 192, 192, 3},
        {256, 256LL * 192 * 9, 1728, PACK_CONV, 192, 192, 3},
        {4096, 4096LL * 57600, 57600, PACK_FC6, 0, 0, 0},
        {4096, 4096LL * 4096, 4096, PACK_PLAIN, 0, 0, 0},
        {400, 400LL * 4096, 4096, PACK_PLAIN, 0, 0, 0},
    };
    for (int i = 0; i < 8; ++i) {
        if (!weights[i] || !biases[i]) { set_error("vpk_cnn_load: layer %d weights/bias NULL", i); return VPK_ERR_ARG; }
        const L& l = layers[i];
        VPK_TRY(ctx->d_misc.ensure(l.src * sizeof(float)));
        VPK_CUDA(cudaMemcpyAsync(ctx->d_misc.p, weights[i], l.src * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        VPK_TRY(s->w[i].ensure((size_t)l.n_out * l.k * 2));
        VPK_TRY(s->b[i].ensure((size_t)l.n_out * sizeof(float)));
        long long total = (long long)l.n_out * l.k;
        {
            KernelScope ks(ctx, "pack_weights");
            pack_weights_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(
                ctx->d_misc.as<float>(), s->w[i].as<__nv_bfloat16>(), l.mode, l.n_out, l.k, l.cin_g, l.cpad, l.ksz);
            VPK_TRY(check_launch("pack_weights"));
        }
        VPK_CUDA(cudaMemcpyAsync(s->b[i].p, biases[i], (size_t)l.n_out * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    s->has_mean = mean != nullptr;
    if (mean) {
        VPK_TRY(s->mean.ensure(250000 * sizeof(float)));
        VPK_CUDA(cudaMemcpyAsync(s->mean.p, mean, 250000 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    s->loaded = true;
    return VPK_OK;
}

int vpk_cnn_forward(vpk_ctx* ctx, const uint8_t* images, int32_t n, float* sigout, float* logits_out) {
    if (!ctx || n < 0 || (n > 0 && (!images || !sigout))) { set_error("vpk_cnn_forward: bad argument"); return VPK_ERR_ARG; }
    if (n == 0) return VPK_OK;
    VPK_CUDA(cudaSetDevice(ctx->device));
    CnnState* s = ctx->cnn;
    if (!s || !s->loaded) { set_error("vpk_cnn_forward: call vpk_cnn_load first"); return VPK_ERR_STATE; }
    const int chunk = 1024;
    for (int i0 = 0; i0 < n; i0 += chunk) {
        int nb = n - i0 < chunk ? n - i0 : chunk;
        VPK_TRY(ensure_activations(ctx, nb));
        VPK_TRY(s->img.ensure((size_t)nb * 250000));
        VPK_CUDA(cudaMemcpyAsync(s->img.p, images + (size_t)i0 * 250000, (size_t)nb * 250000, cudaMemcpyHostToDevice, ctx->stream));
        VPK_TRY(cnn_forward_dev(ctx, s->img.as<uint8_t>(), nb, s->sig.as<float>(), nullptr));
        VPK_CUDA(cudaMemcpyAsync(sigout + (size_t)i0 * 400, s->sig.p, (size_t)nb * 400 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        if (logits_out)
            VPK_CUDA(cudaMemcpyAsync(logits_out + (size_t)i0 * 400, s->logits.p, (size_t)nb * 400 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        VPK_CUDA(cudaStreamSynchronize(ctx->stream));
        s->last_n = nb;
    }
    return VPK_OK;
}

// Diagnostics: raw copy of one activation buffer of the last chunk vpk_cnn_forward ran (layouts in vpk.h).
int vpk_cnn_debug_fetch(vpk_ctx* ctx, int32_t which, int32_t n_images, void* out) {
    if (!ctx || !out || which < 0 || which >= VPK_CNN_NBUF || n_images < 0) { set_error("vpk_cnn_debug_fetch: bad argument"); return VPK_ERR_ARG; }
    CnnState* s = ctx->cnn;
    if (!s || s->last_n <= 0) { set_error("vpk_cnn_debug_fetch: no vpk_cnn_forward since the last load or pipeline run"); return VPK_ERR_STATE; }
    if (n_images > s->last_n) {
        set_error("vpk_cnn_debug_fetch: %d images asked for, the last chunk had %d", n_images, s->last_n);
        return VPK_ERR_ARG;
    }
    // per-image bytes, in the order of the VPK_CNN_BUF_* enum
    static const size_t per_image[VPK_CNN_NBUF] = {15625 * 64 * 2, 123 * 123 * 96 * 2, 65 * 65 * 128 * 2, 61 * 61 * 256 * 2,
                                                   32 * 32 * 256 * 2, 32 * 32 * 384 * 2, 32 * 32 * 384 * 2, 30 * 30 * 256 * 2,
                                                   57600 * 2, 4096 * 2, 4096 * 2, 400 * 4, 400 * 4};
    const DBuf* bufs[VPK_CNN_NBUF] = {&s->a1, &s->c1, &s->a2, &s->c2, &s->a3, &s->a4, &s->a5, &s->c5, &s->a6, &s->f6, &s->f7, &s->logits, &s->sig};
    if (n_images == 0) return VPK_OK;
    VPK_CUDA(cudaSetDevice(ctx->device));
    VPK_CUDA(cudaMemcpyAsync(out, bufs[which]->p, per_image[which] * n_images, cudaMemcpyDeviceToHost, ctx->stream));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    return VPK_OK;
}

// Diagnostics: one plain GEMM through the tcgen05 kernel.  a (m,k), b (n,k) are
// bf16 bit patterns (uint16), bias (n) float32 or NULL, out (m,n) float32.
int vpk_debug_gemm(vpk_ctx* ctx, int32_t m, int32_t n, int32_t k, const uint16_t* a, const uint16_t* b, const float* bias,
                   int32_t relu, int32_t bn, int32_t ksplit, float* out) {
    if (!ctx || !a || !b || !out || m <= 0 || n <= 0 || k <= 0 || k % 64 || bn % 16 || bn < 16 || bn > 256 || n % bn || ksplit < 1) {
        set_error("vpk_debug_gemm: bad argument (k %% 64 == 0, bn %% 16 == 0, n %% bn == 0 required)");
        return VPK_ERR_ARG;
    }
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->cnn) ctx->cnn = new CnnState();
    VPK_TRY(ensure_driver_entry(ctx->cnn));
    DBuf da, db, dbias, dout;
    int rc = VPK_OK;
    do {
        if ((rc = da.ensure((size_t)m * k * 2)) || (rc = db.ensure((size_t)n * k * 2)) || (rc = dout.ensure((size_t)m * n * 4)) ||
            (rc = dbias.ensure((size_t)n * 4))) break;
        cudaMemcpyAsync(da.p, a, (size_t)m * k * 2, cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(db.p, b, (size_t)n * k * 2, cudaMemcpyHostToDevice, ctx->stream);
        if (bias) cudaMemcpyAsync(dbias.p, bias, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream);
        GemmCall c;
        memset(&c, 0, sizeof(c));
        c.name = "gemm_debug"; c.A = da.p; c.a_inner = k; c.a_rows = m; c.a_pitch = (uint64_t)k * 2;
        c.B = db.p; c.b_inner = k; c.b_rows = n; c.groups = 1;
        c.p = plain_params(m, n, k, bn, n, bias ? dbias.as<float>() : nullptr, relu, 1, dout.p);
        if ((rc = launch_gemm_splitk(ctx, c, ksplit, "splitk_debug"))) break;
        cudaMemcpyAsync(out, dout.p, (size_t)m * n * 4, cudaMemcpyDeviceToHost, ctx->stream);
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { set_error("vpk_debug_gemm: %s", cudaGetErrorString(e)); rc = VPK_ERR_CUDA; }
    } while (0);
    da.release(); db.release(); dbias.release(); dout.release();
    return rc;
}

}  // extern "C"
