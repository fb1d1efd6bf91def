// Row N9 of SURVEY.md section 8(f): pipeline input that is already in CUDA memory (photos decoded by another GPU
// decoder, gray planes, segments from a model) and the stream ordering with the caller; DESIGN.md section 4.11.
//
// device_pack gathers B strided caller arrays into the one contiguous buffer the existing stage reads (the photo
// buffer of prep_input, the LSD input buffer of lsd_input, the resident segments).  Item b is a (rows, cols, ch)
// array of esz-byte elements with non-negative byte strides, written row-major at its destination offset.  One CTA
// per tile of rows; a row whose cols * ch elements are consecutive in the source is copied as bytes, 16 at a time
// where the source and destination share their alignment (HWC uint8 rows, contiguous float64 rows); every other
// layout (CHW views, column slices) reads element by element, a thread per (row, column) with the channels in its
// loop.  No byte outside src + sum (extent - 1) * stride (+ the element) is read.  A VPK_DEFINES=VPK_PACK_CHECKS
// build asserts every source and destination index.
#include "vpk_internal.cuh"

#if defined(VPK_PACK_CHECKS)
#include <assert.h>
#define PACK_CHECK(c) assert(c)
#else
#define PACK_CHECK(c) ((void)0)
#endif

namespace vpk {

static constexpr int kPackThreads = 256;
static constexpr int64_t kPackTileBytes = 32 * 1024;   // destination bytes per CTA (at least one row)

__global__ void __launch_bounds__(kPackThreads)
device_pack(const PackItem* __restrict__ items, const int32_t* __restrict__ tile_off, int B, uint8_t* __restrict__ dst,
            int64_t dst_bytes) {
    const int t = blockIdx.x;
    int lo = 0, hi = B - 1;                                 // the item of this tile: last b with tile_off[b] <= t
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (tile_off[mid] <= t) lo = mid; else hi = mid - 1;
    }
    const PackItem it = items[lo];
    const int r0 = (t - tile_off[lo]) * it.rows_per_tile;
    const int r1 = min(r0 + it.rows_per_tile, it.rows);
    const int64_t row_bytes = (int64_t)it.cols * it.ch * it.esz;
    const int64_t span = (int64_t)(it.rows - 1) * it.s0 + (int64_t)(it.cols - 1) * it.s1 + (int64_t)(it.ch - 1) * it.s2 + it.esz;
    PACK_CHECK(r0 < r1 && it.dst + (int64_t)it.rows * row_bytes <= dst_bytes);
    uint8_t* out = dst + it.dst;
    if (it.dense) {
        for (int r = r0; r < r1; ++r) {
            const uint8_t* s = it.src + (int64_t)r * it.s0;
            uint8_t* d = out + (int64_t)r * row_bytes;
            const uintptr_t ms = reinterpret_cast<uintptr_t>(s) & 15, md = reinterpret_cast<uintptr_t>(d) & 15;
            const int64_t head = ms == md ? min(row_bytes, (int64_t)((16 - ms) & 15)) : row_bytes;
            const int64_t nv = (row_bytes - head) >> 4;
            for (int64_t i = threadIdx.x; i < head; i += kPackThreads) {
                PACK_CHECK((int64_t)r * it.s0 + i < span && it.dst + (int64_t)r * row_bytes + i < dst_bytes);
                d[i] = s[i];
            }
            const uint4* sv = reinterpret_cast<const uint4*>(s + head);
            uint4* dv = reinterpret_cast<uint4*>(d + head);
            for (int64_t i = threadIdx.x; i < nv; i += kPackThreads) {
                PACK_CHECK((int64_t)r * it.s0 + head + 16 * i + 15 < span && it.dst + (int64_t)r * row_bytes + head + 16 * i + 15 < dst_bytes);
                dv[i] = __ldg(sv + i);
            }
            for (int64_t i = head + 16 * nv + threadIdx.x; i < row_bytes; i += kPackThreads) {
                PACK_CHECK((int64_t)r * it.s0 + i < span && it.dst + (int64_t)r * row_bytes + i < dst_bytes);
                d[i] = s[i];
            }
        }
        return;
    }
    const int64_t n = (int64_t)(r1 - r0) * it.cols;
    for (int64_t i = threadIdx.x; i < n; i += kPackThreads) {
        const int r = r0 + (int)(i / it.cols), x = (int)(i % it.cols);
        const int64_t so = (int64_t)r * it.s0 + (int64_t)x * it.s1;
        const int64_t dof = ((int64_t)r * it.cols + x) * it.ch * it.esz;
        for (int c = 0; c < it.ch; ++c) {
            const int64_t sc = so + (int64_t)c * it.s2;
            PACK_CHECK(sc + it.esz <= span && it.dst + dof + (int64_t)(c + 1) * it.esz <= dst_bytes);
            if (it.esz == 8) reinterpret_cast<uint64_t*>(out + dof)[c] = *reinterpret_cast<const uint64_t*>(it.src + sc);
            else out[dof + c] = it.src[sc];
        }
    }
}

int pack_dev(vpk_ctx* ctx, std::vector<PackItem>& items, uint8_t* d_dst, int64_t dst_bytes) {
    const int B = (int)items.size();
    std::vector<int32_t> tile_off(B + 1, 0);
    for (int b = 0; b < B; ++b) {
        PackItem& it = items[b];
        const int64_t row_bytes = (int64_t)it.cols * it.ch * it.esz;
        it.rows_per_tile = (int32_t)std::min<int64_t>(it.rows, std::max<int64_t>(1, kPackTileBytes / row_bytes));
        it.dense = (it.ch == 1 || it.s2 == it.esz) && (it.cols == 1 || it.s1 == (int64_t)it.ch * it.esz);
        const int64_t n = (it.rows + it.rows_per_tile - 1) / it.rows_per_tile;
        if (tile_off[b] + n > INT32_MAX) { set_error("device_pack: more than 2^31 row tiles in one call; split the batch"); return VPK_ERR_ARG; }
        tile_off[b + 1] = tile_off[b] + (int32_t)n;
    }
    if (tile_off[B] == 0) return VPK_OK;
    // the descriptors and the tile offsets go to the device in one copy
    const size_t ib = (size_t)B * sizeof(PackItem), tb = (size_t)(B + 1) * sizeof(int32_t);
    std::vector<uint8_t> meta(ib + tb);
    memcpy(meta.data(), items.data(), ib);
    memcpy(meta.data() + ib, tile_off.data(), tb);
    VPK_TRY(ctx->d_pack.ensure(meta.size()));
    VPK_CUDA(cudaMemcpyAsync(ctx->d_pack.p, meta.data(), meta.size(), cudaMemcpyHostToDevice, ctx->stream));
    KernelScope ks(ctx, "device_pack");
    device_pack<<<tile_off[B], kPackThreads, 0, ctx->stream>>>(ctx->d_pack.as<PackItem>(),
                                                               reinterpret_cast<const int32_t*>(ctx->d_pack.as<uint8_t>() + ib), B,
                                                               d_dst, dst_bytes);
    return check_launch("device_pack");
}

int check_device_ptr(vpk_ctx* ctx, const void* p, const char* who, const char* what, const char* host_entry) {
    if (!p) { set_error("%s: %s is NULL", who, what); return VPK_ERR_ARG; }
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        set_error("%s: %s is not a CUDA pointer", who, what);
        return VPK_ERR_ARG;
    }
    if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) {
        set_error("%s: %s is host memory, not device or managed memory; host arrays go to %s", who, what, host_entry);
        return VPK_ERR_ARG;
    }
    if (a.device != ctx->device) {
        set_error("%s: %s is memory of device %d, the context's device is %d", who, what, a.device, ctx->device);
        return VPK_ERR_ARG;
    }
    return VPK_OK;
}

static int io_events(vpk_ctx* ctx) {
    for (auto& e : ctx->io_ev)
        if (!e) VPK_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    return VPK_OK;
}

int stream_enter(vpk_ctx* ctx, void* stream) {
    VPK_TRY(io_events(ctx));
    VPK_CUDA(cudaEventRecord(ctx->io_ev[0], static_cast<cudaStream_t>(stream)));
    VPK_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->io_ev[0], 0));
    return VPK_OK;
}

int stream_leave(vpk_ctx* ctx, void* stream) {
    VPK_TRY(io_events(ctx));
    VPK_CUDA(cudaEventRecord(ctx->io_ev[1], ctx->stream));
    VPK_CUDA(cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), ctx->io_ev[1], 0));
    return VPK_OK;
}

}  // namespace vpk
