// Context, error strings, launch accounting and per-kernel event timing.
#include <stdarg.h>
#include "vpk_internal.cuh"

namespace vpk {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int profile_collect(vpk_ctx* ctx) {
    if (ctx->pending.empty()) return VPK_OK;
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    for (auto& pe : ctx->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, pe.a, pe.b) == cudaSuccess) {
            auto& e = ctx->prof[pe.name];
            e.total_ms += ms;
            e.launches += 1;
        }
        ctx->event_pool.push_back(pe.a);
        ctx->event_pool.push_back(pe.b);
    }
    ctx->pending.clear();
    return VPK_OK;
}

}  // namespace vpk

using namespace vpk;

extern "C" {

int vpk_abi_version(void) { return VPK_ABI_VERSION; }

const char* vpk_last_error(void) { return g_err; }

int vpk_create(int device, vpk_ctx** out) {
    if (!out) { set_error("vpk_create: out is NULL"); return VPK_ERR_ARG; }
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        set_error("vpk_create: no CUDA device (%s); this library has no CPU fallback",
                  e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        return VPK_ERR_CUDA;
    }
    if (device < 0 || device >= n) { set_error("vpk_create: device %d out of range [0,%d)", device, n); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    VPK_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("vpk_create: device %d is sm_%d%d; libvpk is built for sm_100a only", device, prop.major, prop.minor);
        return VPK_ERR_CUDA;
    }
    vpk_ctx* ctx = new vpk_ctx();
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    ctx->l2_bytes = (size_t)prop.l2CacheSize;
    e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { set_error("cudaStreamCreate -> %s", cudaGetErrorString(e)); delete ctx; return VPK_ERR_CUDA; }
    *out = ctx;
    return VPK_OK;
}

int vpk_destroy(vpk_ctx* ctx) {
    if (!ctx) return VPK_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cnn_free(ctx);
    em_free(ctx);
    pipe_free(ctx);
    lsd_free(ctx);
    prep_free(ctx);
    jpeg_free(ctx);
    png_free(ctx);
    for (auto& pe : ctx->pending) { cudaEventDestroy(pe.a); cudaEventDestroy(pe.b); }
    for (auto ev : ctx->event_pool) cudaEventDestroy(ev);
    ctx->d_lines.release(); ctx->d_segments.release(); ctx->d_offsets.release(); ctx->d_work.release();
    ctx->d_hist.release(); ctx->d_img.release(); ctx->d_weights.release(); ctx->d_misc.release(); ctx->d_curves_tab.release();
    ctx->h_stage.release();
    for (auto& e : ctx->marks) if (e) cudaEventDestroy(e);
    ctx->d_pack.release();
    for (auto& e : ctx->io_ev) if (e) cudaEventDestroy(e);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
    return VPK_OK;
}

int vpk_synchronize(vpk_ctx* ctx) {
    if (!ctx) { set_error("null ctx"); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    return VPK_OK;
}

int64_t vpk_launch_count(const vpk_ctx* ctx) { return ctx ? ctx->launches : 0; }

int vpk_mark(vpk_ctx* ctx, int32_t slot) {
    if (!ctx || slot < 0 || slot >= 4) { set_error("vpk_mark: bad argument"); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->marks[slot]) VPK_CUDA(cudaEventCreate(&ctx->marks[slot]));
    VPK_CUDA(cudaEventRecord(ctx->marks[slot], ctx->stream));
    return VPK_OK;
}

int vpk_mark_elapsed(vpk_ctx* from, int32_t slot_from, vpk_ctx* to, int32_t slot_to, float* ms) {
    if (!from || !to || !ms || slot_from < 0 || slot_from >= 4 || slot_to < 0 || slot_to >= 4 || !from->marks[slot_from] ||
        !to->marks[slot_to] || from->device != to->device) {
        set_error("vpk_mark_elapsed: bad argument (both marks must have been recorded, on the same device)");
        return VPK_ERR_ARG;
    }
    VPK_CUDA(cudaSetDevice(from->device));
    VPK_CUDA(cudaEventSynchronize(from->marks[slot_from]));
    VPK_CUDA(cudaEventSynchronize(to->marks[slot_to]));
    VPK_CUDA(cudaEventElapsedTime(ms, from->marks[slot_from], to->marks[slot_to]));
    return VPK_OK;
}

int vpk_profile_enable(vpk_ctx* ctx, int enable) {
    if (!ctx) { set_error("null ctx"); return VPK_ERR_ARG; }
    if (!enable) VPK_TRY(profile_collect(ctx));
    ctx->profiling = enable != 0;
    return VPK_OK;
}

int vpk_profile_reset(vpk_ctx* ctx) {
    if (!ctx) { set_error("null ctx"); return VPK_ERR_ARG; }
    VPK_TRY(profile_collect(ctx));
    ctx->prof.clear();
    return VPK_OK;
}

int vpk_profile_read(vpk_ctx* ctx, int cap, const char** names, double* total_ms, int64_t* launches) {
    if (!ctx) { set_error("null ctx"); return -1; }
    if (profile_collect(ctx) != VPK_OK) return -1;
    int i = 0;
    for (auto& kv : ctx->prof) {
        if (i < cap) {
            if (names) names[i] = kv.first.c_str();
            if (total_ms) total_ms[i] = kv.second.total_ms;
            if (launches) launches[i] = kv.second.launches;
        }
        ++i;
    }
    return i;
}

}  // extern "C"
