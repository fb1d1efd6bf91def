// Whole path on a device-resident ragged batch: segments -> lines -> sphere
// image -> CNN -> EM (reference example.py:37-39 / benchmark.py:59-66 without
// the per-image pickles of evaluation.py:183, 289, 328).  All intermediates
// stay in HBM; only the final per-image results are copied back.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "vpk_internal.cuh"

namespace vpk {

static constexpr int kChunk = 1024;     // images per sphere+CNN pass (bounds the histogram / activation workspaces)
static constexpr int kCells = VPK_GRID * VPK_GRID;

struct PipeState {
    int B = 0;
    int64_t sumN = 0;
    int S = 0;
    std::vector<int32_t> h_offsets;
    DBuf seg, lines, offsets, hist, images, sigout, out_small, out_assoc, horizon, truth;
    HBuf h_horizon, h_small, h_assoc;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    bool have_result = false;
    EmDeviceOut out;
};

void pipe_free(vpk_ctx* ctx) {
    if (!ctx->pipe) return;
    PipeState* p = ctx->pipe;
    p->seg.release(); p->lines.release(); p->offsets.release(); p->hist.release(); p->images.release();
    p->sigout.release(); p->out_small.release(); p->out_assoc.release(); p->horizon.release(); p->truth.release(); p->h_horizon.release(); p->h_small.release(); p->h_assoc.release();
    for (auto& e : p->ev) if (e) cudaEventDestroy(e);
    delete p;
    ctx->pipe = nullptr;
}

// The detector's rows (d_rows, image b's from row_off[b]) into the resident batch: normalised where they are
// (widths / heights: the frames the detector saw), they never leave the device
static int upload_detected(vpk_ctx* ctx, const double* d_rows, const std::vector<int32_t>& row_off, const int32_t* widths,
                           const int32_t* heights, int32_t B) {
    if (!ctx->pipe) {
        ctx->pipe = new PipeState();
        for (auto& e : ctx->pipe->ev) VPK_CUDA(cudaEventCreate(&e));
    }
    PipeState* p = ctx->pipe;
    const int64_t sumN = row_off[B];
    p->B = B; p->sumN = sumN; p->have_result = false;
    p->h_offsets = row_off;
    VPK_TRY(p->seg.ensure((sumN + 1) * 4 * sizeof(double)));
    VPK_TRY(p->lines.ensure((sumN + 1) * 3 * sizeof(double)));
    VPK_TRY(p->offsets.ensure((size_t)(3 * (B + 1)) * sizeof(int32_t)));
    int32_t* d_off = p->offsets.as<int32_t>();
    int32_t* d_w = d_off + (B + 1);
    int32_t* d_h = d_w + (B + 1);
    cudaStream_t st = ctx->stream;
    VPK_CUDA(cudaMemcpyAsync(d_off, row_off.data(), (B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemcpyAsync(d_w, widths, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemcpyAsync(d_h, heights, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    VPK_TRY(segments_from_lsd_dev(ctx, d_rows, 7, d_off, d_w, d_h, B, sumN, p->seg.as<double>(), nullptr));
    VPK_CUDA(cudaStreamSynchronize(st));
    return VPK_OK;
}

}  // namespace vpk

using namespace vpk;

extern "C" {

int vpk_pipeline_upload(vpk_ctx* ctx, const double* segments, const int32_t* offsets, int32_t B) {
    if (!ctx || !offsets || B <= 0 || offsets[0] != 0) { set_error("vpk_pipeline_upload: bad argument"); return VPK_ERR_ARG; }
    for (int b = 0; b < B; ++b) if (offsets[b + 1] < offsets[b]) { set_error("vpk_pipeline_upload: offsets must be non-decreasing"); return VPK_ERR_ARG; }
    const int64_t sumN = offsets[B];
    if (sumN > 0 && !segments) { set_error("vpk_pipeline_upload: segments is NULL"); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->pipe) {
        ctx->pipe = new PipeState();
        for (auto& e : ctx->pipe->ev) VPK_CUDA(cudaEventCreate(&e));
    }
    PipeState* p = ctx->pipe;
    p->B = B; p->sumN = sumN; p->have_result = false;
    p->h_offsets.assign(offsets, offsets + B + 1);
    VPK_TRY(p->seg.ensure((sumN + 1) * 4 * sizeof(double)));
    VPK_TRY(p->lines.ensure((sumN + 1) * 3 * sizeof(double)));
    VPK_TRY(p->offsets.ensure((B + 1) * sizeof(int32_t)));
    if (sumN) VPK_CUDA(cudaMemcpyAsync(p->seg.p, segments, sumN * 4 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    VPK_CUDA(cudaMemcpyAsync(p->offsets.p, offsets, (B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    return VPK_OK;
}

int vpk_pipeline_upload_lsd(vpk_ctx* ctx, const double* lsd, int32_t ncols, const int32_t* offsets, const int32_t* widths,
                            const int32_t* heights, int32_t B) {
    if (!ctx || !offsets || !widths || !heights || B <= 0 || ncols < 4 || offsets[0] != 0) { set_error("vpk_pipeline_upload_lsd: bad argument"); return VPK_ERR_ARG; }
    for (int b = 0; b < B; ++b)
        if (offsets[b + 1] < offsets[b] || widths[b] <= 0 || heights[b] <= 0) { set_error("vpk_pipeline_upload_lsd: bad offsets or image size"); return VPK_ERR_ARG; }
    const int64_t sumN = offsets[B];
    if (sumN > 0 && !lsd) { set_error("vpk_pipeline_upload_lsd: lsd is NULL"); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->pipe) {
        ctx->pipe = new PipeState();
        for (auto& e : ctx->pipe->ev) VPK_CUDA(cudaEventCreate(&e));
    }
    PipeState* p = ctx->pipe;
    p->B = B; p->sumN = sumN; p->have_result = false;
    p->h_offsets.assign(offsets, offsets + B + 1);
    VPK_TRY(p->seg.ensure((sumN + 1) * 4 * sizeof(double)));
    VPK_TRY(p->lines.ensure((sumN + 1) * 3 * sizeof(double)));
    VPK_TRY(p->offsets.ensure((size_t)(3 * (B + 1)) * sizeof(int32_t)));
    VPK_TRY(ctx->d_misc.ensure((size_t)(sumN + 1) * ncols * sizeof(double)));
    int32_t* d_off = p->offsets.as<int32_t>();
    int32_t* d_w = d_off + (B + 1);
    int32_t* d_h = d_w + (B + 1);
    cudaStream_t st = ctx->stream;
    if (sumN) VPK_CUDA(cudaMemcpyAsync(ctx->d_misc.p, lsd, (size_t)sumN * ncols * sizeof(double), cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemcpyAsync(d_off, offsets, (B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemcpyAsync(d_w, widths, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    VPK_CUDA(cudaMemcpyAsync(d_h, heights, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    // the raw LSD rows are normalised where they land: no host loop, no second staging of segments
    VPK_TRY(segments_from_lsd_dev(ctx, ctx->d_misc.as<double>(), ncols, d_off, d_w, d_h, B, sumN, p->seg.as<double>(), nullptr));
    VPK_CUDA(cudaStreamSynchronize(st));
    return VPK_OK;
}

int vpk_pipeline_upload_images(vpk_ctx* ctx, const void* images, int32_t dtype, const int64_t* pixel_offsets, const int32_t* widths,
                               const int32_t* heights, int32_t B, const vpk_lsd_config* cfg, int32_t* counts_out) {
    if (!ctx || !widths || !heights || B <= 0) { set_error("vpk_pipeline_upload_images: bad argument"); return VPK_ERR_ARG; }
    std::vector<int32_t> counts(B), row_off;
    const double* d_rows = nullptr;
    VPK_TRY(lsd_dev(ctx, images, dtype, pixel_offsets, widths, heights, B, cfg, counts.data(), &d_rows, row_off));
    VPK_TRY(upload_detected(ctx, d_rows, row_off, widths, heights, B));
    if (counts_out) memcpy(counts_out, counts.data(), (size_t)B * sizeof(int32_t));
    return VPK_OK;
}

int vpk_pipeline_upload_photos(vpk_ctx* ctx, const uint8_t* rgb, const int64_t* byte_offsets, const int32_t* widths,
                               const int32_t* heights, int32_t B, int32_t target_size, const vpk_lsd_config* cfg,
                               int32_t* counts_out, int32_t* out_widths, int32_t* out_heights) {
    if (!ctx) { set_error("vpk_pipeline_upload_photos: bad argument"); return VPK_ERR_ARG; }
    PrepPlan pp;
    VPK_TRY(prep_plan(rgb, byte_offsets, widths, heights, B, target_size, "vpk_pipeline_upload_photos", pp));
    // the detector reads the prepared planes (float64, x 255) where the preparation kernel writes them
    std::vector<int32_t> counts(B), row_off;
    LsdPlan lp;
    VPK_TRY(lsd_plan(pp.pix_off.data(), pp.W.data(), pp.H.data(), B, VPK_PIX_F64, cfg, counts.data(), lp));
    void* d_in = nullptr;
    VPK_TRY(lsd_input(ctx, lp, &d_in));
    VPK_TRY(prep_run(ctx, pp, rgb, 255.0, static_cast<double*>(d_in)));
    const double* d_rows = nullptr;
    VPK_TRY(lsd_detect(ctx, lp, counts.data(), &d_rows, row_off));
    VPK_TRY(upload_detected(ctx, d_rows, row_off, pp.W.data(), pp.H.data(), B));
    if (counts_out) memcpy(counts_out, counts.data(), (size_t)B * sizeof(int32_t));
    if (out_widths) memcpy(out_widths, pp.W.data(), (size_t)B * sizeof(int32_t));
    if (out_heights) memcpy(out_heights, pp.H.data(), (size_t)B * sizeof(int32_t));
    return VPK_OK;
}

int vpk_pipeline_run(vpk_ctx* ctx, int32_t S, int32_t sphere_mode, double alpha, const vpk_em_config* cfg_in) {
    if (!ctx || !ctx->pipe || ctx->pipe->B <= 0) { set_error("vpk_pipeline_run: no batch uploaded"); return VPK_ERR_STATE; }
    if (S != VPK_CNN_SIZE) { set_error("vpk_pipeline_run: the CNN input is %dx%d (cnn/deploy.prototxt:7); size=%d", VPK_CNN_SIZE, VPK_CNN_SIZE, S); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    PipeState* p = ctx->pipe;
    vpk_em_config cfg;
    if (cfg_in) cfg = *cfg_in; else vpk_em_default_config(&cfg);
    const int B = p->B;
    const size_t plane = (size_t)S * S;
    const int chunk = B < kChunk ? B : kChunk;
    VPK_TRY(p->hist.ensure(sizeof(uint32_t) * plane * chunk));
    VPK_TRY(p->images.ensure(plane * B));
    VPK_TRY(p->sigout.ensure(sizeof(float) * kCells * (size_t)B));
    const size_t n_i32 = 3 * (size_t)B + (size_t)B * VPK_MAX_VP;
    const size_t n_f64 = (size_t)B * VPK_MAX_VP * 5;
    VPK_TRY(p->out_small.ensure(n_f64 * sizeof(double) + n_i32 * sizeof(int32_t) + 64));
    VPK_TRY(p->out_assoc.ensure((p->sumN + 1) * sizeof(int32_t)));
    p->S = S;
    VPK_CUDA(cudaEventRecord(p->ev[0], ctx->stream));
    VPK_TRY(lines_from_segments_dev(ctx, p->seg.as<double>(), p->sumN, p->lines.as<double>()));
    // stage 3, early part: the segment-pair pass of the EM (similarity matrices, line ratings) needs the
    // segments only; it runs on the EM's own streams underneath stages 1 and 2
    EmDeviceOut d;
    double* f = p->out_small.as<double>();
    d.vp = f; f += (size_t)B * VPK_MAX_VP * 3;
    d.sigma = f; f += (size_t)B * VPK_MAX_VP;
    d.counts_weighted = f; f += (size_t)B * VPK_MAX_VP;
    int32_t* ip = reinterpret_cast<int32_t*>(f);
    d.status = ip; ip += B;
    d.n_vp = ip; ip += B;
    d.iterations = ip; ip += B;
    d.counts = ip;
    d.vp_assoc = p->out_assoc.as<int32_t>();
    d.decision_metric = nullptr;
    p->out = d;
    VPK_TRY(em_dev(ctx, p->lines.as<double>(), p->seg.as<double>(), p->offsets.as<int32_t>(), p->h_offsets.data(), B,
                   p->sigout.as<float>(), nullptr, p->images.as<uint8_t>(), S, nullptr, nullptr, &cfg, d, EM_EARLY));
    // stage 1 for the whole batch, chunked
    for (int c0 = 0; c0 < B; c0 += chunk) {
        const int nb = B - c0 < chunk ? B - c0 : chunk;
        uint8_t* img = p->images.as<uint8_t>() + plane * c0;
        VPK_TRY(sphere_map_dev(ctx, p->lines.as<double>(), p->offsets.as<int32_t>() + c0, p->h_offsets.data() + c0, nb, S,
                               sphere_mode, alpha, nullptr, p->hist.as<uint32_t>(), nullptr, img));
        if (sphere_mode == VPK_SPHERE_VOTES)
            VPK_TRY(sphere_votes_finish_dev(ctx, nb, S, p->hist.as<uint32_t>(), nullptr, img, nullptr));
    }
    VPK_CUDA(cudaEventRecord(p->ev[1], ctx->stream));
    // stage 2
    for (int c0 = 0; c0 < B; c0 += chunk) {
        const int nb = B - c0 < chunk ? B - c0 : chunk;
        VPK_TRY(cnn_forward_dev(ctx, p->images.as<uint8_t>() + plane * c0, nb, p->sigout.as<float>() + (size_t)kCells * c0, nullptr));
    }
    VPK_CUDA(cudaEventRecord(p->ev[2], ctx->stream));
    // stage 3 (the rest: initial hypotheses and the supersteps)
    VPK_TRY(em_dev(ctx, p->lines.as<double>(), p->seg.as<double>(), p->offsets.as<int32_t>(), p->h_offsets.data(), B,
                   p->sigout.as<float>(), nullptr, p->images.as<uint8_t>(), S, nullptr, nullptr, &cfg, d));
    VPK_CUDA(cudaEventRecord(p->ev[3], ctx->stream));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    p->have_result = true;
    return VPK_OK;
}

int vpk_pipeline_fetch(vpk_ctx* ctx, vpk_em_result* out, float* sigout, uint8_t* sphere_images) {
    if (!ctx || !ctx->pipe || !ctx->pipe->have_result) { set_error("vpk_pipeline_fetch: nothing to fetch"); return VPK_ERR_STATE; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    PipeState* p = ctx->pipe;
    const size_t B = p->B;
    auto D2H = [&](void* dst, const void* src, size_t bytes) {
        return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream);
    };
    if (out) {
        if (!out->status || !out->n_vp || !out->iterations || !out->vp || !out->sigma || !out->counts || !out->counts_weighted || !out->vp_assoc) {
            set_error("vpk_pipeline_fetch: result arrays must be allocated by the caller"); return VPK_ERR_ARG;
        }
        // the small outputs are one packed block on the device (vp | sigma | counts_weighted | status |
        // n_vp | iterations | counts): one copy into pinned staging instead of seven into pageable memory
        const size_t n_f64 = B * VPK_MAX_VP * 5, n_i32 = 3 * B + B * VPK_MAX_VP;
        const size_t small_bytes = n_f64 * sizeof(double) + n_i32 * sizeof(int32_t);
        VPK_TRY(p->h_small.ensure(small_bytes));
        VPK_TRY(p->h_assoc.ensure((p->sumN + 1) * sizeof(int32_t)));
        VPK_CUDA(D2H(p->h_small.p, p->out_small.p, small_bytes));
        if (p->sumN) VPK_CUDA(D2H(p->h_assoc.p, p->out.vp_assoc, p->sumN * sizeof(int32_t)));
    }
    if (sigout) VPK_CUDA(D2H(sigout, p->sigout.p, B * kCells * sizeof(float)));
    if (sphere_images) VPK_CUDA(D2H(sphere_images, p->images.p, B * (size_t)p->S * p->S));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    if (out) {
        const double* f = p->h_small.as<double>();
        memcpy(out->vp, f, B * VPK_MAX_VP * 3 * sizeof(double)); f += B * VPK_MAX_VP * 3;
        memcpy(out->sigma, f, B * VPK_MAX_VP * sizeof(double)); f += B * VPK_MAX_VP;
        memcpy(out->counts_weighted, f, B * VPK_MAX_VP * sizeof(double)); f += B * VPK_MAX_VP;
        const int32_t* ip = reinterpret_cast<const int32_t*>(f);
        memcpy(out->status, ip, B * sizeof(int32_t)); ip += B;
        memcpy(out->n_vp, ip, B * sizeof(int32_t)); ip += B;
        memcpy(out->iterations, ip, B * sizeof(int32_t)); ip += B;
        memcpy(out->counts, ip, B * VPK_MAX_VP * sizeof(int32_t));
        if (p->sumN) memcpy(out->vp_assoc, p->h_assoc.p, p->sumN * sizeof(int32_t));
    }
    return VPK_OK;
}

int vpk_pipeline_horizon(vpk_ctx* ctx, int32_t maxbest, double theta_vmin, double theta_z, const double* true_horizons,
                         const double* scales, const double* heights, double* points, int32_t* best_combo, double* errors) {
    if (!ctx || !ctx->pipe || !ctx->pipe->have_result) { set_error("vpk_pipeline_horizon: no completed run"); return VPK_ERR_STATE; }
    if (!points || !best_combo || maxbest < 0 || (errors && !(true_horizons && scales && heights))) { set_error("vpk_pipeline_horizon: bad argument"); return VPK_ERR_ARG; }
    VPK_CUDA(cudaSetDevice(ctx->device));
    PipeState* p = ctx->pipe;
    VPK_TRY(p->horizon.ensure(horizon_out_bytes(p->B)));
    VPK_TRY(p->h_horizon.ensure(horizon_out_bytes(p->B)));
    // the EM result stays where the EM wrote it: no host round trip between the two
    const double* d_truth = nullptr;
    if (errors) {
        VPK_TRY(horizon_upload_truth(ctx, p->truth, true_horizons, scales, heights, p->B));
        d_truth = p->truth.as<double>();
    }
    VPK_TRY(horizon_dev(ctx, p->out.vp, p->out.counts, p->out.n_vp, p->B, maxbest, theta_vmin, theta_z, d_truth, p->horizon.p));
    VPK_CUDA(cudaMemcpyAsync(p->h_horizon.p, p->horizon.p, horizon_out_bytes(p->B), cudaMemcpyDeviceToHost, ctx->stream));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    horizon_unpack(p->h_horizon.p, p->B, points, best_combo, errors);
    return VPK_OK;
}

int vpk_pipeline_host(vpk_ctx* ctx, const double* segments, const int32_t* offsets, int32_t B, int32_t S, int32_t sphere_mode,
                      double alpha, const vpk_em_config* cfg, vpk_em_result* out, float* sigout, uint8_t* sphere_images) {
    static const bool trace = getenv("VPK_PIPE_TRACE") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    VPK_TRY(vpk_pipeline_upload(ctx, segments, offsets, B));
    const auto t1 = std::chrono::steady_clock::now();
    VPK_TRY(vpk_pipeline_run(ctx, S, sphere_mode, alpha, cfg));
    const auto t2 = std::chrono::steady_clock::now();
    const int rc = vpk_pipeline_fetch(ctx, out, sigout, sphere_images);
    if (trace) {
        const auto t3 = std::chrono::steady_clock::now();
        auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
            return std::chrono::duration<double, std::milli>(b - a).count();
        };
        float dev[4] = {0, 0, 0, 0};
        vpk_pipeline_stage_ms(ctx, dev);
        fprintf(stderr, "[vpk_pipeline_host] upload %.3f ms, run %.3f ms (device %.3f), fetch %.3f ms\n", ms(t0, t1), ms(t1, t2), dev[3], ms(t2, t3));
    }
    return rc;
}

int vpk_pipeline_stage_ms(vpk_ctx* ctx, float ms[4]) {
    if (!ctx || !ctx->pipe || !ctx->pipe->have_result || !ms) { set_error("vpk_pipeline_stage_ms: no completed run"); return VPK_ERR_STATE; }
    PipeState* p = ctx->pipe;
    VPK_CUDA(cudaEventElapsedTime(&ms[0], p->ev[0], p->ev[1]));
    VPK_CUDA(cudaEventElapsedTime(&ms[1], p->ev[1], p->ev[2]));
    VPK_CUDA(cudaEventElapsedTime(&ms[2], p->ev[2], p->ev[3]));
    VPK_CUDA(cudaEventElapsedTime(&ms[3], p->ev[0], p->ev[3]));
    return VPK_OK;
}

}  // extern "C"
