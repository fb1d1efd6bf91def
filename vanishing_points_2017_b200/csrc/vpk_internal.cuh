// Internal plumbing shared by the libvpk.so translation units: context,
// device workspaces, launch accounting / per-kernel event timing, error strings.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include <map>
#include "../../include/vpk.h"

namespace vpk {

void set_error(const char* fmt, ...);

#define VPK_CUDA(expr)                                                              \
    do {                                                                            \
        cudaError_t _e = (expr);                                                    \
        if (_e != cudaSuccess) {                                                    \
            vpk::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr,             \
                           cudaGetErrorString(_e));                                 \
            return VPK_ERR_CUDA;                                                    \
        }                                                                           \
    } while (0)

#define VPK_TRY(expr)                                                               \
    do {                                                                            \
        int _s = (expr);                                                            \
        if (_s != VPK_OK) return _s;                                                \
    } while (0)

// Growable device workspace.  Steady-state calls never allocate.
struct DBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return VPK_OK;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            set_error("cudaMalloc(%zu) -> %s", want, cudaGetErrorString(e));
            p = nullptr;
            return VPK_ERR_NOMEM;
        }
        cap = want;
        return VPK_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// Pinned host staging buffer (async H2D / D2H need page-locked memory).
struct HBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return VPK_OK;
        if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e != cudaSuccess) {
            set_error("cudaMallocHost(%zu) -> %s", want, cudaGetErrorString(e));
            p = nullptr;
            return VPK_ERR_NOMEM;
        }
        cap = want;
        return VPK_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct ProfEntry {
    double total_ms = 0.0;
    int64_t launches = 0;
};

struct PendingEvent {
    const char* name;
    cudaEvent_t a, b;
};

struct CnnState;   // cnn.cu
struct EmState;    // em.cu
struct PipeState;  // pipeline.cu
struct LsdState;   // lsd.cu
struct PrepState;  // image_prep.cu

}  // namespace vpk

struct vpk_ctx {
    int device = 0;
    int num_sms = 148;
    size_t l2_bytes = 126u << 20;
    cudaStream_t stream = nullptr;
    int64_t launches = 0;
    bool profiling = false;
    std::map<std::string, vpk::ProfEntry> prof;
    std::vector<vpk::PendingEvent> pending;
    std::vector<cudaEvent_t> event_pool;

    // generic workspaces (stage-private buffers live in the stage states)
    vpk::DBuf d_lines, d_segments, d_offsets, d_work, d_hist, d_img, d_weights, d_misc;
    vpk::DBuf d_curves_tab;                 // curves mode: column -> first sample table + coverage LUT for (curves_tab_S, curves_tab_alpha)
    int curves_tab_S = 0;
    double curves_tab_alpha = -1.0;
    size_t curves_band_smem = 0;            // dynamic shared memory the band kernel is opted in for on this device
    vpk::HBuf h_stage;

    cudaEvent_t marks[4] = {nullptr, nullptr, nullptr, nullptr};   // vpk_mark: device timestamps on this context's stream

    vpk::CnnState* cnn = nullptr;
    vpk::EmState* em = nullptr;
    vpk::PipeState* pipe = nullptr;
    vpk::LsdState* lsd = nullptr;
    vpk::PrepState* prep = nullptr;
};

namespace vpk {

// Launch accounting.  Usage:
//   { KernelScope ks(ctx, "name"); kernel<<<g,b,s,ctx->stream>>>(...); }
struct KernelScope {
    vpk_ctx* ctx;
    const char* name;
    cudaEvent_t a = nullptr, b = nullptr;
    bool timed;
    // counted = false: the launch is being captured into a graph (counted when the graph runs, no events)
    KernelScope(vpk_ctx* c, const char* n, bool counted = true) : ctx(c), name(n), timed(counted && c->profiling) {
        if (counted) ctx->launches++;
        if (timed) {
            a = take(); b = take();
            cudaEventRecord(a, ctx->stream);
        }
    }
    ~KernelScope() {
        if (timed) {
            cudaEventRecord(b, ctx->stream);
            ctx->pending.push_back({name, a, b});
        }
    }
    cudaEvent_t take() {
        if (!ctx->event_pool.empty()) {
            cudaEvent_t e = ctx->event_pool.back();
            ctx->event_pool.pop_back();
            return e;
        }
        cudaEvent_t e;
        cudaEventCreate(&e);
        return e;
    }
};

int profile_collect(vpk_ctx* ctx);   // drains ctx->pending into ctx->prof (synchronises)

inline int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("launch %s -> %s", what, cudaGetErrorString(e));
        return VPK_ERR_CUDA;
    }
    return VPK_OK;
}

// ---- stage entry points on DEVICE buffers (used by the public host-buffer
// functions and by the pipeline) -------------------------------------------
int lines_from_segments_dev(vpk_ctx* ctx, const double* d_seg, int64_t n, double* d_lines);

struct SphereWork;  // sphere.cu
int sphere_map_dev(vpk_ctx* ctx, const double* d_lines, const int32_t* d_offsets,
                   const int32_t* h_offsets, int32_t B, int32_t S, int32_t mode, double alpha,
                   const double* d_weights, uint32_t* d_hist, unsigned long long* d_whist,
                   uint8_t* d_img);

int sphere_votes_finish_dev(vpk_ctx* ctx, int32_t B, int32_t S, const uint32_t* d_hist,
                            const unsigned long long* d_whist, uint8_t* d_img, float* d_wout);

int cnn_forward_dev(vpk_ctx* ctx, const uint8_t* d_images, int32_t B, float* d_sigout, float* d_logits);

struct EmDeviceOut {
    int32_t* status; int32_t* n_vp; int32_t* iterations;
    double* vp; double* sigma; int32_t* counts; double* counts_weighted;
    int32_t* vp_assoc; double* decision_metric;
};
int em_dev(vpk_ctx* ctx, const double* d_lines, const double* d_segments, const int32_t* d_offsets,
           const int32_t* h_offsets, int32_t B, const float* d_resp_f32, const double* d_resp_f64,
           const uint8_t* d_sphere, int32_t S, const double* d_init_vp, const int32_t* d_init_off,
           const vpk_em_config* cfg, const EmDeviceOut& out, int phase = 0);
enum { EM_ALL = 0, EM_EARLY = 1 };

int segments_from_lsd_dev(vpk_ctx* ctx, const double* d_lsd, int ncols, const int32_t* d_offsets, const int32_t* d_widths,
                          const int32_t* d_heights, int B, int64_t n, double* d_seg, double* d_nfa);

// horizon.cu: calc_horizon.calculate_horizon_and_ortho_vp for a batch of EM results on the device
int horizon_dev(vpk_ctx* ctx, const double* d_vp, const int32_t* d_counts, const int32_t* d_n_vp, int32_t B, int32_t maxbest,
                double theta_vmin, double theta_z, const double* d_truth, void* d_out);
size_t horizon_out_bytes(int32_t B);
int horizon_upload_truth(vpk_ctx* ctx, DBuf& buf, const double* true_horizons, const double* scales, const double* heights, int32_t B);
void horizon_unpack(const void* h_rec, int32_t B, double* points, int32_t* best_combo, double* errors);

// lsd.cu: the LSD detector on a ragged batch of images; leaves the (sum N, 7) rows on the device (*d_rows,
// image b's rows start at row_offsets[b], which the host also gets) and writes the B counts to counts_out
int lsd_dev(vpk_ctx* ctx, const void* images, int32_t dtype, const int64_t* pixel_offsets, const int32_t* widths,
            const int32_t* heights, int32_t B, const vpk_lsd_config* cfg, int32_t* counts_out, const double** d_rows,
            std::vector<int32_t>& row_offsets);
// The same in three steps, for input that is produced on the device: lsd_plan validates the call and lays out
// its geometry (host only), lsd_input sizes the workspaces and returns the device buffer the detector reads
// (row-major pixels of type `dtype` at pixel_offsets), lsd_detect runs the detector on what was written there.
struct LsdPlan {
    vpk_lsd_config cfg;
    int32_t B = 0, dtype = 0;
    std::vector<int64_t> off64;     // offsets (B+1 each) of the input, x-pass, sampled-pixel and seed-item arrays
    std::vector<int32_t> dims;      // W, H, X, Y (B each)
    int maxX = 0, maxY = 0;
    int64_t max_pix = 0;
};
int lsd_plan(const int64_t* pixel_offsets, const int32_t* widths, const int32_t* heights, int32_t B, int32_t dtype,
             const vpk_lsd_config* cfg, int32_t* counts_out, LsdPlan& plan);
int lsd_input(vpk_ctx* ctx, const LsdPlan& plan, void** d_in);
int lsd_detect(vpk_ctx* ctx, const LsdPlan& plan, int32_t* counts_out, const double** d_rows, std::vector<int32_t>& row_offsets);

// image_prep.cu: resize (INTER_AREA) + rgb2gray of a ragged batch of uint8 RGB photos.  prep_plan validates the
// call and computes the prepared sizes (host only); prep_run copies the photos to the device and writes the float64
// gray planes, multiplied by out_scale, to d_out (image b's W'*H' plane at plan.pix_off[b]).
struct PrepPlan {
    int32_t B = 0;
    std::vector<int32_t> w, h, W, H;
    std::vector<int64_t> src_off;   // B+1 byte offsets of the photos
    std::vector<int64_t> pix_off;   // B+1 pixel offsets of the prepared planes
};
int prep_plan(const uint8_t* rgb, const int64_t* byte_offsets, const int32_t* widths, const int32_t* heights, int32_t B,
              int32_t target_size, const char* who, PrepPlan& plan);
int prep_run(vpk_ctx* ctx, const PrepPlan& plan, const uint8_t* rgb, double out_scale, double* d_out);

void cnn_free(vpk_ctx* ctx);
void em_free(vpk_ctx* ctx);
void pipe_free(vpk_ctx* ctx);
void lsd_free(vpk_ctx* ctx);
void prep_free(vpk_ctx* ctx);

}  // namespace vpk
