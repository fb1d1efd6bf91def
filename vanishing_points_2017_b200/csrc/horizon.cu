// Row N1 of SURVEY.md section 8(f): horizon line and orthogonal VP triplet from the EM result.
//
// Replaces calc_horizon.calculate_horizon_and_ortho_vp (reference calc_horizon.py:19-225), the
// immediate consumer of the EM output in both drivers (example.py:65, benchmark.py:233), for a whole
// batch on the device, so that the resident pipeline can emit horizons without a host round trip.
//
// One CTA per image.  The num_best = min(maxbest, M) VPs with the most lines are ranked
// (numpy.argsort(counts)[::-1], calc_horizon.py:34-36: ascending stable order reversed -- what numpy
// does for up to 16 elements; beyond that numpy's introsort leaves the order of equal counts to the
// platform), every triplet i < j < k of them is scored by one thread (:66-183) and the first triplet
// with the maximal score wins (strict '>' in loop order, :186-192).  float64 throughout, operations in
// the order of the numpy expressions.
#include <math.h>
#include "vpk_internal.cuh"

namespace vpk {

static constexpr int kHorizonThreads = 128;
static constexpr int kHMax = VPK_MAX_VP;

struct HorizonOut { double hP1[3], hP2[3], zVP[3], hVP1[3], hVP2[3], err; int combo[3]; };

struct Triplet {
    double score;
    double zVP[3], hVP1[3], hVP2[3], hlin[3];
};

__device__ __forceinline__ double h_dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
// VPinImage (calc_horizon.py:11-16)
__device__ __forceinline__ bool vp_in_image(const double* v) {
    const double x = v[0] / v[2], y = v[1] / v[2];
    return x <= 1 && x >= -1 && y <= 1 && y >= -1;
}
// hP = cross(hlin, [s, 0, 1]) / its third component (:172-175, :219-222), s = +1 / -1
__device__ __forceinline__ void horizon_point(const double* h, double s, double* p) {
    const double c0 = h[1] * 1.0 - h[2] * 0.0, c1 = h[2] * s - h[0] * 1.0, c2 = h[0] * 0.0 - h[1] * s;
    p[0] = c0 / c2; p[1] = c1 / c2; p[2] = c2 / c2;
}

// one triplet (a, b, c) of ranks into best[] (calc_horizon.py:66-183)
__device__ void eval_triplet(const double (*vps)[3], const int* counts, const int* best, const unsigned char* zen, int a, int b,
                             int c, double costh, Triplet& t) {
    const int ia = best[a], ib = best[b], ic = best[c];
    const double* Va = vps[ia];
    const double* Vb = vps[ib];
    const double* Vc = vps[ic];
    const double AB = fabs(h_dot3(Va, Vb)), BC = fabs(h_dot3(Vb, Vc)), AC = fabs(h_dot3(Va, Vc));
    int num_zenith = 0;
    const double* zenith = Va;
    if (zen[ia]) { ++num_zenith; zenith = Va; }
    if (zen[ib]) { ++num_zenith; zenith = Vb; }
    if (zen[ic]) { ++num_zenith; zenith = Vc; }
    const int num_central = (vp_in_image(Va) ? 1 : 0) + (vp_in_image(Vb) ? 1 : 0) + (vp_in_image(Vc) ? 1 : 0);
    const double* h1v; const double* h2v; const double* zv;
    double h1c, h2c;
    const double ya = fabs(Va[1]), yb = fabs(Vb[1]), yc = fabs(Vc[1]);
    if (ya > yb && ya > yc) { h1v = Vb; h2v = Vc; zv = Va; h1c = counts[ib]; h2c = counts[ic]; }
    else if (yb > ya && yb > yc) { h1v = Va; h2v = Vc; zv = Vb; h1c = counts[ia]; h2c = counts[ic]; }
    else { h1v = Va; h2v = Vb; zv = Vc; h1c = counts[ia]; h2c = counts[ib]; }
    // zlin = cross(zVP, [0,0,1]) / |zlin[0:2]| (:131-132)
    const double z0 = zv[1] * 1.0 - zv[2] * 0.0, z1 = zv[2] * 0.0 - zv[0] * 1.0;
    const double zn = sqrt(z0 * z0 + z1 * z1);
    const double l1 = z0 / zn, l2 = z1 / zn;
    const double v11 = h1v[0], v12 = h1v[1], v13 = h1v[2], v21 = h2v[0], v22 = h2v[1], v23 = h2v[2];
    const double p1x = v11 / v13, p1y = v12 / v13, p1z = v13 / v13, p2x = v21 / v23, p2y = v22 / v23, p2z = v23 / v23;
    const double e1x = 0.0 - p1x, e1y = 0.0 - p1y, e1z = 1.0 - p1z, e2x = 0.0 - p2x, e2y = 0.0 - p2y, e2z = 1.0 - p2z;
    const double d1 = sqrt(e1x * e1x + e1y * e1y + e1z * e1z), d2 = sqrt(e2x * e2x + e2y * e2y + e2z * e2z);
    t.hlin[0] = -l2;
    t.hlin[1] = l1;
    t.hlin[2] = ((v11 * l2 - v12 * l1) / v13 * (d2 * h1c) + (v21 * l2 - v22 * l1) / v23 * (d1 * h2c)) / ((d1 * h2c) + (d2 * h1c));
    // angle of the proposed horizon line (:169-170)
    const double hx = p1x - p2x, hy = p1y - p2y, hz = p1z - p2z;
    const double hn = sqrt(hx * hx + hy * hy + hz * hz);
    const double hang = acos(fabs(hx * 1.0 + hy * 0.0 + hz * 0.0) / hn);
    double hP1[3], hP2[3];
    horizon_point(t.hlin, 1.0, hP1);
    horizon_point(t.hlin, -1.0, hP2);
    double ortho = 0.0;
    if (num_zenith == 1) {
        const double zl = sqrt(h_dot3(zenith, zenith));
        const double cosphi = fabs((hx / hn) * (zenith[0] / zl) + (hy / hn) * (zenith[1] / zl) + (hz / hn) * (zenith[2] / zl));
        double cl = fmin(fmax(cosphi, 0.0), 1.0);
        if (isnan(cosphi)) cl = cosphi;                                   // numpy.clip keeps NaN
        ortho = 1.0 - cl;
    }
    const int zenith_pos = zv[1] > 0 ? 1 : -1;
    const int hor_pos = (hP1[1] + hP2[1]) / 2 < 0 ? 1 : -1;
    const bool ok = AB < costh && BC < costh && AC < costh && num_zenith == 1 && num_central <= 1 &&
                    hang < 30 * 3.14159265358979323846 / 180 && zenith_pos * hor_pos == 1;
    const double weight = (double)(counts[ia] + counts[ib] + counts[ic]);
    t.score = (ok ? 1.0 : 0.0) * weight * ortho;
    for (int k = 0; k < 3; ++k) { t.zVP[k] = zv[k]; t.hVP1[k] = h1v[k]; t.hVP2[k] = h2v[k]; }
}

__device__ __forceinline__ void unrank_triplet(int idx, int n, int& a, int& b, int& c) {
    int r = idx;
    a = 0;
    while (true) { const int m = n - 1 - a, cnt = m * (m - 1) / 2; if (r < cnt) break; r -= cnt; ++a; }
    b = a + 1;
    while (true) { const int cnt = n - 1 - b; if (r < cnt) break; r -= cnt; ++b; }
    c = b + 1 + r;
}

__global__ void __launch_bounds__(kHorizonThreads) horizon_kernel(const double* __restrict__ vp, const int32_t* __restrict__ counts,
                                                                  const int32_t* __restrict__ n_vp, int maxbest, double costh,
                                                                  double sin_tz, const double* __restrict__ true_h,
                                                                  const double* __restrict__ scales, const double* __restrict__ heights,
                                                                  HorizonOut* __restrict__ out) {
    __shared__ double s_vp[kHMax][3];
    __shared__ int s_cnt[kHMax], s_best[kHMax];
    __shared__ unsigned char s_zen[kHMax];
    __shared__ double s_score[kHorizonThreads];
    __shared__ int s_idx[kHorizonThreads];
    const int img = blockIdx.x, tid = threadIdx.x;
    const int M = min(max(n_vp[img], 0), kHMax);
    for (int m = tid; m < M; m += kHorizonThreads) {
        for (int k = 0; k < 3; ++k) s_vp[m][k] = vp[((size_t)img * kHMax + m) * 3 + k];
        s_cnt[m] = counts[(size_t)img * kHMax + m];
        s_zen[m] = fabs(s_vp[m][1]) > sin_tz ? 1 : 0;                      // :31
    }
    __syncthreads();
    const int nb = min(maxbest, M);
    // argsort(counts)[::-1][:num_best] (:34-36): stable ascending rank, reversed
    for (int m = tid; m < M; m += kHorizonThreads) {
        int pos = 0;
        for (int q = 0; q < M; ++q) pos += (s_cnt[q] < s_cnt[m] || (s_cnt[q] == s_cnt[m] && q < m)) ? 1 : 0;
        const int rpos = M - 1 - pos;
        if (rpos < nb) s_best[rpos] = m;
    }
    __syncthreads();
    HorizonOut o;
    for (int k = 0; k < 3; ++k) o.combo[k] = -1;
    double hlin[3];
    if (nb > 2) {
        const int ncomb = nb * (nb - 1) * (nb - 2) / 6;
        // first triplet with the maximal score (:186-192); NaN scores never win
        double bs = -1.0;
        int bi = -1;
        for (int idx = tid; idx < ncomb; idx += kHorizonThreads) {
            int a, b, c;
            unrank_triplet(idx, nb, a, b, c);
            Triplet t;
            eval_triplet(s_vp, s_cnt, s_best, s_zen, a, b, c, costh, t);
            if (t.score > bs) { bs = t.score; bi = idx; }
        }
        s_score[tid] = bs; s_idx[tid] = bi;
        __syncthreads();
        for (int o2 = kHorizonThreads / 2; o2 > 0; o2 >>= 1) {
            if (tid < o2) {
                const double s2 = s_score[tid + o2];
                const int i2 = s_idx[tid + o2];
                if (i2 >= 0 && (s_idx[tid] < 0 || s2 > s_score[tid] || (s2 == s_score[tid] && i2 < s_idx[tid]))) {
                    s_score[tid] = s2; s_idx[tid] = i2;
                }
            }
            __syncthreads();
        }
        if (tid != 0) return;
        const int win = s_idx[0] >= 0 ? s_idx[0] : 0;      // every score NaN: the reference leaves the outputs unbound; triplet 0 here
        int a, b, c;
        unrank_triplet(win, nb, a, b, c);
        Triplet t;
        eval_triplet(s_vp, s_cnt, s_best, s_zen, a, b, c, costh, t);
        for (int k = 0; k < 3; ++k) { o.zVP[k] = t.zVP[k]; o.hVP1[k] = t.hVP1[k]; o.hVP2[k] = t.hVP2[k]; hlin[k] = t.hlin[k]; }
        o.combo[0] = s_best[a]; o.combo[1] = s_best[b]; o.combo[2] = s_best[c];
    } else {
        if (tid != 0) return;
        const double up[3] = {0.0, 1.0, 0.0};
        for (int k = 0; k < 3; ++k) o.zVP[k] = up[k];
        if (nb > 1) {                                                      // :195-200
            for (int k = 0; k < 3; ++k) { o.hVP1[k] = s_vp[0][k]; o.hVP2[k] = s_vp[1][k]; }
            o.combo[0] = 0; o.combo[1] = 1;
            const double* p = s_vp[0];
            const double* q = s_vp[1];
            hlin[0] = p[1] * q[2] - p[2] * q[1]; hlin[1] = p[2] * q[0] - p[0] * q[2]; hlin[2] = p[0] * q[1] - p[1] * q[0];
        } else {
            if (nb > 0) { for (int k = 0; k < 3; ++k) { o.hVP1[k] = s_vp[0][k]; o.hVP2[k] = s_vp[0][k]; } }   // :201-206
            else { o.hVP1[0] = -1.0; o.hVP1[1] = 0.0; o.hVP1[2] = 0.0; o.hVP2[0] = 1.0; o.hVP2[1] = 0.0; o.hVP2[2] = 0.0; }   // :207-212
            o.combo[0] = 0; o.combo[1] = 0;
            hlin[0] = 0.0; hlin[1] = 1.0; hlin[2] = 0.0;                    // cross([0,0,1], [1,0,1])
        }
    }
    horizon_point(hlin, 1.0, o.hP1);                                       // :219-222
    horizon_point(hlin, -1.0, o.hP2);
    // horizon error against the ground-truth horizon (benchmark.py:247-253), NaN without one
    o.err = nan("");
    if (true_h) {
        double t1[3], t2[3];
        horizon_point(true_h + 3 * (size_t)img, 1.0, t1);
        horizon_point(true_h + 3 * (size_t)img, -1.0, t2);
        o.err = fmax(fabs(o.hP1[1] - t1[1]), fabs(o.hP2[1] - t2[1])) / 2 * scales[img] * 1.0 / heights[img];
    }
    out[img] = o;
}

int horizon_dev(vpk_ctx* ctx, const double* d_vp, const int32_t* d_counts, const int32_t* d_n_vp, int32_t B, int32_t maxbest,
                double theta_vmin, double theta_z, const double* d_truth, void* d_out) {
    if (B <= 0) return VPK_OK;
    KernelScope ks(ctx, "horizon");
    // d_truth: nullptr or (B,3) true horizons | (B) scales | (B) image heights, contiguous
    horizon_kernel<<<B, kHorizonThreads, 0, ctx->stream>>>(d_vp, d_counts, d_n_vp, maxbest, cos(theta_vmin), sin(theta_z), d_truth,
                                                          d_truth ? d_truth + 3 * (size_t)B : nullptr,
                                                          d_truth ? d_truth + 4 * (size_t)B : nullptr,
                                                          static_cast<HorizonOut*>(d_out));
    return check_launch("horizon");
}

size_t horizon_out_bytes(int32_t B) { return sizeof(HorizonOut) * (size_t)B; }

// (B,3) true horizons | (B) scales | (B) heights -> one device block
int horizon_upload_truth(vpk_ctx* ctx, DBuf& buf, const double* true_horizons, const double* scales, const double* heights, int32_t B) {
    VPK_TRY(buf.ensure(5 * (size_t)B * sizeof(double)));
    double* d = buf.as<double>();
    VPK_CUDA(cudaMemcpyAsync(d, true_horizons, 3 * (size_t)B * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    VPK_CUDA(cudaMemcpyAsync(d + 3 * (size_t)B, scales, (size_t)B * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    VPK_CUDA(cudaMemcpyAsync(d + 4 * (size_t)B, heights, (size_t)B * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    return VPK_OK;
}

// unpack HorizonOut records (host copy) into the caller's arrays
void horizon_unpack(const void* h_rec, int32_t B, double* points, int32_t* best_combo, double* errors) {
    const HorizonOut* r = static_cast<const HorizonOut*>(h_rec);
    for (int b = 0; b < B; ++b) {
        const double* src[5] = {r[b].hP1, r[b].hP2, r[b].zVP, r[b].hVP1, r[b].hVP2};
        for (int q = 0; q < 5; ++q)
            for (int k = 0; k < 3; ++k) points[((size_t)b * 5 + q) * 3 + k] = src[q][k];
        for (int k = 0; k < 3; ++k) best_combo[(size_t)b * 3 + k] = r[b].combo[k];
        if (errors) errors[b] = r[b].err;
    }
}

// the same on the device, one thread per image, into the caller's device arrays
__global__ void horizon_unpack_kernel(const HorizonOut* __restrict__ r, int32_t B, double* __restrict__ points,
                                      int32_t* __restrict__ best_combo, double* __restrict__ errors) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double* src[5] = {r[b].hP1, r[b].hP2, r[b].zVP, r[b].hVP1, r[b].hVP2};
    for (int q = 0; q < 5; ++q)
        for (int k = 0; k < 3; ++k) points[((size_t)b * 5 + q) * 3 + k] = src[q][k];
    for (int k = 0; k < 3; ++k) best_combo[(size_t)b * 3 + k] = r[b].combo[k];
    if (errors) errors[b] = r[b].err;
}

int horizon_unpack_dev(vpk_ctx* ctx, const void* d_rec, int32_t B, double* d_points, int32_t* d_best_combo, double* d_errors) {
    if (B <= 0) return VPK_OK;
    KernelScope ks(ctx, "horizon_unpack");
    horizon_unpack_kernel<<<(B + 127) / 128, 128, 0, ctx->stream>>>(static_cast<const HorizonOut*>(d_rec), B, d_points, d_best_combo,
                                                                      d_errors);
    return check_launch("horizon_unpack");
}

}  // namespace vpk

using namespace vpk;

extern "C" {

int vpk_horizon(vpk_ctx* ctx, const double* vp, const int32_t* counts, const int32_t* n_vp, int32_t n_images, int32_t maxbest,
                double theta_vmin, double theta_z, const double* true_horizons, const double* scales, const double* heights,
                double* points, int32_t* best_combo, double* errors) {
    if (!ctx || n_images < 0 || maxbest < 0 || (n_images > 0 && (!vp || !counts || !n_vp || !points || !best_combo)) ||
        (errors && !(true_horizons && scales && heights))) {
        set_error("vpk_horizon: bad argument");
        return VPK_ERR_ARG;
    }
    if (n_images == 0) return VPK_OK;
    VPK_CUDA(cudaSetDevice(ctx->device));
    const size_t B = (size_t)n_images;
    DBuf dvp, dc, dn, dout, dtruth;
    HBuf hout;
    int rc = VPK_OK;
    do {
        if ((rc = dvp.ensure(B * kHMax * 3 * sizeof(double))) || (rc = dc.ensure(B * kHMax * sizeof(int32_t))) ||
            (rc = dn.ensure(B * sizeof(int32_t))) || (rc = dout.ensure(horizon_out_bytes(n_images))) ||
            (rc = hout.ensure(horizon_out_bytes(n_images)))) break;
        cudaMemcpyAsync(dvp.p, vp, B * kHMax * 3 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(dc.p, counts, B * kHMax * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(dn.p, n_vp, B * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream);
        const double* d_truth = nullptr;
        if (errors) {
            if ((rc = horizon_upload_truth(ctx, dtruth, true_horizons, scales, heights, n_images))) break;
            d_truth = dtruth.as<double>();
        }
        if ((rc = horizon_dev(ctx, dvp.as<double>(), dc.as<int32_t>(), dn.as<int32_t>(), n_images, maxbest, theta_vmin, theta_z, d_truth, dout.p))) break;
        cudaMemcpyAsync(hout.p, dout.p, horizon_out_bytes(n_images), cudaMemcpyDeviceToHost, ctx->stream);
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { set_error("vpk_horizon: %s", cudaGetErrorString(e)); rc = VPK_ERR_CUDA; break; }
        horizon_unpack(hout.p, n_images, points, best_combo, errors);
    } while (0);
    dvp.release(); dc.release(); dn.release(); dout.release(); dtruth.release(); hout.release();
    return rc;
}

}  // extern "C"
