// Stage 3 core: the per-image logic of the EM vanishing-point localisation
// (reference vp_localisation.py:168-450 and what it calls in
// probability_functions.py / coordinate_conversion.py), written against a
// small "team" abstraction so that the very same source is
//   * the body of the CUDA kernels in em.cu (team = one CTA), and
//   * a single-threaded host build used ONLY by tests/hostsim (team = 1 thread)
//     to check the control flow against the golden vectors on a box without a
//     GPU.  The host build is test infrastructure; libvpk.so never contains it.
//
// Execution model (em.cu): every image owns a slot.  The reference's control
// flow is a sequence of "E-step, weight matrix, then a reduction over the lines
// and a discrete decision"; it is restated here as a state machine.  One
// superstep = E kernel (all lines of all active slots) -> W kernel (the
// (M x N)(N x N) weight-matrix products, tiled over the whole GPU) -> POST
// kernel (one CTA per slot: reductions, 3x3 eigen-solves, pruning / split /
// merge decisions, choice of the next superstep).  `phase` says what POST does
// with the fresh E/W results.
#pragma once
#if defined(VPK_HOST_TRACE)
#include <cstdio>
#endif
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include "../../include/vpk.h"

#if defined(__CUDACC__)
#define VPK_DEV __device__ __forceinline__
#define VPK_DEVFN __device__
#define VPK_HD __host__ __device__ __forceinline__
#else
#include <cmath>
#define VPK_DEV inline
#define VPK_DEVFN inline
#define VPK_HD inline
#endif

namespace vpk {
namespace em {

#if !defined(__CUDACC__)
using std::isinf;
using std::isnan;
inline double rsqrt(double x) { return 1.0 / sqrt(x); }
#endif

constexpr int kMaxM = VPK_MAX_VP;
constexpr int kMaxComp = 100;              // probability_functions.py:87
constexpr int kCells = VPK_GRID * VPK_GRID;
constexpr int kTK = 64;                    // columns per similarity slab (W kernel tile)
constexpr int kMP = 32;                    // VP rows per weight-matrix pass (up to four 8-row tensor-core tiles)
constexpr int kMPS = kMP + 4;              // largest row stride of the W operand wt (8 * tiles + 4 doubles: conflict-free fragments)
constexpr int kPostThreads = 512;
constexpr int kK1 = 10;                    // kNN rating: nearest by distance (vp_localisation.py:34)
constexpr double kPi = 3.141592653589793;

// what POST does with the E/W results of the superstep that just ran
enum Phase : int32_t {
    PH_INIT_COUNTS = 0,   // :245-251  counts of the initial hypotheses, drop < 3 lines
    PH_SPLIT,             // :262-269  split_best_vp
    PH_MSTEP,             // :284-333  M-step
    PH_MERGE_EVAL,        // :649-681  one merge trial of merge_vps
    PH_HARD_REFIT,        // :344-396  hard-assignment refit
    PH_KEEP_WINNERS,      // :398-413  keep VPs that win a line
    PH_FINAL_COUNTS,      // :415-437  counts, drop VPs with too few lines
    PH_DONE,
    // control states (no E/W needed to enter them)
    CT_ITER_BEGIN, CT_MERGE_LOOP, CT_ADVANCE, CT_FINAL_A
};

struct Team { int tid, nthreads, warp, lane, nwarps, lanes; };

#if defined(__CUDACC__)
VPK_DEV Team make_team() {
    Team T;
    T.tid = threadIdx.x; T.nthreads = blockDim.x; T.warp = T.tid >> 5; T.lane = T.tid & 31;
    T.nwarps = T.nthreads >> 5; T.lanes = 32;
    return T;
}
VPK_DEV void team_sync() { __syncthreads(); }
VPK_DEV double warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
VPK_DEV int warp_sum_i(int v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
VPK_DEV int warp_max_i(int v) {
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
VPK_DEV long long warp_sum_ll(long long v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
VPK_DEV bool warp_any(bool p) { return __any_sync(0xffffffffu, p) != 0; }
// number of lanes below this one with p set; total = lanes with p set
VPK_DEV int warp_rank(bool p, int& total) {
    const unsigned m = __ballot_sync(0xffffffffu, p);
    total = __popc(m);
    return __popc(m & ((1u << (threadIdx.x & 31)) - 1u));
}
// max that propagates NaN like numpy.max
VPK_DEV double warp_max_nanprop(double v) {
    for (int o = 16; o > 0; o >>= 1) {
        double t = __shfl_xor_sync(0xffffffffu, v, o);
        v = (isnan(v) || isnan(t)) ? nan("") : (t > v ? t : v);
    }
    return v;
}
#else
inline Team make_team() { return Team{0, 1, 0, 0, 1, 1}; }
inline void team_sync() {}
inline double warp_sum(double v) { return v; }
inline int warp_sum_i(int v) { return v; }
inline int warp_max_i(int v) { return v; }
inline long long warp_sum_ll(long long v) { return v; }
inline bool warp_any(bool p) { return p; }
inline int warp_rank(bool p, int& total) { total = p ? 1 : 0; return 0; }
inline double warp_max_nanprop(double v) { return v; }
#endif

VPK_DEV double nanmax(double a, double b) { return (isnan(a) || isnan(b)) ? nan("") : (b > a ? b : a); }
VPK_DEV double sign_np(double x) { return x > 0 ? 1.0 : (x < 0 ? -1.0 : 0.0); }   // numpy.sign
VPK_DEV int imin(int a, int b) { return a < b ? a : b; }

// ---------------------------------------------------------------------------
// per-slot state (global memory; POST works on a shared-memory copy)
// ---------------------------------------------------------------------------
struct EmSlot {
    int32_t img, N, base, phase, iter, M, vsel, run_e, run_w, done, status, iters_out;
    int32_t merge_j, merge_k, after_merge, vidx, npdf, cap_hit;   // cap_hit: a hypothesis was dropped because kMaxM were live
    double merge_thresh, sigma_prior;
    unsigned long long ws_off;             // doubles from the workspace base
    double cur[kMaxM][3], nxt[kMaxM][3], s[kMaxM];
    // constants of the E-step on the selected VP set (prepare_estep)
    double pv[kMaxM], vx[kMaxM], vy[kMaxM], inv2s[kMaxM], coef[kMaxM];
    double cw[kMaxM];
    int32_t cnt[kMaxM];
    double pdf_a[kMaxComp], pdf_b[kMaxComp], pdf_w[kMaxComp];
};

struct EmOut {
    int32_t* status; int32_t* n_vp; int32_t* iterations;
    double* vp; double* sigma; int32_t* counts; double* counts_weighted;
    int32_t* vp_assoc; double* decision_metric;
};

// per-image view of the slot workspace
struct Img {
    int N;
    const double* lp;      // (N,4) segments (input)
    double* lsim;          // slab-major similarity matrix: element (j,k) at lsim_index(N,j,k)
    double* ln;            // (N,3) unit lines
    double* lweight;       // (N)
    double* colsum;        // (N)
    double* langle;        // (N)
    int* assoc;            // (N)
    double* lvsq;          // (kMaxM,N)  -- lvsq|pvl|w|wt are contiguous: split scratch
    double* pvl;           // (kMaxM,N)
    double* w;             // (kMaxM,N)
    double* wt;            // pvl*lweight, the A operand of the W kernel: pass p (VP rows 32p..32p+31) at
                           // wt + p*N*kMPS, line n of the pass at stride wpass_stride(M, p) (rows padded with zeros)
    size_t scratch_cap;    // doubles available from lvsq on
};

VPK_HD size_t lsim_doubles(int N) { return (size_t)((N + kTK - 1) / kTK) * kTK * (size_t)N; }
// Element (j,k) of the similarity matrix: 64-column slabs, each N x 64 contiguous; inside a row the column is
// XOR-swizzled with the row index (bits 2-3) so that the FP64 tensor-core B fragments of the W kernel (4 rows x 8
// columns per instruction, read straight from the bulk-copied rows) hit 16 different shared-memory bank pairs.
VPK_HD int lsim_swz(int j, int col) { return col ^ ((j & 3) << 2); }
VPK_HD size_t lsim_index(int N, int j, int k) { return ((size_t)(k / kTK) * N + j) * kTK + lsim_swz(j, k % kTK); }
// Pass p of the weight-matrix product for M hypotheses covers the VP rows 32p .. 32p+31 as wpass_tiles() tiles of
// 8 rows (m8n8k4 FP64 mma); line n of the pass stores its 8 * tiles operands (rows >= M are zeros) at a stride
// of 8 * tiles + 4 doubles (= 4 mod 8: the A fragments are conflict-free too).
VPK_HD int wpass_tiles(int M, int p) {
    int mp = M - p * kMP;
    if (mp > kMP) mp = kMP;
    if (mp < 1) mp = 1;
    return (mp + 7) / 8;
}
VPK_HD int wpass_stride(int M, int p) { return 8 * wpass_tiles(M, p) + 4; }
VPK_HD size_t wt_index(int N, int n, int m, int M) {
    const int p = m / kMP;
    return (size_t)p * N * kMPS + (size_t)n * wpass_stride(M, p) + (m % kMP);
}
VPK_HD size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

VPK_HD size_t slot_doubles(int N) {
    size_t n = (size_t)N;
    return align16(lsim_doubles(N)) + align16(3 * n) + 3 * align16(n) + align16((n + 1) / 2 + 1) + 3 * align16((size_t)kMaxM * n) +
           align16((size_t)(kMaxM / kMP) * kMPS * n) + 16;
}

// (host-callable too: vpk_em_debug_fetch finds the buffers of a slot with it)
VPK_HD Img make_img(int N, double* ws, const double* lp) {
    Img im;
    size_t n = (size_t)N;
    im.N = N; im.lp = lp;
    double* p = ws;
    im.lsim = p; p += align16(lsim_doubles(N));
    im.ln = p; p += align16(3 * n);
    im.lweight = p; p += align16(n);
    im.colsum = p; p += align16(n);
    im.langle = p; p += align16(n);
    im.assoc = reinterpret_cast<int*>(p); p += align16((n + 1) / 2 + 1);
    im.lvsq = p; p += align16((size_t)kMaxM * n);
    im.pvl = p; p += align16((size_t)kMaxM * n);
    im.w = p; p += align16((size_t)kMaxM * n);
    im.wt = p; p += align16((size_t)(kMaxM / kMP) * kMPS * n);
    im.scratch_cap = 3 * align16((size_t)kMaxM * n) + align16((size_t)(kMaxM / kMP) * kMPS * n);
    return im;
}

// ---------------------------------------------------------------------------
// segment-pair geometry (vp_localisation.py:700-762)
// ---------------------------------------------------------------------------
struct Seg { double x1, y1, x2, y2; };
VPK_DEV Seg load_seg(const double* lp, int n) {
    const double* p = lp + 4 * (size_t)n;
    Seg s; s.x1 = p[0]; s.y1 = p[1]; s.x2 = p[2]; s.y2 = p[3];
    return s;
}
// line_segment_point_distance (:743-758), squared; note the squared *norm* of :747
VPK_DEV double psd2(const Seg& s, double px, double py) {
    double dx = s.x2 - s.x1, dy = s.y2 - s.y1;
    double nrm = sqrt(dx * dx + dy * dy);
    double param = ((px - s.x1) * dx + (py - s.y1) * dy) / (nrm * nrm);
    double cx, cy;
    if (param < 0) { cx = s.x1; cy = s.y1; }
    else if (param > 1) { cx = s.x2; cy = s.y2; }
    else { cx = s.x1 + param * dx; cy = s.y1 + param * dy; }
    double ex = cx - px, ey = cy - py;
    return ex * ex + ey * ey;
}
// line_distance_closest (:727-740).  sqrt is monotone and correctly rounded, so the minimum of
// the four distances is the root of the minimum of the four squared distances, bit for bit.
VPK_DEV double seg_distance(const Seg& a, const Seg& b) {
    double d1 = psd2(a, b.x1, b.y1), d2 = psd2(a, b.x2, b.y2), d4 = psd2(b, a.x1, a.y1), d5 = psd2(b, a.x2, a.y2);
    return sqrt(fmin(fmin(d1, d2), fmin(d4, d5)));
}
VPK_DEV double seg_len(const Seg& a) {
    double dx = a.x1 - a.x2, dy = a.y1 - a.y2;
    return sqrt(dx * dx + dy * dy);
}
// cos(clip(f * acos(c), -pi/2, pi/2)) for c = |cos| in [0, 1] (:720-724).  For the two factors the
// reference uses (f = 9 in lines_similarity / line_rating_knn, f = 2 in split_best_vp) the Chebyshev
// polynomial T_f(c), written in u = 1 - c and evaluated by Horner's rule, replaces acos + cos: inside the
// clip range u <= 1 - cos(pi / 2f) is small, the evaluation is as accurate as the libm pair (2e-16
// against 3e-16 absolute, checked against 40-digit arithmetic) and costs a tenth of the instructions.
// Outside the range the clip gives cos(pi/2), 6.1e-17 in float64.
VPK_DEV double cos_clipped_multiple(double c, double f) {
    const double kAtClip = 6.123233995736766e-17;
    const double u = 1.0 - fmin(c, 1.0);
#if !defined(VPK_NO_CHEB)
    if (f == 9.0 && !isnan(c)) {
        if (u > 1.0 - 0.984807753012208) return kAtClip;          // 9 acos(c) > pi/2
        const double t = 1.0 + u * (-81.0 + u * (1080.0 + u * (-5544.0 + u * (14256.0 + u * (-20592.0 + u * (17472.0 + u * (-8640.0 +
                         u * (2304.0 - 256.0 * u))))))));
        return fmax(t, kAtClip);
    }
    if (f == 2.0 && !isnan(c)) {
        if (u > 1.0 - 0.7071067811865476) return kAtClip;         // 2 acos(c) > pi/2
        return fmax(1.0 + u * (-4.0 + 2.0 * u), kAtClip);
    }
#endif
    double dphi = fabs(acos(fmin(fmax(c, -1.0), 1.0)));
    if (isnan(c)) dphi = c;
    return cos(fmin(fmax(f * dphi, -0.5 * kPi), 0.5 * kPi));
}
// lines_points_cosangle (:715-724), literally: no polynomial shortcut, and on the device every operation
// individually rounded (nvcc would otherwise contract a*b + c*d into a fused multiply-add and move the
// last bit of c, which is what decides near-ties)
VPK_DEV double cosangle_reference_order(const Seg& a, const Seg& b, double f) {
    double v1x = a.x1 - a.x2, v1y = a.y1 - a.y2, v2x = b.x1 - b.x2, v2y = b.y1 - b.y2;
#if defined(__CUDA_ARCH__)
    const double dot = __dadd_rn(__dmul_rn(v1x, v2x), __dmul_rn(v1y, v2y));
    const double n1 = __dsqrt_rn(__dadd_rn(__dmul_rn(v1x, v1x), __dmul_rn(v1y, v1y)));
    const double n2 = __dsqrt_rn(__dadd_rn(__dmul_rn(v2x, v2x), __dmul_rn(v2y, v2y)));
    double c = fabs(__ddiv_rn(dot, __dmul_rn(n1, n2)));
    double dphi = fabs(acos(fmin(fmax(c, -1.0), 1.0)));
    if (isnan(c)) dphi = c;
    return cos(fmin(fmax(__dmul_rn(f, dphi), -0.5 * kPi), 0.5 * kPi));
#else
    double c = fabs((v1x * v2x + v1y * v2y) / (sqrt(v1x * v1x + v1y * v1y) * sqrt(v2x * v2x + v2y * v2y)));
    double dphi = fabs(acos(fmin(fmax(c, -1.0), 1.0)));
    if (isnan(c)) dphi = c;
    return cos(fmin(fmax(f * dphi, -0.5 * kPi), 0.5 * kPi));
#endif
}
// lines_points_cosangle (:715-724)
VPK_DEV double cosangle(const Seg& a, const Seg& b, double f) {
    double v1x = a.x1 - a.x2, v1y = a.y1 - a.y2, v2x = b.x1 - b.x2, v2y = b.y1 - b.y2;
    double c = fabs((v1x * v2x + v1y * v2y) / (sqrt(v1x * v1x + v1y * v1y) * sqrt(v2x * v2x + v2y * v2y)));
    return cos_clipped_multiple(c, f);
}
// lines_proximity (:708-712), sigma = 1
VPK_DEV double proximity(const Seg& a, const Seg& b, double d) {
    double sg = fmin(seg_len(a), seg_len(b));
    return exp(-(d * d) / (2 * sg * sg));
}
// lines_similarity (:700-705)
VPK_DEV double similarity(const Seg& a, const Seg& b, double d) { return cosangle(a, b, 9.0) * proximity(a, b, d); }

// ---- the O(N^2) pair pass works on per-segment constants so that a pair costs no division or
// square root: reciprocals are taken once per segment (results differ from the reference's
// per-pair divisions by rounding only, ~1e-16 relative).
struct SegPre { double x1, y1, x2, y2, dx, dy, inv_nn, inv_len, h; };
VPK_DEV SegPre seg_pre(const Seg& s) {
    SegPre p;
    p.x1 = s.x1; p.y1 = s.y1; p.x2 = s.x2; p.y2 = s.y2;
    p.dx = s.x2 - s.x1; p.dy = s.y2 - s.y1;
    const double nrm = sqrt(p.dx * p.dx + p.dy * p.dy);
    p.inv_nn = 1.0 / (nrm * nrm);          // line_segment_point_distance :747
    p.inv_len = 1.0 / nrm;                 // lines_points_cosangle :719
    p.h = 1.0 / (2 * nrm * nrm);           // lines_proximity :711 with sigma = 1
    return p;
}
VPK_DEV double psd2_pre(const SegPre& s, double px, double py) {
    const double param = ((px - s.x1) * s.dx + (py - s.y1) * s.dy) * s.inv_nn;
    // branch-free: the interior point is always formed and replaced by an end point outside [0, 1] (same values as
    // the reference's if / elif / else, :750-756; a NaN parameter takes the interior expression like the reference)
    double cx = s.x1 + param * s.dx, cy = s.y1 + param * s.dy;
    const bool lo = param < 0, hi = param > 1;
    cx = hi ? s.x2 : cx; cy = hi ? s.y2 : cy;
    cx = lo ? s.x1 : cx; cy = lo ? s.y1 : cy;
    const double ex = cx - px, ey = cy - py;
    return ex * ex + ey * ey;
}
// squared closest distance of two segments (line_distance_closest :727-740)
VPK_DEV double seg_distance2(const SegPre& a, const SegPre& b) {
    return fmin(fmin(psd2_pre(a, b.x1, b.y1), psd2_pre(a, b.x2, b.y2)), fmin(psd2_pre(b, a.x1, a.y1), psd2_pre(b, a.x2, a.y2)));
}
// cos(clip(9 acos(c), +-pi/2)), c = |cos| of the angle between the segments (:715-724 with f = 9).
// For 9 acos(c) >= pi/2 the reference evaluates cos(pi/2) = 6.123e-17; below that
// cos(9 t) = T3(T3(cos t)) with T3(x) = 4x^3 - 3x (no acos / cos evaluation).
VPK_DEV double cos9_pre(const SegPre& a, const SegPre& b) {
    double c = fabs((a.dx * b.dx + a.dy * b.dy) * (a.inv_len * b.inv_len));
    c = c > 1.0 ? 1.0 : c;                 // NaN stays NaN
    // branch-free (nine of ten pairs are clipped, so nearly every warp would run both sides of a branch anyway)
    const double t = c * (4.0 * c * c - 3.0);
    double r = t * (4.0 * t * t - 3.0);
    r = r < 6.123233995736766e-17 ? 6.123233995736766e-17 : r;
    return c <= 0.984807753012208 ? 6.123233995736766e-17 : r;
}
VPK_DEV double prox_pre(const SegPre& a, const SegPre& b, double d2) { return exp(-(d2 * fmax(a.h, b.h))); }
// lines_similarity (:700-705) from the squared distance
VPK_DEV double similarity_pre(const SegPre& a, const SegPre& b, double d2) { return cos9_pre(a, b) * prox_pre(a, b, d2); }

// E4 tail (vp_localisation.py:50-72, :230-233): line score from the k1 nearest segments
// cj/cd2 (ascending squared distance, ties by index; the line itself enters with distance 4, :82).
VPK_DEVFN double rate_line(const double* lp, int i, const int* cj, const double* cd2, int cnt, int N) {
    const int k2 = imin(4, N);
    const SegPre si = seg_pre(load_seg(lp, i));
    double c[kK1], px[kK1];
    for (int q = 0; q < cnt; ++q) {
        const SegPre sj = seg_pre(load_seg(lp, cj[q]));
        // The k2 neighbours are SELECTED by this value (:57-59) and real LSD output is full of exactly
        // parallel segments, whose cosangles are equal up to the last bits: the value is computed with the
        // reference's own expression and operation order (division by the product of the two norms, acos,
        // cos; lines_points_cosangle :715-724), not with the reciprocal / Chebyshev form used for the N^2
        // entries of the similarity matrix, so that near-ties fall the way they do in the reference.
        double cc = cosangle_reference_order(load_seg(lp, i), load_seg(lp, cj[q]), 9.0);
        double d2true = (cj[q] == i) ? seg_distance2(si, sj) : cd2[q];     // :65 recomputes the true distance
        px[q] = prox_pre(si, sj, d2true);
        c[q] = isnan(cc) ? -INFINITY : cc;
    }
    // the k2 largest cosangles, descending; argsort()[::-1] puts the later of equal values first (:57-59)
    double score = 0.0;
    for (int r = 0; r < k2 && r < cnt; ++r) {
        int who = 0;
        for (int q = 1; q < cnt; ++q)
            if (c[q] >= c[who]) who = q;
        score += px[who] * c[who];
        c[who] = -INFINITY;
    }
    score /= (double)k2;
    double ls = fmin(fmax(score, 0.2), 1.0);      // :231
    if (isnan(score)) ls = score;
    const Seg s0 = load_seg(lp, i);
    return seg_len(s0) * ls;                      // :232-233
}

// insert (d, j) into an ascending candidate list of capacity kK1 (ties: smaller j first).
// stride: element q of the list lives at kd[q * stride], kj[q * stride].
VPK_DEV void knn_insert(double* kd, int* kj, int stride, int& cnt, double d, int j) {
    if (isnan(d)) d = INFINITY;
    int pos;
    if (cnt < kK1) pos = cnt++;
    else {
        double ld = kd[(kK1 - 1) * stride];
        int lj = kj[(kK1 - 1) * stride];
        if (!(d < ld || (d == ld && j < lj))) return;
        pos = kK1 - 1;
    }
    while (pos > 0) {
        double pd = kd[(pos - 1) * stride];
        int pj = kj[(pos - 1) * stride];
        if (!(pd > d || (pd == d && pj > j))) break;
        kd[pos * stride] = pd; kj[pos * stride] = pj;
        --pos;
    }
    kd[pos * stride] = d; kj[pos * stride] = j;
}

// ---------------------------------------------------------------------------
// Eigen-decomposition of the symmetric 3x3 matrix [g0 g1 g2; g1 g3 g4; g2 g4 g5] (cyclic Jacobi,
// float64): eigenvalues ascending in eval (scaled by 1 / trace), eigenvectors in the columns of evec
// in the same order.  false if not finite.  relative: stop on |a_pq| <= 1e-16 sqrt(a_pp a_qq) instead of
// an absolute threshold -- Jacobi then resolves the small eigenpairs of a GRADED matrix to high relative
// accuracy (Demmel & Veselic), which the refinement of ill-conditioned fits below relies on.
// Replaces SVD(diag(w) l) of calc_new_vanishing_point (vp_localisation.py:453-479).
// ---------------------------------------------------------------------------
VPK_DEVFN bool jacobi_eig3(const double g[6], bool relative, double evec[3][3], double eval[3]) {
    double tr = g[0] + g[3] + g[5];
    if (!(tr > 0.0) || isinf(tr)) return false;
    double sc = 1.0 / tr;
    double a[3][3] = {{g[0] * sc, g[1] * sc, g[2] * sc}, {g[1] * sc, g[3] * sc, g[4] * sc}, {g[2] * sc, g[4] * sc, g[5] * sc}};
    double v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            if (isnan(a[i][j])) return false;
    for (int sweep = 0; sweep < (relative ? 40 : 24); ++sweep) {
        if (relative) {
            const double tol = 1e-32;
            if (a[0][1] * a[0][1] <= tol * fabs(a[0][0] * a[1][1]) && a[0][2] * a[0][2] <= tol * fabs(a[0][0] * a[2][2]) &&
                a[1][2] * a[1][2] <= tol * fabs(a[1][1] * a[2][2])) break;
        } else {
            double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2];
            if (off < 1e-36) break;             // off-diagonal below 1e-18 of the trace: converged in float64
        }
#pragma unroll
        for (int pq = 0; pq < 3; ++pq) {
            const int p = pq == 2 ? 1 : 0, q = pq == 0 ? 1 : 2;
            double apq = a[p][q];
            if (apq == 0.0) continue;
            // tan of the rotation angle, t = sgn(theta) / (|theta| + sqrt(theta^2 + 1)) with
            // theta = (aqq - app) / (2 apq), written with one square root and one division
            const double d = a[q][q] - a[p][p], b2 = 2.0 * apq;
            const double den = fabs(d) + sqrt(d * d + b2 * b2);
            const double t = den > 0.0 ? (d >= 0 ? b2 : -b2) / den : 1.0;      // den == 0: underflow, theta = 0
            const double c = rsqrt(t * t + 1.0), sn = t * c;
            double app = a[p][p], aqq = a[q][q];
            a[p][p] = app - t * apq;
            a[q][q] = aqq + t * apq;
            a[p][q] = a[q][p] = 0.0;
            const int r = 3 - p - q;
            double arp = a[r][p], arq = a[r][q];
            a[r][p] = a[p][r] = c * arp - sn * arq;
            a[r][q] = a[q][r] = sn * arp + c * arq;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                double vkp = v[k][p], vkq = v[k][q];
                v[k][p] = c * vkp - sn * vkq;
                v[k][q] = sn * vkp + c * vkq;
            }
        }
    }
    // ascending order of the diagonal (first one on ties); selects instead of dynamic indexing
    const double d0 = a[0][0], d1 = a[1][1], d2 = a[2][2];
    int lo = 0;
    if (d1 < d0) lo = 1;
    if (d2 < (lo == 0 ? d0 : d1)) lo = 2;
    int hi = lo == 0 ? 1 : 0;                                   // largest of the other two (first on ties)
    {
        const int o1 = lo == 0 ? 1 : 0, o2 = lo == 2 ? 1 : 2;
        const double e1 = o1 == 0 ? d0 : d1, e2 = o2 == 1 ? d1 : d2;
        hi = e2 > e1 ? o2 : o1;
    }
    const int mid = 3 - lo - hi;
    const int order[3] = {lo, mid, hi};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int m = order[c];
        eval[c] = m == 0 ? d0 : (m == 1 ? d1 : d2);
#pragma unroll
        for (int k = 0; k < 3; ++k) evec[k][c] = m == 0 ? v[k][0] : (m == 1 ? v[k][1] : v[k][2]);
    }
    return true;
}
VPK_DEVFN bool smallest_eigvec3(const double g[6], double out[3]) {
    double evec[3][3], eval[3];
    if (!jacobi_eig3(g, false, evec, eval)) return false;
    const double x = evec[0][0], y = evec[1][0], z = evec[2][0];
    double n = sqrt(x * x + y * y + z * z);
    if (!(n > 0.0)) return false;
    out[0] = x / n; out[1] = y / n; out[2] = z / n;
    return true;
}

// ---------------------------------------------------------------------------
// scratch of the per-slot kernels (shared memory on the device)
// ---------------------------------------------------------------------------
constexpr int kLinkMax = 512;              // clusterings up to this size keep their bookkeeping in shared memory
struct PostScratch {
    double redv[kPostThreads];
    int redi[kPostThreads], redj[kPostThreads];
    // average-linkage bookkeeping (split_best_vp)
    double l_nnd[kLinkMax], l_csize[kLinkMax], l_height[kLinkMax];
    int l_nn[kLinkMax], l_mate[kLinkMax], l_rep[kLinkMax], l_act[kLinkMax], l_keep[kLinkMax / 2];
    int l_nflag;
    double ang[kMaxM], err[kMaxM], nv[kMaxM][3];
    int ok[kMaxM], rem[kMaxM];
    int ia, ib, flag, flag2;
    double da;
#if defined(VPK_EM_MARKS)
    long long mark[16], mark_t;        // cycles of thread 0 between the markers of post_slot (diagnostic builds)
#endif
};
#if defined(__CUDACC__) && defined(VPK_EM_MARKS)
#define VPK_MARK(sc, T, k) do { if ((T).tid == 0) { long long c_ = clock64(); (sc).mark[k] += c_ - (sc).mark_t; (sc).mark_t = c_; } } while (0)
#else
#define VPK_MARK(sc, T, k) do {} while (0)
#endif

// Block-wide arg-min of (v, i) pairs: smallest v, ties -> smallest i; i < 0 = no candidate.
// Result in sc.da / sc.ia (ia < 0: no candidate at all).  Deterministic.
#if defined(__CUDACC__)
VPK_DEVFN void team_min_pair(double v, int i, PostScratch& sc, const Team& T) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ov = __shfl_xor_sync(0xffffffffu, v, o);
        int oi = __shfl_xor_sync(0xffffffffu, i, o);
        if (oi >= 0 && (i < 0 || ov < v || (ov == v && oi < i))) { v = ov; i = oi; }
    }
    if (T.lane == 0) { sc.redv[T.warp] = v; sc.redi[T.warp] = i; }
    __syncthreads();
    if (T.warp == 0) {
        v = T.lane < T.nwarps ? sc.redv[T.lane] : 0.0;
        i = T.lane < T.nwarps ? sc.redi[T.lane] : -1;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double ov = __shfl_xor_sync(0xffffffffu, v, o);
            int oi = __shfl_xor_sync(0xffffffffu, i, o);
            if (oi >= 0 && (i < 0 || ov < v || (ov == v && oi < i))) { v = ov; i = oi; }
        }
        if (T.lane == 0) { sc.da = v; sc.ia = i; }
    }
    __syncthreads();
}
// warp-wide version, result in every lane
VPK_DEV void warp_min_pair(double& v, int& i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ov = __shfl_xor_sync(0xffffffffu, v, o);
        int oi = __shfl_xor_sync(0xffffffffu, i, o);
        if (oi >= 0 && (i < 0 || ov < v || (ov == v && oi < i))) { v = ov; i = oi; }
    }
}
#else
inline void team_min_pair(double v, int i, PostScratch& sc, const Team&) { sc.da = v; sc.ia = i; }
inline void warp_min_pair(double&, int&) {}
#endif

struct InitScratch {
    double resp[kCells];
    double cand[kCells][3];
    int keep[kCells], ismax[kCells], has[kCells];
};

// ---------------------------------------------------------------------------
// per-line constants: unit lines (:186/:226), segment angles (:765-776)
// ---------------------------------------------------------------------------
VPK_DEVFN void line_constants(const Img& im, const double* lines, const Team& T) {
    const int N = im.N;
    for (int n = T.tid; n < N; n += T.nthreads) {
        const double* l = lines + 3 * (size_t)n;
        double a = l[0], bb = l[1], c = l[2];
        double nr = sqrt(a * a + bb * bb + c * c);
        a /= nr; bb /= nr; c /= nr;
        nr = sqrt(a * a + bb * bb + c * c);               // the reference normalises twice
        im.ln[3 * (size_t)n] = a / nr; im.ln[3 * (size_t)n + 1] = bb / nr; im.ln[3 * (size_t)n + 2] = c / nr;
        Seg sg = load_seg(im.lp, n);
        double vx = sg.x1 - sg.x2, vy = sg.y1 - sg.y2;
        vx = vx / sqrt(vx * vx + vy * vy);
        double phi = fabs(acos(fmin(fmax(vx, -1.0), 1.0)));
        im.langle[n] = phi > 0.5 * kPi ? kPi - phi : phi;
    }
}

// ---------------------------------------------------------------------------
// E0/E1/E2: prior mixture and initial VPs.  resp: this image's (20,20) response
// already staged in sc.resp.  Sets st.npdf/pdf_*/sigma_prior and, unless
// have_init, st.cur / st.M.
// ---------------------------------------------------------------------------
VPK_DEVFN void init_prior_and_vps(EmSlot& st, InitScratch& sc, const uint8_t* img, int S, int num_init_vp,
                                  bool have_init, const Team& T) {
    const int G = VPK_GRID;
    // --- E2 pdf_params (probability_functions.py:62-96): top-100 cells
    for (int c = T.tid; c < kCells; c += T.nthreads) {
        double v = sc.resp[c];
        int rank = 0;
        for (int o = 0; o < kCells; ++o) {
            double u = sc.resp[o];
            rank += (u > v) || (u == v && o > c);
        }
        sc.keep[c] = rank < kMaxComp;
    }
    team_sync();
    if (T.tid == 0) {
        double sum = 0.0;
        for (int c = 0; c < kCells; ++c) if (sc.keep[c]) sum += sc.resp[c];
        double sigma = kPi / (1.282 * G);
        st.sigma_prior = sigma;
        int n = 0;
        for (int c = 0; c < kCells; ++c) {
            if (!sc.keep[c]) continue;
            double w = sc.resp[c] / sum / (2 * kPi * sigma * sigma);
            if (!(w > 0)) continue;                    // calc_pdf skips weights <= 0 (:21)
            int a = c % G, bb = c / G;
            // numpy.linspace(-(G-1)/G*pi/2, (G-1)/G*pi/2, G)
            double lo = -(G - 1.0) / G * kPi / 2, hi = (G - 1.0) / G * kPi / 2, stp = (hi - lo) / (G - 1);
            st.pdf_a[n] = a == G - 1 ? hi : a * stp + lo;
            st.pdf_b[n] = bb == G - 1 ? hi : bb * stp + lo;
            st.pdf_w[n] = w;
            ++n;
        }
        st.npdf = n;
    }
    team_sync();
    if (have_init) return;
    // --- E0 find_maxima (vp_localisation.py:13-31, border quirk included)
    for (int c = T.tid; c < kCells; c += T.nthreads) {
        int a = c % G, bb = c / G;
        double vm = sc.resp[c];
        double vu = a + 1 < G ? sc.resp[bb * G + a + 1] : 0.0;
        double vd = a - 1 > 0 ? sc.resp[bb * G + a - 1] : 0.0;
        double vl = bb - 1 > 0 ? sc.resp[(bb - 1) * G + a] : 0.0;
        double vr = bb + 1 < G ? sc.resp[(bb + 1) * G + a] : 0.0;
        sc.ismax[c] = (vm > vu && vm > vd && vm > vl && vm > vr) ? 1 : 0;
    }
    team_sync();
    // keep the num_init_vp strongest maxima (:121-126)
    for (int c = T.tid; c < kCells; c += T.nthreads) {
        if (!sc.ismax[c]) { sc.keep[c] = 0; continue; }
        double v = sc.resp[c];
        int rank = 0;
        for (int o = 0; o < kCells; ++o)
            if (sc.ismax[o]) { double u = sc.resp[o]; rank += (u > v) || (u == v && o > c); }
        sc.keep[c] = rank < num_init_vp;
    }
    team_sync();
    // --- E1: per kept cell, mean index of the brightest pixels of the flipped sphere slice
    for (int c = T.warp; c < kCells; c += T.nwarps) {
        if (!sc.keep[c]) { if (T.lane == 0) sc.has[c] = 0; continue; }
        int ra = c / G, rb = c % G;      // ra: row of the response (beta), rb: column (alpha)
        int r0 = ra * S / G, r1 = (ra + 1) * S / G, c0 = rb * S / G, c1 = (rb + 1) * S / G;
        int w = c1 - c0, npx = (r1 - r0) * w;
        int mx = 0;
        for (int e = T.lane; e < npx; e += T.lanes) {
            int r = r0 + e / w, cc = c0 + e % w;
            int px = (int)img[(size_t)(S - 1 - r) * S + cc];      // flipped vertically (:114)
            mx = px > mx ? px : mx;
        }
        mx = warp_max_i(mx);
        long long sr = 0, scol = 0;
        int cnt = 0;
        if (mx > 0)
            for (int e = T.lane; e < npx; e += T.lanes) {
                int r = e / w, cc = e % w;
                if ((int)img[(size_t)(S - 1 - (r0 + r)) * S + c0 + cc] == mx) { sr += r; scol += cc; ++cnt; }
            }
        sr = warp_sum_ll(sr); scol = warp_sum_ll(scol); cnt = warp_sum_i(cnt);
        if (T.lane == 0) {
            sc.has[c] = cnt > 0;
            if (cnt > 0) {
                double idx0 = (double)scol / (double)cnt + c0;   // :158
                double idx1 = (double)sr / (double)cnt + r0;     // :157
                double alpha = (idx0 - 0.5 * S + 0.5) * kPi / S; // index_to_angle
                double beta = (idx1 - 0.5 * S + 0.5) * kPi / S;
                double x = sin(alpha) * cos(beta), y = sin(beta), z = cos(alpha) * cos(beta);
                double sg = sign_np(z);                          // angle_to_point :48
                sc.cand[c][0] = x * sg; sc.cand[c][1] = y * sg; sc.cand[c][2] = z * sg;
            }
        }
    }
    team_sync();
    if (T.tid == 0) {
        int M = 0;
        for (int c = 0; c < kCells; ++c)
            if (sc.keep[c] && sc.has[c]) {
                if (M >= kMaxM) { st.cap_hit = 1; break; }       // num_init_vp > 64 maxima: reported as VPK_EM_CAPACITY
                st.cur[M][0] = sc.cand[c][0]; st.cur[M][1] = sc.cand[c][1]; st.cur[M][2] = sc.cand[c][2];
                ++M;
            }
        st.M = M;
#if defined(VPK_HOST_TRACE)
        printf("[trace] initial VPs M=%d\n", M);
        for (int m = 0; m < M; ++m) printf("[trace]   %d: %.9f %.9f %.9f\n", m, st.cur[m][0], st.cur[m][1], st.cur[m][2]);
#endif
    }
    team_sync();
}

// ---------------------------------------------------------------------------
// E5 part 1: constants of the E-step for the VP set `v` (prior at the VP angles:
// calc_angles probability_functions.py:252-259 + calc_pdf :8-40; the in-place
// clamp of s in calc_plv :139).
// ---------------------------------------------------------------------------
VPK_DEVFN void prepare_estep(EmSlot& st, const double (*v)[3], const Team& T) {
    const int M = st.M;
    for (int m = T.warp; m < M; m += T.nwarps) {
        double beta = asin(v[m][1]);
        double inner = v[m][0] / cos(beta);
        inner = fmax(fmin(inner, 1.0), -1.0);
        if (isnan(v[m][0] / cos(beta))) inner = nan("");
        double x = asin(inner), y = beta;
        const double k = -0.5 / (st.sigma_prior * st.sigma_prior);
        double acc = 0.0;
        for (int n = T.lane; n < st.npdf; n += T.lanes) {
            double mx = st.pdf_a[n], my = st.pdf_b[n];
            double d1 = (x - mx) * (x - mx) + (y - my) * (y - my);
            double d2 = (x - mx + kPi) * (x - mx + kPi) + (y + my) * (y + my);
            double d3 = (x - mx - kPi) * (x - mx - kPi) + (y + my) * (y + my);
            double d4 = (x + mx) * (x + mx) + (y - my - kPi) * (y - my - kPi);
            double p = exp(d1 * k) + exp(d2 * k) + exp(d3 * k) + exp(d4 * k) + exp(d4 * k);   // 4th == 5th (:25-26)
            acc += p * st.pdf_w[n];
        }
        acc = warp_sum(acc);
        if (T.lane == 0) {
            st.pv[m] = acc;
            st.vx[m] = v[m][0] / v[m][2];
            st.vy[m] = v[m][1] / v[m][2];
            double sm = st.s[m] > 1e-200 ? st.s[m] : 1e-200;    // calc_plv mutates s (:139)
            if (isnan(st.s[m])) sm = 1e-200;
            st.s[m] = sm;
            st.inv2s[m] = 1.0 / (2.0 * sm);
            st.coef[m] = 1.0 / sqrt(2.0 * kPi * sm);
        }
    }
    team_sync();
}

// E5 part 2 (probability_functions.py:99-147).  Per-line constants of calc_lvsq_angle (:157-176):
struct LineGeom { double mx, my, bx, by, inv_nb; };
VPK_DEV LineGeom line_geom(const double* lp, int n) {
    Seg sg = load_seg(lp, n);
    LineGeom g;
    g.mx = 0.5 * (sg.x1 + sg.x2); g.my = 0.5 * (sg.y1 + sg.y2);
    g.bx = sg.x1 - sg.x2; g.by = sg.y1 - sg.y2;
    g.inv_nb = 1.0 / sqrt(g.bx * g.bx + g.by * g.by);
    return g;
}
// one (line, VP) pair: lvsq (:174) and p(l|v) (calc_plv :140-145).  The divisions of the reference
// are multiplications by reciprocals taken once per line / per VP (rounding-level difference).
VPK_DEV void estep_nm(const LineGeom& g, double vx, double vy, double inv2s, double coef, double& lvsq, double& plv) {
    double ax = g.mx - vx, ay = g.my - vy;
    double c = (ax * g.bx + ay * g.by) * (rsqrt(ax * ax + ay * ay) * g.inv_nb);
    double q = 1.0 - fabs(c);
    lvsq = q * q;
    plv = exp(-(lvsq * inv2s)) * coef;
}
// whole line (host build): lvsq, p(v|l), and the W-kernel operand wt = p(v|l) * lweight
VPK_DEV void estep_line(const Img& im, int M, const double* pv, const double* vx, const double* vy, const double* inv2s,
                        const double* coef, int n) {
    const int N = im.N;
    const LineGeom g = line_geom(im.lp, n);
    double pl = 0.0;
    for (int m = 0; m < M; ++m) {
        double lvsq, plv;
        estep_nm(g, vx[m], vy[m], inv2s[m], coef[m], lvsq, plv);
        im.lvsq[(size_t)m * N + n] = lvsq;
        im.pvl[(size_t)m * N + n] = plv;
        pl += plv * pv[m];
    }
    if (pl < 1e-12) pl = 1e-12;                                         // :117 (NaN stays NaN)
    const double inv_pl = 1.0 / pl;
    const double lw = im.lweight[n];
    const int passes = (M + kMP - 1) / kMP;
    for (int p = 0; p < passes; ++p) {
        const int rows = 8 * wpass_tiles(M, p);
        for (int mm = 0; mm < rows; ++mm) {
            const int m = p * kMP + mm;
            double x = 0.0;
            if (m < M) {
                x = im.pvl[(size_t)m * N + n] * pv[m] * inv_pl;         // calc_pvl (:128)
                im.pvl[(size_t)m * N + n] = x;
                x *= lw;                                                // weight_matrix :517
            }
            im.wt[wt_index(N, n, m, M)] = x;
        }
    }
}

// E6 epilogue (vp_localisation.py:519-523): acc = sum_j wt[j,m] * lsim[j,k]
VPK_DEV double wmat_finish(double wt_mk, double lw_k, double colsum_k, double acc, double bias) {
    return (wt_mk + bias * lw_k * acc) / (1 + bias * lw_k * colsum_k);
}

// ---------------------------------------------------------------------------
// reductions over the lines used by POST
// ---------------------------------------------------------------------------
// assoc[n] = argmax_m w[m,n] (first maximum, numpy.argmax; NaN counts as max)
VPK_DEVFN void argmax_assoc(const Img& im, int M, const Team& T) {
    const int N = im.N;
    for (int n = T.tid; n < N; n += T.nthreads) {
        int best = 0;
        double bv = M > 0 ? im.w[n] : 0.0;
        for (int m = 1; m < M; ++m) {
            double x = im.w[(size_t)m * N + n];
            if (isnan(bv)) break;
            if (x > bv || isnan(x)) { bv = x; best = m; }
        }
        im.assoc[n] = best;
    }
    team_sync();
}

// E9: calc_vp_line_counts (vp_localisation.py:482-512).  lvsq must have been
// computed (E-step) for the same VP set that is being counted.
VPK_DEVFN void line_counts(const Img& im, EmSlot& st, double thresh, const Team& T) {
    const int M = st.M, N = im.N;
    argmax_assoc(im, M, T);
    for (int n = T.tid; n < N; n += T.nthreads) {
        int m = im.assoc[n];
        double dist = im.lvsq[(size_t)m * N + n];
        if (dist > thresh * sqrt(st.s[m]) || im.lweight[n] == 0.0) im.assoc[n] = -1;
    }
    team_sync();
    for (int m = T.warp; m < M; m += T.nwarps) {
        int c = 0;
        double cw = 0.0;
        for (int n = T.lane; n < N; n += T.lanes)
            if (im.assoc[n] == m) { ++c; cw += im.lweight[n]; }
        c = warp_sum_i(c);
        cw = warp_sum(cw);
        if (T.lane == 0) { st.cnt[m] = c; st.cw[m] = cw; }
    }
    team_sync();
}

// E7 + E8 in two parts, so that the dependent scalar chains of all VPs (3x3 eigen-solve, log/exp)
// run side by side instead of once per warp round:
//   refit_sums  : one warp sweeps the lines twice (row maximum, then every sum at once) -> RefitAcc
//   refit_finish: one thread per VP solves, another one evaluates sigma
// E7: smallest eigenvector of sum (w/max w)^2 l l^T over the selected lines (sel < 0: all lines;
// sel >= 0: only lines with assoc == sel, the final refit).  wrow2: optional second weight row
// added to the first (merge).  ok = 0 where calc_new_vanishing_point returns None.
// E8: sv = exp(log(sum lvsq*pvl) - log(sum pvl)) over ALL lines for VP row vm
// (vp_localisation.py:301-304), or the pooled form of merge_vps (:663-664) if vm2 >= 0.
struct RefitAcc {
    double g[6], num, den, a1[3];      // a1: the only selected row, scaled (rows == 1)
    double nv[3], sv;                  // results
    double q[6];                       // refinement: the other two eigenvectors of the first solve
    int rows, fit, any, ok, refine;
};
VPK_DEVFN void refit_sums(const Img& im, const double* wrow, const double* wrow2, int sel, int vm, int vm2, RefitAcc& acc,
                          const Team& T) {
    const int N = im.N;
    // One sweep: the row maximum and the unscaled sums side by side; the scatter matrix of the rows
    // (w / max w) l is the unscaled one times 1 / (max w)^2 (rounding-level difference, same eigenvectors).
    double mx = -INFINITY;
    bool any = false;
    const double* p1 = im.pvl + (size_t)vm * N;
    const double* q1 = im.lvsq + (size_t)vm * N;
    const double* p2 = vm2 >= 0 ? im.pvl + (size_t)vm2 * N : nullptr;
    const double* q2 = vm2 >= 0 ? im.lvsq + (size_t)vm2 * N : nullptr;
    double g[6] = {0, 0, 0, 0, 0, 0};
    double num = 0.0, den = 0.0;
    int rows = 0, only = -1;
#pragma unroll 4
    for (int n = T.lane; n < N; n += T.lanes) {
        double p = p1[n], q = q1[n];
        if (p2) { p += p2[n]; q = 0.5 * (q2[n] + q); }
        num += q * p;
        den += p;
        const double x = wrow[n] + (wrow2 ? wrow2[n] : 0.0);
        const double l0 = im.ln[3 * (size_t)n], l1 = im.ln[3 * (size_t)n + 1], l2 = im.ln[3 * (size_t)n + 2];
        const bool use = sel < 0 || im.assoc[n] == sel;
        if (use) {
            any = true;
            mx = nanmax(mx, x);
            const double a = x * l0, b = x * l1, c = x * l2;
            g[0] += a * a; g[1] += a * b; g[2] += a * c; g[3] += b * b; g[4] += b * c; g[5] += c * c;
            ++rows; only = n;
        }
    }
    mx = warp_max_nanprop(mx);
    any = warp_any(any);
    const bool fit = !(!any || mx == 0.0 || isnan(mx) || isinf(mx));     // :456-460 / LinAlgError
#if defined(VPK_FORCE_SCALED)
    if (fit) {
#else
    if (fit && (mx < 1e-140 || mx > 1e140)) {
#endif
        // the squares would leave the float64 range: scale the rows first (second sweep, rare)
#pragma unroll
        for (int k = 0; k < 6; ++k) g[k] = 0.0;
        for (int n = T.lane; n < N; n += T.lanes) {
            if (!(sel < 0 || im.assoc[n] == sel)) continue;
            const double x = (wrow[n] + (wrow2 ? wrow2[n] : 0.0)) / mx;
            const double a = x * im.ln[3 * (size_t)n], b = x * im.ln[3 * (size_t)n + 1], c = x * im.ln[3 * (size_t)n + 2];
            g[0] += a * a; g[1] += a * b; g[2] += a * c; g[3] += b * b; g[4] += b * c; g[5] += c * c;
        }
    } else {
        const double inv = fit ? 1.0 / mx : 0.0, inv2 = inv * inv;
#pragma unroll
        for (int k = 0; k < 6; ++k) g[k] *= inv2;
    }
    if (!fit) rows = 0;
    num = warp_sum(num);
    den = warp_sum(den);
#pragma unroll
    for (int k = 0; k < 6; ++k) g[k] = warp_sum(g[k]);
    rows = warp_sum_i(rows);
    only = warp_max_i(only);
    if (T.lane == 0) {
#pragma unroll
        for (int k = 0; k < 6; ++k) acc.g[k] = g[k];
        acc.num = num; acc.den = den; acc.rows = rows; acc.fit = fit ? 1 : 0; acc.any = any ? 1 : 0;
        if (fit && rows == 1) {
            const double x = (wrow[only] + (wrow2 ? wrow2[only] : 0.0)) / mx;
            acc.a1[0] = x * im.ln[3 * (size_t)only]; acc.a1[1] = x * im.ln[3 * (size_t)only + 1]; acc.a1[2] = x * im.ln[3 * (size_t)only + 2];
        }
    }
}
// The 3x3 scatter matrix squares the singular values of diag(w / max w) l.  When one line dominates the
// fit (sigma_2 / sigma_1 tiny: a hypothesis supported by very few lines) the smallest eigenvector of the
// matrix formed in the ORIGINAL basis is only good to eps * lambda_1 / (lambda_2 - lambda_3), far worse than
// the reference's SVD.  Such fits are refined: a second sweep forms the scatter matrix in the eigenbasis
// of the first solve -- there it is graded, its small entries are sums of small numbers instead of
// differences of large ones -- and a Jacobi solve with a relative stopping rule resolves the small
// eigenpair to high relative accuracy.
constexpr double kRefineGap = 1e-9;    // refine if (lambda_2 - lambda_3) < kRefineGap * lambda_1 (first solve worse than ~1e-7 rad)

VPK_DEVFN void refit_solve(RefitAcc& acc) {
    acc.ok = 0;
    acc.refine = 0;
    if (!acc.fit) return;
    double e[3];
    bool okv;
    if (acc.rows == 1) {
        // A single 1x3 row has a 2-D null space; LAPACK's full SVD (what numpy.linalg.svd runs,
        // vp_localisation.py:466) completes V with the Householder reflector of dgelqf/dlarfg:
        // V[:,2] = row 3 of H = I - tau v v^T, v = (1, a2/(a1-beta), a3/(a1-beta)).
        const double a1 = acc.a1[0], a2 = acc.a1[1], a3 = acc.a1[2];
        double nrm = sqrt(a1 * a1 + a2 * a2 + a3 * a3);
        double beta = -copysign(nrm, a1);
        double tau = (beta - a1) / beta;
        double v2 = a2 / (a1 - beta), v3 = a3 / (a1 - beta);
        e[0] = -tau * v3; e[1] = -tau * v3 * v2; e[2] = 1.0 - tau * v3 * v3;
        double n2 = sqrt(e[0] * e[0] + e[1] * e[1] + e[2] * e[2]);
        okv = n2 > 0.0 && !isnan(n2);
        if (okv) { e[0] /= n2; e[1] /= n2; e[2] /= n2; }
    } else {
        double evec[3][3], eval[3];
        okv = jacobi_eig3(acc.g, false, evec, eval);
        if (okv) {
            const double n = sqrt(evec[0][0] * evec[0][0] + evec[1][0] * evec[1][0] + evec[2][0] * evec[2][0]);
            okv = n > 0.0;
            if (okv) {
                e[0] = evec[0][0] / n; e[1] = evec[1][0] / n; e[2] = evec[2][0] / n;
                if (eval[1] - eval[0] < kRefineGap * eval[2]) {
                    acc.refine = 1;
                    for (int k = 0; k < 3; ++k) { acc.q[k] = evec[k][2]; acc.q[3 + k] = evec[k][1]; }
                }
            }
        }
    }
    if (!okv) return;
    if (acc.refine) { acc.nv[0] = e[0]; acc.nv[1] = e[1]; acc.nv[2] = e[2]; acc.ok = 1; return; }   // sign after the refinement
    double sg = sign_np(e[2]);                                           // :474
    acc.nv[0] = e[0] * sg; acc.nv[1] = e[1] * sg; acc.nv[2] = e[2] * sg;
    acc.ok = 1;
}
// second sweep of a refined fit (one warp): scatter matrix of the selected rows in the basis (q1, q2, nv)
VPK_DEVFN void refit_sums_rotated(const Img& im, const double* wrow, const double* wrow2, int sel, RefitAcc& acc, const Team& T) {
    const int N = im.N;
    const double q1[3] = {acc.q[0], acc.q[1], acc.q[2]}, q2[3] = {acc.q[3], acc.q[4], acc.q[5]},
                 q3[3] = {acc.nv[0], acc.nv[1], acc.nv[2]};
    double g[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll 4
    for (int n = T.lane; n < N; n += T.lanes) {
        if (!(sel < 0 || im.assoc[n] == sel)) continue;
        const double x = wrow[n] + (wrow2 ? wrow2[n] : 0.0);
        const double l0 = im.ln[3 * (size_t)n], l1 = im.ln[3 * (size_t)n + 1], l2 = im.ln[3 * (size_t)n + 2];
        const double a = x * (l0 * q1[0] + l1 * q1[1] + l2 * q1[2]), b = x * (l0 * q2[0] + l1 * q2[1] + l2 * q2[2]),
                     c = x * (l0 * q3[0] + l1 * q3[1] + l2 * q3[2]);
        g[0] += a * a; g[1] += a * b; g[2] += a * c; g[3] += b * b; g[4] += b * c; g[5] += c * c;
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) g[k] = warp_sum(g[k]);
    if (T.lane == 0) {
#pragma unroll
        for (int k = 0; k < 6; ++k) acc.g[k] = g[k];
    }
}
VPK_DEVFN void refit_refine(RefitAcc& acc) {
    double evec[3][3], eval[3];
    double e[3] = {acc.nv[0], acc.nv[1], acc.nv[2]};
    if (jacobi_eig3(acc.g, true, evec, eval)) {
        // smallest eigenvector in the rotated basis -> original coordinates
        const double c1 = evec[0][0], c2 = evec[1][0], c3 = evec[2][0];
        double r[3];
        for (int k = 0; k < 3; ++k) r[k] = c1 * acc.q[k] + c2 * acc.q[3 + k] + c3 * acc.nv[k];
        const double n = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
        if (n > 0.0 && !isnan(n)) { e[0] = r[0] / n; e[1] = r[1] / n; e[2] = r[2] / n; }
    }
    double sg = sign_np(e[2]);                                           // :474
    acc.nv[0] = e[0] * sg; acc.nv[1] = e[1] * sg; acc.nv[2] = e[2] * sg;
}
// the scalar tails of `count` refits: thread q < kMaxM solves VP q, thread kMaxM + q evaluates its sigma;
// then the refinement of the ill-conditioned ones.  Fit m uses the weight row w0 + m * stride (+ w1, merge)
// and, hard = true, only the lines assigned to VP m.
VPK_DEVFN void refit_finish(RefitAcc* acc, int count, const Img& im, const double* w0, size_t stride, const double* w1, bool hard,
                            int& any_refine, const Team& T) {
    if (T.tid == 0) any_refine = 0;
    team_sync();
    for (int q = T.tid; q < 2 * kMaxM; q += T.nthreads) {
        const int m = q % kMaxM;
        if (m >= count) continue;
        if (q < kMaxM) {
            refit_solve(acc[m]);
            if (acc[m].refine) any_refine = 1;
        } else acc[m].sv = exp(log(acc[m].num) - log(acc[m].den));
    }
    team_sync();
    if (!any_refine) return;
    for (int m = T.warp; m < count; m += T.nwarps)
        if (acc[m].refine) refit_sums_rotated(im, w0 + (size_t)m * stride, w1, hard ? m : -1, acc[m], T);
    team_sync();
    for (int m = T.tid; m < count; m += T.nthreads)
        if (acc[m].refine) refit_refine(acc[m]);
    team_sync();
}

// the accumulators live on the (idle) average-linkage bookkeeping of the POST scratch
static_assert(sizeof(RefitAcc) * kMaxM <= 3 * kLinkMax * sizeof(double), "RefitAcc overlay");
VPK_DEV RefitAcc* refit_acc(PostScratch& sc) { return reinterpret_cast<RefitAcc*>(sc.l_nnd); }

// remove the VPs flagged in rem[] from cur / nxt / s (numpy.delete along the VP axis)
VPK_DEVFN void compact_vps(EmSlot& st, const int* rem, const Team& T) {
    team_sync();
    if (T.tid == 0) {
        int k = 0;
        for (int m = 0; m < st.M; ++m) {
            if (rem[m]) continue;
            if (k != m) {
                for (int c = 0; c < 3; ++c) { st.cur[k][c] = st.cur[m][c]; st.nxt[k][c] = st.nxt[m][c]; }
                st.s[k] = st.s[m];
            }
            ++k;
        }
        st.M = k;
    }
    team_sync();
}

// ---------------------------------------------------------------------------
// E11: split_best_vp (vp_localisation.py:527-630)
// ---------------------------------------------------------------------------
// UPGMA (average linkage) down to two clusters on the n x n matrix D -- what
// scikit-learn's AgglomerativeClustering(linkage='average', n_clusters=2)
// computes on a complete connectivity graph.  The dendrogram is built by rounds
// of *reciprocal nearest neighbour* merges instead of one merge at a time:
// average linkage is reducible, so every pair of clusters that are each other's
// nearest neighbour is a node of the UPGMA tree and all such pairs can be merged
// in the same round (Lance-Williams update in the order the sequential
// algorithm would apply it, so only rounding-level differences).  A round never
// takes the count below two, and the two survivors are the children of the
// root.  ~log(n) rounds of block-wide work replace n - 2 dependent merges.
// Ties: nearest neighbour under the total order (distance, smaller index, larger
// index), which keeps the globally closest pair reciprocal (progress).
// Labels follow _hc_cut: label 0 = the root's child with the larger node id,
// i.e. the one formed later = with the larger merge height (a leaf: its index).
// have_nn: nn / nnd of the first round are already filled in (the caller found them while writing D).
VPK_DEVFN void average_linkage_two(double* D, int n, int* rep, int* mate, double* csize, double* nnd, int* nn,
                                    int* act, double* height, int* keep, PostScratch& sc, const Team& T, bool have_nn = false) {
    const int tid = T.tid, NT = T.nthreads;
    for (int i = tid; i < n; i += NT) { rep[i] = i; csize[i] = 1.0; height[i] = -INFINITY; act[i] = i; }
    team_sync();
    int nact = n;
    while (nact > 2) {
        // 1. nearest neighbour of every active cluster, one warp per row, eight loads per lane in flight (the
        //    matrix lives in the L2).  act is ascending, so the first minimum along a row is the tie-break by index.
        for (int f = T.warp; f < nact && !have_nn; f += T.nwarps) {
            const int a = act[f];
            const double* row = D + (size_t)a * n;
            double bd = INFINITY;
            int bb = -1;
            for (int g0 = T.lane; g0 < nact; g0 += 8 * T.lanes) {
                double v[8];
                int b[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int g = g0 + u * T.lanes;
                    b[u] = g < nact ? act[g] : a;
                    v[u] = b[u] != a ? row[b[u]] : INFINITY;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    if (b[u] == a) continue;
                    const double x = isnan(v[u]) ? INFINITY : v[u];
                    if (bb < 0 || x < bd) { bd = x; bb = b[u]; }
                }
            }
            warp_min_pair(bd, bb);
            if (T.lane == 0) { nn[a] = bb; nnd[a] = bd; }
        }
        have_nn = false;
        team_sync();
        // 2. reciprocal pairs; the smaller index of a pair keeps the merged cluster (ordered list `keep`)
        if (T.warp == 0) {
            int k = 0;
            for (int f0 = 0; f0 < nact; f0 += T.lanes) {
                const int f = f0 + T.lane;
                bool kp = false;
                int a = -1;
                if (f < nact) {
                    a = act[f];
                    const int b = nn[a];
                    const bool rec = nn[b] == a;
                    mate[a] = rec ? b : -1;
                    kp = rec && a < b;
                }
                int tot;
                const int pos = warp_rank(kp, tot);
                if (kp) keep[k + pos] = a;
                k += tot;
            }
            if (T.lane == 0) sc.l_nflag = k;
        }
        team_sync();
        const int k = sc.l_nflag;
        // 3. distances of the merged clusters to every surviving cluster: one warp per merged cluster, four columns
        //    per lane in flight.  Each new entry depends on old entries that no other thread of this round writes.
        for (int q = T.warp; q < k; q += T.nwarps) {
            const int X = keep[q], b = mate[X];
            const double na = csize[X], nb = csize[b];
            double* rx = D + (size_t)X * n;
            const double* rb = D + (size_t)b * n;
            for (int f0 = T.lane; f0 < nact; f0 += 4 * T.lanes) {
                int Y[4], my[4];
                bool go[4];
                double x1[4], x2[4], y1[4], y2[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int f = f0 + u * T.lanes;
                    Y[u] = f < nact ? act[f] : X;
                    my[u] = mate[Y[u]];
                    // skipped: itself / Y is absorbed this round / pair of merged clusters, done by (Y, X)
                    go[u] = !(Y[u] == X || (my[u] >= 0 && my[u] < Y[u]) || (my[u] > Y[u] && Y[u] < X));
                    x1[u] = x2[u] = y1[u] = y2[u] = 0.0;
                    if (go[u]) {
                        x1[u] = rx[Y[u]]; x2[u] = rb[Y[u]];
                        if (my[u] > Y[u]) { y1[u] = rx[my[u]]; y2[u] = rb[my[u]]; }
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (!go[u]) continue;
                    double v = (na * x1[u] + nb * x2[u]) / (na + nb);                             // average_merge
                    if (my[u] > Y[u]) {
                        const double v2 = (na * y1[u] + nb * y2[u]) / (na + nb);
                        const double nc = csize[Y[u]], nd = csize[my[u]];
                        v = (nc * v + nd * v2) / (nc + nd);
                    }
                    rx[Y[u]] = v;
                    D[(size_t)Y[u] * n + X] = v;
                }
            }
        }
        team_sync();
        // 4. bookkeeping, then drop the absorbed clusters from the active list (order kept)
        for (int q = tid; q < k; q += NT) {
            const int a = keep[q], b = mate[a];
            height[a] = nnd[a];
            csize[a] += csize[b];
        }
        for (int i = tid; i < n; i += NT) {
            const int r = rep[i], m = mate[r];
            if (m >= 0 && m < r) rep[i] = m;
        }
        if (T.warp == 0) {
            int k2 = 0;
            for (int f0 = 0; f0 < nact; f0 += T.lanes) {
                const int f = f0 + T.lane;
                bool kp = false;
                int a = -1;
                if (f < nact) { a = act[f]; const int m = mate[a]; kp = !(m >= 0 && m < a); }
                int tot;
                const int pos = warp_rank(kp, tot);
                if (kp) act[k2 + pos] = a;                       // k2 + pos <= f: in place
                k2 += tot;
            }
            if (T.lane == 0) sc.ia = k2;
        }
        team_sync();
        nact = sc.ia;
        team_sync();
    }
    // the two survivors; label 0 = formed later
    const int a0 = act[0], a1 = nact > 1 ? act[1] : act[0];
    int c0 = a1;                                                 // equal heights (two leaves): the larger index
    if (height[a0] > height[a1]) c0 = a0;
    team_sync();
    for (int i = tid; i < n; i += NT) rep[i] = (rep[i] == c0) ? 0 : 1;
    team_sync();
}

// Returns -1 if nothing was touched (no VP qualifies), 0 if the scratch (E/W results) was
// overwritten but the hypothesis set is unchanged, 1 if it changed.  big/big_cap: scratch used when the
// clustering of the chosen VP does not fit the slot's own scratch (nullptr: skip).
VPK_DEVFN int split_best_vp(const Img& im, EmSlot& st, PostScratch& sc, double min_diff, double* big, size_t big_cap,
                            int* big_lock, const Team& T) {
    const int M = st.M, N = im.N, tid = T.tid;
    VPK_MARK(sc, T, 10);
    argmax_assoc(im, M, T);
    // global maximum of w (weightMatrix.max(), :539) only decides the sign of the greedy entries
    double lm = -INFINITY;
    for (size_t e = tid; e < (size_t)M * N; e += T.nthreads) lm = nanmax(lm, im.w[e]);
    lm = warp_max_nanprop(lm);
    if (T.lane == 0) sc.redv[T.warp] = lm;
    team_sync();
    if (tid == 0) {
        double g = sc.redv[0];
        for (int k = 1; k < T.nwarps; ++k) g = nanmax(g, sc.redv[k]);
        sc.da = g;
    }
    team_sync();
    const double wmax = sc.da;
    // std of the segment angles of the lines greedily assigned to each VP (:541-544), lines per VP
    for (int m = T.warp; m < M; m += T.nwarps) {
        double sum = 0.0;
        int c = 0, call = 0;
        for (int n = T.lane; n < N; n += T.lanes) {
            if (im.assoc[n] != m) continue;
            ++call;
            if ((im.w[(size_t)m * N + n] / wmax) > 0) { sum += im.langle[n]; ++c; }
        }
        sum = warp_sum(sum);
        c = warp_sum_i(c);
        call = warp_sum_i(call);
        double mean = sum / c, var = 0.0;
        for (int n = T.lane; n < N; n += T.lanes)
            if (im.assoc[n] == m && (im.w[(size_t)m * N + n] / wmax) > 0) { double d = im.langle[n] - mean; var += d * d; }
        var = warp_sum(var);
        if (T.lane == 0) { sc.ang[m] = c > 0 ? sqrt(var / c) : nan(""); st.cnt[m] = call; }
    }
    team_sync();
    VPK_MARK(sc, T, 11);
    if (tid == 0) {
        // argsort(std)[::-1]: ascending, NaN last, stable; then reversed (:546-547)
        int ord[kMaxM];
        for (int m = 0; m < M; ++m) ord[m] = m;
        for (int i = 1; i < M; ++i) {
            int x = ord[i];
            double kx = isnan(sc.ang[x]) ? INFINITY : sc.ang[x];
            bool nx = isnan(sc.ang[x]);
            int p = i;
            while (p > 0) {
                int y = ord[p - 1];
                double ky = isnan(sc.ang[y]) ? INFINITY : sc.ang[y];
                bool ny = isnan(sc.ang[y]);
                bool greater = (ny && !nx) || (!ny && !nx && ky > kx);
                if (!greater) break;
                ord[p] = y; --p;
            }
            ord[p] = x;
        }
        int worst = -1;
        for (int m = 0; m < M; ++m) {
            int cand = ord[M - 1 - m];
            double px = st.cur[m][0] / st.cur[m][2], py = st.cur[m][1] / st.cur[m][2];     // row m, not cand (:557)
            if (st.cnt[cand] > 8 && px > -1 && py > -1 && px < 1 && py < 1) { worst = cand; break; }
        }
        sc.ia = worst;
    }
    team_sync();
    const int worst = sc.ia;
    VPK_MARK(sc, T, 12);
    if (worst < 0) return -1;
    const int nw = st.cnt[worst];
    // scratch layout (doubles): D[nw*nw] | csize nnd height [nw each] | ints: idx rep mate nn act [nw each] keep [nw/2]
    // (the bookkeeping arrays live in shared memory when nw <= kLinkMax)
    size_t need = (size_t)nw * nw + 3 * (size_t)nw + (11 * (size_t)nw / 2 + 3) / 2 + 4;
    double* scratch = im.lvsq;
    bool locked = false;
    // the line -> VP association and the line weights live outside the scratch region; the E/W
    // results in it are dead after this point (the next superstep recomputes them)
    if (need > im.scratch_cap) {
        if (!big || need > big_cap) return -1;           // cannot split: leave the hypothesis set unchanged
        scratch = big;
        locked = true;
#if defined(__CUDACC__)
        // one clustering at a time in the shared overflow buffer
        if (tid == 0) { while (atomicCAS(big_lock, 0, 1) != 0) __nanosleep(200); __threadfence(); }
        team_sync();
#endif
    }
    double* D = scratch;
    double* csize = D + (size_t)nw * nw;
    double* nnd = csize + nw;
    double* height = nnd + nw;
    int* idx = reinterpret_cast<int*>(height + nw);
    int* rep = idx + nw;
    int* mate = rep + nw;
    int* nn = mate + nw;
    int* act = nn + nw;
    int* keep = act + nw;
    if (nw <= kLinkMax) {
        csize = sc.l_csize; nnd = sc.l_nnd; height = sc.l_height; rep = sc.l_rep; mate = sc.l_mate; nn = sc.l_nn;
        act = sc.l_act; keep = sc.l_keep;
    }
    if (T.warp == 0) {
        // lines of the worst VP in ascending order (warp-wide stream compaction)
        int k = 0;
        for (int n0 = 0; n0 < N; n0 += T.lanes) {
            const int n = n0 + T.lane;
            const bool f = n < N && im.assoc[n] == worst;
            int tot;
            const int r = warp_rank(f, tot);
            if (f) idx[k + r] = n;
            k += tot;
        }
    }
    team_sync();
    // Ldist = 1 - cosangle(f = 2) (:572), one warp per row.  Direction and length of every line are taken once (the
    // expressions of cosangle(), so every entry has the bits of the per-pair evaluation); they sit in the three
    // float64 arrays the clustering initialises later.  While a row is written its nearest neighbour is found, which
    // is the first round of the clustering (kept in redv until the rows are done: nnd holds the directions).
    static_assert(kLinkMax <= kPostThreads, "redv holds the first nearest-neighbour distances");
    double* dir_x = nnd; double* dir_y = csize; double* dir_n = height;
    for (int q = tid; q < nw; q += T.nthreads) {
        const Seg sg = load_seg(im.lp, idx[q]);
        const double vx = sg.x1 - sg.x2, vy = sg.y1 - sg.y2;
        dir_x[q] = vx; dir_y[q] = vy; dir_n[q] = sqrt(vx * vx + vy * vy);
    }
    team_sync();
    const bool fuse_nn = nw <= kLinkMax && nw > 2;
    for (int a = T.warp; a < nw; a += T.nwarps) {
        const double v1x = dir_x[a], v1y = dir_y[a], n1 = dir_n[a];
        double* row = D + (size_t)a * nw;
        double bd = INFINITY;
        int bb = -1;
        for (int b = T.lane; b < nw; b += T.lanes) {
            double d = 0.0;
            if (a != b) {
                const double v2x = dir_x[b], v2y = dir_y[b];
                const double c = fabs((v1x * v2x + v1y * v2y) / (n1 * dir_n[b]));
                d = 1.0 - cos_clipped_multiple(c, 2.0);
                const double x = isnan(d) ? INFINITY : d;
                if (bb < 0 || x < bd) { bd = x; bb = b; }
            }
            row[b] = d;
        }
        if (fuse_nn) {
            warp_min_pair(bd, bb);
            if (T.lane == 0) { nn[a] = bb; sc.redv[a] = bd; }
        }
    }
    team_sync();
    if (fuse_nn)
        for (int q = tid; q < nw; q += T.nthreads) nnd[q] = sc.redv[q];
    team_sync();
    VPK_MARK(sc, T, 13);
    average_linkage_two(D, nw, rep, mate, csize, nnd, nn, act, height, keep, sc, T, fuse_nn);
    VPK_MARK(sc, T, 14);
    // per cluster: smallest right-singular vector of the lweight-scaled lines (:580-602)
    for (int c = T.warp; c < 2; c += T.nwarps) {
        double g[6] = {0, 0, 0, 0, 0, 0};
        int cnt = 0;
        for (int q = T.lane; q < nw; q += T.lanes) {
            if (rep[q] != c) continue;
            int n = idx[q];
            double lw = im.lweight[n];
            double a = im.ln[3 * (size_t)n] * lw, b = im.ln[3 * (size_t)n + 1] * lw, cc = im.ln[3 * (size_t)n + 2] * lw;
            g[0] += a * a; g[1] += a * b; g[2] += a * cc; g[3] += b * b; g[4] += b * cc; g[5] += cc * cc;
            ++cnt;
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) g[k] = warp_sum(g[k]);
        cnt = warp_sum_i(cnt);
        double e[3] = {0, 0, 0};
        bool okv = cnt >= 3 && smallest_eigvec3(g, e);
        if (T.lane == 0) {
            sc.ok[c] = okv;
            double sg = e[2] < 0 ? -1.0 : 1.0;
            sc.nv[c][0] = e[0] * sg; sc.nv[c][1] = e[1] * sg; sc.nv[c][2] = e[2] * sg;
        }
    }
    team_sync();
#if defined(__CUDACC__)
    if (locked && tid == 0) { __threadfence(); atomicExch(big_lock, 0); }
#else
    (void)locked; (void)big_lock;
#endif
    if (tid == 0) {
        sc.flag = 0;
        if (sc.ok[0] && sc.ok[1]) {
            double c = sc.nv[0][0] * sc.nv[1][0] + sc.nv[0][1] * sc.nv[1][1] + sc.nv[0][2] * sc.nv[1][2];
            c = fmin(fmax(c, -1.0), 1.0);
            double ang = fabs(acos(fmin(fmax(fabs(c), -1.0), 1.0)));
            if (ang > min_diff && st.M >= kMaxM) st.cap_hit = 1;      // the reference would append; reported as VPK_EM_CAPACITY
            if (ang > min_diff && st.M < kMaxM) {
                double stdd = st.s[worst] / 2;
                for (int k = 0; k < 3; ++k) { st.cur[worst][k] = sc.nv[0][k]; st.cur[st.M][k] = sc.nv[1][k]; st.nxt[st.M][k] = 0.0; }
                st.s[worst] = stdd;
                st.s[st.M] = stdd;
                st.M += 1;
                sc.flag = 1;
            }
        }
    }
    team_sync();
    VPK_MARK(sc, T, 15);
    return sc.flag != 0 ? 1 : 0;
}

// ---------------------------------------------------------------------------
// result (vp_localisation.py:441-442)
// ---------------------------------------------------------------------------
VPK_DEVFN void write_result(const EmOut& out, const Img& im, EmSlot& st, int status, int iters, bool have_vps, const Team& T) {
    const int N = im.N, b = st.img, base = st.base;
    if (status == VPK_EM_OK && st.cap_hit) status = VPK_EM_CAPACITY;
    if (T.tid == 0) {
        out.status[b] = status;
        out.iterations[b] = iters;
        out.n_vp[b] = have_vps ? st.M : 0;
    }
    for (int m = T.tid; m < kMaxM; m += T.nthreads) {
        bool live = have_vps && m < st.M;
        for (int c = 0; c < 3; ++c) out.vp[((size_t)b * kMaxM + m) * 3 + c] = live ? st.nxt[m][c] : 0.0;
        out.sigma[(size_t)b * kMaxM + m] = live ? st.s[m] : 0.0;
        out.counts[(size_t)b * kMaxM + m] = live ? st.cnt[m] : 0;
        out.counts_weighted[(size_t)b * kMaxM + m] = live ? st.cw[m] : 0.0;
    }
    for (int n = T.tid; n < N; n += T.nthreads) out.vp_assoc[base + n] = have_vps ? im.assoc[n] : -1;
    if (out.decision_metric && have_vps) {
        double* dm = out.decision_metric + (size_t)kMaxM * base;
        for (size_t e = T.tid; e < (size_t)st.M * N; e += T.nthreads) dm[e] = im.w[e];
    }
    team_sync();
    if (T.tid == 0) { st.phase = PH_DONE; st.run_e = 0; st.run_w = 0; st.done = 1; st.status = status; st.iters_out = iters; }
    team_sync();
}

// ask for an E-step (and weight matrix) on cur (vsel 0) or nxt (vsel 1); POST resumes in `phase`
VPK_DEVFN void request(EmSlot& st, int vsel, int phase, const Team& T, PostScratch* msc = nullptr) {
    team_sync();
    if (T.tid == 0) { st.vsel = vsel; st.phase = phase; st.run_e = 1; st.run_w = 1; }
#if defined(VPK_EM_MARKS)
    if (msc) VPK_MARK(*msc, T, 8);
#endif
    prepare_estep(st, vsel ? st.nxt : st.cur, T);
#if defined(VPK_EM_MARKS)
    if (msc) VPK_MARK(*msc, T, 9);
#endif
    (void)msc;
}

// ---------------------------------------------------------------------------
// INIT: per-line constants are done by the caller; this sets up the hypotheses
// and asks for the first superstep.  Returns false if the slot finished.
// ---------------------------------------------------------------------------
VPK_DEVFN bool init_slot(EmSlot& st, InitScratch& isc, const Img& im, const EmOut& out, const vpk_em_config& cfg,
                         const uint8_t* sphere, int S, const double* init_vp, int n_init, const Team& T) {
    if (T.tid == 0) { st.M = 0; st.done = 0; st.iter = 0; st.vidx = 0; st.run_e = 0; st.run_w = 0; st.iters_out = 0; st.cap_hit = 0; }
    team_sync();
    if (im.N == 0) { write_result(out, im, st, VPK_EM_NO_INITIAL_VPS, 0, false, T); return false; }
    const bool have_init = init_vp != nullptr;
    // more hypotheses than the slot holds (the reference has no cap): reported, never truncated
    if (have_init && n_init > kMaxM) { write_result(out, im, st, VPK_EM_CAPACITY, 0, false, T); return false; }
    init_prior_and_vps(st, isc, sphere, S, cfg.num_init_vp, have_init, T);
    if (have_init) {
        if (T.tid == 0) {
            int M = imin(n_init, kMaxM);
            for (int m = 0; m < M; ++m) {
                const double* v = init_vp + 3 * (size_t)m;
                double nr = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
                st.cur[m][0] = v[0] / nr; st.cur[m][1] = v[1] / nr; st.cur[m][2] = v[2] / nr;
            }
            st.M = M;
        }
        team_sync();
    }
    if (st.M == 0) { write_result(out, im, st, VPK_EM_NO_INITIAL_VPS, 0, false, T); return false; }
    for (int m = T.tid; m < kMaxM; m += T.nthreads) {
        st.s[m] = st.sigma_prior * 1e-6;                  // s_init (:219)
        st.nxt[m][0] = st.nxt[m][1] = st.nxt[m][2] = 0.0;
    }
    request(st, 0, PH_INIT_COUNTS, T);
    return true;
}

// ---------------------------------------------------------------------------
// POST: consume the E/W results of the superstep according to st.phase and run
// the reference's control flow until the next E-step is needed or the image is
// finished.
// ---------------------------------------------------------------------------
// presummed: the entry phase is PH_MSTEP and the caller has already filled refit_acc(sc)[0 .. M) with the sums
// of refit_sums (the fused kernel spreads them over the warps of a whole cluster).
VPK_DEVFN void post_slot(EmSlot& st, PostScratch& sc, const Img& im, const EmOut& out, const vpk_em_config& cfg,
                         double* big, size_t big_cap, int* big_lock, const Team& T, bool presummed = false) {
    const int N = im.N;
    const double max_stdd = 1e-6;            // angle mode (:197)
    int ph = st.phase;
    VPK_MARK(sc, T, 0);
    while (true) {
        team_sync();
        switch (ph) {
        case PH_INIT_COUNTS: {
            line_counts(im, st, cfg.outlier_thresh, T);
            for (int m = T.tid; m < st.M; m += T.nthreads) sc.rem[m] = st.cnt[m] < 3;
            compact_vps(st, sc.rem, T);
            if (T.tid == 0) st.iter = 0;
            ph = CT_ITER_BEGIN;
            break;
        }
        case CT_ITER_BEGIN: {
            const int i = st.iter;
            if (i >= cfg.num_iter || st.M == 0) {             // "No VPs left!" (:258) / loop exhausted (:450)
                write_result(out, im, st, VPK_EM_NO_VPS_LEFT, 0, false, T);
                return;
            }
            if (i % cfg.split_merge_freq == 0 && i > 0 && i < 100 && cfg.do_split) {     // :262
                request(st, 0, PH_SPLIT, T, &sc);
                return;
            }
            VPK_MARK(sc, T, 5);
            request(st, 0, PH_MSTEP, T, &sc);                       // :273, :282
            return;
        }
        case PH_SPLIT: {
            int changed = split_best_vp(im, st, sc, cfg.merge_thresh, big, big_cap, big_lock, T);
            // no candidate: the E/W results of this superstep are exactly what :273/:282 recompute
            if (changed < 0) { ph = PH_MSTEP; break; }
            // otherwise the split scratch has overwritten lvsq/pvl/w
            request(st, 0, PH_MSTEP, T, &sc);
            return;
        }
        case PH_MSTEP: {
            // ---- M-step (:284-322): sums by one warp per VP, then the scalar tails side by side
            const int M = st.M;
            RefitAcc* acc = refit_acc(sc);
            if (cfg.do_iterations) {
                VPK_MARK(sc, T, 1);
                if (!presummed)
                    for (int m = T.warp; m < M; m += T.nwarps) refit_sums(im, im.w + (size_t)m * N, nullptr, -1, m, -1, acc[m], T);
                team_sync();
                VPK_MARK(sc, T, 2);
                refit_finish(acc, M, im, im.w, (size_t)N, nullptr, false, sc.flag2, T);
                VPK_MARK(sc, T, 3);
            }
            for (int m = T.tid; m < M; m += T.nthreads) {
                if (!cfg.do_iterations) {
                    sc.rem[m] = 0; sc.err[m] = 0.0;
                    for (int c = 0; c < 3; ++c) st.nxt[m][c] = st.cur[m][c];
                    continue;
                }
                int rem = 0;
                double err = 0.0;
                if (!acc[m].ok) rem = 1;
                else {
                    const double* nv = acc[m].nv;
                    double sv = acc[m].sv;
                    st.nxt[m][0] = nv[0]; st.nxt[m][1] = nv[1]; st.nxt[m][2] = nv[2];
                    sv = isnan(sv) ? sv : fmin(sv, max_stdd);                  // :306
                    sv = isnan(sv) ? sv : fmax(sv, cfg.s_thresh);              // :307
                    st.s[m] = sv;
                    if (isnan(sv)) rem = 1;
                    else {
                        double d = fabs(st.cur[m][0] * nv[0] + st.cur[m][1] * nv[1] + st.cur[m][2] * nv[2]);
                        err = acos(fmin(d, 1.0));                               // :312
                        if (isnan(d)) err = d;
                        if (err > 1.5) rem = 1;
                    }
                }
                sc.rem[m] = rem;
                sc.err[m] = err;
            }
            team_sync();
            if (T.tid == 0) {
                double mx = 0.0;
                for (int m = 0; m < M; ++m) {
                    double e = sc.err[m];
                    if (isnan(e) || isnan(mx)) mx = nan("");      // numpy.maximum propagates NaN
                    else if (e > mx) mx = e;
                }
                sc.da = mx;
            }
            team_sync();
            const double max_err = sc.da;
            compact_vps(st, sc.rem, T);
            // the E-step of :332 only clamps s in place (calc_plv :139); its probabilities are
            // recomputed before every use (:273, :344, merge_vps :650)
            for (int m = T.tid; m < st.M; m += T.nthreads) {
                double sm = st.s[m] > 1e-200 ? st.s[m] : 1e-200;
                if (isnan(st.s[m])) sm = 1e-200;
                st.s[m] = sm;
            }
            team_sync();
            VPK_MARK(sc, T, 4);
            const int i = st.iter;
            if (max_err < cfg.final_convergence || i == cfg.num_iter - 1 || !cfg.do_iterations) {   // :335
                if (cfg.do_merge) {                                                  // :339
                    if (T.tid == 0) { st.merge_thresh = cfg.merge_thresh * 10; st.after_merge = CT_FINAL_A; }
                    ph = CT_MERGE_LOOP;
                } else ph = CT_FINAL_A;
                break;
            }
            if (i % cfg.split_merge_freq == 0 && i > 0 && i <= 100 + cfg.split_merge_freq && cfg.do_merge) {   // :444
                if (T.tid == 0) { st.merge_thresh = cfg.merge_thresh; st.after_merge = CT_ADVANCE; }
                ph = CT_MERGE_LOOP;
                break;
            }
            ph = CT_ADVANCE;
            break;
        }
        case CT_MERGE_LOOP: {
            // E10: merge_vps (vp_localisation.py:633-684) on the nxt row set
            const int M = st.M;
            if (M <= 1) { ph = st.after_merge; break; }
            // closest pair: first minimum in row-major order of the (M,M) angle matrix (diag = pi);
            // numpy.argmin returns the first NaN if there is one (key -inf)
            {
                double bv = INFINITY;
                int be = -1;
                for (int e = T.tid; e < M * M; e += T.nthreads) {
                    const int j = e / M, k = e % M;
                    double a;
                    if (j == k) a = kPi;
                    else {
                        double c = st.nxt[k][0] * st.nxt[j][0] + st.nxt[k][1] * st.nxt[j][1] + st.nxt[k][2] * st.nxt[j][2];
                        c = fmin(fmax(c, -1.0), 1.0);
                        a = fabs(acos(fmin(fmax(fabs(c), -1.0), 1.0)));
                        if (isnan(c)) a = c;
                    }
                    if (isnan(a)) a = -INFINITY;
                    if (be < 0 || a < bv) { bv = a; be = e; }
                }
                team_min_pair(bv, be, sc, T);
                if (T.tid == 0) {
                    const int e = sc.ia;
                    sc.ib = e % M; sc.ia = e / M;
                    if (sc.da == -INFINITY) sc.da = nan("");
                }
                team_sync();
            }
            if (!(sc.da < st.merge_thresh)) { ph = st.after_merge; break; }
            if (T.tid == 0) { st.merge_j = sc.ia; st.merge_k = sc.ib; }
            request(st, 1, PH_MERGE_EVAL, T, &sc);
            return;
        }
        case PH_MERGE_EVAL: {
            const int j = st.merge_j, k = st.merge_k, M = st.M;
            RefitAcc* acc = refit_acc(sc);
            if (T.warp == 0) refit_sums(im, im.w + (size_t)j * N, im.w + (size_t)k * N, -1, k, j, acc[0], T);
            refit_finish(acc, 1, im, im.w + (size_t)j * N, (size_t)N, im.w + (size_t)k * N, false, sc.flag2, T);
            if (T.tid == 0) {
                const double sk = acc[0].sv;
                st.s[k] = sk;                                  // assigned before the test (:666)
                sc.flag = (acc[0].ok && !(sk > 0.01)) ? 1 : 0;       // max_stdd = 0.01 (:633, :668)
                if (sc.flag) { st.nxt[k][0] = acc[0].nv[0]; st.nxt[k][1] = acc[0].nv[1]; st.nxt[k][2] = acc[0].nv[2]; }
            }
            team_sync();
            if (!sc.flag) { ph = st.after_merge; break; }
            for (int m = T.tid; m < M; m += T.nthreads) sc.rem[m] = (m == j);
            compact_vps(st, sc.rem, T);
            ph = CT_MERGE_LOOP;
            break;
        }
        case CT_ADVANCE: {
            // v[i+1] becomes the current set
            for (int m = T.tid; m < st.M; m += T.nthreads)
                for (int c = 0; c < 3; ++c) { st.cur[m][c] = st.nxt[m][c]; st.nxt[m][c] = 0.0; }
            team_sync();
            if (T.tid == 0) st.iter += 1;
            ph = CT_ITER_BEGIN;
            break;
        }
        case CT_FINAL_A: {
            request(st, 0, PH_HARD_REFIT, T, &sc);                   // :344 (index i, sic)
            return;
        }
        case PH_HARD_REFIT: {
            argmax_assoc(im, st.M, T);
#if defined(VPK_HOST_TRACE)
            { int bc[kMaxM] = {0}; for (int n = 0; n < N; ++n) bc[im.assoc[n]]++; printf("[trace] HARD_REFIT M=%d assoc bincount:", st.M); for (int m = 0; m < st.M; ++m) printf(" %d", bc[m]); printf("\n"); }
#endif
            // hard-assignment refit (:353-392)
            const int M2 = st.M;
            RefitAcc* acc = refit_acc(sc);
            for (int m = T.warp; m < M2; m += T.nwarps) refit_sums(im, im.w + (size_t)m * N, nullptr, m, m, -1, acc[m], T);
            refit_finish(acc, M2, im, im.w, (size_t)N, nullptr, true, sc.flag2, T);
            for (int m = T.tid; m < M2; m += T.nthreads) {
                if (!acc[m].any) { sc.rem[m] = 0; continue; }              // no line assigned: left as it is (:354-356)
                int rem = 0;
                if (!acc[m].ok) rem = 1;
                else {
                    const double* nv = acc[m].nv;
                    double sv = acc[m].sv;
                    st.nxt[m][0] = nv[0]; st.nxt[m][1] = nv[1]; st.nxt[m][2] = nv[2];
                    sv = isnan(sv) ? sv : fmin(sv, max_stdd);               // :377
                    st.s[m] = sv;
                    if (isnan(sv) || sv < cfg.s_thresh) rem = 1;            // :379
                    else {
                        double d = fabs(st.cur[m][0] * nv[0] + st.cur[m][1] * nv[1] + st.cur[m][2] * nv[2]);
                        double err = acos(fmin(d, 1.0));
                        if (err > 1.5) rem = 1;
                    }
                }
                sc.rem[m] = rem;
            }
#if defined(VPK_HOST_TRACE)
            printf("[trace] HARD_REFIT removed:"); for (int m = 0; m < M2; ++m) if (sc.rem[m]) printf(" %d", m); printf("  s:"); for (int m = 0; m < M2; ++m) printf(" %.6e", st.s[m]); printf("\n");
#endif
            compact_vps(st, sc.rem, T);
            if (st.M == 0) {                                    // "decision metric is empty" (:400-404)
                write_result(out, im, st, VPK_EM_NO_VPS_LEFT, 0, false, T);
                return;
            }
            request(st, 0, PH_KEEP_WINNERS, T, &sc);                 // :398
            return;
        }
        case PH_KEEP_WINNERS: {
            // keep only the VPs that win at least one line (:406-413)
            argmax_assoc(im, st.M, T);
            for (int m = T.tid; m < st.M; m += T.nthreads) sc.rem[m] = 1;
            team_sync();
            for (int n = T.tid; n < N; n += T.nthreads) sc.rem[im.assoc[n]] = 0;
#if defined(VPK_HOST_TRACE)
            { int bc[kMaxM] = {0}; for (int n = 0; n < N; ++n) bc[im.assoc[n]]++; printf("[trace] KEEP_WINNERS M=%d bincount:", st.M); for (int m = 0; m < st.M; ++m) printf(" %d", bc[m]); printf("\n"); }
#endif
            compact_vps(st, sc.rem, T);
            if (T.tid == 0) st.vidx = 0;
            request(st, 1, PH_FINAL_COUNTS, T, &sc);                 // :415 (index i+1)
            return;
        }
        case PH_FINAL_COUNTS: {
            line_counts(im, st, cfg.outlier_thresh, T);
#if defined(VPK_HOST_TRACE)
            printf("[trace] FINAL_COUNTS M=%d counts:", st.M); for (int m = 0; m < st.M; ++m) printf(" %d", st.cnt[m]); printf("\n");
#endif
            // drop VPs with too few lines, front to back (:423-437)
            if (T.tid == 0) {
                int v = st.vidx;
                while (v < st.M && !(st.cnt[v] < cfg.num_min_lines)) ++v;
                st.vidx = v;
            }
            team_sync();
            const int v = st.vidx;
            if (v >= st.M) {
                const bool ok = st.M > 0;
                write_result(out, im, st, ok ? VPK_EM_OK : VPK_EM_NO_VPS_LEFT, st.iter, ok, T);
                return;
            }
            for (int m = T.tid; m < st.M; m += T.nthreads) sc.rem[m] = (m == v);
            compact_vps(st, sc.rem, T);
            if (st.M == 0) {                                    // the reference crashes here (argmax of an empty axis)
                write_result(out, im, st, VPK_EM_NO_VPS_LEFT, st.iter, false, T);
                return;
            }
            request(st, 1, PH_FINAL_COUNTS, T, &sc);
            return;
        }
        default:
            return;
        }
    }
}

}  // namespace em
}  // namespace vpk
