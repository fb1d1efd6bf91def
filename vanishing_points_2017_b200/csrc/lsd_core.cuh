// Row N4: the sequential part of the LSD line segment detector 1.6 (Grompone von Gioi et al., IPOL 2012; the
// detector behind lsd.detect_line_segments, reference evaluation.py:227-251): region growing, region2rect /
// get_theta, refine / reduce_region_radius, rect_improve / rect_nfa / nfa / log_gamma, restated from
// oracle/lsd_detector_oracle.py.  The same source is
//   * the body of the region kernel in lsd.cu (team = one warp per image: every lane runs the same control flow
//     on the same data, lane 0 alone writes the `used` bitmap, the region list and the rows, and the lanes
//     share out the columns of the rectangle in rect_nfa, whose aligned-pixel count is an integer sum), and
//   * a single-threaded host build, tests/hostsim/lsd_hostsim.cpp (TEST INFRASTRUCTURE, never in libvpk.so).
// Floating point: every operation is a single correctly rounded float64 operation in the oracle's order (on the
// device through __dmul_rn & co, so nothing is contracted into an FMA; the host build uses -ffp-contract=off),
// and every floating-point sum runs in the oracle's order (region sums in pixel-insertion order).
#pragma once
#include <math.h>
#include <stdint.h>
#if defined(VPK_LSD_CHECKS)
#include <assert.h>
#define LSD_CHECK(c) assert(c)
#else
#define LSD_CHECK(c) ((void)0)
#endif

#if defined(__CUDACC__)
#define LSD_HD __host__ __device__ __forceinline__
#else
#define LSD_HD inline
#endif

namespace vpk {
namespace lsd {

constexpr double kNotDef = -1024.0;
constexpr double kPi = 3.14159265358979323846;
constexpr double k3_2Pi = 4.71238898038;       // lsd.c's own truncated constants
constexpr double k2Pi = 6.28318530718;
constexpr double kLn10 = 2.30258509299404568402;
constexpr double kDblEps = 2.220446049250313e-16;
constexpr double kDblMin = 2.2250738585072014e-308;

#if defined(__CUDA_ARCH__)
LSD_HD double add(double a, double b) { return __dadd_rn(a, b); }
LSD_HD double sub(double a, double b) { return __dsub_rn(a, b); }
LSD_HD double mul(double a, double b) { return __dmul_rn(a, b); }
LSD_HD double dv(double a, double b) { return __ddiv_rn(a, b); }
LSD_HD double sqr(double a) { return __dsqrt_rn(a); }
#else
LSD_HD double add(double a, double b) { return a + b; }
LSD_HD double sub(double a, double b) { return a - b; }
LSD_HD double mul(double a, double b) { return a * b; }
LSD_HD double dv(double a, double b) { return a / b; }
LSD_HD double sqr(double a) { return sqrt(a); }
#endif

// One image as the region stage sees it.  used: one bit per pixel (shared memory on the device where it fits);
// reg: the region's pixels, x in the low and y in the high 16 bits.
struct View {
    const double* ang;     // level-line angle or kNotDef, x + y * X
    const double* mod;     // gradient norm
    uint32_t* used;
    uint32_t* reg;
    int X, Y;
};

struct Rect { double x1, y1, x2, y2, width, x, y, theta, dx, dy, prec, p; };

#if defined(__CUDA_ARCH__)
LSD_HD int lane() { return threadIdx.x & 31; }
LSD_HD int nlanes() { return 32; }
LSD_HD void tsync() { __syncwarp(); }
LSD_HD int tsum(int v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
#else
inline int lane() { return 0; }
inline int nlanes() { return 1; }
inline void tsync() {}
inline int tsum(int v) { return v; }
#endif

LSD_HD bool used_get(const View& v, int i) { return (v.used[i >> 5] >> (i & 31)) & 1u; }
// writers: lane 0 only, followed by tsync() before anyone reads
LSD_HD void used_set(View& v, int i) {
    LSD_CHECK(i >= 0 && i < v.X * v.Y);
    v.used[i >> 5] |= 1u << (i & 31);
}
LSD_HD void used_clear(View& v, int i) {
    LSD_CHECK(i >= 0 && i < v.X * v.Y);
    v.used[i >> 5] &= ~(1u << (i & 31));
}
LSD_HD void reg_put(View& v, int k, int x, int y) {
    LSD_CHECK(k >= 0 && k < v.X * v.Y);
    v.reg[k] = (uint32_t)x | ((uint32_t)y << 16);
}
LSD_HD int reg_x(const View& v, int k) { return (int)(v.reg[k] & 0xffffu); }
LSD_HD int reg_y(const View& v, int k) { return (int)(v.reg[k] >> 16); }

LSD_HD bool double_equal(double a, double b) {
    if (a == b) return true;
    const double abs_diff = fabs(sub(a, b));
    const double aa = fabs(a), bb = fabs(b);
    double abs_max = aa > bb ? aa : bb;
    if (abs_max < kDblMin) abs_max = kDblMin;
    return dv(abs_diff, abs_max) <= mul(100.0, kDblEps);
}

LSD_HD double dist(double x1, double y1, double x2, double y2) {
    return sqr(add(mul(sub(x2, x1), sub(x2, x1)), mul(sub(y2, y1), sub(y2, y1))));
}

LSD_HD double angle_diff_signed(double a, double b) {
    a = sub(a, b);
    while (a <= -kPi) a = add(a, k2Pi);
    while (a > kPi) a = sub(a, k2Pi);
    return a;
}
LSD_HD double angle_diff(double a, double b) { return fabs(angle_diff_signed(a, b)); }

LSD_HD bool isaligned(const View& v, int i, double theta, double prec) {
    const double a = v.ang[i];
    if (a == kNotDef) return false;
    theta = sub(theta, a);
    if (theta < 0.0) theta = -theta;
    if (theta > k3_2Pi) {
        theta = sub(theta, k2Pi);
        if (theta < 0.0) theta = -theta;
    }
    return theta <= prec;
}

LSD_HD double log_gamma(double x) {
    if (x > 15.0)   // Windschitl
        return add(sub(add(0.918938533204673, mul(sub(x, 0.5), log(x))), x),
                   mul(mul(0.5, x), log(add(mul(x, sinh(dv(1.0, x))), dv(1.0, mul(810.0, pow(x, 6.0)))))));
    const double q[7] = {75122.6331530, 80916.6278952, 36308.2951477, 8687.24529705, 1168.92649479, 83.8676043424,
                         2.50662827511};
    double a = sub(mul(add(x, 0.5), log(add(x, 5.5))), add(x, 5.5));   // Lanczos
    double b = 0.0;
    for (int n = 0; n < 7; ++n) {
        a = sub(a, log(add(x, (double)n)));
        b = add(b, mul(q[n], pow(x, (double)n)));
    }
    return add(a, log(b));
}

LSD_HD double nfa(int n, int k, double p, double logNT) {
    if (n == 0 || k == 0) return -logNT;
    if (n == k) return sub(-logNT, mul((double)n, log10(p)));
    const double p_term = dv(p, sub(1.0, p));
    const double log1term = add(add(sub(sub(log_gamma(add((double)n, 1.0)), log_gamma(add((double)k, 1.0))),
                                        log_gamma(add((double)(n - k), 1.0))),
                                    mul((double)k, log(p))),
                                mul((double)(n - k), log(sub(1.0, p))));
    double term = exp(log1term);
    if (double_equal(term, 0.0)) {
        if ((double)k > mul((double)n, p)) return sub(dv(-log1term, kLn10), logNT);
        return -logNT;
    }
    double bin_tail = term;
    for (int i = k + 1; i <= n; ++i) {
        const double bin_term = mul((double)(n - i + 1), dv(1.0, (double)i));
        const double mult_term = mul(bin_term, p_term);
        term = mul(term, mult_term);
        bin_tail = add(bin_tail, term);
        if (bin_term < 1.0) {
            const double err = mul(term, sub(dv(sub(1.0, pow(mult_term, (double)(n - i + 1))), sub(1.0, mult_term)), 1.0));
            if (err < mul(mul(0.1, fabs(sub(-log10(bin_tail), logNT))), bin_tail)) break;
        }
    }
    return sub(-log10(bin_tail), logNT);
}

// region_grow: neighbours xx outer, yy inner; the region angle after every accepted pixel.  Returns the size.
LSD_HD int region_grow(View& v, int x, int y, double prec, double* reg_angle) {
    int size = 1;
    if (lane() == 0) { reg_put(v, 0, x, y); used_set(v, x + y * v.X); }
    tsync();
    double ra = v.ang[x + y * v.X];
    double sumdx = cos(ra), sumdy = sin(ra);
    for (int i = 0; i < size; ++i) {
        const int rx = reg_x(v, i), ry = reg_y(v, i);
        for (int xx = rx - 1; xx <= rx + 1; ++xx)
            for (int yy = ry - 1; yy <= ry + 1; ++yy) {
                if (xx < 0 || yy < 0 || xx >= v.X || yy >= v.Y) continue;
                const int k = xx + yy * v.X;
                if (used_get(v, k) || !isaligned(v, k, ra, prec)) continue;
                if (lane() == 0) { used_set(v, k); reg_put(v, size, xx, yy); }
                tsync();
                ++size;
                sumdx = add(sumdx, cos(v.ang[k]));
                sumdy = add(sumdy, sin(v.ang[k]));
                ra = atan2(sumdy, sumdx);
            }
    }
    *reg_angle = ra;
    return size;
}

LSD_HD double get_theta(const View& v, int n, double x, double y, double reg_angle, double prec) {
    double Ixx = 0.0, Iyy = 0.0, Ixy = 0.0;
    for (int i = 0; i < n; ++i) {
        const double rx = (double)reg_x(v, i), ry = (double)reg_y(v, i);
        const double w = v.mod[reg_x(v, i) + reg_y(v, i) * v.X];
        Ixx = add(Ixx, mul(mul(sub(ry, y), sub(ry, y)), w));
        Iyy = add(Iyy, mul(mul(sub(rx, x), sub(rx, x)), w));
        Ixy = sub(Ixy, mul(mul(sub(rx, x), sub(ry, y)), w));
    }
    const double lambda = mul(0.5, sub(add(Ixx, Iyy), sqr(add(mul(sub(Ixx, Iyy), sub(Ixx, Iyy)), mul(mul(4.0, Ixy), Ixy)))));
    double theta = fabs(Ixx) > fabs(Iyy) ? atan2(sub(lambda, Ixx), Ixy) : atan2(Ixy, sub(lambda, Iyy));
    if (angle_diff(theta, reg_angle) > prec) theta = add(theta, kPi);
    return theta;
}

LSD_HD void region2rect(const View& v, int n, double reg_angle, double prec, double p, Rect& r) {
    double x = 0.0, y = 0.0, sum = 0.0;
    for (int i = 0; i < n; ++i) {
        const double w = v.mod[reg_x(v, i) + reg_y(v, i) * v.X];
        x = add(x, mul((double)reg_x(v, i), w));
        y = add(y, mul((double)reg_y(v, i), w));
        sum = add(sum, w);
    }
    x = dv(x, sum);
    y = dv(y, sum);
    const double theta = get_theta(v, n, x, y, reg_angle, prec);
    const double dx = cos(theta), dy = sin(theta);
    double l_min = 0.0, l_max = 0.0, w_min = 0.0, w_max = 0.0;
    for (int i = 0; i < n; ++i) {
        const double ex = sub((double)reg_x(v, i), x), ey = sub((double)reg_y(v, i), y);
        const double l = add(mul(ex, dx), mul(ey, dy));
        const double w = add(mul(-ex, dy), mul(ey, dx));
        if (l > l_max) l_max = l;
        if (l < l_min) l_min = l;
        if (w > w_max) w_max = w;
        if (w < w_min) w_min = w;
    }
    r.x1 = add(x, mul(l_min, dx)); r.y1 = add(y, mul(l_min, dy));
    r.x2 = add(x, mul(l_max, dx)); r.y2 = add(y, mul(l_max, dy));
    r.width = sub(w_max, w_min);
    r.x = x; r.y = y; r.theta = theta; r.dx = dx; r.dy = dy; r.prec = prec; r.p = p;
    if (r.width < 1.0) r.width = 1.0;
}

LSD_HD double inter_low(double x, double x1, double y1, double x2, double y2) {
    if (double_equal(x1, x2) && y1 < y2) return y1;
    if (double_equal(x1, x2) && y1 > y2) return y2;
    return add(y1, dv(mul(sub(x, x1), sub(y2, y1)), sub(x2, x1)));
}
LSD_HD double inter_hi(double x, double x1, double y1, double x2, double y2) {
    if (double_equal(x1, x2) && y1 < y2) return y2;
    if (double_equal(x1, x2) && y1 > y2) return y1;
    return add(y1, dv(mul(sub(x, x1), sub(y2, y1)), sub(x2, x1)));
}

// rect_nfa over the pixels of lsd.c's rectangle iterator (ri_ini / ri_inc): columns x = ceil(vx[0]) .. while
// x <= vx[2], in each y = ceil(ys) .. while y <= ye.  The lanes take every nlanes()-th column; the counts are
// integers, so their sum does not depend on that split.
LSD_HD double rect_nfa(const View& v, const Rect& r, double logNT) {
    const double hw = dv(r.width, 2.0);
    double cx[4], cy[4];
    cx[0] = sub(r.x1, mul(r.dy, hw)); cy[0] = add(r.y1, mul(r.dx, hw));
    cx[1] = sub(r.x2, mul(r.dy, hw)); cy[1] = add(r.y2, mul(r.dx, hw));
    cx[2] = add(r.x2, mul(r.dy, hw)); cy[2] = sub(r.y2, mul(r.dx, hw));
    cx[3] = add(r.x1, mul(r.dy, hw)); cy[3] = sub(r.y1, mul(r.dx, hw));
    int off;
    if (r.x1 < r.x2 && r.y1 <= r.y2) off = 0;
    else if (r.x1 >= r.x2 && r.y1 < r.y2) off = 1;
    else if (r.x1 > r.x2 && r.y1 >= r.y2) off = 2;
    else off = 3;
    double vx[4], vy[4];
    for (int n = 0; n < 4; ++n) { vx[n] = cx[(off + n) & 3]; vy[n] = cy[(off + n) & 3]; }
    int pts = 0, alg = 0;
    for (int x = (int)ceil(vx[0]) + lane(); (double)x <= vx[2]; x += nlanes()) {
        const double fx = (double)x;
        const double ys = fx < vx[3] ? inter_low(fx, vx[0], vy[0], vx[3], vy[3]) : inter_low(fx, vx[3], vy[3], vx[2], vy[2]);
        const double ye = fx < vx[1] ? inter_hi(fx, vx[0], vy[0], vx[1], vy[1]) : inter_hi(fx, vx[1], vy[1], vx[2], vy[2]);
        if (x < 0 || x >= v.X) continue;
        for (int y = (int)ceil(ys); (double)y <= ye; ++y) {
            if (y < 0 || y >= v.Y) continue;
            ++pts;
            if (isaligned(v, x + y * v.X, r.theta, r.prec)) ++alg;
        }
    }
    return nfa(tsum(pts), tsum(alg), r.p, logNT);
}

LSD_HD double rect_improve(const View& v, Rect& rec, double logNT, double log_eps) {
    const double delta = 0.5, delta_2 = dv(delta, 2.0);
    double log_nfa = rect_nfa(v, rec, logNT);
    if (log_nfa > log_eps) return log_nfa;
    Rect r = rec;
    for (int n = 0; n < 5; ++n) {                    // finer precisions
        r.p = dv(r.p, 2.0);
        r.prec = mul(r.p, kPi);
        const double nw = rect_nfa(v, r, logNT);
        if (nw > log_nfa) { log_nfa = nw; rec = r; }
    }
    if (log_nfa > log_eps) return log_nfa;
    r = rec;
    for (int n = 0; n < 5; ++n) {                    // reduce width
        if (sub(r.width, delta) >= 0.5) {
            r.width = sub(r.width, delta);
            const double nw = rect_nfa(v, r, logNT);
            if (nw > log_nfa) { rec = r; log_nfa = nw; }
        }
    }
    if (log_nfa > log_eps) return log_nfa;
    for (int side = 0; side < 2; ++side) {           // reduce one side, then the other
        r = rec;
        for (int n = 0; n < 5; ++n) {
            if (sub(r.width, delta) >= 0.5) {
                const double ox = mul(-r.dy, delta_2), oy = mul(r.dx, delta_2);
                if (side == 0) {
                    r.x1 = add(r.x1, ox); r.y1 = add(r.y1, oy); r.x2 = add(r.x2, ox); r.y2 = add(r.y2, oy);
                } else {
                    r.x1 = sub(r.x1, ox); r.y1 = sub(r.y1, oy); r.x2 = sub(r.x2, ox); r.y2 = sub(r.y2, oy);
                }
                r.width = sub(r.width, delta);
                const double nw = rect_nfa(v, r, logNT);
                if (nw > log_nfa) { rec = r; log_nfa = nw; }
            }
        }
        if (log_nfa > log_eps) return log_nfa;
    }
    r = rec;
    for (int n = 0; n < 5; ++n) {                    // even finer precisions
        r.p = dv(r.p, 2.0);
        r.prec = mul(r.p, kPi);
        const double nw = rect_nfa(v, r, logNT);
        if (nw > log_nfa) { log_nfa = nw; rec = r; }
    }
    return log_nfa;
}

LSD_HD double density(int n, const Rect& r) { return dv((double)n, mul(dist(r.x1, r.y1, r.x2, r.y2), r.width)); }

LSD_HD bool reduce_region_radius(View& v, int* n, double reg_angle, double prec, double p, Rect& rec, double density_th) {
    double d = density(*n, rec);
    if (d >= density_th) return true;
    const double xc = (double)reg_x(v, 0), yc = (double)reg_y(v, 0);
    const double rad1 = dist(xc, yc, rec.x1, rec.y1), rad2 = dist(xc, yc, rec.x2, rec.y2);
    double rad = rad1 > rad2 ? rad1 : rad2;
    while (d < density_th) {
        rad = mul(rad, 0.75);
        for (int i = 0; i < *n; ++i)
            if (dist(xc, yc, (double)reg_x(v, i), (double)reg_y(v, i)) > rad) {
                if (lane() == 0) {                   // swap with the last point, as lsd.c does
                    used_clear(v, reg_x(v, i) + reg_y(v, i) * v.X);
                    v.reg[i] = v.reg[*n - 1];
                }
                tsync();
                --*n;
                --i;
            }
        if (*n < 2) return false;
        region2rect(v, *n, reg_angle, prec, p, rec);
        d = density(*n, rec);
    }
    return true;
}

LSD_HD bool refine(View& v, int* n, double reg_angle, double prec, double p, Rect& rec, double density_th) {
    if (density(*n, rec) >= density_th) return true;
    const int x0 = reg_x(v, 0), y0 = reg_y(v, 0);
    const double xc = (double)x0, yc = (double)y0;
    const double ang_c = v.ang[x0 + y0 * v.X];
    double sum = 0.0, s_sum = 0.0;
    int cnt = 0;
    for (int i = 0; i < *n; ++i) {
        const int rx = reg_x(v, i), ry = reg_y(v, i);
        if (dist(xc, yc, (double)rx, (double)ry) < rec.width) {
            const double ang_d = angle_diff_signed(v.ang[rx + ry * v.X], ang_c);
            sum = add(sum, ang_d);
            s_sum = add(s_sum, mul(ang_d, ang_d));
            ++cnt;
        }
    }
    if (lane() == 0)
        for (int i = 0; i < *n; ++i) used_clear(v, reg_x(v, i) + reg_y(v, i) * v.X);
    tsync();
    const double mean_angle = dv(sum, (double)cnt);
    const double tau = mul(2.0, sqr(add(dv(sub(s_sum, mul(mul(2.0, mean_angle), sum)), (double)cnt), mul(mean_angle, mean_angle))));
    *n = region_grow(v, x0, y0, tau, &reg_angle);
    if (*n < 2) return false;
    region2rect(v, *n, reg_angle, prec, p, rec);
    if (density(*n, rec) < density_th) return reduce_region_radius(v, n, reg_angle, prec, p, rec, density_th);
    return true;
}

// ---- data-parallel steps (one output pixel each) ----------------------------------------------------------
// gaussian_sampler (lsd.c :611): the kernel of output position x depends on x, scale and sigma only, so one table
// of kernels serves every image and both passes; it is computed on the host with the C library's exp.
inline int sampler_half(double scale, double sigma_scale) {
    const double sigma = scale < 1.0 ? sigma_scale / scale : sigma_scale;
    return (int)ceil(sigma * sqrt(2.0 * 2.0 * log(10.0)));
}
inline void sampler_table(double scale, double sigma_scale, int positions, double* k /* positions * (2h+1) */) {
    const double sigma = scale < 1.0 ? sigma_scale / scale : sigma_scale;
    const int h = sampler_half(scale, sigma_scale), n = 2 * h + 1;
    for (int x = 0; x < positions; ++x) {
        const double xx = (double)x / scale;
        const int xc = (int)floor(xx + 0.5);
        const double mean = (double)h + xx - (double)xc;
        double* kv = k + (size_t)x * n;
        double sum = 0.0;
        for (int i = 0; i < n; ++i) {
            const double val = ((double)i - mean) / sigma;
            kv[i] = exp(-0.5 * val * val);
            sum += kv[i];
        }
        if (sum >= 0.0)
            for (int i = 0; i < n; ++i) kv[i] /= sum;
    }
}
LSD_HD int sampler_centre(int x, double scale) { return (int)floor(add(dv((double)x, scale), 0.5)); }
// symmetric boundary condition of gaussian_sampler
LSD_HD int mirror(int j, int size) {
    const int dbl = 2 * size;
    while (j < 0) j += dbl;
    while (j >= dbl) j -= dbl;
    if (j >= size) j = dbl - 1 - j;
    return j;
}
// ll_angle (lsd.c :752) on the 2x2 window  A B / C D  at (x, y)
LSD_HD double gradient(double A, double B, double C, double D, double rho, double* ang) {
    const double com1 = sub(D, A), com2 = sub(B, C);
    const double gx = add(com1, com2), gy = sub(com1, com2);
    const double norm = sqr(dv(add(mul(gx, gx), mul(gy, gy)), 4.0));
    *ang = norm <= rho ? kNotDef : atan2(gx, -gy);
    return norm;
}
LSD_HD int grad_bin(double norm, int n_bins, double max_grad) {
    unsigned i = (unsigned)dv(mul(norm, (double)n_bins), max_grad);
    return i >= (unsigned)n_bins ? n_bins - 1 : (int)i;
}

struct Params { double scale, prec, p, log_eps, density_th, logNT; int min_reg_size; };

LSD_HD Params make_params(double scale, double ang_th, double log_eps, double density_th, int X, int Y) {
    Params q;
    q.scale = scale;
    q.prec = dv(mul(kPi, ang_th), 180.0);
    q.p = dv(ang_th, 180.0);
    q.log_eps = log_eps;
    q.density_th = density_th;
    q.logNT = add(dv(mul(5.0, add(log10((double)X), log10((double)Y))), 2.0), log10(11.0));
    q.min_reg_size = (int)dv(-q.logNT, log10(q.p));
    return q;
}

// One seed of LineSegmentDetection's search loop (lsd.c :2126-2190), for a seed that is not used and not NOTDEF.
// Returns true and the row x1, y1, x2, y2, width, p, -log10(NFA) when it yields a segment.
LSD_HD bool process_seed(View& v, int x, int y, const Params& q, double row[7]) {
    double reg_angle;
    int n = region_grow(v, x, y, q.prec, &reg_angle);
    if (n < q.min_reg_size) return false;
    Rect rec;
    region2rect(v, n, reg_angle, q.prec, q.p, rec);
    if (!refine(v, &n, reg_angle, q.prec, q.p, rec, q.density_th)) return false;
    const double log_nfa = rect_improve(v, rec, q.logNT, q.log_eps);
    if (log_nfa <= q.log_eps) return false;
    row[0] = add(rec.x1, 0.5); row[1] = add(rec.y1, 0.5); row[2] = add(rec.x2, 0.5); row[3] = add(rec.y2, 0.5);
    row[4] = rec.width;
    if (q.scale != 1.0)
        for (int c = 0; c < 5; ++c) row[c] = dv(row[c], q.scale);
    row[5] = rec.p;
    row[6] = log_nfa;
    return true;
}

}  // namespace lsd
}  // namespace vpk
