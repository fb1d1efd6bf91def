// TEST INFRASTRUCTURE ONLY.  Single-threaded host build of the LSD detector from the same source the CUDA kernels
// use (vanishing_points_2017_b200/csrc/lsd_core.cuh, team = 1 thread), so that the whole sequential algorithm can
// be checked against oracle/lsd_detector_oracle.py on a box without a GPU.  The data-parallel steps (sampler,
// gradient, pseudo-ordering) are plain loops here, in the order the kernels' per-pixel functions define.
// Never linked into libvpk.so, never imported by the package.
#include <algorithm>
#include <vector>
#include "../../vanishing_points_2017_b200/csrc/lsd_core.cuh"

using namespace vpk::lsd;

// image (H, W) row-major float64.  Returns the number of rows; writes at most `cap` rows of 7 into `rows`.
extern "C" int hostsim_lsd(const double* image, int W, int H, double scale, double sigma_scale, double quant, double ang_th,
                           double log_eps, double density_th, int n_bins, double* rows, int cap) {
    std::vector<double> img(image, image + (size_t)W * H);
    int X = W, Y = H;
    if (scale != 1.0) {
        X = (int)ceil(W * scale);
        Y = (int)ceil(H * scale);
        const int h = sampler_half(scale, sigma_scale), n = 2 * h + 1;
        std::vector<double> k((size_t)std::max(X, Y) * n);
        sampler_table(scale, sigma_scale, std::max(X, Y), k.data());
        std::vector<double> aux((size_t)X * H), out((size_t)X * Y);
        for (int x = 0; x < X; ++x)
            for (int y = 0; y < H; ++y) {
                const int xc = sampler_centre(x, scale);
                double s = 0.0;
                for (int i = 0; i < n; ++i) s = add(s, mul(img[mirror(xc - h + i, W) + (size_t)y * W], k[(size_t)x * n + i]));
                aux[x + (size_t)y * X] = s;
            }
        for (int y = 0; y < Y; ++y)
            for (int x = 0; x < X; ++x) {
                const int yc = sampler_centre(y, scale);
                double s = 0.0;
                for (int i = 0; i < n; ++i) s = add(s, mul(aux[x + (size_t)mirror(yc - h + i, H) * X], k[(size_t)y * n + i]));
                out[x + (size_t)y * X] = s;
            }
        img.swap(out);
    }
    const double prec = dv(mul(kPi, ang_th), 180.0);
    const double rho = dv(quant, sin(prec));
    std::vector<double> ang((size_t)X * Y, kNotDef), mod((size_t)X * Y, 0.0);
    double max_grad = 0.0;
    for (int y = 0; y + 1 < Y; ++y)
        for (int x = 0; x + 1 < X; ++x) {
            const size_t a = x + (size_t)y * X;
            double an;
            mod[a] = gradient(img[a], img[a + 1], img[a + X], img[a + X + 1], rho, &an);
            ang[a] = an;
            if (an != kNotDef && mod[a] > max_grad) max_grad = mod[a];
        }
    // pseudo-ordering: traversal x outer / y inner, stable by descending bin; only defined pixels seed
    std::vector<std::pair<int, int>> seeds;     // (n_bins - 1 - bin, pixel)
    for (int x = 0; x + 1 < X; ++x)
        for (int y = 0; y + 1 < Y; ++y) {
            const size_t a = x + (size_t)y * X;
            if (ang[a] != kNotDef) seeds.push_back({n_bins - 1 - grad_bin(mod[a], n_bins, max_grad), (int)a});
        }
    std::stable_sort(seeds.begin(), seeds.end(), [](const std::pair<int, int>& p, const std::pair<int, int>& q) { return p.first < q.first; });
    std::vector<uint32_t> used(((size_t)X * Y + 31) / 32, 0u), reg((size_t)X * Y);
    View v{ang.data(), mod.data(), used.data(), reg.data(), X, Y};
    const Params q = make_params(scale, ang_th, log_eps, density_th, X, Y);
    int count = 0;
    for (const auto& s : seeds) {
        if (used_get(v, s.second)) continue;
        double row[7];
        if (!process_seed(v, s.second % X, s.second / X, q, row)) continue;
        if (count < cap)
            for (int c = 0; c < 7; ++c) rows[7 * count + c] = row[c];
        ++count;
    }
    return count;
}
