"""TEST INFRASTRUCTURE ONLY -- float64 restatement of the LSD line segment detector 1.6 (R. Grompone von Gioi,
J. Jakubowicz, J.-M. Morel, G. Randall, "LSD: a Line Segment Detector", IPOL 2012; the reference calls it through
lsdpython: lsd.detect_line_segments, evaluation.py:227-251, with the defaults of lsdpython/lsd.pyx:17-18).

Followed step for step, in lsd.c's own order of operations:
  gaussian_sampler   per-output-position Gaussian kernel, symmetric boundary, x pass then y pass
  ll_angle           2x2 gradient, NOTDEF below rho = quant / sin(prec), pseudo-ordering into n_bins bins
                     (traversal x outer / y inner, bins from the highest down)
  region_grow        neighbours xx outer / yy inner, region angle atan2(sum sin, sum cos) after every pixel
  region2rect / get_theta, refine / reduce_region_radius, rect_improve / rect_nfa (rectangle iterator) / nfa
  with lsd.c's log_gamma (Lanczos at or below 15, Windschitl above).
Output rows: x1, y1, x2, y2, width, p, -log10(NFA) in pixels of the input image, in seed order.

Parity with the lsd.c binary is UNPINNED: neither lsd.c nor the reference's images are available; the cross-check
is OpenCV's independent port (tests/test_oracle_lsd_detector.py).  Transcendentals go through `math` (the C
library), the same functions the host build of csrc/lsd_core.cuh calls.  Never imported by the package."""
import math

import numpy as np

NOTDEF = -1024.0
M_PI = 3.14159265358979323846
M_3_2_PI = 4.71238898038          # lsd.c's own truncated constants
M_2__PI = 6.28318530718
M_LN10 = 2.30258509299404568402
DBL_EPSILON = 2.220446049250313e-16
DBL_MIN = 2.2250738585072014e-308
TABSIZE = 100000


def double_equal(a, b):
    if a == b:
        return True
    abs_diff = abs(a - b)
    aa, bb = abs(a), abs(b)
    abs_max = aa if aa > bb else bb
    if abs_max < DBL_MIN:
        abs_max = DBL_MIN
    return (abs_diff / abs_max) <= (100.0 * DBL_EPSILON)


def dist(x1, y1, x2, y2):
    return math.sqrt((x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1))


def angle_diff_signed(a, b):
    a -= b
    while a <= -M_PI:
        a += M_2__PI
    while a > M_PI:
        a -= M_2__PI
    return a


def angle_diff(a, b):
    return abs(angle_diff_signed(a, b))


def log_gamma(x):
    if x > 15.0:
        return 0.918938533204673 + (x - 0.5) * math.log(x) - x + 0.5 * x * math.log(x * math.sinh(1 / x) + 1 / (810.0 * math.pow(x, 6.0)))
    q = (75122.6331530, 80916.6278952, 36308.2951477, 8687.24529705, 1168.92649479, 83.8676043424, 2.50662827511)
    a = (x + 0.5) * math.log(x + 5.5) - (x + 5.5)
    b = 0.0
    for n in range(7):
        a -= math.log(x + float(n))
        b += q[n] * math.pow(x, float(n))
    return a + math.log(b)


def nfa(n, k, p, logNT):
    if n == 0 or k == 0:
        return -logNT
    if n == k:
        return -logNT - float(n) * math.log10(p)
    p_term = p / (1.0 - p)
    log1term = (log_gamma(float(n) + 1.0) - log_gamma(float(k) + 1.0) - log_gamma(float(n - k) + 1.0)
                + float(k) * math.log(p) + float(n - k) * math.log(1.0 - p))
    term = math.exp(log1term)
    if double_equal(term, 0.0):
        if float(k) > float(n) * p:
            return -log1term / M_LN10 - logNT
        return -logNT
    bin_tail = term
    for i in range(k + 1, n + 1):
        bin_term = float(n - i + 1) * (1.0 / float(i))
        mult_term = bin_term * p_term
        term *= mult_term
        bin_tail += term
        if bin_term < 1.0:
            err = term * ((1.0 - math.pow(mult_term, float(n - i + 1))) / (1.0 - mult_term) - 1.0)
            if err < 0.1 * abs(-math.log10(bin_tail) - logNT) * bin_tail:
                break
    return -math.log10(bin_tail) - logNT


def gaussian_kernel(n, sigma, mean):
    vals = []
    s = 0.0
    for i in range(n):
        val = (float(i) - mean) / sigma
        v = math.exp(-0.5 * val * val)
        vals.append(v)
        s += v
    if s >= 0.0:
        vals = [v / s for v in vals]
    return vals


def sampler_taps(size_in, size_out, scale, sigma_scale):
    """Per output position: the source indices (symmetric boundary) and the kernel of gaussian_sampler."""
    sigma = sigma_scale / scale if scale < 1.0 else sigma_scale
    h = int(math.ceil(sigma * math.sqrt(2.0 * 2.0 * math.log(10.0))))
    n = 1 + 2 * h
    dbl = 2 * size_in
    J = np.empty((size_out, n), np.int64)
    K = np.empty((size_out, n), np.float64)
    for x in range(size_out):
        xx = float(x) / scale
        xc = int(math.floor(xx + 0.5))
        K[x] = gaussian_kernel(n, sigma, float(h) + xx - float(xc))
        for i in range(n):
            j = xc - h + i
            while j < 0:
                j += dbl
            while j >= dbl:
                j -= dbl
            if j >= size_in:
                j = dbl - 1 - j
            J[x, i] = j
    return J, K


def gaussian_sampler(img, scale, sigma_scale):
    Y, X = img.shape
    N = int(math.ceil(X * scale))
    M = int(math.ceil(Y * scale))
    Jx, Kx = sampler_taps(X, N, scale, sigma_scale)
    aux = np.zeros((Y, N))
    for i in range(Jx.shape[1]):                       # tap by tap: sum = ((0 + t0) + t1) + ...
        aux = aux + img[:, Jx[:, i]] * Kx[None, :, i]
    Jy, Ky = sampler_taps(Y, M, scale, sigma_scale)
    out = np.zeros((M, N))
    for i in range(Jy.shape[1]):
        out = out + aux[Jy[:, i], :] * Ky[:, i, None]
    return out


def ll_angle(img, rho, n_bins):
    """angles (flat, x + y*X), modgrad (flat), and the seed list (flat indices of non-NOTDEF pixels in
    lsd.c's pseudo-order)."""
    Y, X = img.shape
    ang = np.full(X * Y, NOTDEF)
    mod = np.zeros(X * Y)
    if X < 2 or Y < 2:
        return ang.tolist(), mod.tolist(), []
    A, B, C, D = img[:-1, :-1], img[:-1, 1:], img[1:, :-1], img[1:, 1:]
    com1 = D - A
    com2 = B - C
    gx = com1 + com2
    gy = com1 - com2
    norm = np.sqrt((gx * gx + gy * gy) / 4.0)
    defined = norm > rho
    ys, xs = np.nonzero(defined)
    idx = xs + ys * X
    mod2 = mod.reshape(Y, X)
    mod2[:-1, :-1] = norm
    ang[idx] = [math.atan2(a, b) for a, b in zip(gx[ys, xs].tolist(), (-gy[ys, xs]).tolist())]
    if not defined.any():
        return ang.tolist(), mod.tolist(), []
    max_grad = float(norm[defined].max())
    # traversal order x outer, y inner; bins from the highest; only defined pixels can seed
    nT = norm.T                                        # (X-1, Y-1): row = x
    dT = defined.T
    b = np.floor(nT * float(n_bins) / max_grad)
    b = np.minimum(b, n_bins - 1).astype(np.int64)
    t = np.arange(nT.size).reshape(nT.shape)
    tsel, bsel = t[dT], b[dT]
    order = tsel[np.argsort(-bsel, kind="stable")]
    sx, sy = order // (Y - 1), order % (Y - 1)
    return ang.tolist(), mod.tolist(), (sx + sy * X).tolist()


class _Img:
    pass


def isaligned(I, idx, theta, prec):
    a = I.ang[idx]
    if a == NOTDEF:
        return False
    theta -= a
    if theta < 0.0:
        theta = -theta
    if theta > M_3_2_PI:
        theta -= M_2__PI
        if theta < 0.0:
            theta = -theta
    return theta <= prec


def region_grow(I, x, y, reg, prec):
    X, Y, used, ang = I.X, I.Y, I.used, I.ang
    del reg[:]
    reg.append((x, y))
    reg_angle = ang[x + y * X]
    sumdx = math.cos(reg_angle)
    sumdy = math.sin(reg_angle)
    used[x + y * X] = 1
    i = 0
    while i < len(reg):
        rx, ry = reg[i]
        for xx in range(rx - 1, rx + 2):
            for yy in range(ry - 1, ry + 2):
                if 0 <= xx < X and 0 <= yy < Y:
                    k = xx + yy * X
                    if used[k] != 1 and isaligned(I, k, reg_angle, prec):
                        used[k] = 1
                        reg.append((xx, yy))
                        sumdx += math.cos(ang[k])
                        sumdy += math.sin(ang[k])
                        reg_angle = math.atan2(sumdy, sumdx)
        i += 1
    return reg_angle


def get_theta(I, reg, x, y, reg_angle, prec):
    Ixx = Iyy = Ixy = 0.0
    for rx, ry in reg:
        w = I.mod[rx + ry * I.X]
        Ixx += (float(ry) - y) * (float(ry) - y) * w
        Iyy += (float(rx) - x) * (float(rx) - x) * w
        Ixy -= (float(rx) - x) * (float(ry) - y) * w
    lam = 0.5 * (Ixx + Iyy - math.sqrt((Ixx - Iyy) * (Ixx - Iyy) + 4.0 * Ixy * Ixy))
    theta = math.atan2(lam - Ixx, Ixy) if abs(Ixx) > abs(Iyy) else math.atan2(Ixy, lam - Iyy)
    if angle_diff(theta, reg_angle) > prec:
        theta += M_PI
    return theta


def region2rect(I, reg, reg_angle, prec, p):
    x = y = s = 0.0
    for rx, ry in reg:
        w = I.mod[rx + ry * I.X]
        x += float(rx) * w
        y += float(ry) * w
        s += w
    x /= s
    y /= s
    theta = get_theta(I, reg, x, y, reg_angle, prec)
    dx = math.cos(theta)
    dy = math.sin(theta)
    l_min = l_max = w_min = w_max = 0.0
    for rx, ry in reg:
        l = (float(rx) - x) * dx + (float(ry) - y) * dy
        w = -(float(rx) - x) * dy + (float(ry) - y) * dx
        if l > l_max:
            l_max = l
        if l < l_min:
            l_min = l
        if w > w_max:
            w_max = w
        if w < w_min:
            w_min = w
    r = {"x1": x + l_min * dx, "y1": y + l_min * dy, "x2": x + l_max * dx, "y2": y + l_max * dy,
         "width": w_max - w_min, "x": x, "y": y, "theta": theta, "dx": dx, "dy": dy, "prec": prec, "p": p}
    if r["width"] < 1.0:
        r["width"] = 1.0
    return r


def inter_low(x, x1, y1, x2, y2):
    if double_equal(x1, x2) and y1 < y2:
        return y1
    if double_equal(x1, x2) and y1 > y2:
        return y2
    return y1 + (x - x1) * (y2 - y1) / (x2 - x1)


def inter_hi(x, x1, y1, x2, y2):
    if double_equal(x1, x2) and y1 < y2:
        return y2
    if double_equal(x1, x2) and y1 > y2:
        return y1
    return y1 + (x - x1) * (y2 - y1) / (x2 - x1)


def rect_corners(r):
    hw = r["width"] / 2.0
    vx = [r["x1"] - r["dy"] * hw, r["x2"] - r["dy"] * hw, r["x2"] + r["dy"] * hw, r["x1"] + r["dy"] * hw]
    vy = [r["y1"] + r["dx"] * hw, r["y2"] + r["dx"] * hw, r["y2"] - r["dx"] * hw, r["y1"] - r["dx"] * hw]
    x1, y1, x2, y2 = r["x1"], r["y1"], r["x2"], r["y2"]
    if x1 < x2 and y1 <= y2:
        off = 0
    elif x1 >= x2 and y1 < y2:
        off = 1
    elif x1 > x2 and y1 >= y2:
        off = 2
    else:
        off = 3
    return [vx[(off + n) % 4] for n in range(4)], [vy[(off + n) % 4] for n in range(4)]


def rect_pixels(r):
    """The pixels ri_ini / ri_inc visit, in their order: columns x = ceil(vx0) .. while x <= vx2, in each
    y = ceil(ys) .. while y <= ye."""
    vx, vy = rect_corners(r)
    x = int(math.ceil(vx[0]))
    while float(x) <= vx[2]:
        ys = inter_low(float(x), vx[0], vy[0], vx[3], vy[3]) if float(x) < vx[3] else inter_low(float(x), vx[3], vy[3], vx[2], vy[2])
        ye = inter_hi(float(x), vx[0], vy[0], vx[1], vy[1]) if float(x) < vx[1] else inter_hi(float(x), vx[1], vy[1], vx[2], vy[2])
        y = int(math.ceil(ys))
        while float(y) <= ye:
            yield x, y
            y += 1
        x += 1


def rect_nfa(I, r, logNT):
    pts = alg = 0
    X, Y = I.X, I.Y
    theta, prec = r["theta"], r["prec"]
    for x, y in rect_pixels(r):
        if 0 <= x < X and 0 <= y < Y:
            pts += 1
            if isaligned(I, x + y * X, theta, prec):
                alg += 1
    return nfa(pts, alg, r["p"], logNT)


def rect_improve(I, rec, logNT, log_eps):
    delta, delta_2 = 0.5, 0.25
    log_nfa = rect_nfa(I, rec, logNT)
    if log_nfa > log_eps:
        return log_nfa, rec

    def finer(rec, log_nfa):
        r = dict(rec)
        for _ in range(5):
            r["p"] /= 2.0
            r["prec"] = r["p"] * M_PI
            new = rect_nfa(I, r, logNT)
            if new > log_nfa:
                log_nfa, rec = new, dict(r)
        return rec, log_nfa

    rec, log_nfa = finer(rec, log_nfa)
    if log_nfa > log_eps:
        return log_nfa, rec
    r = dict(rec)
    for _ in range(5):
        if (r["width"] - delta) >= 0.5:
            r["width"] -= delta
            new = rect_nfa(I, r, logNT)
            if new > log_nfa:
                rec, log_nfa = dict(r), new
    if log_nfa > log_eps:
        return log_nfa, rec
    for sgn in (1.0, -1.0):
        r = dict(rec)
        for _ in range(5):
            if (r["width"] - delta) >= 0.5:
                if sgn > 0:
                    r["x1"] += -r["dy"] * delta_2
                    r["y1"] += r["dx"] * delta_2
                    r["x2"] += -r["dy"] * delta_2
                    r["y2"] += r["dx"] * delta_2
                else:
                    r["x1"] -= -r["dy"] * delta_2
                    r["y1"] -= r["dx"] * delta_2
                    r["x2"] -= -r["dy"] * delta_2
                    r["y2"] -= r["dx"] * delta_2
                r["width"] -= delta
                new = rect_nfa(I, r, logNT)
                if new > log_nfa:
                    rec, log_nfa = dict(r), new
        if log_nfa > log_eps:
            return log_nfa, rec
    rec, log_nfa = finer(rec, log_nfa)
    return log_nfa, rec


def density(reg, r):
    return float(len(reg)) / (dist(r["x1"], r["y1"], r["x2"], r["y2"]) * r["width"])


def reduce_region_radius(I, reg, reg_angle, prec, p, rec, density_th):
    d = density(reg, rec)
    if d >= density_th:
        return True, rec
    xc, yc = float(reg[0][0]), float(reg[0][1])
    rad1 = dist(xc, yc, rec["x1"], rec["y1"])
    rad2 = dist(xc, yc, rec["x2"], rec["y2"])
    rad = rad1 if rad1 > rad2 else rad2
    while d < density_th:
        rad *= 0.75
        i = 0
        while i < len(reg):                            # swap-with-last removal, as lsd.c does
            if dist(xc, yc, float(reg[i][0]), float(reg[i][1])) > rad:
                I.used[reg[i][0] + reg[i][1] * I.X] = 0
                reg[i] = reg[-1]
                reg.pop()
            else:
                i += 1
        if len(reg) < 2:
            return False, rec
        rec = region2rect(I, reg, reg_angle, prec, p)
        d = density(reg, rec)
    return True, rec


def refine(I, reg, reg_angle, prec, p, rec, density_th):
    if density(reg, rec) >= density_th:
        return True, rec
    xc, yc = float(reg[0][0]), float(reg[0][1])
    ang_c = I.ang[reg[0][0] + reg[0][1] * I.X]
    s = s_sum = 0.0
    n = 0
    for rx, ry in reg:
        I.used[rx + ry * I.X] = 0
        if dist(xc, yc, float(rx), float(ry)) < rec["width"]:
            ang_d = angle_diff_signed(I.ang[rx + ry * I.X], ang_c)
            s += ang_d
            s_sum += ang_d * ang_d
            n += 1
    mean_angle = s / float(n)
    tau = 2.0 * math.sqrt((s_sum - 2.0 * mean_angle * s) / float(n) + mean_angle * mean_angle)
    reg_angle = region_grow(I, reg[0][0], reg[0][1], reg, tau)
    if len(reg) < 2:
        return False, rec
    rec = region2rect(I, reg, reg_angle, prec, p)
    if density(reg, rec) < density_th:
        return reduce_region_radius(I, reg, reg_angle, prec, p, rec, density_th)
    return True, rec


def detect_line_segments(image, scale=0.8, sigma_scale=0.6, quant=2.0, ang_th=22.5, log_eps=0.0, density_th=0.7,
                         n_bins=1024):
    """lsd.detect_line_segments (lsdpython/lsd.pyx:17-18 defaults): image (H, W) gray values; returns (N, 7)
    float64 rows x1, y1, x2, y2, width, p, -log10(NFA)."""
    img = np.asarray(image, dtype=np.float64)
    prec = M_PI * ang_th / 180.0
    p = ang_th / 180.0
    rho = quant / math.sin(prec)
    if scale != 1.0:
        img = gaussian_sampler(img, scale, sigma_scale)
    Y, X = img.shape
    I = _Img()
    I.X, I.Y = X, Y
    I.ang, I.mod, seeds = ll_angle(img, rho, n_bins)
    I.used = [0] * (X * Y)
    logNT = 5.0 * (math.log10(float(X)) + math.log10(float(Y))) / 2.0 + math.log10(11.0)
    min_reg_size = int(-logNT / math.log10(p))
    out = []
    reg = []
    for s in seeds:
        if I.used[s] != 0:
            continue
        x, y = s % X, s // X
        reg_angle = region_grow(I, x, y, reg, prec)
        if len(reg) < min_reg_size:
            continue
        rec = region2rect(I, reg, reg_angle, prec, p)
        ok, rec = refine(I, reg, reg_angle, prec, p, rec, density_th)
        if not ok:
            continue
        log_nfa, rec = rect_improve(I, rec, logNT, log_eps)
        if log_nfa <= log_eps:
            continue
        x1, y1, x2, y2, w = rec["x1"] + 0.5, rec["y1"] + 0.5, rec["x2"] + 0.5, rec["y2"] + 0.5, rec["width"]
        if scale != 1.0:
            x1, y1, x2, y2, w = x1 / scale, y1 / scale, x2 / scale, y2 / scale, w / scale
        out.append((x1, y1, x2, y2, w, rec["p"], log_nfa))
    return np.array(out, dtype=np.float64).reshape(-1, 7)
