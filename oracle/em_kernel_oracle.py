"""ORACLE (test infrastructure, not product code) -- the EM's data-parallel kernels checked one by one.

em_pair, em_estep and em_wmat (csrc/em.cu) are each recomputed from the DEVICE'S OWN input to that kernel (the
buffers vpk_em_debug_fetch returns), so an error in one cannot hide behind, or be absorbed by, the kernels and the
discrete decisions after it.  Layouts (lsim_index, wt_index of csrc/em_core.cuh) are unpacked by
vanishing_points_2017_b200.vp_localisation; the packers here are their inverses, used by `emulate_*`.

u = 2^-53.  gamma(n) = n u / (1 - n u).  "LD" = numpy.longdouble (64-bit mantissa on x86: its own rounding is 2^11
times smaller than u, and every bound below keeps more than that as slack).

em_pair (reference: vp_oracle.calc_lsim(sigma=1) / line_rating_knn(k1=10, k2=4), what expectation_maximisation
passes, evaluated in LD)
  lsim    exactly symmetric with an exactly zero diagonal (the pair arithmetic is symmetric in its two segments and
          fmin / fmax / products commute, so any contraction the compiler picks is the same for (j, k) and (k, j));
          per element
              |dev - ref| <= prox (81 dc + 64 u) + cos9 dprox + u lsim
          * c = |cos| of the angle.  The device forms c from per-segment reciprocals: every component product and
            the norms carry a few roundings, so dc = 8 u (|a_x b_x| + |a_y b_y|) / (|a||b|) + 6 u c.
          * cos 9 theta = T9(c) (Chebyshev, evaluated as T3(T3(c))): |T9'(c)| <= 81 on the unclipped range
            c > cos(pi/18), which amplifies dc; the two Horner steps add at most 9 * 5 u + 5 u < 64 u absolute.
            The clip at c = cos(pi/18) is continuous (T9 = 0 there, the device returns cos(fl(pi/2)) = 6.1e-17 like
            the reference), so pairs on both sides of it are covered by the same 81 dc.
          * prox = exp(-x), x = d^2 h, h = 1 / (2 min(len)^2).  The squared distance cancels when the closest point
            is near the other segment: its error is absolute, |d(d^2)| <= 4 d D + D^2 + 3 u d^2 with
            D = 16 u S, S = the largest coordinate magnitude of the two segments plus both lengths and d; h has
            6 u.  So dx = h |d(d^2)| + 8 u x and dprox = prox (dx + 2 u) (exp: 1 ulp, the product 1 more).
  colsum  the four row-class partials and their sum add non-negative terms: |dev - sum_j lsim_dev[j, k]| <=
          gamma(N) colsum, in any order (the exact sum is taken in LD from the device's own lsim).
  lweight the kNN selection is discrete.  The reference ranks the candidates by (distance, index) and the chosen k2
          by (cosangle, later list position first), in LD; a line whose k1-th / (k1+1)-th distance or k2-th /
          (k2+1)-th cosangle differ by more than 0 and less than the two values' error bounds is a NEAR-TIE: it is
          listed and counted, not compared (exact ties are resolved by the same rule on both sides).  Otherwise
              |dev - ref| <= len / k2 * sum_sel (prox (81 dc + 8 u) + cos9 dprox + 2 u prox cos9) + 4 u lweight
          (the rating's cosangle is the reference's own acos / cos expression: libm's 2 ulp each, and the
          composite slope in c is again |T9'| <= 81).  The clip to [0.2, 1] is 1-Lipschitz.
em_estep (reference: probability_functions.calc_probabilities from the segments, the fetched lweight and the fetched
ESTEP constants vx, vy, inv2s, coef, pv, in LD)
  lvsq    q = 1 - |c| cancels, so the bound is absolute in c:
              |d lvsq| <= 2 q dc + dc^2 + 3 u lvsq,
              dc = 8 u (|a_x b_x| + |a_y b_y|) / (|a||b|) + 6 u |c| + 4 u (|m_x| + |m_y|) / |a|
          (a = midpoint - VP, b = the segment; the last term is the rounding of the midpoint m; rsqrt is 1 ulp).
  p(l|v)  rel <= |d lvsq| inv2s + 3 u lvsq inv2s + 4 u.
          exp's result below the normal range has an absolute error of a few subnormal ulps, TINY = 2^-1070, which
          the product with coef = 1 / sqrt(2 pi s) scales (by 1e6 and more for the small s of a tight hypothesis):
          |d p(l|v)| <= p(l|v) rel + TINY coef.
  p(v|l)  p(l) = max(sum_m p(l|v) pv, 1e-12): |d p(l)| <= sum_m |d p(l|v)| pv + gamma(M + 1) p(l) (positive terms,
          any order; the clamp is 1-Lipschitz); |d p(v|l)| <= |d p(l|v)| pv / p(l) + p(v|l) (rel(p(l)) + 4 u).  The
          clamp at 1e-12 multiplies the subnormal error by up to pv 1e12: measured on the B200, a fixed TINY on
          p(v|l) instead of TINY coef on p(l|v) was exceeded 2e4-fold at N = 3073.
  wt      == fl(pvl * lweight) BIT FOR BIT (one correctly rounded product), rows M .. of the last pass exactly 0.
  ESTEP   vx = vp0 / vp2, vy = vp1 / vp2, inv2s = 1 / (2 sigma), coef = 1 / sqrt(2 pi sigma) of the result's vp and
          sigma: correctly rounded operations in the same order, BIT FOR BIT.  pv against
          vp_oracle.calc_pdf(pdf_params(resp), calc_angles(vp)): a positive sum of exponentials, each exp(k d_i) with
          d_i = e_x^2 + e_y^2 a squared angle distance and |k| = 1 / (2 sigma_prior^2): rel_i = |k| dd_i + 4 u,
          dd_i = 2 (|e_x| (dx + 8 u) + |e_y| (dy + 8 u)) + 4 u d_i, where dx, dy are the angles' errors: asin and cos
          are 2 ulp each, amplified by asin's slope 1 / sqrt(1 - t^2), which is large for a VP far from the image
          (v2 -> 0, v0 / cos(beta) -> +-1: measured 2e-10 relative in pv at v2 ~ 1e-5, beyond a fixed 64 u); plus
          gamma(5 * 100 + 10) for the sums and the weight normalisation.
em_wmat (reference: acc = wt @ lsim in float64 from the fetched wt, lsim; w = (wt + b lw acc) / (1 + b lw colsum))
  wt >= 0 and lsim >= 0, so acc is a sum of non-negative terms and |d acc| <= gamma(N) acc for ANY summation tree,
  the FP64 tensor core's included; the reference's own float64 product obeys the same, so |dev - ref| of acc is
  within 2 gamma(N) acc.  Then
      |dev - ref| <= (b lw (2.01 gamma(N) acc + 4 u acc) + 2 u wt) / (1 + b lw colsum) + 6 u w + TINY.
  Rigorous, and a dropped 32-row chunk moves acc by orders of magnitude more.

`emulate_pair`, `emulate_estep`, `emulate_wmat` are float64 numpy emulations of the kernels in their device layouts
and summation orders (the reciprocal / Chebyshev forms, the four colsum partials, the per-group kNN lists, the eight
p(l) partials, 32-row chunks in two row halves of four k-steps, rank-ordered chunk ranges).  They pass every check;
the planted bugs (BUGS) are applied to them and each must fail its own kernel's check.
"""
import numpy as np

from oracle import vp_oracle as vo
from vanishing_points_2017_b200.synth import lines_from_segments
from vanishing_points_2017_b200.vp_localisation import lsim_index, unpack_lsim, unpack_wt, wpass_tiles, wt_index, wt_rows

U = 2.0 ** -53
TINY = 2.0 ** -1070
LD = np.longdouble
K1, K2 = 10, 4                       # line_rating_knn(k1=10, k2=4) as expectation_maximisation calls it (:230)
TK, JR, MP, MPS = 64, 32, 32, 36     # csrc/em_core.cuh kTK, em.cu kJR, em_core.cuh kMP, kMPS
CLIP_C = 0.984807753012208           # cos(pi / 18) as the device writes it
AT_CLIP = 6.123233995736766e-17      # cos(fl(pi / 2))

# planted bugs: name -> kernel whose check must fail
BUGS = {
    "lsim_unswizzled": "lsim", "prox_longer_segment": "lsim", "clip_0_99": "lsim", "colsum_drop_partial": "colsum",
    "knn_ties_larger_index": "lweight", "pl_seven_partials": "pvl", "pass1_reads_pass0": "w",
    "stale_rows": "w", "rank_range_off_by_one": "w", "wbias_twice": "w",
}


def gamma(n):
    return n * U / (1 - n * U)


def _worst(err, bound):
    """max err / bound; a NaN anywhere is a failure (inf)."""
    with np.errstate(over="ignore"):
        r = np.asarray(err / bound, np.float64)
    return float("inf") if np.isnan(r).any() else float(r.max(initial=0.0))


def wmat_split(N):
    """CTAs per slab of em_wmat (em.cu wmat_split)."""
    return 1 if N <= 1536 else (2 if N <= 3072 else 4)


def lsim_doubles(N):
    return (N + TK - 1) // TK * TK * N


def pack_lsim(L, swizzle=True):
    N = L.shape[0]
    raw = np.full(lsim_doubles(N), np.nan)
    j, k = np.meshgrid(np.arange(N), np.arange(N), indexing="ij")
    idx = lsim_index(N, j, k) if swizzle else ((k // TK) * N + j) * TK + k % TK
    raw[idx] = L
    return raw


def pack_wt(wt, N, M):
    """(wt_rows(M), N) -> WT buffer; the never-written 4 doubles per line (and the unused tail) are NaN."""
    raw = np.full((M + MP - 1) // MP * N * MPS, np.nan)
    m, n = np.meshgrid(np.arange(wt_rows(M)), np.arange(N), indexing="ij")
    raw[wt_index(N, n, m, M)] = wt
    return raw


# ---------------------------------------------------------------------------------------------------------------
# test scenes
# ---------------------------------------------------------------------------------------------------------------
def vp_scene(seed, N, M, width=800, height=600, jitter=1e-3):
    """N segments, every one on a line through one of M vanishing points (each VP gets N // M or more, shuffled),
    turned by up to `jitter` rad about its midpoint.  Given as init_vp with do_iterations / do_merge / do_split off
    and num_min_lines = 0, every hypothesis keeps its own lines, so the last superstep runs on M hypotheses."""
    rs = np.random.RandomState(seed)
    # far VPs in directions pi / M apart (as seen from the image): no line is close to a second VP's direction
    th = np.pi * (np.arange(M) + rs.uniform(0.3, 0.7, M)) / max(M, 1)
    r = 10.0 ** rs.uniform(4.3, 6.0, M)
    vps = np.stack([0.5 * width + r * np.cos(th), 0.5 * height + r * np.sin(th), np.ones(M)], 1)
    owner = rs.permutation(np.arange(N) % max(M, 1))
    mid = np.stack([rs.uniform(0, width, N), rs.uniform(0, height, N)], 1)
    d = vps[owner, :2] - mid
    ang = np.arctan2(d[:, 1], d[:, 0]) + rs.uniform(-jitter, jitter, N)
    half = 0.5 * rs.uniform(15, 70, N)
    e = np.stack([np.cos(ang), np.sin(ang)], 1) * half[:, None]
    seg = np.concatenate([mid - e, mid + e], 1)
    v = vps / np.linalg.norm(vps, axis=1, keepdims=True)
    return {"segments": seg, "lines": lines_from_segments(seg), "vps": v}


def tie_scene(seed, N):
    """axis-parallel segments on a 3-pixel lattice, one in eight an exact duplicate: distances and cosangles tie
    exactly (in float64 as in LD), so the kNN ranking rests on its index rules alone."""
    rs = np.random.RandomState(seed)
    n0 = N - N // 8
    p = rs.randint(0, 40, (n0, 2)).astype(np.float64) * 3
    d = np.array([[1, 0], [0, 1]], np.float64)[rs.randint(0, 2, n0)] * rs.randint(2, 6, n0)[:, None] * 3
    seg = np.concatenate([p, p + d], 1)
    seg = np.concatenate([seg, seg[rs.randint(0, n0, N - n0)]])[rs.permutation(N)]
    return {"segments": seg, "lines": lines_from_segments(seg)}


# ---------------------------------------------------------------------------------------------------------------
# em_pair
# ---------------------------------------------------------------------------------------------------------------
def _pair_terms(lp, rows):
    """LD reference terms and device error bounds of the pairs (rows x all columns)."""
    A, B = lp[rows].astype(LD), lp.astype(LD)
    d = vo.segment_distance(A, B)
    v1x, v1y = (A[:, 0] - A[:, 2])[:, None], (A[:, 1] - A[:, 3])[:, None]
    v2x, v2y = (B[:, 0] - B[:, 2])[None, :], (B[:, 1] - B[:, 3])[None, :]
    n1, n2 = np.sqrt(v1x * v1x + v1y * v1y), np.sqrt(v2x * v2x + v2y * v2y)
    c = np.minimum(np.abs((v1x * v2x + v1y * v2y) / (n1 * n2)), LD(1))
    th9 = 9 * np.arccos(c)
    cos9 = np.where(th9 < np.pi / LD(2), np.cos(th9), LD(AT_CLIP))
    ln = np.minimum(n1, n2)
    h = 1 / (2 * ln * ln)
    x = d * d * h
    prox = np.exp(-x)
    dc = 8 * U * (np.abs(v1x * v2x) + np.abs(v1y * v2y)) / (n1 * n2) + 6 * U * c
    S = np.maximum(np.abs(A).max(1)[:, None], np.abs(B).max(1)[None, :]) + n1 + n2 + d
    D = 16 * U * S
    dd2 = 4 * d * D + D * D + 3 * U * d * d
    dprox = prox * (h * dd2 + 8 * U * x + 2 * U)
    return {"d": d, "dd2": dd2, "c": c, "dc": dc, "cos9": cos9, "prox": prox, "dprox": dprox}


def sample_rows(N, limit, seed=0):
    """all rows up to `limit`, else a seeded sample that keeps the first / last row of every 64-row slab."""
    if N <= limit:
        return np.arange(N)
    edges = np.unique(np.concatenate([np.arange(0, N, TK), np.minimum(np.arange(TK - 1, N + TK - 1, TK), N - 1)]))
    rs = np.random.RandomState(seed)
    extra = rs.choice(N, max(limit - edges.size, 0), replace=False)
    return np.unique(np.concatenate([edges[:limit], extra]))


def check_lsim(lp, L, rows):
    """L: the device's (N, N) lsim -> max |dev - ref| / bound over `rows`."""
    t = _pair_terms(lp, rows)
    ref = t["cos9"] * t["prox"]
    ref[np.arange(rows.size), rows] = 0
    bound = t["prox"] * (81 * t["dc"] + 64 * U) + t["cos9"] * t["dprox"] + U * ref + TINY
    return _worst(np.abs(L[rows].astype(LD) - ref), bound)


def assert_lsim_exact(L):
    assert np.array_equal(L, L.T), "lsim is not exactly symmetric"
    assert np.all(np.diag(L) == 0.0), "lsim diagonal is not exactly zero"


def check_colsum(L, colsum):
    exact = np.sum(L.astype(LD), axis=0)
    bound = gamma(L.shape[0]) * exact + TINY
    return _worst(np.abs(colsum.astype(LD) - exact), bound)


def check_lweight(lp, lweight, rows):
    """-> (max ratio over the lines without a near-tie, list of near-tie lines)."""
    N = lp.shape[0]
    t = _pair_terms(lp, rows)
    k1, k2 = min(K1, N), min(K2, N)
    seglen = vo.seg_length(lp.astype(LD))
    worst, ties = 0.0, []
    for r, i in enumerate(rows):
        d = t["d"][r].copy()
        d[i] = 4
        d2 = d * d
        order = np.lexsort((np.arange(N), d2))
        near = order[:k1]
        tie = False
        if k1 < N:
            a, b = order[k1 - 1], order[k1]
            gap = d2[b] - d2[a]
            tie |= 0 < gap <= t["dd2"][r][a] + t["dd2"][r][b]
        cosv = t["cos9"][r][near]
        ecos = 81 * t["dc"][r][near] + 8 * U
        # argsort()[::-1] of the reference: largest first, of equal values the later list position first
        pos = np.arange(near.size)
        sel = np.lexsort((-pos, -cosv))
        if k2 < near.size:
            a, b = sel[k2 - 1], sel[k2]
            gap = cosv[a] - cosv[b]
            tie |= 0 < gap <= ecos[a] + ecos[b]
        if tie:
            ties.append(int(i))
            continue
        best = sel[:k2]
        j = near[best]
        prox = t["prox"][r][j].copy()
        dprox = t["dprox"][r][j].copy()
        prox[j == i], dprox[j == i] = 1, 0
        score = np.sum(prox * cosv[best]) / k2
        ref = seglen[i] * np.clip(score, LD(0.2), LD(1))
        bound = seglen[i] / k2 * np.sum(prox * ecos[best] + cosv[best] * dprox + 2 * U * prox * cosv[best]) + 4 * U * ref + TINY
        worst = max(worst, _worst(abs(LD(lweight[i]) - ref), bound))
    return worst, ties


def _segpre(lp):
    x1, y1, x2, y2 = lp.T
    dx, dy = x2 - x1, y2 - y1
    nrm = np.sqrt(dx * dx + dy * dy)
    return {"x1": x1, "y1": y1, "x2": x2, "y2": y2, "dx": dx, "dy": dy, "inv_nn": 1.0 / (nrm * nrm),
            "inv_len": 1.0 / nrm, "h": 1.0 / (2 * nrm * nrm)}


def _psd2_pre(s, px, py):
    """psd2_pre of segments s (column vectors) to points (row vectors)."""
    param = ((px - s["x1"]) * s["dx"] + (py - s["y1"]) * s["dy"]) * s["inv_nn"]
    cx, cy = s["x1"] + param * s["dx"], s["y1"] + param * s["dy"]
    cx, cy = np.where(param > 1, s["x2"], cx), np.where(param > 1, s["y2"], cy)
    cx, cy = np.where(param < 0, s["x1"], cx), np.where(param < 0, s["y1"], cy)
    ex, ey = cx - px, cy - py
    return ex * ex + ey * ey


def _cosangle_reference_order(a, b):
    v1x, v1y, v2x, v2y = a[0] - a[2], a[1] - a[3], b[..., 0] - b[..., 2], b[..., 1] - b[..., 3]
    c = np.abs((v1x * v2x + v1y * v2y) / (np.sqrt(v1x * v1x + v1y * v1y) * np.sqrt(v2x * v2x + v2y * v2y)))
    dphi = np.abs(np.arccos(np.clip(c, -1.0, 1.0)))
    return np.cos(np.clip(9.0 * dphi, -0.5 * np.pi, 0.5 * np.pi))


def emulate_pair(lp, bug=None):
    """em_pair in float64 -> (LSIM buffer, colsum, lweight)."""
    N = lp.shape[0]
    P = _segpre(lp)
    col = {k: v[None, :] for k, v in P.items()}           # segment k (column)
    row = {k: v[:, None] for k, v in P.items()}           # segment j (row)
    with np.errstate(all="ignore"):
        d2 = np.fmin(np.fmin(_psd2_pre(row, col["x1"], col["y1"]), _psd2_pre(row, col["x2"], col["y2"])),
                     np.fmin(_psd2_pre(col, row["x1"], row["y1"]), _psd2_pre(col, row["x2"], row["y2"])))
        c = np.abs((row["dx"] * col["dx"] + row["dy"] * col["dy"]) * (row["inv_len"] * col["inv_len"]))
        c = np.where(c > 1.0, 1.0, c)
        t = c * (4.0 * c * c - 3.0)
        r = t * (4.0 * t * t - 3.0)
        r = np.where(r < AT_CLIP, AT_CLIP, r)
        cos9 = np.where(c <= (0.99 if bug == "clip_0_99" else CLIP_C), AT_CLIP, r)
        hh = np.fmin(row["h"], col["h"]) if bug == "prox_longer_segment" else np.fmax(row["h"], col["h"])
        L = cos9 * np.exp(-(d2 * hh))
    np.fill_diagonal(L, 0.0)
    np.fill_diagonal(d2, 16.0)
    # colsum: four partials, rows j = g (mod 4) ascending, added in group order
    part = np.zeros((4, N))
    for j in range(N):
        part[j % 4] += L[j]
    colsum = 0.0 + part[0]
    for g in range(1, 4):
        if not (bug == "colsum_drop_partial" and g == 3):
            colsum = colsum + part[g]
    # kNN: the k1 nearest by (squared distance, index), then rate_line
    key = np.where(np.isnan(d2), np.inf, d2)
    lweight = np.empty(N)
    k2 = min(K2, N)
    for k in range(N):
        idx = np.arange(N)
        order = np.lexsort((-idx if bug == "knn_ties_larger_index" else idx, key[:, k]))[:min(K1, N)]
        cc = _cosangle_reference_order(lp[k], lp[order])
        d2t = np.where(order == k, 0.0, key[order, k])
        px = np.exp(-(d2t * np.fmax(P["h"][k], P["h"][order])))
        cv = np.where(np.isnan(cc), -np.inf, cc)
        score = 0.0
        for _ in range(k2):
            who = 0
            for q in range(1, cv.size):
                if cv[q] >= cv[who]:
                    who = q
            score += px[who] * cv[who]
            cv[who] = -np.inf
        score /= k2
        ls = min(max(score, 0.2), 1.0)
        dx, dy = lp[k, 0] - lp[k, 2], lp[k, 1] - lp[k, 3]
        lweight[k] = np.sqrt(dx * dx + dy * dy) * ls
    return pack_lsim(L, swizzle=bug != "lsim_unswizzled"), colsum, lweight


# ---------------------------------------------------------------------------------------------------------------
# em_estep
# ---------------------------------------------------------------------------------------------------------------
def estep_constants(vp, sigma, pv):
    """the slot's E-step constants as prepare_estep forms them from the result's vp / sigma (pv given)."""
    s = np.maximum(sigma, 1e-200)
    return {"pv": np.asarray(pv, np.float64), "vx": vp[:, 0] / vp[:, 2], "vy": vp[:, 1] / vp[:, 2],
            "inv2s": 1.0 / (2.0 * s), "coef": 1.0 / np.sqrt(2.0 * np.pi * s)}


def check_estep_constants(est, vp, sigma, resp):
    """vx, vy, inv2s, coef bit for bit; -> max |pv - calc_pdf| / bound."""
    want = estep_constants(vp, sigma, est["pv"])
    for k in ("vx", "vy", "inv2s", "coef"):
        assert np.array_equal(est[k], want[k]), k
    par = vo.pdf_params(np.array(resp, np.float64))
    ang = vo.calc_angles(vp)
    x, y = ang[:, 0], ang[:, 1]
    ref = vo.calc_pdf(par, x, y)
    # the angles' errors: asin / cos are 2 ulp each, amplified by asin's slope 1 / sqrt(1 - t^2) (a VP far from the
    # image has v2 -> 0 and v0 / cos(beta) -> +-1)
    v1 = np.abs(vp[:, 1])
    dy = 2 * U * v1 / np.sqrt(np.maximum(1 - v1 * v1, U)) + 2 * U * np.abs(y)
    inner = np.abs(np.clip(vp[:, 0] / np.cos(y), -1, 1))
    dinner = inner * (3 * U + np.abs(np.tan(y)) * dy)
    dx = dinner / np.sqrt(np.maximum(1 - inner * inner, dinner)) + 2 * U * np.abs(x)
    k = 0.5 / (par.sigma * par.sigma)
    PI = np.pi
    err = np.zeros_like(ref)
    for n in np.nonzero(par.weights > 0)[0]:
        mx, my = par.means[n]
        for ex, ey in (((x - mx), (y - my)), ((x - mx + PI), (y + my)), ((x - mx - PI), (y + my)),
                       ((x + mx), (y - my - PI)), ((x + mx), (y - my - PI))):
            di = ex * ex + ey * ey
            ddi = 2 * (np.abs(ex) * (dx + 8 * U) + np.abs(ey) * (dy + 8 * U)) + 4 * U * di
            err += par.weights[n] * np.exp(-k * di) * (k * ddi + 4 * U)
    bound = err + gamma(5 * 100 + 10) * ref + TINY
    return _worst(np.abs(est["pv"] - ref), bound)


def ref_estep(lp, lweight, est):
    """LD lvsq and p(v|l) (M, N) with their bounds."""
    E = {k: np.asarray(v, np.float64).astype(LD)[:, None] for k, v in est.items()}
    A = lp.astype(LD)
    mx, my = ((A[:, 0] + A[:, 2]) / 2)[None, :], ((A[:, 1] + A[:, 3]) / 2)[None, :]
    bx, by = (A[:, 0] - A[:, 2])[None, :], (A[:, 1] - A[:, 3])[None, :]
    ax, ay = mx - E["vx"], my - E["vy"]
    na, nb = np.sqrt(ax * ax + ay * ay), np.sqrt(bx * bx + by * by)
    c = (ax * bx + ay * by) / (na * nb)
    q = 1 - np.abs(c)
    lvsq = q * q
    dc = 8 * U * (np.abs(ax * bx) + np.abs(ay * by)) / (na * nb) + 6 * U * np.abs(c) + 4 * U * (np.abs(mx) + np.abs(my)) / na
    dl = 2 * q * dc + dc * dc + 3 * U * lvsq
    plv = np.exp(-(lvsq * E["inv2s"])) * E["coef"]
    rel = dl * E["inv2s"] + 3 * U * lvsq * E["inv2s"] + 4 * U
    M = lvsq.shape[0]
    eplv = plv * rel + TINY * E["coef"]            # exp's result below the normal range, then scaled by coef
    terms = plv * E["pv"]
    pl = np.maximum(np.sum(terms, axis=0), LD(1e-12))[None, :]
    rel_pl = (np.sum(eplv * E["pv"], axis=0)[None, :] + TINY) / pl + gamma(M + 1)
    pvl = terms / pl
    bpvl = eplv * E["pv"] / pl + pvl * (rel_pl + 4 * U) + TINY
    return {"lvsq": lvsq, "b_lvsq": dl + TINY, "pvl": pvl, "b_pvl": bpvl}


def assert_wt_exact(wt, pvl, lweight):
    M, N = pvl.shape
    want = np.zeros((wt_rows(M), N))
    want[:M] = pvl * lweight[None, :]
    assert np.array_equal(wt, want), "wt != fl(pvl * lweight) or padding rows not zero"


def check_estep(lp, lweight, est, lvsq, pvl):
    """-> {"lvsq": ratio, "pvl": ratio}."""
    M, N = lvsq.shape
    if M == 0:
        return {"lvsq": 0.0, "pvl": 0.0}
    r = ref_estep(lp, lweight, est)
    return {"lvsq": _worst(np.abs(lvsq.astype(LD) - r["lvsq"]), r["b_lvsq"]),
            "pvl": _worst(np.abs(pvl.astype(LD) - r["pvl"]), r["b_pvl"])}


def emulate_estep(lp, lweight, est, bug=None):
    """em_estep in float64 -> (lvsq, pvl, WT buffer)."""
    M, N = est["pv"].size, lp.shape[0]
    x1, y1, x2, y2 = lp.T
    mx, my, bx, by = 0.5 * (x1 + x2), 0.5 * (y1 + y2), x1 - x2, y1 - y2
    inv_nb = 1.0 / np.sqrt(bx * bx + by * by)
    lvsq, plv = np.empty((M, N)), np.empty((M, N))
    part = np.zeros((8, N))
    with np.errstate(under="ignore"):
        for m in range(M):
            ax, ay = mx - est["vx"][m], my - est["vy"][m]
            c = (ax * bx + ay * by) * ((1.0 / np.sqrt(ax * ax + ay * ay)) * inv_nb)
            q = 1.0 - np.abs(c)
            lvsq[m] = q * q
            plv[m] = np.exp(-(lvsq[m] * est["inv2s"][m])) * est["coef"][m]
            part[m % 8] += plv[m] * est["pv"][m]
        pl = np.zeros(N)
        for w in range(7 if bug == "pl_seven_partials" else 8):
            pl = pl + part[w]
        pl = np.where(pl < 1e-12, 1e-12, pl)
        pvl = plv * est["pv"][:, None] * (1.0 / pl)[None, :]
    wt = np.zeros((wt_rows(M), N))
    wt[:M] = pvl * lweight[None, :]
    return lvsq, pvl, pack_wt(wt, N, M)


# ---------------------------------------------------------------------------------------------------------------
# em_wmat
# ---------------------------------------------------------------------------------------------------------------
def check_w(wt, L, lweight, colsum, w, wbias, use_weights=True):
    """wt: dense (wt_rows, N); L: (N, N) or None without weights.  -> max |dev - ref| / bound."""
    M, N = w.shape
    if M == 0:
        return 0.0
    a = wt[:M]
    acc = a @ L if use_weights else np.zeros((M, N))
    tl = wbias * lweight[None, :]
    den = 1 + tl * colsum[None, :]
    ref = (a + tl * acc) / den
    bound = (tl * (2.01 * gamma(N) * acc + 4 * U * acc) + 2 * U * a) / den + 6 * U * ref + TINY
    return _worst(np.abs(w - ref), bound)


def emulate_wmat(wt_raw, lsim_raw, lweight, colsum, N, M, wbias, use_weights=True, bug=None):
    """em_wmat in float64 -> w (M, N)."""
    L = unpack_lsim(lsim_raw, N) if use_weights else None
    nch = (N + JR - 1) // JR
    cs = wmat_split(N)
    ranges = [(nch * r // cs, nch * (r + 1) // cs) for r in range(cs)] if use_weights else [(0, 0)]
    if bug == "rank_range_off_by_one" and cs > 1:
        ranges[1] = (ranges[1][0] + 1, ranges[1][1])
    bias = wbias * wbias if bug == "wbias_twice" else wbias
    w = np.empty((M, N))
    for p in range((M + MP - 1) // MP):
        mt = wpass_tiles(M, p)
        ws = 8 * mt + 4
        base = 0 if bug == "pass1_reads_pass0" else p * N * MPS
        A = wt_raw[base + np.arange(N)[:, None] * ws + np.arange(8 * mt)[None, :]]      # (N, rows of the pass)
        total = None
        for c0, c1 in ranges:
            halves = [np.zeros((8 * mt, N)), np.zeros((8 * mt, N))]
            for ch in range(c0, c1):
                j0 = ch * JR
                jn = min(JR, N - j0)
                for hf in range(2):
                    for ks in range(JR // 8):
                        j = j0 + (JR // 2) * hf + 4 * ks + np.arange(4)
                        ok = j < j0 + jn
                        if bug == "stale_rows" and j0 >= JR:
                            src = np.where(ok, j, j - JR)
                            a4, l4 = A[src], L[src]
                        else:
                            jj = np.minimum(j, N - 1)
                            a4, l4 = np.where(ok[:, None], A[jj], 0.0), np.where(ok[:, None], L[jj], 0.0)
                        halves[hf] += a4.T @ l4
            part = halves[0] + halves[1]
            total = part if total is None else total + part
        m = p * MP + np.arange(8 * mt)
        keep = m < M
        a = A[:, :8 * mt].T
        tl = bias * lweight[None, :]
        w[m[keep]] = ((a + tl * total) / (1 + tl * colsum[None, :]))[keep]
    return w


def emulate(lp, est, wbias=1.0, use_weights=True, bug=None):
    """all three kernels -> the buffers vpk_em_debug_fetch returns (dense where the wrapper unpacks)."""
    N, M = lp.shape[0], est["pv"].size
    if use_weights:
        lsim_raw, colsum, lweight = emulate_pair(lp, bug)
    else:
        lsim_raw, colsum, lweight = np.full(lsim_doubles(N), np.nan), np.zeros(N), np.ones(N)
    lvsq, pvl, wt_raw = emulate_estep(lp, lweight, est, bug)
    w = emulate_wmat(wt_raw, lsim_raw, lweight, colsum, N, M, wbias, use_weights, bug)
    return {"lsim": unpack_lsim(lsim_raw, N), "colsum": colsum, "lweight": lweight, "lvsq": lvsq, "pvl": pvl,
            "wt": unpack_wt(wt_raw, N, M), "w": w, "estep": est}


def check_all(lp, buf, wbias=1.0, use_weights=True, row_limit=1100, seed=0, exact=True):
    """every check on a set of fetched (or emulated) buffers -> {kernel check: worst ratio}, near-tie lines.
    exact: also assert the bit-exact properties (lsim symmetric with zero diagonal, wt)."""
    N = lp.shape[0]
    out, ties = {}, []
    rows = sample_rows(N, row_limit, seed)
    if use_weights:
        if exact:
            assert_lsim_exact(buf["lsim"])
        out["lsim"] = check_lsim(lp, buf["lsim"], rows)
        out["colsum"] = check_colsum(buf["lsim"], buf["colsum"])
        out["lweight"], ties = check_lweight(lp, buf["lweight"], rows)
    else:
        assert np.all(buf["colsum"] == 0.0) and np.all(buf["lweight"] == 1.0)
    if "w" in buf:
        if exact:
            assert_wt_exact(buf["wt"], buf["pvl"], buf["lweight"])
        out.update(check_estep(lp, buf["lweight"], buf["estep"], buf["lvsq"], buf["pvl"]))
        out["w"] = check_w(buf["wt"], buf["lsim"] if use_weights else None, buf["lweight"], buf["colsum"], buf["w"],
                           wbias, use_weights)
    return out, ties
