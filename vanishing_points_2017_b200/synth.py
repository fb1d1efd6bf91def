"""Seeded synthetic Manhattan scenes for the lines->VPs hot path.

The reference ships no datasets offline; BASELINE.json's configs are shapes
(YUD / ECD / HLW / stress).  This module generates line segments with the
coordinate frame of ``evaluation.detect_lsd_lines`` (reference
evaluation.py:233-249: centre origin, divided by max(w,h)/2, y up) and the
homogeneous lines of evaluation.py:158-168 (``l = [x1,y1,1] x [x2,y2,1]``).

Pure numpy, host side only; used identically by the oracle, the tests and
bench.py so both arms always see the same inputs.
"""
import numpy as np

CONFIGS = {
    # id: (name, n_images, N mean, N std, N min, N max, aspects)
    2: ("yud", 102, 500, 75, 250, 900, ((640, 480),)),
    3: ("ecd", 103, 1500, 300, 600, 3000,
        ((800, 600), (600, 800), (800, 533), (533, 800), (800, 450))),
    4: ("hlw", 2018, 800, 200, 200, 2000,
        ((800, 600), (600, 800), (800, 533), (533, 800), (800, 450))),
    5: ("stress", 10000, None, None, 200, 5000,
        ((800, 600), (600, 800), (800, 533), (533, 800), (800, 450))),
}


def _rot(yaw, pitch, roll):
    cy, sy = np.cos(yaw), np.sin(yaw)
    cp, sp = np.cos(pitch), np.sin(pitch)
    cr, sr = np.cos(roll), np.sin(roll)
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rx = np.array([[1, 0, 0], [0, cp, -sp], [0, sp, cp]])
    Rz = np.array([[cr, -sr, 0], [sr, cr, 0], [0, 0, 1]])
    return Rz @ Rx @ Ry


def make_scene(seed, n_segments, width=640, height=480, outlier_frac=0.15,
               noise_deg=0.5, extra_vps=0):
    """One synthetic image: returns dict(segments (N,4) f64, lines (N,3) f64,
    vps (K,3) unit z>=0, width, height)."""
    rs = np.random.RandomState(seed)
    yaw = rs.uniform(-np.pi, np.pi)
    pitch = rs.normal(0.0, np.deg2rad(10.0))
    roll = rs.normal(0.0, np.deg2rad(5.0))
    f = rs.uniform(0.8, 2.5)
    R = _rot(yaw, pitch, roll)
    K = np.diag([f, f, 1.0])
    vps = [K @ R[:, k] for k in range(3)]
    for _ in range(extra_vps):
        a = rs.uniform(-np.pi, np.pi)
        d = R @ np.array([np.cos(a), 0.0, np.sin(a)])
        vps.append(K @ d)
    vps = np.array(vps)
    vps /= np.linalg.norm(vps, axis=1, keepdims=True)
    vps[vps[:, 2] < 0] *= -1.0

    s = float(max(width, height))
    xr, yr = width / s, height / s
    N = int(n_segments)
    n_out = int(round(outlier_frac * N))
    n_in = N - n_out
    probs = np.array([0.4, 0.35, 0.25] + [0.0] * extra_vps)
    if extra_vps:
        probs = np.array([0.34, 0.3, 0.2] + [0.16 / extra_vps] * extra_vps)
    which = rs.choice(len(vps), size=n_in, p=probs / probs.sum())
    mid = np.stack([rs.uniform(-xr, xr, N), rs.uniform(-yr, yr, N)], axis=1)
    length = np.clip(np.exp(rs.normal(np.log(0.06), 0.6, N)), 0.02, 0.9)
    ang = np.empty(N)
    for n in range(n_in):
        v = vps[which[n]]
        # direction from the midpoint towards the (possibly infinite) VP
        d = v[0:2] - v[2] * mid[n]
        ang[n] = np.arctan2(d[1], d[0]) + np.deg2rad(noise_deg) * rs.normal()
    ang[n_in:] = rs.uniform(0.0, np.pi, n_out)
    half = 0.5 * length[:, None] * np.stack([np.cos(ang), np.sin(ang)], axis=1)
    seg = np.concatenate([mid - half, mid + half], axis=1)
    perm = rs.permutation(N)
    seg = np.ascontiguousarray(seg[perm])
    return {"segments": seg, "lines": lines_from_segments(seg), "vps": vps,
            "width": width, "height": height}


def lines_from_segments(seg):
    """evaluation.py:161-168: line = cross([x1,y1,1],[x2,y2,1]) (vectorised)."""
    seg = np.asarray(seg, dtype=np.float64)
    x1, y1, x2, y2 = seg[:, 0], seg[:, 1], seg[:, 2], seg[:, 3]
    return np.stack([y1 - y2, x2 - x1, x1 * y2 - y1 * x2], axis=1)


def _pixel_segments(sc, width, height):
    """make_scene's segments in pixels (inverse of evaluation.py:240-249)."""
    s = float(max(width, height))
    seg = sc["segments"].copy()
    seg[:, [0, 2]] = seg[:, [0, 2]] * (s / 2.0) + width / 2.0
    seg[:, [1, 3]] = -seg[:, [1, 3]] * (s / 2.0) + height / 2.0
    return seg


def _bars(seg, width, height, line_width):
    """(rows, cols, coverage) of every anti-aliased bar `line_width` px wide along seg (pixels); coverage falls off
    linearly over one pixel at the border.  Segments outside the image yield nothing."""
    hw = 0.5 * line_width
    for k, (x1, y1, x2, y2) in enumerate(seg):
        x0, x9 = int(max(np.floor(min(x1, x2) - hw - 1), 0)), int(min(np.ceil(max(x1, x2) + hw + 1), width - 1))
        y0, y9 = int(max(np.floor(min(y1, y2) - hw - 1), 0)), int(min(np.ceil(max(y1, y2) + hw + 1), height - 1))
        if x9 < x0 or y9 < y0:
            continue
        yy, xx = np.mgrid[y0:y9 + 1, x0:x9 + 1].astype(np.float64)
        dx, dy = x2 - x1, y2 - y1
        L2 = dx * dx + dy * dy
        t = np.clip(((xx - x1) * dx + (yy - y1) * dy) / max(L2, 1e-12), 0.0, 1.0)
        d = np.hypot(xx - (x1 + t * dx), yy - (y1 + t * dy))
        yield k, slice(y0, y9 + 1), slice(x0, x9 + 1), np.clip(hw + 0.5 - d, 0.0, 1.0)


def render_scene(seed, n_segments, width=640, height=480, noise_sigma=2.0, line_width=2.5):
    """A grayscale (height, width) float64 image of make_scene(seed, n_segments, width, height)'s segments: each is
    an anti-aliased bar `line_width` px wide (coverage falls off linearly over one pixel at its border) darker or
    brighter than a uniform background by a random contrast, plus Gaussian noise of `noise_sigma`, clipped to
    0..255.  Integer-valued (rounded), so the uint8 and float64 copies of it are the same image.  The LSD tests and
    tools/lsd_bench.py render their inputs here."""
    sc = make_scene(seed, n_segments, width, height)
    rs = np.random.RandomState(seed + 7919)
    seg = _pixel_segments(sc, width, height)
    img = np.full((height, width), rs.uniform(70.0, 180.0))
    contrast = rs.uniform(25.0, 70.0, seg.shape[0]) * rs.choice([-1.0, 1.0], seg.shape[0])
    for k, ys, xs, cov in _bars(seg, width, height, line_width):
        img[ys, xs] += contrast[k] * cov
    img += rs.normal(0.0, noise_sigma, img.shape)
    return np.clip(np.round(img), 0.0, 255.0)


def render_photo(seed, n_segments, width=2000, height=1333, noise_sigma=2.0, line_width=None):
    """An RGB (height, width, 3) uint8 photo of make_scene(seed, n_segments, width, height)'s segments:
    render_scene's bars (`line_width` defaults to 2.5 px per 640 px of the longer side, so the scene looks the same
    after resizing to 640) on a uniform background of a random colour, each bar with its own contrast per channel,
    plus independent Gaussian noise of `noise_sigma` per channel, rounded and clipped to 0..255.  The photo
    preparation tests and tools/image_prep_bench.py render their inputs here."""
    sc = make_scene(seed, n_segments, width, height)
    rs = np.random.RandomState(seed + 7927)
    if line_width is None:
        line_width = 2.5 * max(width, height) / 640.0
    seg = _pixel_segments(sc, width, height)
    img = np.empty((height, width, 3))
    img[:] = rs.uniform(70.0, 180.0, 3)
    contrast = rs.uniform(25.0, 70.0, (seg.shape[0], 3)) * rs.choice([-1.0, 1.0], (seg.shape[0], 1))
    for k, ys, xs, cov in _bars(seg, width, height, line_width):
        img[ys, xs, :] += cov[:, :, None] * contrast[k]
    img += rs.normal(0.0, noise_sigma, img.shape)
    return np.clip(np.round(img), 0.0, 255.0).astype(np.uint8)


def ideal_response(vps, grid=20, seed=0, peak=0.9, noise=0.05):
    """A CNN-like (grid,grid) response: `peak` at each true VP's cell,
    U(0,noise) elsewhere.  Row index <-> beta, column index <-> alpha, index 0
    = most negative angle (probability_functions.py:73-94 cell-centre means)."""
    rs = np.random.RandomState(seed)
    resp = rs.uniform(0.0, noise, (grid, grid))
    for v in vps:
        v = v / np.linalg.norm(v)
        if v[2] < 0:
            v = -v
        beta = np.arcsin(v[1])
        alpha = np.arcsin(np.clip(v[0] / np.cos(beta), -1, 1))
        a = int(np.clip(np.floor(alpha * grid / np.pi + grid / 2), 0, grid - 1))
        b = int(np.clip(np.floor(beta * grid / np.pi + grid / 2), 0, grid - 1))
        resp[b, a] = peak
    return resp


def config_sizes(cfg, n_images=None):
    """Per-image segment counts and (w,h) of BASELINE.json config `cfg`."""
    name, B, mu, sd, lo, hi, aspects = CONFIGS[cfg]
    if n_images is not None:
        B = n_images
    rs = np.random.RandomState(1_000_003 * cfg)
    if mu is None:
        n = np.exp(rs.uniform(np.log(lo), np.log(hi), B))
    else:
        n = rs.normal(mu, sd, B)
    n = np.clip(np.round(n), lo, hi).astype(np.int64)
    asp = [aspects[i] for i in rs.randint(0, len(aspects), B)]
    return n, asp


def make_batch(cfg, n_images=None, n_override=None):
    """Ragged batch for a config: returns dict(segments (sumN,4), lines
    (sumN,3), offsets (B+1,) int32, vps list, name)."""
    n, asp = config_sizes(cfg, n_images)
    if n_override is not None:
        n[:] = n_override
    segs, vps = [], []
    for idx in range(len(n)):
        sc = make_scene(1_000_003 * cfg + idx, int(n[idx]), asp[idx][0], asp[idx][1])
        segs.append(sc["segments"])
        vps.append(sc["vps"])
    offsets = np.zeros(len(n) + 1, dtype=np.int32)
    offsets[1:] = np.cumsum(n)
    seg = np.concatenate(segs, axis=0)
    return {"segments": seg, "lines": lines_from_segments(seg), "offsets": offsets,
            "vps": vps, "name": CONFIGS[cfg][0]}
