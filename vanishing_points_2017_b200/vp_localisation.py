"""Drop-in for the reference's vp_localisation.expectation_maximisation
(stage 3) on the B200.

Same positional order, keyword names, defaults and result-dict keys as
reference vp_localisation.py:168-172 / :441-442; a failed image returns the
reference's skeleton dict of None (:205-206).  The whole EM (pair similarity,
kNN line rating, E/M steps, split, merge, final refit) runs inside one
persistent CUDA kernel behind libvpk.so's C ABI (`vpk_em`).
"""
import collections
import ctypes as C

import numpy as np

from . import _lib

# the reference's probability_functions.PDF (probability_functions.py:5): type of result['distribution']
PDF = collections.namedtuple("PDF", "v lv vl l lvsq angles")


def em_distribution(image, n_vp, n_lines, ctx=None):
    """result['distribution'] of image `image` of the LAST EM call on `ctx` (vp_localisation.py:441-442): evaluated on
    the device from the planes of the last E-step (`vpk_em_distribution`); ask before the next EM call."""
    ctx = ctx or _lib.default_context()
    M, N = int(n_vp), int(n_lines)
    a = {"v": np.empty(M), "lv": np.empty((N, M)), "vl": np.empty((M, N)), "l": np.empty(N), "lvsq": np.empty((N, M)),
         "angles": np.empty((M, 2))}
    _lib.check(ctx.lib.vpk_em_distribution(ctx.h, int(image), M, N, _lib.ptr(a["v"]), _lib.ptr(a["lv"]), _lib.ptr(a["vl"]),
                                           _lib.ptr(a["l"]), _lib.ptr(a["lvsq"]), _lib.ptr(a["angles"])), "vpk_em_distribution")
    return PDF(**a)


# vpk_em_debug_fetch buffer names (include/vpk.h, VPK_EM_BUF_*)
EM_BUFFERS = ["lsim", "colsum", "lweight", "lvsq", "pvl", "w", "wt", "estep"]
_TK, _MP, _MPS = 64, 32, 36          # csrc/em_core.cuh kTK, kMP, kMPS


def lsim_index(N, j, k):
    """csrc/em_core.cuh lsim_index: 64-column slabs of N x 64, the column XOR-swizzled with bits 0-1 of the row."""
    j, k = np.asarray(j, np.int64), np.asarray(k, np.int64)
    return ((k // _TK) * N + j) * _TK + ((k % _TK) ^ ((j & 3) << 2))


def wpass_tiles(M, p):
    """csrc/em_core.cuh wpass_tiles: 8-row tiles of pass p (VP rows 32p .. 32p+31) for M hypotheses."""
    return (min(max(M - p * _MP, 1), _MP) + 7) // 8


def wt_index(N, n, m, M):
    """csrc/em_core.cuh wt_index: pass p = m // 32 at p*N*36, line n of the pass at stride 8 * tiles + 4."""
    n, m = np.asarray(n, np.int64), np.asarray(m, np.int64)
    p = m // _MP
    stride = np.array([8 * wpass_tiles(M, q) + 4 for q in range(int(p.max(initial=0)) + 1)], np.int64)[p]
    return p * N * _MPS + n * stride + m % _MP


def wt_rows(M):
    """rows of the W operand for M hypotheses: every pass but the last has 32, the last 8 * its tiles."""
    passes = (M + _MP - 1) // _MP
    return 0 if M == 0 else _MP * (passes - 1) + 8 * wpass_tiles(M, passes - 1)


def unpack_lsim(raw, N):
    """(N, N) similarity matrix from the LSIM buffer."""
    j, k = np.meshgrid(np.arange(N), np.arange(N), indexing="ij")
    return raw[lsim_index(N, j, k)]


def unpack_wt(raw, N, M):
    """(wt_rows(M), N) W operand from the WT buffer: rows M .. of the last pass are its zero padding."""
    m, n = np.meshgrid(np.arange(wt_rows(M)), np.arange(N), indexing="ij")
    return raw[wt_index(N, n, m, M)] if m.size else np.zeros((wt_rows(M), N))


def _em_fetch_raw(ctx, image, which):
    n = C.c_int64(0)
    _lib.check(ctx.lib.vpk_em_debug_fetch(ctx.h, int(image), int(which), None, 0, C.byref(n)), "vpk_em_debug_fetch")
    out = np.empty(n.value)
    _lib.check(ctx.lib.vpk_em_debug_fetch(ctx.h, int(image), int(which), _lib.ptr(out), out.size, None), "vpk_em_debug_fetch")
    return out


def em_debug_fetch(image, name, ctx=None, raw=False):
    """Buffer `name` (EM_BUFFERS) of image `image`'s EM workspace as the LAST EM call on `ctx` left it
    (`vpk_em_debug_fetch`, diagnostics).  raw=True: the device layout; otherwise dense arrays: lsim (N, N),
    colsum / lweight (N), lvsq / pvl / w (M, N), wt (wt_rows(M), N), estep a dict of pv, vx, vy, inv2s, coef (M)."""
    ctx = ctx or _lib.default_context()
    out = _em_fetch_raw(ctx, image, EM_BUFFERS.index(name))
    if raw or name in ("colsum", "lweight"):
        return out
    if name == "estep":
        return dict(zip(("pv", "vx", "vy", "inv2s", "coef"), out.reshape(5, -1)))
    N = _em_fetch_raw(ctx, image, EM_BUFFERS.index("colsum")).size
    if name == "lsim":
        return unpack_lsim(out, N)
    M = _em_fetch_raw(ctx, image, EM_BUFFERS.index("estep")).size // 5
    return unpack_wt(out, N, M) if name == "wt" else out.reshape(M, N)


_SKELETON = {"vp_assoc": None, "vp": None, "counts": None, "count_id": None, "decision_metric": None,
             "iterations": 0}


def _alloc_result(B, sumN, want_dm):
    M = _lib.VPK_MAX_VP
    arrs = {
        # every entry the caller reads is written by the library (rows beyond n_vp are never read)
        "status": np.empty(B, np.int32), "n_vp": np.empty(B, np.int32), "iterations": np.empty(B, np.int32),
        "vp": np.empty((B, M, 3), np.float64), "sigma": np.empty((B, M), np.float64),
        "counts": np.empty((B, M), np.int32), "counts_weighted": np.empty((B, M), np.float64),
        "vp_assoc": np.empty(max(sumN, 1), np.int32),
        "decision_metric": np.zeros(max(M * sumN, 1), np.float64) if want_dm else None,
    }
    res = _lib.EmResult()
    for k, a in arrs.items():
        setattr(res, k, None if a is None else a.ctypes.data)
    return arrs, res


def unpack_results(arrs, offsets):
    """Per-image reference-style dicts from the flat result arrays."""
    out = []
    M = _lib.VPK_MAX_VP
    for b in range(len(offsets) - 1):
        if arrs["status"][b] != _lib.EM_OK:
            d = dict(_SKELETON)
            d["status"] = int(arrs["status"][b])
            out.append(d)
            continue
        m = int(arrs["n_vp"][b])
        o0, o1 = int(offsets[b]), int(offsets[b + 1])
        dm = None
        if arrs.get("decision_metric") is not None:
            dm = arrs["decision_metric"][M * o0:M * o0 + m * (o1 - o0)].reshape(m, o1 - o0).copy()
        out.append({"vp_assoc": arrs["vp_assoc"][o0:o1].astype(np.int64), "vp": arrs["vp"][b, :m].copy(),
                    "counts": arrs["counts"][b, :m].astype(np.float64),
                    "counts_weighted": arrs["counts_weighted"][b, :m].copy(), "count_id": None,
                    "decision_metric": dm, "iterations": int(arrs["iterations"][b]),
                    "sigma": arrs["sigma"][b, :m].copy(), "status": 0})
    return out


def expectation_maximisation_batch(lines, segments, offsets, responses, sphere_images, init_vp=None,
                                   init_vp_offsets=None, want_decision_metric=False, ctx=None, **kwargs):
    """Ragged batch form: lines (sumN,3), segments (sumN,4), offsets (B+1),
    responses (B,20,20), sphere_images (B,S,S) uint8 -> list of result dicts."""
    ctx = ctx or _lib.default_context()
    dm = kwargs.pop("distance_measure", "angle")
    if dm != "angle":
        if dm in ("dotprod", "area"):
            raise NotImplementedError("only distance_measure='angle' (the value every reference caller passes: "
                                      "example.py:28, benchmark.py:51) is built")
        assert False        # vp_localisation.py:203
    cfg = _lib.em_config(**{k: (int(v) if isinstance(v, (bool, np.bool_)) else v) for k, v in kwargs.items()})
    lines = _lib.as_f64(lines, 3)
    segments = _lib.as_f64(segments, 4)
    off = _lib.as_offsets(offsets)
    B = off.size - 1
    if off[-1] != lines.shape[0] or lines.shape[0] != segments.shape[0]:
        raise ValueError("offsets / lines / segments disagree")
    resp = np.ascontiguousarray(responses, dtype=np.float64).reshape(B, _lib.VPK_GRID, _lib.VPK_GRID)
    sph = None
    S = 1
    if sphere_images is not None:
        sph = np.ascontiguousarray(sphere_images, dtype=np.uint8)
        sph = sph.reshape(B, sph.shape[-2], sph.shape[-1])
        if sph.shape[1] != sph.shape[2]:
            raise ValueError("sphere images must be square")
        S = sph.shape[1]
    iv = ioff = None
    if init_vp is not None:
        iv = _lib.as_f64(init_vp, 3)
        if init_vp_offsets is None and B != 1:
            raise ValueError("init_vp for a batch of %d images needs init_vp_offsets (B + 1 entries)" % B)
        ioff = _lib.as_offsets(init_vp_offsets if init_vp_offsets is not None else [0, iv.shape[0]])
        if ioff.size != B + 1 or ioff[-1] != iv.shape[0]:
            raise ValueError("init_vp_offsets must have B + 1 = %d entries ending at %d, got %r" % (B + 1, iv.shape[0], ioff))
    arrs, res = _alloc_result(B, int(off[-1]), want_decision_metric)
    _lib.check(ctx.lib.vpk_em(ctx.h, _lib.ptr(lines), _lib.ptr(segments), _lib.ptr(off), B, _lib.ptr(resp),
                              _lib.ptr(sph), S, _lib.ptr(iv), _lib.ptr(ioff), C.byref(cfg), C.byref(res)),
               "vpk_em")
    return unpack_results(arrs, off)


def expectation_maximisation(l, lp, cnn_response, num_iter=100, sphere_image=None,
                             init_vp=None, do_merge=True, do_split=True, do_iterations=True,
                             distance_measure="angle", use_weights=True, wbias=1, num_init_vp=25, split_merge_freq=10,
                             merge_thresh=1e-3, outlier_thresh=1.96 ** 2, final_convergence=5e-3,
                             s_thresh=1e-200, num_min_lines=3, ctx=None):
    """vp_localisation.expectation_maximisation (reference vp_localisation.py:168-450).

    Like the reference, `l` is row-normalised in place (:186, :226) so callers
    that re-pickle it (evaluation.py:350) see the same array."""
    N = l.shape[0]
    res = expectation_maximisation_batch(
        l, lp, [0, N], np.asarray(cnn_response)[None], None if sphere_image is None else sphere_image[None],
        init_vp=init_vp, want_decision_metric=True, ctx=ctx, num_iter=num_iter, do_merge=do_merge,
        do_split=do_split, do_iterations=do_iterations, distance_measure=distance_measure, use_weights=use_weights,
        wbias=float(wbias), num_init_vp=num_init_vp, split_merge_freq=split_merge_freq, merge_thresh=merge_thresh,
        outlier_thresh=outlier_thresh, final_convergence=final_convergence, s_thresh=s_thresh,
        num_min_lines=num_min_lines)[0]
    if N:
        nr = np.sqrt(np.sum(l * l, axis=1))
        l /= nr[:, None]
        l /= np.sqrt(np.sum(l * l, axis=1))[:, None]
    if res["vp"] is None:
        return {k: res[k] for k in _SKELETON}
    res.pop("status", None)
    res["distribution"] = em_distribution(0, res["vp"].shape[0], N, ctx)       # the PDF tuple of the last E-step (:441-442)
    return res
