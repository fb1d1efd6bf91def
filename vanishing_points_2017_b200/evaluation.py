"""Host mirror of the parts of the reference's evaluation.py that sit between the LSD detector and the
hot path (SURVEY.md section 8(f), row N2): the normalisation of the raw LSD rows
(`detect_lsd_lines`, evaluation.py:227-251, everything after the `lsd.detect_line_segments` call) and the
line construction (evaluation.py:158-168), on the device through the C ABI (`vpk_segments_from_lsd`), and
`detect_lsd_lines` itself with the detector on the device too (row N4, `vpk_lsd`).  No CPU fallback."""
import numpy as np

from . import _lib


def segments_from_lsd_batch(lsd_rows, image_shapes, want_lines=True, ctx=None):
    """lsd_rows: list of (N_b, >=4) arrays as lsd.detect_line_segments returns them (pixels);
    image_shapes: list of (height, width[, ...]) like `image.shape`.
    Returns dict(segments (sum N,4), lines (sum N,3) | None, nfa (sum N,) | None, offsets (B+1,) int32)."""
    ctx = ctx or _lib.default_context()
    B = len(lsd_rows)
    rows = [np.asarray(r, np.float64).reshape(-1, np.asarray(r).shape[-1] if np.asarray(r).ndim == 2 else 7) for r in lsd_rows]
    ncols = rows[0].shape[1] if B else 7
    if any(r.shape[1] != ncols for r in rows) or ncols < 4:
        raise ValueError("all LSD arrays must have the same number of columns (>= 4)")
    off = np.concatenate([[0], np.cumsum([r.shape[0] for r in rows])]).astype(np.int32)
    flat = np.ascontiguousarray(np.concatenate(rows) if B else np.zeros((0, ncols)))
    widths = np.array([s[1] for s in image_shapes], np.int32)
    heights = np.array([s[0] for s in image_shapes], np.int32)
    n = int(off[-1])
    seg = np.empty((n, 4), np.float64)
    lines = np.empty((n, 3), np.float64) if want_lines else None
    nfa = np.empty(n, np.float64) if ncols >= 7 else None
    _lib.check(ctx.lib.vpk_segments_from_lsd(ctx.h, _lib.ptr(flat), ncols, _lib.ptr(off), _lib.ptr(widths), _lib.ptr(heights), B,
                                             _lib.ptr(seg), _lib.ptr(lines), _lib.ptr(nfa)), "vpk_segments_from_lsd")
    return {"segments": seg, "lines": lines, "nfa": nfa, "offsets": off}


def segments_from_lsd(lsd_lines, image_shape):
    """What detect_lsd_lines returns for one image (evaluation.py:251): {'segments': (N,4), 'nfa': (N,)}."""
    out = segments_from_lsd_batch([lsd_lines], [image_shape], want_lines=False)
    return {"segments": out["segments"], "nfa": out["nfa"]}


def detect_lsd_lines(image):
    """evaluation.detect_lsd_lines (reference evaluation.py:227-251) for a 2-D grayscale image: gray values as
    float64, scaled by 255 when the image's maximum is at most 1, LSD with lsd.pyx's defaults, then the
    normalisation above.  Returns {'segments': (N,4), 'nfa': (N,)}.  (RGB -> gray stays with the caller.)"""
    from . import lsd
    gray = np.array(image, dtype=np.float64)
    if gray.ndim != 2:
        raise ValueError("detect_lsd_lines takes a 2-D grayscale image, got shape %r" % (gray.shape,))
    if gray.max() <= 1:
        gray *= 255
    return segments_from_lsd(lsd.detect_line_segments(gray), gray.shape)


# ---------------------------------------------------------------------------------------------------
# Row N3: the stage hand-off.  The reference passes one pickle per image from stage to stage
# (evaluation.py:152-183 writes {'lines': datum, 'sphere_image'}, :283-289 adds 'cnn_prediction',
# :344-349 adds 'EM_result'); the pipeline keeps everything in HBM instead.  For the reference's own
# consumers (example.py:62-65, benchmark.py:228-241, result_plotting) the same dicts can be exported.
# ---------------------------------------------------------------------------------------------------
def reference_data(results, segments, offsets, sphere_images, cnn_predictions, image_shapes=None, images=None,
                   extra=None):
    """One dict per image with the layout of the reference's per-image pickle after run_em
    (evaluation.py:349): {'lines': {'image_shape', 'image', 'line_segments', 'lines', ...},
    'sphere_image' (S,S) uint8, 'cnn_prediction' (20,20) float32, 'EM_result' dict | None}.

    'lines'['lines'] holds the ROW-NORMALISED homogeneous lines: the reference's EM normalises the array it
    is given in place (vp_localisation.py:186, :226) and run_em_single stores that very array back
    (evaluation.py:350).  A failed image gets the reference's skeleton dict with None entries
    (vp_localisation.py:205-206); `status` is dropped (not a key of the reference)."""
    seg = np.asarray(segments, np.float64).reshape(-1, 4)
    off = np.asarray(offsets).astype(np.int64)
    B = off.size - 1
    out = []
    for b in range(B):
        s = seg[off[b]:off[b + 1]].copy()
        p1 = np.concatenate([s[:, 0:2], np.ones((s.shape[0], 1))], axis=1)
        p2 = np.concatenate([s[:, 2:4], np.ones((s.shape[0], 1))], axis=1)
        lines = np.cross(p1, p2)                                              # evaluation.py:161-168
        em = None
        if results[b] is not None:
            em = {k: v for k, v in results[b].items() if k != "status"}
            em.setdefault("distribution", None)
            if lines.shape[0]:
                lines = lines / np.sqrt(np.sum(lines * lines, axis=1))[:, None]  # the EM's in-place normalisation
        datum = {"image_shape": None if image_shapes is None else tuple(image_shapes[b]),
                 "image": None if images is None else images[b], "line_segments": s, "lines": lines}
        if extra is not None:
            datum.update(extra[b])                                            # e.g. 'dataset', 'image_file' (:152)
        out.append({"lines": datum, "sphere_image": None if sphere_images is None else np.asarray(sphere_images[b]),
                    "cnn_prediction": None if cnn_predictions is None else np.asarray(cnn_predictions[b], np.float32),
                    "EM_result": em})
    return out


def dump_reference_pickles(data, paths):
    """Write the dicts of reference_data() as the reference writes them (evaluation.py:182-183:
    pickle.dump(..., -1) under Python 2, i.e. protocol 2, which Python 2 and 3 both read)."""
    import pickle
    for d, p in zip(data, paths):
        with open(p, "wb") as fh:
            pickle.dump(d, fh, 2)
