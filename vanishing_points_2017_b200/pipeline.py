"""The whole hot path for a ragged batch, and its sharding over the GPUs of one box.

segments -> lines -> sphere image -> CNN -> EM -> VPs with every intermediate
resident in HBM (reference example.py:37-39 / benchmark.py:59-66, which
round-trip through per-image pickles instead).  Images are independent
(reference loops per file: evaluation.py:126, 271, 309), so multi-GPU is a
cost-balanced partition of the batch with no collective on the data path; the
only exchange is the final gather of the small per-image results.
"""
import ctypes as C

import numpy as np

from . import _lib
from . import cnn as _cnn
from .vp_localisation import _alloc_result, unpack_results


class Pipeline:
    """One context (GPU) running the path; CNN weights loaded once."""

    def __init__(self, device=0, weights=None, biases=None, mean=None, sphere_mode=None, alpha=0.1, size=500,
                 ctx=None, **em_kwargs):
        """weights: list of the eight Caffe-layout weight blobs (with `biases`), or anything
        cnn.load_weights takes (a .caffemodel / .npz path or dict).  sphere_mode: "curves" is the
        reference's great-circle line plot (sphere_mapping.py:36-72), what the TRAINED net expects;
        "votes" is north_star's pairwise-intersection histogram.  Default: "curves" with real
        weights; without weights the random fillers are used (benchmarks / tests; a RuntimeWarning is
        raised unless sphere_mode is given explicitly) and the mode defaults to "votes"."""
        self.ctx = ctx if ctx is not None else _lib.default_context(device)
        if weights is None or isinstance(weights, (str, dict)) or hasattr(weights, "files"):
            explicit = sphere_mode is not None
            if sphere_mode is None:
                sphere_mode = "votes" if weights is None else "curves"
            weights, biases = _cnn.load_weights(weights, allow_random=explicit)
        elif sphere_mode is None:
            sphere_mode = "curves"
        self.net = _cnn.Net(self.ctx, weights, biases)
        if mean is not None:
            self.net.set_mean(mean)
        self.mode = {"votes": _lib.SPHERE_VOTES, "curves": _lib.SPHERE_CURVES}[sphere_mode]
        self.alpha = float(alpha)
        self.size = int(size)
        self.cfg = _lib.em_config(**em_kwargs)
        self._B = 0
        self._off = None

    # -- the three steps of include/vpk.h, so callers can time them separately
    def upload(self, segments, offsets, stream=None):
        """segments (sum N, 4) float64 with image b's rows offsets[b] .. offsets[b+1]-1.  Segments in CUDA memory
        (anything exposing __cuda_array_interface__, e.g. a torch CUDA tensor or a column slice of a wider one) are
        gathered on the device, ordered after the work queued on `stream` (see _lib.call_stream); offsets may then be
        host or device memory, the latter costing one device-to-host copy on that stream."""
        if _lib.is_cuda_array(segments):
            return self._upload_device(segments, offsets, stream)
        seg = _lib.as_f64(segments, 4)
        off = _lib.as_offsets(offsets)
        if off[-1] != seg.shape[0]:
            raise ValueError("offsets[-1] must equal the number of segments")
        self._B, self._off = off.size - 1, off
        _lib.check(self.ctx.lib.vpk_pipeline_upload(self.ctx.h, _lib.ptr(seg), _lib.ptr(off), self._B),
                   "vpk_pipeline_upload")

    def _upload_device(self, segments, offsets, stream):
        a = _lib.cuda_array(segments, (_lib.F64,), (2,))
        if a.shape[1] != 4:
            raise ValueError("expected a (N,4) array, got %r" % (a.shape,))
        dev = self.ctx.device
        if _lib.is_cuda_array(offsets):
            st = _lib.call_stream(stream, dev, [a, _lib.cuda_array(offsets, (_lib.I32, _lib.I64), (1,))])
            import torch
            with torch.cuda.stream(_lib.torch_stream(st, dev)):
                offsets = torch.as_tensor(offsets, device=torch.device("cuda", dev)).to("cpu").numpy()
        else:
            st = _lib.call_stream(stream, dev, [a])
        off = _lib.as_offsets(offsets)
        if off[-1] != a.shape[0]:
            raise ValueError("offsets[-1] must equal the number of segments")
        self._B, self._off = off.size - 1, off
        _lib.check(self.ctx.lib.vpk_pipeline_upload_device(self.ctx.h, a.ptr, a.strides[0] // 8, a.strides[1] // 8, _lib.ptr(off),
                                                           self._B, st), "vpk_pipeline_upload_device")

    def upload_lsd(self, lsd_rows, offsets, widths, heights):
        """upload() for raw LSD rows (flat (sum N, ncols) array, pixels): normalised on the device
        (evaluation.py:240-249) into the resident batch."""
        lsd = np.ascontiguousarray(lsd_rows, dtype=np.float64)
        off = _lib.as_offsets(offsets)
        if lsd.ndim != 2 or off[-1] != lsd.shape[0]:
            raise ValueError("lsd_rows must be (sum N, ncols) with offsets[-1] == sum N")
        w = np.ascontiguousarray(widths, dtype=np.int32)
        h = np.ascontiguousarray(heights, dtype=np.int32)
        self._B, self._off = off.size - 1, off
        _lib.check(self.ctx.lib.vpk_pipeline_upload_lsd(self.ctx.h, _lib.ptr(lsd), lsd.shape[1], _lib.ptr(off), _lib.ptr(w),
                                                        _lib.ptr(h), self._B), "vpk_pipeline_upload_lsd")

    def upload_images(self, images, stream=None, **lsd_kwargs):
        """upload() from grayscale images (a list of 2-D arrays of any sizes, uint8 or float64 gray values): the
        LSD detector (lsd.detect_line_segments with `lsd_kwargs`, lsd.pyx's defaults otherwise) and the
        normalisation of evaluation.py:240-249 run on the device into the resident batch; only the per-image
        segment counts come back.  Returns them.  Images in CUDA memory (__cuda_array_interface__: torch CUDA tensors,
        strided views included; all uint8 or all float64) are gathered on the device, ordered after the work queued
        on `stream` (see _lib.call_stream)."""
        from .lsd import pack_images
        if len(images) == 0:
            raise ValueError("upload_images needs at least one image")
        cfg = _lib.lsd_config(**lsd_kwargs)
        counts = np.empty(len(images), np.int32)
        dev = _device_arrays(images, "images", (_lib.U8, _lib.F64), (2,))
        if dev is not None:
            if len({a.typestr for a in dev}) != 1:
                raise ValueError("images in CUDA memory must be all uint8 or all float64")
            ptrs = (C.c_void_p * len(dev))(*[a.ptr for a in dev])
            es = 1 if dev[0].typestr == _lib.U8 else 8
            strides = np.array([[a.strides[0] // es, a.strides[1] // es] for a in dev], np.int64)
            h, w = (np.array([a.shape[k] for a in dev], np.int32) for k in (0, 1))
            st = _lib.call_stream(stream, self.ctx.device, dev)
            _lib.check(self.ctx.lib.vpk_pipeline_upload_images_device(
                self.ctx.h, ptrs, _lib.ptr(strides), _lib.ptr(w), _lib.ptr(h), len(dev), _lib.PIX_U8 if es == 1 else _lib.PIX_F64,
                C.byref(cfg), st, _lib.ptr(counts)), "vpk_pipeline_upload_images_device")
        else:
            flat, dt, off, w, h = pack_images(images)
            _lib.check(self.ctx.lib.vpk_pipeline_upload_images(self.ctx.h, _lib.ptr(flat), dt, _lib.ptr(off), _lib.ptr(w), _lib.ptr(h),
                                                               len(images), C.byref(cfg), _lib.ptr(counts)), "vpk_pipeline_upload_images")
        self._B = len(images)
        self._off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
        return counts

    def upload_photos(self, photos, target_size=None, stream=None, **lsd_kwargs):
        """upload_images() from RGB photos (a list of (H, W, 3) uint8 arrays of any sizes): the preparation of
        evaluation.py:139-154 (images.prepare_images: resize to `target_size`, rgb2gray), LSD on the gray planes
        times 255 and the normalisation run on the device; the photos cross PCIe as uint8 RGB and nothing but the
        per-image counts and sizes comes back.  Returns (counts, shapes): shapes are the prepared (H', W') pairs,
        the frames the segments are normalised in (horizons(image_heights=...), evaluation.reference_data).
        Photos in CUDA memory (__cuda_array_interface__, e.g. torchvision.io.decode_jpeg(..., device="cuda") output)
        are gathered on the device, ordered after the work queued on `stream` (see _lib.call_stream): (H, W, 3) uint8
        views of any strides (a CHW tensor passed as t.permute(1, 2, 0), crops), or (H, W) uint8 gray photos, which
        are prepared as upload_files prepares gray files."""
        from .images import pack_photos, _target
        dev = _device_arrays(photos, "photos", (_lib.U8,), (2, 3))
        if dev is not None:
            return self._upload_photos_device(dev, _target(target_size), stream, lsd_kwargs)
        flat, off, w, h = pack_photos(photos)
        if len(w) == 0:
            raise ValueError("upload_photos needs at least one photo")
        cfg = _lib.lsd_config(**lsd_kwargs)
        B = len(w)
        counts = np.empty(B, np.int32)
        ow = np.empty(B, np.int32)
        oh = np.empty(B, np.int32)
        _lib.check(self.ctx.lib.vpk_pipeline_upload_photos(self.ctx.h, _lib.ptr(flat), _lib.ptr(off), _lib.ptr(w), _lib.ptr(h), B,
                                                           _target(target_size), C.byref(cfg), _lib.ptr(counts), _lib.ptr(ow),
                                                           _lib.ptr(oh)), "vpk_pipeline_upload_photos")
        self._B = B
        self._off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
        return counts, [(int(a), int(b)) for a, b in zip(oh, ow)]

    def _upload_photos_device(self, dev, target, stream, lsd_kwargs):
        cfg = _lib.lsd_config(**lsd_kwargs)
        B = len(dev)
        ptrs = (C.c_void_p * B)(*[a.ptr for a in dev])
        strides = np.array([list(a.strides) + [0] * (3 - len(a.shape)) for a in dev], np.int64)
        h, w = (np.array([a.shape[k] for a in dev], np.int32) for k in (0, 1))
        ch = np.array([a.shape[2] if len(a.shape) == 3 else 1 for a in dev], np.int32)
        counts, ow, oh = (np.empty(B, np.int32) for _ in range(3))
        st = _lib.call_stream(stream, self.ctx.device, dev)
        _lib.check(self.ctx.lib.vpk_pipeline_upload_photos_device(self.ctx.h, ptrs, _lib.ptr(strides), _lib.ptr(w), _lib.ptr(h),
                                                                  _lib.ptr(ch), B, target, C.byref(cfg), st, _lib.ptr(counts),
                                                                  _lib.ptr(ow), _lib.ptr(oh)), "vpk_pipeline_upload_photos_device")
        self._B = B
        self._off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
        return counts, [(int(a), int(b)) for a, b in zip(oh, ow)]

    def upload_jpegs(self, blobs, target_size=None, **lsd_kwargs):
        """upload_photos() from JPEG files (a list of bytes or 1-D uint8 arrays of the file contents): the files are
        decoded on the device (images.decode_jpegs) where the preparation kernel reads them, so only the files cross
        PCIe.  Returns (counts, shapes, status): as upload_photos, plus an int32 status per file (0, or
        _lib.JPEG_CORRUPT: inconsistent entropy-coded data, whose rows come from unspecified pixels).  A refused or
        1-component (gray) file raises VpkError naming its index and reason."""
        from .images import pack_jpegs, _target
        flat, off = pack_jpegs(blobs)
        B = len(off) - 1
        if B == 0:
            raise ValueError("upload_jpegs needs at least one file")
        cfg = _lib.lsd_config(**lsd_kwargs)
        counts = np.empty(B, np.int32)
        ow = np.empty(B, np.int32)
        oh = np.empty(B, np.int32)
        status = np.empty(B, np.int32)
        _lib.check(self.ctx.lib.vpk_pipeline_upload_jpegs(self.ctx.h, _lib.ptr(flat), _lib.ptr(off), B, _target(target_size),
                                                          C.byref(cfg), _lib.ptr(counts), _lib.ptr(ow), _lib.ptr(oh),
                                                          _lib.ptr(status)), "vpk_pipeline_upload_jpegs")
        self._B = B
        self._off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
        return counts, [(int(a), int(b)) for a, b in zip(oh, ow)], status

    def upload_pngs(self, blobs, target_size=None, **lsd_kwargs):
        """upload_photos() from PNG files (a list of bytes or 1-D uint8 arrays of the file contents): the files are
        decoded on the device (images.decode_pngs) where the preparation kernel reads them, so only the files cross
        PCIe.  Returns (counts, shapes, status): as upload_photos, plus an int32 status per file (0, or
        _lib.PNG_CORRUPT: a damaged stream, whose rows come from unspecified pixels).  A refused or gray (colour type 0
        or 4) file raises VpkError naming its index and reason."""
        from .images import pack_jpegs, _target
        flat, off = pack_jpegs(blobs, "PNG")
        B = len(off) - 1
        if B == 0:
            raise ValueError("upload_pngs needs at least one file")
        cfg = _lib.lsd_config(**lsd_kwargs)
        counts = np.empty(B, np.int32)
        ow = np.empty(B, np.int32)
        oh = np.empty(B, np.int32)
        status = np.empty(B, np.int32)
        _lib.check(self.ctx.lib.vpk_pipeline_upload_pngs(self.ctx.h, _lib.ptr(flat), _lib.ptr(off), B, _target(target_size),
                                                         C.byref(cfg), _lib.ptr(counts), _lib.ptr(ow), _lib.ptr(oh),
                                                         _lib.ptr(status)), "vpk_pipeline_upload_pngs")
        self._B = B
        self._off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
        return counts, [(int(a), int(b)) for a, b in zip(oh, ow)], status

    def upload_files(self, blobs, target_size=None, **lsd_kwargs):
        """upload_photos() from a mixed batch of files (a list of bytes or 1-D uint8 arrays): JPEG, PNG and binary PGM,
        colour or gray, as evaluation.get_data_list lists them.  Each format's files are decoded on the device by its
        decoder; colour files are prepared as upload_photos does, gray ones as the reference does (the resized uint8
        plane, times 255 only if its maximum is at most 1), and LSD and the normalisation follow for the whole batch in
        input order.  Only the files cross PCIe.  Returns (counts, shapes, status) as upload_jpegs, status being each
        format's own code (0, _lib.JPEG_CORRUPT or _lib.PNG_CORRUPT).  A refused or unknown file raises VpkError
        naming its index, format and reason (images.file_info tells them beforehand)."""
        from .images import pack_jpegs, _target
        flat, off = pack_jpegs(blobs, "image")
        B = len(off) - 1
        if B == 0:
            raise ValueError("upload_files needs at least one file")
        cfg = _lib.lsd_config(**lsd_kwargs)
        counts = np.empty(B, np.int32)
        ow = np.empty(B, np.int32)
        oh = np.empty(B, np.int32)
        status = np.empty(B, np.int32)
        _lib.check(self.ctx.lib.vpk_pipeline_upload_files(self.ctx.h, _lib.ptr(flat), _lib.ptr(off), B, _target(target_size),
                                                          C.byref(cfg), _lib.ptr(counts), _lib.ptr(ow), _lib.ptr(oh),
                                                          _lib.ptr(status)), "vpk_pipeline_upload_files")
        self._B = B
        self._off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
        return counts, [(int(a), int(b)) for a, b in zip(oh, ow)], status

    def run(self):
        _lib.check(self.ctx.lib.vpk_pipeline_run(self.ctx.h, self.size, self.mode, self.alpha, C.byref(self.cfg)),
                   "vpk_pipeline_run")

    def fetch(self, want_response=False, want_sphere=False, raw=False, device=False, stream=None):
        """The EM results of the last run(): per-image dicts (raw=False) or the flat arrays (raw=True), plus the CNN
        responses and sphere images when asked for -> (results, sig, sphere).  device=True returns torch CUDA tensors
        of the flat arrays instead (a dict with the keys of pipeline.RAW_PER_IMAGE and "vp_assoc"; sig (B, 20, 20)
        float32, sphere (B, S, S) uint8), written on the device without blocking the host and ordered before the work
        queued on `stream` after the call (see _lib.call_stream)."""
        if device:
            return self._fetch_device(want_response, want_sphere, stream)
        arrs, res = _alloc_result(self._B, int(self._off[-1]), False)
        sig = np.empty((self._B, 20, 20), np.float32) if want_response else None
        sph = np.empty((self._B, self.size, self.size), np.uint8) if want_sphere else None
        _lib.check(self.ctx.lib.vpk_pipeline_fetch(self.ctx.h, C.byref(res), _lib.ptr(sig), _lib.ptr(sph)),
                   "vpk_pipeline_fetch")
        out = arrs if raw else unpack_results(arrs, self._off)
        return (out, sig, sph) if (want_response or want_sphere) else out

    def _fetch_device(self, want_response, want_sphere, stream):
        import torch
        dev = torch.device("cuda", self.ctx.device)
        st = _lib.call_stream(stream, self.ctx.device)
        B, n = self._B, int(self._off[-1])
        tdt = {np.int32: torch.int32, np.float64: torch.float64}
        with torch.cuda.stream(_lib.torch_stream(st, self.ctx.device)):       # the tensors belong to that stream
            out = {k: torch.empty((B,) + _RAW_TAIL[k], dtype=tdt[_RAW_DTYPES[k]], device=dev) for k in RAW_PER_IMAGE}
            out["vp_assoc"] = torch.empty(n, dtype=torch.int32, device=dev)
            sig = torch.empty((B, 20, 20), dtype=torch.float32, device=dev) if want_response else None
            sph = torch.empty((B, self.size, self.size), dtype=torch.uint8, device=dev) if want_sphere else None
        res = _lib.EmResult(*[out[k].data_ptr() for k in ("status", "n_vp", "iterations", "vp", "sigma", "counts", "counts_weighted",
                                                          "vp_assoc")], None)
        _lib.check(self.ctx.lib.vpk_pipeline_fetch_device(self.ctx.h, C.byref(res), None if sig is None else sig.data_ptr(),
                                                          None if sph is None else sph.data_ptr(), st), "vpk_pipeline_fetch_device")
        return (out, sig, sph) if (want_response or want_sphere) else out

    def horizons(self, maxbest=10, theta_vmin=np.pi / 10., theta_z=np.pi / 4., true_horizons=None, scales=None,
                 image_heights=None, device=False, stream=None):
        """calc_horizon.calculate_horizon_and_ortho_vp (calc_horizon.py:19-225) on the device-resident EM
        result of the last run(): one (hP1, hP2, zVP, hVP1, hVP2, best_combo) tuple per image; with ground-truth
        horizons also the horizon errors of benchmark.py:247-253 -> (tuples, errors).  device=True returns torch
        CUDA tensors (points (B, 5, 3) float64 = hP1, hP2, zVP, hVP1, hVP2; best_combo (B, 3) int32, -1 where fewer
        than three VPs take part; errors (B) float64 or None), written without blocking the host and ordered before
        the work queued on `stream` after the call (see _lib.call_stream); the ground truth may then be host or
        device arrays."""
        if device:
            return self._horizons_device(maxbest, theta_vmin, theta_z, true_horizons, scales, image_heights, stream)
        from . import calc_horizon
        points = np.empty((self._B, 5, 3), np.float64)
        combo = np.empty((self._B, 3), np.int32)
        th, sc, hh, err = calc_horizon._truth(true_horizons, scales, image_heights, self._B)
        _lib.check(self.ctx.lib.vpk_pipeline_horizon(self.ctx.h, int(maxbest), float(theta_vmin), float(theta_z), _lib.ptr(th),
                                                     _lib.ptr(sc), _lib.ptr(hh), _lib.ptr(points), _lib.ptr(combo),
                                                     _lib.ptr(err)), "vpk_pipeline_horizon")
        n_vp = np.array([3 if c[2] >= 0 else 0 for c in combo])
        out = calc_horizon._unpack(points, combo, n_vp, 3)
        return out if err is None else (out, err)

    def _horizons_device(self, maxbest, theta_vmin, theta_z, true_horizons, scales, image_heights, stream):
        import torch
        dev = torch.device("cuda", self.ctx.device)
        B = self._B
        arrays = [_lib.cuda_array(a, (_lib.F64, _lib.I32, _lib.I64), (1, 2)) for a in (true_horizons, scales, image_heights) if _lib.is_cuda_array(a)]
        st = _lib.call_stream(stream, self.ctx.device, arrays)
        with torch.cuda.stream(_lib.torch_stream(st, self.ctx.device)):
            points = torch.empty((B, 5, 3), dtype=torch.float64, device=dev)
            combo = torch.empty((B, 3), dtype=torch.int32, device=dev)
            truth, err = [None] * 3, None
            if true_horizons is not None:
                f64 = lambda a: torch.as_tensor(a, dtype=torch.float64, device=dev)   # noqa: E731
                truth = [f64(true_horizons).reshape(B, 3).contiguous(), f64(scales).expand(B).contiguous(),
                         f64(image_heights).expand(B).contiguous()]
                err = torch.empty(B, dtype=torch.float64, device=dev)
        ptr = lambda t: None if t is None else t.data_ptr()   # noqa: E731
        _lib.check(self.ctx.lib.vpk_pipeline_horizon_device(self.ctx.h, int(maxbest), float(theta_vmin), float(theta_z),
                                                            *[ptr(t) for t in truth], ptr(points), ptr(combo), ptr(err), st),
                   "vpk_pipeline_horizon_device")
        return points, combo, err

    def stage_ms(self):
        ms = (C.c_float * 4)()
        _lib.check(self.ctx.lib.vpk_pipeline_stage_ms(self.ctx.h, ms), "vpk_pipeline_stage_ms")
        return {"sphere": ms[0], "cnn": ms[1], "em": ms[2], "total": ms[3]}

    def __call__(self, segments, offsets, want_response=False, want_sphere=False, raw=False):
        """End to end from host buffers in ONE library call (vpk_pipeline_host: H2D, path, D2H)."""
        seg = _lib.as_f64(segments, 4)
        off = _lib.as_offsets(offsets)
        if off[-1] != seg.shape[0]:
            raise ValueError("offsets[-1] must equal the number of segments")
        self._B, self._off = off.size - 1, off
        arrs, res = _alloc_result(self._B, int(off[-1]), False)
        sig = np.empty((self._B, 20, 20), np.float32) if want_response else None
        sph = np.empty((self._B, self.size, self.size), np.uint8) if want_sphere else None
        _lib.check(self.ctx.lib.vpk_pipeline_host(self.ctx.h, _lib.ptr(seg), _lib.ptr(off), self._B, self.size, self.mode,
                                                  self.alpha, C.byref(self.cfg), C.byref(res), _lib.ptr(sig), _lib.ptr(sph)),
                   "vpk_pipeline_host")
        out = arrs if raw else unpack_results(arrs, self._off)
        return (out, sig, sph) if (want_response or want_sphere) else out


class StreamedPipeline:
    """`depth` batches in flight on one GPU: one library context (own streams, own workspaces, own copy of the CNN
    weights) and one host thread per batch in flight.  The EM stage of a batch is a chain of dependent supersteps
    that leaves most SMs idle towards its end; the sphere mapping / CNN / pair pass of the next batches fill them
    (measured on the 102-image YUD-shaped batch: +29 % images/s with two batches in flight, +38 % with three;
    nothing on the 2018-image HLW-shaped batch, which already fills the GPU).  Results are bit-identical to
    Pipeline's: every batch still runs alone on its context.

    submit(segments, offsets) returns a concurrent.futures.Future of Pipeline.__call__'s result; batches are dealt
    round-robin to the contexts, and a context runs its batches in submission order."""

    def __init__(self, device=0, weights=None, biases=None, depth=2, **kwargs):
        from concurrent.futures import ThreadPoolExecutor
        if weights is None or isinstance(weights, (str, dict)) or hasattr(weights, "files"):
            if kwargs.get("sphere_mode") is None:
                kwargs["sphere_mode"] = "votes" if weights is None else "curves"
                weights, biases = _cnn.load_weights(weights)
            else:
                weights, biases = _cnn.load_weights(weights, allow_random=True)
        self.pipes = [Pipeline(device, weights, biases, ctx=_lib.Context(device), **kwargs) for _ in range(int(depth))]
        self._workers = [ThreadPoolExecutor(max_workers=1) for _ in self.pipes]
        self._next = 0

    @property
    def depth(self):
        return len(self.pipes)

    def submit(self, segments, offsets, **kwargs):
        k = self._next
        self._next = (k + 1) % len(self.pipes)
        return self._workers[k].submit(self.pipes[k].__call__, segments, offsets, **kwargs)

    def map(self, batches, **kwargs):
        """Results of an iterable of (segments, offsets) batches, in order, at most `depth` in flight."""
        from collections import deque
        pending = deque()
        for seg, off in batches:
            if len(pending) >= len(self.pipes):
                yield pending.popleft().result()
            pending.append(self.submit(seg, off, **kwargs))
        while pending:
            yield pending.popleft().result()

    def each(self, fn):
        """fn(pipe) on every context's own thread, concurrently; returns the results (benchmarks: resident loops)."""
        return [f.result() for f in [w.submit(fn, p) for w, p in zip(self._workers, self.pipes)]]

    def close(self):
        for w in self._workers:
            w.shutdown(wait=True)
        for p in self.pipes:
            p.ctx.close()


def image_cost(n):
    """Relative cost model of one image: the O(N^2) pair/weight-matrix work
    dominates, plus the constant CNN cost expressed in the same unit."""
    n = np.asarray(n, dtype=np.float64)
    return n * n + 250_000.0


def shard_batch(offsets, world_size, rank):
    """Cost-balanced partition: images sorted by descending cost are dealt to
    the currently lightest rank (LPT).  Returns the sorted image indices of `rank`."""
    n = np.diff(np.asarray(offsets, dtype=np.int64))
    cost = image_cost(n)
    order = np.argsort(-cost, kind="stable")
    load = np.zeros(world_size)
    owner = np.empty(len(n), dtype=np.int64)
    for i in order:
        r = int(np.argmin(load))
        owner[i] = r
        load[r] += cost[i]
    return np.sort(np.where(owner == rank)[0])


def take_images(segments, offsets, idx):
    """Sub-batch (segments, offsets) of the images `idx`."""
    offsets = np.asarray(offsets, dtype=np.int64)
    segs = [segments[offsets[i]:offsets[i + 1]] for i in idx]
    n = np.array([s.shape[0] for s in segs], dtype=np.int64)
    off = np.zeros(len(idx) + 1, dtype=np.int32)
    off[1:] = np.cumsum(n)
    seg = np.concatenate(segs, axis=0) if segs else np.zeros((0, 4))
    return np.ascontiguousarray(seg), off


def gather_results(local_results, idx, n_images, world_size, dist=None):
    """Final result gather (rank 0 gets the full list): the only inter-rank
    exchange of the path.  `dist` is torch.distributed or None (single rank)."""
    if dist is None or world_size == 1:
        out = [None] * n_images
        for i, r in zip(idx, local_results):
            out[int(i)] = r
        return out
    payload = [(int(i), r) for i, r in zip(idx, local_results)]
    gathered = [None] * world_size if dist.get_rank() == 0 else None
    dist.gather_object(payload, gathered, dst=0)
    if dist.get_rank() != 0:
        return None
    out = [None] * n_images
    for part in gathered:
        for i, r in part:
            out[i] = r
    return out


RAW_PER_IMAGE = ("status", "n_vp", "iterations", "vp", "sigma", "counts", "counts_weighted")
_RAW_DTYPES = {"status": np.int32, "n_vp": np.int32, "iterations": np.int32, "vp": np.float64, "sigma": np.float64,
               "counts": np.int32, "counts_weighted": np.float64}
_RAW_TAIL = {"status": (), "n_vp": (), "iterations": (), "vp": (_lib.VPK_MAX_VP, 3), "sigma": (_lib.VPK_MAX_VP,),
             "counts": (_lib.VPK_MAX_VP,), "counts_weighted": (_lib.VPK_MAX_VP,)}
_gather_cache = {}


def _device_arrays(items, what, typestrs, ndims):
    """CudaArrays of a list whose members expose __cuda_array_interface__, None if none does (the host route)."""
    if isinstance(items, np.ndarray) or not hasattr(items, "__len__"):
        return None
    flags = [_lib.is_cuda_array(x) for x in items]
    if not any(flags):
        return None
    if not all(flags):
        raise ValueError("%s must be all in CUDA memory or all host arrays" % what)
    return [_lib.cuda_array(x, typestrs, ndims) for x in items]


def _blob_layout(n_img, n_seg):
    """Byte offsets of the flat result arrays of a shard inside its gather blob (8-byte aligned fields)."""
    lay, pos = {}, 0
    for k in RAW_PER_IMAGE:
        nb = n_img * int(np.prod(_RAW_TAIL[k], dtype=np.int64)) * np.dtype(_RAW_DTYPES[k]).itemsize
        lay[k] = (pos, nb)
        pos += (nb + 7) // 8 * 8
    lay["vp_assoc"] = (pos, n_seg * 4)
    pos += (n_seg * 4 + 7) // 8 * 8
    return lay, pos


_plan_cache = {}


def _gather_plan(offsets_all, world_size):
    """Everything about a sharded batch that does not change from step to step (cached on the offsets)."""
    offsets_all = np.ascontiguousarray(offsets_all, dtype=np.int64)
    key = (offsets_all.tobytes(), world_size)
    plan = _plan_cache.get(key)
    if plan is None:
        n_all = np.diff(offsets_all)
        shards = [shard_batch(offsets_all, world_size, r) for r in range(world_size)]
        sizes = [(len(ix), int(n_all[ix].sum())) for ix in shards]
        layouts = [_blob_layout(*sz) for sz in sizes]
        # vp_assoc stays in rank-major order (the blobs as they arrive); image i starts at assoc_start[i]
        assoc_start = np.empty(n_all.shape[0], dtype=np.int64)
        base = 0
        for ix, (_, n_seg) in zip(shards, sizes):
            assoc_start[ix] = base + np.concatenate([[0], np.cumsum(n_all[ix])])[:-1]
            base += n_seg
        plan = {"n": n_all, "shards": shards, "sizes": sizes, "layouts": layouts, "assoc_start": assoc_start,
                "nbytes": max(l[1] for l in layouts)}
        _plan_cache.clear()
        _plan_cache[key] = plan
    return plan


def gather_raw(arrs, offsets_all, world_size, rank, dist=None, group=None):
    """The path's only inter-rank exchange, for the flat result arrays (`raw=True`) of the shards
    `shard_batch(offsets_all, world_size, r)`: ONE fixed-size `torch.distributed.gather` of a byte blob per rank
    (every rank can compute every shard's sizes from the batch offsets, so nothing else is exchanged; `group`: the
    process group to use -- the results are in host memory when a step returns, so a gloo group keeps the exchange
    off the GPU, whose streams are busy with the next batches; with an NCCL group the blobs go over NVLink).
    Rank 0 returns the per-image arrays in the batch's image order, "vp_assoc" in rank-major order with
    "assoc_start" (image i owns vp_assoc[assoc_start[i] : assoc_start[i] + n[i]]) and "n"; the other ranks None."""
    import torch
    plan = _gather_plan(offsets_all, world_size)
    shards, sizes, layouts, nbytes = plan["shards"], plan["sizes"], plan["layouts"], plan["nbytes"]
    n_images = plan["n"].shape[0]
    use_cuda = dist is not None and world_size > 1 and dist.get_backend(group) == "nccl"
    key = (nbytes, world_size, rank, use_cuda)
    buf = _gather_cache.get(key)
    if buf is None:
        _gather_cache.clear()
        host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=use_cuda)
        buf = {"host": host}
        if use_cuda:
            buf["dev"] = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
            if rank == 0:
                buf["dev_all"] = torch.empty(world_size * nbytes, dtype=torch.uint8, device="cuda")
                buf["host_all"] = torch.empty(world_size * nbytes, dtype=torch.uint8, pin_memory=True)
        elif rank == 0:
            buf["host_all"] = torch.empty(world_size * nbytes, dtype=torch.uint8)
        _gather_cache[key] = buf
    # pack this rank's arrays
    lay, _ = layouts[rank]
    hv = buf["host"].numpy()
    n_img, n_seg = sizes[rank]
    for k in RAW_PER_IMAGE:
        pos, nb = lay[k]
        hv[pos:pos + nb] = np.ascontiguousarray(arrs[k][:n_img], dtype=_RAW_DTYPES[k]).view(np.uint8).reshape(-1)
    pos, nb = lay["vp_assoc"]
    hv[pos:pos + nb] = np.ascontiguousarray(arrs["vp_assoc"][:n_seg], dtype=np.int32).view(np.uint8)
    if dist is None or world_size == 1:
        allv = hv[None, :]
    elif use_cuda:
        buf["dev"].copy_(buf["host"], non_blocking=True)
        parts = list(buf["dev_all"].view(world_size, nbytes).unbind(0)) if rank == 0 else None
        dist.gather(buf["dev"], parts, dst=0, group=group)
        if rank != 0:
            return None
        buf["host_all"].copy_(buf["dev_all"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        allv = buf["host_all"].numpy().reshape(world_size, nbytes)
    else:
        parts = list(buf["host_all"].view(world_size, nbytes).unbind(0)) if rank == 0 else None
        dist.gather(buf["host"], parts, dst=0, group=group)
        if rank != 0:
            return None
        allv = buf["host_all"].numpy().reshape(world_size, nbytes)
    # per-image arrays in image order; the line associations stay where they arrived
    out = {k: np.empty((n_images,) + _RAW_TAIL[k], dtype=_RAW_DTYPES[k]) for k in RAW_PER_IMAGE}
    assoc = []
    for r in range(world_size):
        lay, _ = layouts[r]
        n_img, n_seg = sizes[r]
        for k in RAW_PER_IMAGE:
            pos, nb = lay[k]
            out[k][shards[r]] = allv[r, pos:pos + nb].view(_RAW_DTYPES[k]).reshape((n_img,) + _RAW_TAIL[k])
        pos, nb = lay["vp_assoc"]
        assoc.append(allv[r, pos:pos + nb].view(np.int32))
    out["vp_assoc"] = np.concatenate(assoc) if len(assoc) > 1 else assoc[0].copy()
    out["assoc_start"] = plan["assoc_start"]
    out["n"] = plan["n"]
    return out
