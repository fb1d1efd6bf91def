"""Photo preparation on the device (vpk_prepare_images / Pipeline.upload_photos, row N5) against the host path
(cv2.resize INTER_AREA + numpy gray on all host cores), on the same rendered photos in the same run.

Batches (synth.render_photo, `--segments` bars each):
  example-shaped  102 photos 2000x1333 / 1333x2000 (mixed orientation), target 640 (example.py:37)
  HLW-shaped      2018 photos with longer side 1200 (the aspects of synth.CONFIGS[4] times 1.5), target 800
                  (benchmark.py:59-60; factor 1.5, generic path); 64 distinct photos cycled to keep host memory
                  near 6.5 GB

Reported per batch: the image_prep kernel's time (CUDA events of vpk_profile around every launch, over `--reps`
calls); its algorithmic bytes (sum 3wh read + sum 8W'H' written) over that time, against a device-to-device copy
measured in the same run (torch, read + write bytes) and against the data sheet's 7.7 TB/s; the split of one
upload_photos call (device marks around the call; kernels from vpk_profile; the host-to-device copy of the same
pageable bytes timed on its own); photos -> horizons end to end; the host baseline; the card and its power limit.

    python tools/image_prep_bench.py --out profiles/r4_image_prep_bench.json
"""
import argparse
import ctypes as C
import json
import os
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from multiprocessing import Pool

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from lsd_bench import card  # noqa: E402
from vanishing_points_2017_b200 import _lib, images, pipeline, synth  # noqa: E402
from vanishing_points_2017_b200 import cnn as vcnn  # noqa: E402

DATASHEET_HBM_TBPS = 7.7      # NVIDIA HGX B200 data sheet, one GPU


def _render(args):
    return synth.render_photo(*args)


def example_batch(n, segments):
    shapes = [(2000, 1333) if k % 2 == 0 else (1333, 2000) for k in range(n)]
    with Pool(min(16, os.cpu_count() or 1)) as pool:
        return pool.map(_render, [(90_000 + k, segments, w, h) for k, (w, h) in enumerate(shapes)])


def hlw_batch(n, segments, distinct=64):
    _, _, _, _, _, _, aspects = synth.CONFIGS[4]
    rs = np.random.RandomState(4_000_037)
    shapes = [aspects[i] for i in rs.randint(0, len(aspects), n)]
    shapes = [(int(round(w * 1.5)), int(round(h * 1.5))) for w, h in shapes]
    keys = sorted(set(shapes))
    per = max(1, distinct // len(keys))
    with Pool(min(16, os.cpu_count() or 1)) as pool:
        rendered = pool.map(_render, [(95_000 + 100 * i + j, segments, w, h) for i, (w, h) in enumerate(keys) for j in range(per)])
    by_shape = {k: rendered[i * per:(i + 1) * per] for i, k in enumerate(keys)}
    return [by_shape[s][k % per] for k, s in enumerate(shapes)]


def d2d_copy_tbps(nbytes=4 << 30, reps=10):
    """Device-to-device copy bandwidth (bytes read + bytes written per second) with torch, median of `reps`."""
    import torch
    a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    del a, b
    torch.cuda.empty_cache()
    return 2 * nbytes / float(np.median(ts)) / 1e12


def h2d_ms(flat, reps=3):
    """The host-to-device copy of the packed photos from the same pageable memory, on its own."""
    import torch
    src = torch.from_numpy(flat)
    dst = torch.empty(flat.nbytes, dtype=torch.uint8, device="cuda")
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dst.copy_(src)
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    del dst
    torch.cuda.empty_cache()
    return float(np.median(ts))


def prep_kernel(ctx, photos, target, reps):
    flat, off, w, h = images.pack_photos(photos)
    sizes = [images.prepared_size(a, b, target) for a, b in zip(w, h)]
    n_out = sum(W * H for W, H in sizes)
    out = np.empty(n_out, np.float64)
    ow, oh = np.empty(len(w), np.int32), np.empty(len(w), np.int32)

    def call():
        _lib.check(ctx.lib.vpk_prepare_images(ctx.h, _lib.ptr(flat), _lib.ptr(off), _lib.ptr(w), _lib.ptr(h), len(w), target,
                                              _lib.ptr(ow), _lib.ptr(oh), _lib.ptr(out)), "vpk_prepare_images")
    call()                                      # warm-up: module, workspaces
    ctx.profile_reset()
    ctx.profile_enable(True)
    for _ in range(reps):
        call()
    ctx.synchronize()
    prof = ctx.profile_read()["image_prep"]
    ctx.profile_enable(False)
    ms = prof["ms"] / prof["launches"]
    in_bytes, out_bytes = int(flat.nbytes), 8 * int(n_out)
    return flat, {"launches": prof["launches"], "kernel_ms_mean": round(ms, 3), "bytes_read": in_bytes, "bytes_written": out_bytes,
                  "algorithmic_tbps": round((in_bytes + out_bytes) / (ms * 1e-3) / 1e12, 3)}


def host_baseline(photos, target, reps):
    import cv2
    from oracle import image_prep_oracle as P
    cv2.setNumThreads(1)

    def one(p):
        W, H = images.prepared_size(p.shape[1], p.shape[0], target)
        r = p if (W, H) == (p.shape[1], p.shape[0]) else cv2.resize(p, (W, H), interpolation=cv2.INTER_AREA)
        return P.rgb2gray(r)
    n = os.cpu_count()
    with ThreadPoolExecutor(max_workers=n) as ex:
        list(ex.map(one, photos[:2 * n]))
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            list(ex.map(one, photos))
            ts.append(time.perf_counter() - t0)
    med = float(np.median(ts))
    return {"threads": n, "s_median": round(med, 4), "images_per_s": round(len(photos) / med, 1)}


def upload_split(pipe, flat, photos, target):
    ctx = pipe.ctx
    pipe.upload_photos(photos, target)          # warm-up
    ctx.profile_reset()
    ctx.profile_enable(True)
    ctx.mark(0)
    counts, _ = pipe.upload_photos(photos, target)
    ctx.mark(1)
    ctx.synchronize()
    total = ctx.elapsed_ms(0, ctx, 1)
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    prep = prof["image_prep"]["ms"]
    lsd = sum(v["ms"] for k, v in prof.items() if k.startswith("lsd_"))
    return {"call_device_ms": round(total, 3), "h2d_ms_same_bytes_alone": round(h2d_ms(flat), 3), "image_prep_ms": round(prep, 3),
            "lsd_ms": round(lsd, 3), "rest_ms": round(total - prep - lsd, 3), "segments": int(counts.sum()),
            "kernels_ms": {k: round(v["ms"], 3) for k, v in prof.items()}}


def end_to_end(pipe, photos, target, reps):
    def step():
        _, shapes = pipe.upload_photos(photos, target)
        pipe.run()
        return pipe.horizons()
    step()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    med = float(np.median(ts))
    return {"s_median": round(med, 4), "images_per_s": round(len(photos) / med, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/image_prep_bench.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--segments", type=int, default=300)
    ap.add_argument("--example-images", type=int, default=102)
    ap.add_argument("--hlw-images", type=int, default=2018)
    a = ap.parse_args()
    res = {"card": card(), "host_cpus": os.cpu_count(), "reps": a.reps, "segments_per_photo_rendered": a.segments}
    ctx = _lib.default_context(0)
    res["d2d_copy_tbps_read_plus_write"] = round(d2d_copy_tbps(), 3)
    res["datasheet_hbm_tbps"] = DATASHEET_HBM_TBPS
    ws, bs = vcnn.random_weights(0, scale=3.0)
    pipe = pipeline.Pipeline(0, ws, bs, sphere_mode="votes", ctx=ctx)
    for key, make, target in (("example", lambda: example_batch(a.example_images, a.segments), 640),
                              ("hlw", lambda: hlw_batch(a.hlw_images, a.segments), 800)):
        t0 = time.time()
        photos = make()
        r = {"photos": len(photos), "target_size": target, "render_s": round(time.time() - t0, 1)}
        flat, r["image_prep"] = prep_kernel(ctx, photos, target, a.reps)
        k = r["image_prep"]
        k["share_of_measured_copy"] = round(k["algorithmic_tbps"] / res["d2d_copy_tbps_read_plus_write"], 3)
        k["share_of_datasheet_7.7TBps"] = round(k["algorithmic_tbps"] / DATASHEET_HBM_TBPS, 3)
        r["upload_photos_split"] = upload_split(pipe, flat, photos, target)
        r["photos_to_horizons"] = end_to_end(pipe, photos, target, max(1, a.reps // 2))
        r["host_cv2_area_numpy_gray_all_cores"] = host_baseline(photos, target, max(1, a.reps // 2))
        res[key] = r
        print(key, json.dumps(r), flush=True)
        del photos, flat
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"card": res["card"], "copy_tbps": res["d2d_copy_tbps_read_plus_write"],
                      "example_kernel_ms": res["example"]["image_prep"]["kernel_ms_mean"],
                      "hlw_kernel_ms": res["hlw"]["image_prep"]["kernel_ms_mean"],
                      "hlw_share_of_copy": res["hlw"]["image_prep"]["share_of_measured_copy"]}))


if __name__ == "__main__":
    main()
