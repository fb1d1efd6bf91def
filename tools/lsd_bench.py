"""Throughput of the device LSD detector (vpk_lsd, row N4) against OpenCV's LSD on all host cores, on the same
rendered images in the same run, plus images -> horizons end to end through Pipeline.upload_images.

Batches: YUD-shaped (102 images 640x480) and HLW-shaped (2018 images, max side 800, the aspects of
synth.CONFIGS[4]), rendered by synth.render_scene with `--segments` bars each.  vpk_lsd is timed between device
marks around the whole call (host-to-device copy of the images included, bytes reported separately), uint8 and
float64 input; per-kernel times come from a separate profiled call.  OpenCV runs LSD_REFINE_ADV with its default
scale 0.8 (the same work), one detector per thread, os.cpu_count() threads.

    python tools/lsd_bench.py --out profiles/r3_lsd_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vanishing_points_2017_b200 import _lib, lsd, pipeline, synth  # noqa: E402
from vanishing_points_2017_b200 import cnn as vcnn  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:                      # noqa: BLE001
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def batch(cfg, n_segments, n_images=None):
    name, B, _, _, _, _, aspects = synth.CONFIGS[cfg]
    B = n_images or B
    rs = np.random.RandomState(1_000_003 * cfg)
    shapes = [aspects[i] for i in rs.randint(0, len(aspects), B)]
    return [synth.render_scene(77_000 * cfg + k, n_segments, w, h).astype(np.uint8) for k, (w, h) in enumerate(shapes)]


def time_vpk_lsd(ctx, imgs, reps):
    flat, dt, off, w, h = lsd.pack_images(imgs)
    cfg = _lib.lsd_config()
    counts = np.empty(len(imgs), np.int32)
    import ctypes as C

    def call():
        _lib.check(ctx.lib.vpk_lsd(ctx.h, _lib.ptr(flat), dt, _lib.ptr(off), _lib.ptr(w), _lib.ptr(h), len(imgs), C.byref(cfg),
                                   _lib.ptr(counts)), "vpk_lsd")
    call()
    call()                                      # warm-up: modules, workspaces, CUB temp storage
    ms = []
    for _ in range(reps):
        ctx.mark(0)
        call()
        ctx.mark(1)
        ms.append(ctx.elapsed_ms(0, ctx, 1))
    ctx.profile_reset()
    ctx.profile_enable(True)
    call()
    ctx.synchronize()
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    kernels = {k: round(v["ms"], 3) for k, v in prof.items() if k.startswith("lsd_")}
    med = float(np.median(ms))
    return {"ms_median": round(med, 3), "ms_all": [round(x, 3) for x in ms], "images_per_s": round(len(imgs) / med * 1e3, 1),
            "h2d_bytes": int(flat.nbytes), "segments": int(counts.sum()), "kernel_ms": kernels}


def time_opencv(imgs, reps):
    import cv2
    cv2.setNumThreads(1)
    n = os.cpu_count()
    import threading
    local = threading.local()

    def one(im):
        d = getattr(local, "d", None)
        if d is None:
            d = local.d = cv2.createLineSegmentDetector(cv2.LSD_REFINE_ADV)
        r = d.detect(im)[0]
        return 0 if r is None else r.shape[0]
    with ThreadPoolExecutor(max_workers=n) as ex:
        list(ex.map(one, imgs[: 2 * n]))
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            segs = sum(ex.map(one, imgs))
            ts.append(time.perf_counter() - t0)
    med = float(np.median(ts))
    return {"threads": n, "s_median": round(med, 4), "images_per_s": round(len(imgs) / med, 1), "segments": int(segs)}


def time_end_to_end(pipe, imgs, reps):
    def step():
        pipe.upload_images(imgs)
        pipe.run()
        return pipe.horizons()
    step()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    med = float(np.median(ts))
    return {"s_median": round(med, 4), "images_per_s": round(len(imgs) / med, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/lsd_bench.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--segments", type=int, default=300)
    ap.add_argument("--hlw-images", type=int, default=None, help="fewer HLW-shaped images (rehearsal only)")
    a = ap.parse_args()
    res = {"card": card(), "host_cpus": os.cpu_count(), "segments_per_image_rendered": a.segments, "reps": a.reps}
    ctx = _lib.default_context(0)
    ws, bs = vcnn.random_weights(0, scale=3.0)
    pipe = pipeline.Pipeline(0, ws, bs, sphere_mode="votes", ctx=ctx)
    for cfg, key, n in ((2, "yud", None), (4, "hlw", a.hlw_images)):
        t0 = time.time()
        imgs = batch(cfg, a.segments, n)
        r = {"images": len(imgs), "render_s": round(time.time() - t0, 1)}
        r["gpu_uint8"] = time_vpk_lsd(ctx, imgs, a.reps)
        r["gpu_float64"] = time_vpk_lsd(ctx, [im.astype(np.float64) for im in imgs], a.reps)
        r["opencv_all_cores"] = time_opencv(imgs, max(1, a.reps // 2))
        r["gpu_over_opencv"] = round(r["gpu_uint8"]["images_per_s"] / r["opencv_all_cores"]["images_per_s"], 2)
        r["end_to_end_images_to_horizons"] = time_end_to_end(pipe, imgs, max(1, a.reps // 2))
        res[key] = r
        print(key, json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"card": res["card"], "yud_ratio": res["yud"]["gpu_over_opencv"], "hlw_ratio": res["hlw"]["gpu_over_opencv"]}))


if __name__ == "__main__":
    main()
