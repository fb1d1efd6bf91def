"""Pipeline I/O in CUDA memory (row N9, DESIGN.md section 4.11) against the host routes, in one run.

Batch: the HLW-shaped photo batch of tools/image_prep_bench.py (2018 photos with longer side 1200, target 800; 64
distinct photos cycled), resident in torch as (H, W, 3) uint8 CUDA tensors (one per distinct photo, the batch list
refers to them), and as numpy arrays for the host route.

Reported:
  upload_photos     from the device tensors vs from numpy (host clock around calls that end in a synchronise, median of
                    --reps, the two routes alternated)
  device_pack       kernel time (CUDA events of vpk_profile) and bytes/s (bytes read + written) for HWC tensors and for
                    CHW tensors passed as t.permute(1, 2, 0), against a device-to-device copy measured in the same run
  fetch             fetch(device=True) (ends in torch.cuda.synchronize) vs fetch(raw=True) and fetch() on the run of
                    that batch, median of --fetch-reps
  the card's name and power limit.

    python tools/device_io_bench.py --out profiles/r8_device_io_bench.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from image_prep_bench import d2d_copy_tbps, hlw_batch  # noqa: E402
from lsd_bench import card  # noqa: E402
from vanishing_points_2017_b200 import pipeline  # noqa: E402
from vanishing_points_2017_b200 import cnn as vcnn  # noqa: E402


def wall(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), [round(t, 6) for t in ts]


def pack_kernel(pipe, photos, target, reps):
    ctx = pipe.ctx
    pipe.upload_photos(photos, target)                      # warm-up
    ctx.profile_reset()
    ctx.profile_enable(True)
    for _ in range(reps):
        pipe.upload_photos(photos, target)
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    ms = prof["device_pack"]["ms"] / prof["device_pack"]["launches"]
    nbytes = 2 * sum(int(p.numel()) for p in photos)          # read + written
    return {"ms": round(ms, 4), "bytes_read_plus_written": nbytes, "tbps": round(nbytes / (ms * 1e-3) / 1e12, 3),
            "image_prep_ms": round(prof["image_prep"]["ms"] / prof["image_prep"]["launches"], 4)}


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/device_io_bench.json")
    ap.add_argument("--images", type=int, default=2018)
    ap.add_argument("--segments", type=int, default=300)
    ap.add_argument("--target", type=int, default=800)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--pack-reps", type=int, default=5)
    ap.add_argument("--fetch-reps", type=int, default=21)
    args = ap.parse_args()
    res = {"card": card(), "images": args.images, "target": args.target}
    photos = hlw_batch(args.images, args.segments)
    distinct = {}
    for p in photos:
        if id(p) not in distinct:
            distinct[id(p)] = torch.from_numpy(p).cuda()
    dev = [distinct[id(p)] for p in photos]
    chw_store = {k: t.permute(2, 0, 1).contiguous() for k, t in distinct.items()}
    chw = [chw_store[id(p)].permute(1, 2, 0) for p in photos]
    res["distinct_photos"] = len(distinct)
    res["photo_bytes"] = int(sum(p.size for p in photos))
    ws, bs = vcnn.random_weights(0, scale=3.0)
    pipe = pipeline.Pipeline(0, ws, bs, sphere_mode="votes")

    # the two routes must agree before they are timed
    c_dev, s_dev = pipe.upload_photos(dev, args.target)
    c_host, s_host = pipe.upload_photos(photos, args.target)
    c_chw, s_chw = pipe.upload_photos(chw, args.target)
    assert c_dev.tolist() == c_host.tolist() == c_chw.tolist() and s_dev == s_host == s_chw
    res["segments_detected"] = int(c_dev.sum())

    times = {"device": [], "host": []}
    for _ in range(args.reps):
        for k, batch in (("device", dev), ("host", photos)):
            t0 = time.perf_counter()
            pipe.upload_photos(batch, args.target)
            times[k].append(time.perf_counter() - t0)
    res["upload_photos_s"] = {k: {"median": round(float(np.median(v)), 4), "all": [round(t, 4) for t in v]} for k, v in times.items()}
    res["upload_photos_speedup"] = round(res["upload_photos_s"]["host"]["median"] / res["upload_photos_s"]["device"]["median"], 3)
    print("upload_photos", json.dumps(res["upload_photos_s"]), flush=True)

    res["d2d_copy_tbps_read_plus_write"] = round(d2d_copy_tbps(), 3)
    res["device_pack_hwc"] = pack_kernel(pipe, dev, args.target, args.pack_reps)
    res["device_pack_chw"] = pack_kernel(pipe, chw, args.target, args.pack_reps)
    print("device_pack", json.dumps({"hwc": res["device_pack_hwc"], "chw": res["device_pack_chw"],
                                     "copy_tbps": res["d2d_copy_tbps_read_plus_write"]}), flush=True)

    pipe.upload_photos(dev, args.target)
    pipe.run()
    host = pipe.fetch(raw=True)
    d = pipe.fetch(device=True)
    torch.cuda.synchronize()
    for k in pipeline.RAW_PER_IMAGE + ("vp_assoc",):
        assert np.array_equal(d[k].cpu().numpy(), host[k]), k

    def fetch_device():
        pipe.fetch(device=True)
        torch.cuda.synchronize()

    fetch_device()
    t_dev, all_dev = wall(fetch_device, args.fetch_reps)
    t_host, all_host = wall(lambda: pipe.fetch(raw=True), args.fetch_reps)
    t_dicts, _ = wall(pipe.fetch, args.fetch_reps)
    res["fetch_ms"] = {"device": round(t_dev * 1e3, 4), "host_raw": round(t_host * 1e3, 4), "host_dicts": round(t_dicts * 1e3, 4),
                       "device_all": all_dev, "host_raw_all": all_host}
    print("fetch", json.dumps(res["fetch_ms"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"card": res["card"], "upload_photos_s": {k: v["median"] for k, v in res["upload_photos_s"].items()},
                      "device_pack_hwc": res["device_pack_hwc"], "device_pack_chw": res["device_pack_chw"],
                      "fetch_ms": {k: res["fetch_ms"][k] for k in ("device", "host_raw", "host_dicts")}}))


if __name__ == "__main__":
    main()
