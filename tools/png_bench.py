"""PNG decoding on the device (vpk_decode_pngs / Pipeline.upload_pngs, row N7) against host decoding (cv2.imdecode on
all host cores) and the host-decode + upload_photos path, on the same files in the same run.

Batches (oracle.jpeg_oracle.photo: synth.render_photo plus uniform noise texture of +-`--texture`; cv2.imencode with
its defaults):
  HLW-shaped      2018 files with longer side 1200 (the aspects of synth.CONFIGS[4] times 1.5), target 800;
                  64 distinct files cycled
  example-shaped  102 files 2000x1333 / 1333x2000, target 640; 32 distinct files cycled
  one 6000x4000   a single file, target 640: the weak case of one warp per file

Reported per batch: compressed size and bits per pixel; every decode kernel's time (CUDA events of vpk_profile over
`--reps` calls) and decoded megapixels per second of their sum; one decode_pngs call on the host clock (host walk,
copies and pixels back included); cv2.imdecode on all host cores; PNGs -> horizons photos/s through upload_pngs
against host decode + upload_photos.  Also one 640x480 file's decode kernels beside the LSD kernels of the same
image, and the card and its power limit.

    python tools/png_bench.py --out profiles/r6_png_bench.json
"""
import argparse
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
from oracle import png_oracle as P  # noqa: E402
from vanishing_points_2017_b200 import _lib, images, pipeline, synth  # noqa: E402
from vanishing_points_2017_b200 import cnn as vcnn  # noqa: E402

TEXTURE = 12


def _encode(args):
    seed, w, h, texture = args
    return P.encode_cv2(P.photo(seed, w, h, texture=texture))


def encode_many(specs):
    with Pool(min(16, os.cpu_count() or 1)) as pool:
        return pool.map(_encode, specs)


def hlw_batch(n, texture, distinct=64):
    _, _, _, _, _, _, aspects = synth.CONFIGS[4]
    rs = np.random.RandomState(4_000_037)
    shapes = [aspects[i] for i in rs.randint(0, len(aspects), n)]
    shapes = [(int(round(w * 1.5)), int(round(h * 1.5))) for w, h in shapes]
    keys = sorted(set(shapes))
    per = max(1, distinct // len(keys))
    files = encode_many([(95_000 + 100 * i + j, w, h, texture) for i, (w, h) in enumerate(keys) for j in range(per)])
    by_shape = {k: files[i * per:(i + 1) * per] for i, k in enumerate(keys)}
    return [by_shape[s][k % per] for k, s in enumerate(shapes)]


def example_batch(n, texture, distinct=32):
    files = encode_many([(90_000 + k, 2000, 1333, texture) if k % 2 == 0 else (90_000 + k, 1333, 2000, texture)
                         for k in range(distinct)])
    return [files[k % distinct] for k in range(n)]


def pixels(files):
    return sum(w * h for w, h, _, _ in images.png_info(files))


def kernel_times(ctx, fn, reps, prefix):
    fn()                                            # warm-up
    ctx.profile_reset()
    ctx.profile_enable(True)
    for _ in range(reps):
        fn()
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    return {k: round(v["ms"] / reps, 3) for k, v in prof.items() if k.startswith(prefix)}


def decode_call(files, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        _, st = images.decode_pngs(files)
        ts.append(time.perf_counter() - t0)
    assert not st.any()
    return round(float(np.median(ts)), 4)


def host_decode(files, reps):
    import cv2
    cv2.setNumThreads(1)
    flags = cv2.IMREAD_COLOR | cv2.IMREAD_IGNORE_ORIENTATION

    def one(b):
        return cv2.imdecode(np.frombuffer(b, np.uint8), flags)[:, :, ::-1]
    n = os.cpu_count()
    with ThreadPoolExecutor(max_workers=n) as ex:
        list(ex.map(one, files[:2 * n]))
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            list(ex.map(one, files))
            ts.append(time.perf_counter() - t0)
    med = float(np.median(ts))
    return {"threads": n, "s_median": round(med, 4), "images_per_s": round(len(files) / med, 1)}, one


def end_to_end(pipe, files, target, reps, host_one):
    n = os.cpu_count()

    def via_pngs():
        pipe.upload_pngs(files, target)
        pipe.run()
        return pipe.horizons()

    def via_host():
        with ThreadPoolExecutor(max_workers=n) as ex:
            photos = list(ex.map(host_one, files))
        pipe.upload_photos(photos, target)
        pipe.run()
        return pipe.horizons()
    out = {}
    for name, fn in (("pngs_to_horizons", via_pngs), ("host_decode_then_upload_photos", via_host)):
        fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        med = float(np.median(ts))
        out[name] = {"s_median": round(med, 4), "images_per_s": round(len(files) / med, 1)}
    return out


def run_batch(ctx, pipe, files, target, reps):
    px = pixels(files)
    nbytes = sum(len(b) for b in files)
    ks = kernel_times(ctx, lambda: images.decode_pngs(files), reps, "png_")
    dec_ms = sum(ks.values())
    host, one = host_decode(files, reps)
    return {"files": len(files), "megapixels": round(px / 1e6, 2), "png_mb": round(nbytes / 1e6, 2),
            "bits_per_pixel": round(8.0 * nbytes / px, 3), "kernels_ms": ks, "decode_kernels_ms": round(dec_ms, 3),
            "decode_mp_per_s": round(px / 1e6 / (dec_ms * 1e-3), 1), "decode_call_s_median": decode_call(files, reps),
            "host_cv2_imdecode": host, "end_to_end": end_to_end(pipe, files, target, reps, one), "target": target}


def single_640x480(ctx, pipe, texture, reps):
    """one 640x480 file: the decode kernels against the LSD kernels of the same image (upload_photos, no resize)"""
    blob = _encode((91, 640, 480, texture))
    dec = kernel_times(ctx, lambda: images.decode_pngs([blob]), reps, "png_")
    photo = P.decode(blob)
    lsd = kernel_times(ctx, lambda: pipe.upload_photos([photo], None), reps, "lsd_")
    return {"png_bytes": len(blob), "decode_kernels_ms": round(sum(dec.values()), 3), "kernels_ms": dec,
            "lsd_kernels_ms": round(sum(lsd.values()), 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/png_bench.json")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--texture", type=int, default=TEXTURE)
    ap.add_argument("--hlw-images", type=int, default=2018)
    ap.add_argument("--example-images", type=int, default=102)
    ap.add_argument("--batches", default="one_640x480,hlw_shaped,example_shaped,one_6000x4000",
                    help="comma-separated subset of the batches to run")
    a = ap.parse_args()
    want = set(a.batches.split(","))
    res = {"card": card(), "host_cores": os.cpu_count(), "texture": a.texture, "reps": a.reps}
    ctx = _lib.default_context()
    ws, bs = vcnn.random_weights(0, scale=3.0)
    pipe = pipeline.Pipeline(0, ws, bs, sphere_mode="votes")
    if "one_640x480" in want:
        res["one_640x480"] = single_640x480(ctx, pipe, a.texture, a.reps)
        print("one_640x480", json.dumps(res["one_640x480"]), flush=True)
    batches = [("hlw_shaped", lambda: hlw_batch(a.hlw_images, a.texture), 800),
               ("example_shaped", lambda: example_batch(a.example_images, a.texture), 640),
               ("one_6000x4000", lambda: [_encode((7, 6000, 4000, a.texture))], 640)]
    for key, make, target in batches:
        if key not in want:
            continue
        files = make()
        r = run_batch(ctx, pipe, files, target, a.reps)
        res[key] = r
        print(key, json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
