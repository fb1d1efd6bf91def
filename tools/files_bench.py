"""Mixed batches of files on the device (Pipeline.upload_files, row N8) against the per-format calls on the same files
in the same run, and the preparation kernel on gray photos against RGB photos of equal sizes.

Batch (HLW-shaped, target 800): `--files` files whose longer side is drawn from 800 to 2000 with the aspects of
synth.CONFIGS[4]; about 70 % colour JPEG, 10 % gray JPEG, 15 % colour PNG, 4 % gray PNG and 1 % PGM, in a shuffled
order (oracle.jpeg_oracle.photo content, cv2.imencode defaults; `--distinct` distinct files per kind, cycled).

Reported: the files' sizes; Pipeline.upload_files on the host clock around the call, which ends in a device
synchronise (median of `--reps`); beside it the per-format path a caller had before: upload_jpegs on the colour JPEG
files, upload_pngs on the colour PNG files and, for the gray files, the host decode (cv2.imdecode) and resize
(cv2.resize INTER_AREA) followed by upload_images, each call timed the same way and summed; then the image_prep kernel
(CUDA events of vpk_profile) on `--prep-photos` photos as RGB (vpk_prepare_images) and as gray PGM files of the same
sizes (vpk_prepare_files), and the card and its power limit.

    python tools/files_bench.py --out profiles/r7_files_bench.json
"""
import argparse
import json
import os
import sys
import time
from multiprocessing import Pool

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from lsd_bench import card  # noqa: E402
from oracle import files_oracle as F  # noqa: E402
from oracle import jpeg_oracle as J  # noqa: E402
from oracle import png_oracle as G  # noqa: E402
from vanishing_points_2017_b200 import images, pipeline, synth  # noqa: E402
from vanishing_points_2017_b200 import cnn as vcnn  # noqa: E402

KINDS = [("jpeg_rgb", 0.70), ("jpeg_gray", 0.10), ("png_rgb", 0.15), ("png_gray", 0.04), ("pgm", 0.01)]
TEXTURE = 12


def _encode(args):
    kind, seed, w, h = args
    img = J.photo(seed, w, h, texture=TEXTURE)
    if kind == "jpeg_rgb":
        return J.encode_cv2(img)
    gray = np.ascontiguousarray(img[:, :, 1])
    if kind == "jpeg_gray":
        import cv2
        return cv2.imencode(".jpg", gray, [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes()
    if kind == "png_rgb":
        return G.encode_cv2(img)
    if kind == "png_gray":
        return G.encode_cv2(gray)
    return F.write_pgm(gray)


def shapes(n, seed):
    _, _, _, _, _, _, aspects = synth.CONFIGS[4]
    rs = np.random.RandomState(seed)
    out = []
    for i, side in zip(rs.randint(0, len(aspects), n), rs.randint(800, 2001, n)):
        w, h = aspects[i]
        s = side / max(w, h)
        out.append((max(1, int(round(w * s))), max(1, int(round(h * s)))))
    return out


def mixed_batch(n, distinct):
    rs = np.random.RandomState(7_000_001)
    kinds = []
    for name, share in KINDS:
        kinds += [name] * max(1, int(round(n * share)))
    kinds = [kinds[i] for i in rs.permutation(len(kinds))][:n]
    specs = []
    for k, (name, _) in enumerate(KINDS):
        specs += [(name, 97_000 + 1000 * k + j, w, h) for j, (w, h) in enumerate(shapes(distinct, 11 + k))]
    with Pool(min(16, os.cpu_count() or 1)) as pool:
        files = pool.map(_encode, specs)
    by_kind = {name: files[k * distinct:(k + 1) * distinct] for k, (name, _) in enumerate(KINDS)}
    count = {name: 0 for name, _ in KINDS}
    batch = []
    for name in kinds:
        batch.append(by_kind[name][count[name] % distinct])
        count[name] += 1
    return batch, kinds


def timed(fn, reps):
    fn()                                            # warm-up: modules, workspaces
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def host_gray(files, target):
    import cv2
    out = []
    for b in files:
        g = cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_UNCHANGED)
        W, H = images.prepared_size(g.shape[1], g.shape[0], target)
        out.append(g if (W, H) == (g.shape[1], g.shape[0]) else cv2.resize(g, (W, H), interpolation=cv2.INTER_AREA))
    return out


def prep_kernel_ms(ctx, fn, reps):
    fn()
    ctx.profile_reset()
    ctx.profile_enable(True)
    for _ in range(reps):
        fn()
    ctx.synchronize()
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    p = prof["image_prep"]
    return round(p["ms"] / p["launches"], 3), {k: round(v["ms"] / reps, 3) for k, v in prof.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/files_bench.json")
    ap.add_argument("--files", type=int, default=2000)
    ap.add_argument("--distinct", type=int, default=24)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--prep-photos", type=int, default=256)
    ap.add_argument("--target", type=int, default=800)
    a = ap.parse_args()
    res = {"card": card(), "host_cpus": os.cpu_count(), "reps": a.reps, "target_size": a.target}
    t0 = time.time()
    batch, kinds = mixed_batch(a.files, a.distinct)
    info = images.file_info(batch)
    res["batch"] = {"files": len(batch), "encode_s": round(time.time() - t0, 1),
                    "per_kind": {name: kinds.count(name) for name, _ in KINDS},
                    "megapixels": round(sum(w * h for _, w, h, _, _ in info) / 1e6, 1),
                    "file_mb": round(sum(len(b) for b in batch) / 1e6, 1)}
    ws, bs = vcnn.random_weights(0, scale=3.0)
    pipe = pipeline.Pipeline(0, ws, bs, sphere_mode="votes")
    ctx = pipe.ctx
    T = a.target

    def mixed():
        counts, _, st = pipe.upload_files(batch, T)
        assert not st.any()
    res["upload_files_s_median"] = round(timed(mixed, a.reps), 4)
    jr = [b for b, k in zip(batch, kinds) if k == "jpeg_rgb"]
    pr = [b for b, k in zip(batch, kinds) if k == "png_rgb"]
    gr = [b for b, k in zip(batch, kinds) if k in ("jpeg_gray", "png_gray", "pgm")]
    split = {"upload_jpegs_s_median": round(timed(lambda: pipe.upload_jpegs(jr, T), a.reps), 4),
             "upload_pngs_s_median": round(timed(lambda: pipe.upload_pngs(pr, T), a.reps), 4),
             "gray_host_decode_resize_then_upload_images_s_median":
                 round(timed(lambda: pipe.upload_images(host_gray(gr, T)), a.reps), 4)}
    split["sum_s"] = round(sum(split.values()), 4)
    res["per_format_calls"] = split
    res["upload_files_over_per_format"] = round(res["upload_files_s_median"] / split["sum_s"], 3)
    # the preparation kernel: the same photos as RGB and as gray
    sh = shapes(a.prep_photos, 3)
    photos = [J.photo(50_000 + k, w, h, texture=TEXTURE) for k, (w, h) in enumerate(sh[:16])]
    photos = [photos[k % len(photos)] for k in range(a.prep_photos)]
    pgms = [F.write_pgm(np.ascontiguousarray(p[:, :, 1])) for p in photos]
    rgb_ms, _ = prep_kernel_ms(ctx, lambda: images.prepare_images(photos, T, ctx=ctx), a.reps)
    gray_ms, gray_all = prep_kernel_ms(ctx, lambda: images.prepare_files(pgms, T, ctx=ctx), a.reps)
    px = sum(w * h for w, h in (p.shape[1::-1] for p in photos))
    res["image_prep"] = {"photos": a.prep_photos, "megapixels": round(px / 1e6, 1), "rgb_kernel_ms": rgb_ms,
                         "gray_kernel_ms": gray_ms, "gray_over_rgb": round(gray_ms / rgb_ms, 3),
                         "bytes_read_rgb": 3 * px, "bytes_read_gray": px}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
