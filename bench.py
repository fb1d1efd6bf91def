#!/usr/bin/env python
"""bench.py -- images/sec of the lines->VPs hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config C] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the path (segments -> lines -> sphere votes -> CNN ->
EM -> VPs) over one synthetic batch of BASELINE.json config C.
  N = 1 (default config 2): the YUD-shaped batch, 102 images 640x480, ~500 segments, single B200.
  N > 1 (default config 4, launched by torch.distributed.run, one rank per GPU): STRONG scaling of
        the ONE HLW-shaped batch of 2018 images (BASELINE.json configs[3], "sharded across 1/2/4/8
        B200"; the reference loops per file, evaluation.py:126, 271, 309): rank r runs
        pipeline.shard_batch(offsets, N, r) (cost-balanced, images are independent, no data-path
        collective) and the per-image results are gathered on rank 0 INSIDE the timed e2e region;
        value = 2018 / (max over ranks of the step time).  `--weak` restores the fixed-per-GPU-work mode
        (every rank runs its own copy of the batch); `--strong` with N = 1 gives the one-GPU figure
        of the same workload.

value    : whole-job images/s over K steps with the batch already resident in HBM, `--inflight` (default 4)
           steps in flight per GPU -- one library context and host thread each (pipeline.StreamedPipeline):
           the EM of a batch is a chain of dependent supersteps that leaves SMs idle, the next batches'
           sphere mapping / CNN / pair pass fill them.  Device time between CUDA events on the library's
           streams (first start mark -> last end mark), max over ranks.  `serial` is the same with ONE batch at a
           time (the latency of a batch).
e2e      : same metric through the public API from pinned HOST buffers, H2D and D2H (and, with several ranks,
           the result gather) inside the timed region, the same number of calls in flight.
roofline : dominant kernel of the step vs the measured peak in MEASURED_PEAKS.json.
cpu_baseline / --impl reference : the CPU oracle (numpy/torch restatement of the
           reference path, oracle/) on a bounded sample of the same batch.
--dump-outputs DIR : the EM result of the last end-to-end step (after the gather, with several ranks) as
           DIR/<name>.npy; the inputs depend on the arguments only, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from vanishing_points_2017_b200 import synth  # noqa: E402

METRIC = "images/sec end-to-end (lines->VPs)"
UNIT = "images/s"
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}

# algorithmic MACs per image of cnn/deploy.prototxt (SURVEY.md section 8(a))
CNN_MACS = {"gemm_conv1": 175_738_464, "gemm_conv2": 1_143_091_200, "gemm_conv3": 796_262_400,
            "gemm_conv4": 597_196_800, "gemm_conv5": 398_131_200, "gemm_fc6": 235_929_600,
            "gemm_fc7": 16_777_216, "gemm_fc8": 1_638_400}


def ncu_traffic(workload, kernel):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of `kernel` from the committed
    `ncu --set full` capture of this workload (profiles/ncu_traffic.json, written by tools/ncu_summary.py)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return float(json.load(open(p))[workload][kernel]["dram_bytes_per_launch"])
    except Exception:
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            d["_source"] = "measured"
            return d
        except Exception:
            pass
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region.  Sampled in-process through NVML
    (pynvml) so that no `nvidia-smi` process is spawned beside a launch-heavy timed region;
    falls back to nvidia-smi if NVML cannot be loaded."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.period = index, [], False, period
        self.nv = self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[index])
            except Exception:
                pass
        return index

    def _sample_nvml(self):
        nv = self.nv
        mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
        flags = [bool(r & 0x8), bool(r & 0x40), bool(r & 0x20), bool(r & 0x4)]   # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
        return [str(mhz), str(self.max_mhz)] + ["Active" if f else "Not Active" for f in flags]

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        parts = [x.strip() for x in out.strip().split(",")]
        return parts if len(parts) >= 6 else None

    def run(self):
        while not self.stop_flag:
            try:
                parts = self._sample_nvml() if self.nv else self._sample_smi()
                if parts:
                    self.samples.append(parts)
            except Exception:
                pass
            time.sleep(self.period if self.nv else max(self.period, 0.2))

    def summary(self):
        self.stop_flag = True
        self.join(timeout=3)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = [n for k, n in enumerate(self.NAMES) if any(s[2 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(self.samples), "source": "nvml" if self.nv else "nvidia-smi"}


def make_workload(cfg, rank, n_images=None):
    """The batch of config `cfg` for this rank (rank r draws seeds disjoint from rank 0's)."""
    name, B = synth.CONFIGS[cfg][0], synth.CONFIGS[cfg][1]
    if n_images is not None:
        B = n_images
    n, asp = synth.config_sizes(cfg, B)
    segs = []
    for idx in range(B):
        sc = synth.make_scene(1_000_003 * cfg + 100_000 * rank + idx, int(n[idx]), asp[idx][0], asp[idx][1])
        segs.append(sc["segments"])
    off = np.zeros(B + 1, dtype=np.int32)
    off[1:] = np.cumsum(n)
    return name, np.concatenate(segs, axis=0), off


DUMP_LIMIT_BYTES = 60_000_000          # array data; with the .npy headers the files stay below 64 MB


def dump_outputs(dirname, res, off):
    """The flat EM result arrays of one step (Pipeline(..., raw=True), or pipeline.gather_raw's with several ranks) as
    DIR/<name>.npy in float64.  Entries the library leaves undefined (VP rows beyond n_vp; every field but `status`
    of an image without VPs) are stored as 0, so that two runs compare byte for byte; `vp_assoc` is in image order.
    Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of the images is stored; `image_index` lists the images stored."""
    B, M = len(off) - 1, res["vp"].shape[1]
    n = np.diff(off).astype(np.int64)
    start = np.asarray(res.get("assoc_start", off[:-1]), dtype=np.int64)
    keep = np.arange(B)
    per_image = 8 * (4 + 6 * M + n)
    if per_image.sum() > DUMP_LIMIT_BYTES:
        order = np.random.RandomState(0).permutation(B)
        keep = np.sort(order[:np.searchsorted(np.cumsum(per_image[order]), DUMP_LIMIT_BYTES, side="right")])
    ok = res["status"][keep] == 0
    n_vp = np.where(ok, res["n_vp"][keep], 0)
    rows = np.arange(M)[None, :] < n_vp[:, None]
    out = {"image_index": keep, "status": res["status"][keep], "n_vp": n_vp,
           "iterations": np.where(ok, res["iterations"][keep], 0), "vp": np.where(rows[:, :, None], res["vp"][keep], 0.0)}
    for k in ("sigma", "counts", "counts_weighted"):
        out[k] = np.where(rows, res[k][keep], 0)
    out["vp_assoc"] = np.concatenate([np.zeros(0)] + [res["vp_assoc"][start[i]:start[i] + n[i]] if good else np.zeros(n[i])
                                                      for i, good in zip(keep, ok)])
    os.makedirs(dirname, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(dirname, k + ".npy"), np.asarray(a, dtype=np.float64))


# ------------------------------------------------------------------ CPU oracle arm
def oracle_pipeline(seg, off, idx, weights, biases):
    """The CPU restatement of the reference path on images `idx`: numpy sphere votes,
    torch-CPU fp32 CNN, numpy EM (oracle/)."""
    from oracle import cnn_oracle, sphere_oracle, vp_oracle
    n_ok = 0
    for i in idx:
        s = seg[off[i]:off[i + 1]]
        lines = synth.lines_from_segments(s)
        img = sphere_oracle.votes_to_image(sphere_oracle.sphere_votes(lines, 500))
        sig, _ = cnn_oracle.forward(img[None], weights, biases)
        try:
            res = vp_oracle.expectation_maximisation(lines, s.copy(), sig[0], sphere_image=img)
            n_ok += res["vp"] is not None
        except ValueError:
            pass
    return n_ok


def time_oracle(seg, off, weights, biases, sample, repeats=1):
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    idx = np.linspace(0, len(off) - 2, sample).astype(int)
    t0 = time.perf_counter()
    for _ in range(repeats):
        oracle_pipeline(seg, off, idx, weights, biases)
    dt = (time.perf_counter() - t0) / repeats
    return sample / dt, dt


def time_reference_em(seg, off, weights, biases, sample):
    """The reference's OWN EM (vp_localisation.expectation_maximisation, Python-3-patched copy in the
    git-ignored baseline/_ref/, written by __graft_entry__.build() where /root/reference exists; BASELINE.md
    section 3) on `sample` images of the batch, joblib on all host cores like the original.  Sphere image and
    CNN response come from the port (matplotlib / Caffe are not installable).  None if baseline/_ref is absent."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref_dir, "vp_localisation.py")):
        return None
    import contextlib
    import io
    import warnings
    from oracle import cnn_oracle, ref_patch, sphere_oracle
    try:
        vp, _ = ref_patch.load(ref_dir)
    except Exception as e:                       # e.g. sklearn / joblib missing on the box
        return {"unavailable": "%s: %s" % (type(e).__name__, e)}
    idx = np.linspace(0, len(off) - 2, sample).astype(int)
    prep = []
    for i in idx:
        sgm = seg[off[i]:off[i + 1]]
        lines = synth.lines_from_segments(sgm)
        img = sphere_oracle.votes_to_image(sphere_oracle.sphere_votes(lines, 500))
        sig, _ = cnn_oracle.forward(img[None], weights, biases)
        prep.append((lines, sgm.copy(), sig[0].astype(np.float64), img))
    t0 = time.perf_counter()
    with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
        warnings.simplefilter("ignore")
        for lines, sgm, sig, img in prep:
            try:
                vp.expectation_maximisation(lines, sgm, sig, sphere_image=img, distance_measure="angle", use_weights=True,
                                            do_split=True, do_merge=True)
            except ValueError:
                pass
    dt = time.perf_counter() - t0
    return {"value": sample / dt, "unit": "images/s (EM stage only)", "seconds": dt, "images": int(sample),
            "segments": [int(off[i + 1] - off[i]) for i in idx], "cores": os.cpu_count() or 1,
            "what": "UNMODIFIED arithmetic of the reference's vp_localisation.expectation_maximisation "
                    "(five mechanical Python-3 patches, baseline/_ref/), joblib over all cores"}


def run_reference(args, rank, world):
    """--impl reference: the CPU path on the box's host cores, rank 0 only."""
    if rank != 0:
        return
    from oracle import cnn_oracle
    name, seg, off = make_workload(args.config, 0, args.images)
    ws, bs = cnn_oracle.random_weights(0, scale=args.weight_scale)
    sample = 2
    for _ in range(args.warmup):
        time_oracle(seg, off, ws, bs, sample)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        time_oracle(seg, off, ws, bs, sample)
    dt = (time.perf_counter() - t0) / args.steps
    v = sample / dt
    cores = os.cpu_count() or 1
    ref_em = None if args.no_reference_em else time_reference_em(seg, off, ws, bs, 2)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s-shaped synthetic batch (BASELINE.json configs[%d])" % (name, args.config - 1),
                       "sample": "%d images per step, evenly spaced over the %d-image batch" % (sample, len(off) - 1)},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d images/step of the same batch; numpy+torch CPU oracle (oracle/), "
                                       "BLAS/torch threads = %d" % (sample, cores),
                             "reference_em": ref_em},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------ GPU arm
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from vanishing_points_2017_b200 import cnn as vcnn, pipeline

    torch.cuda.set_device(local_rank)
    host_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # the result gather runs over host memory (gloo): the results are on the host when a step returns and the GPU's
        # streams are busy with the next batches -- no NCCL on the path (north_star)
        host_group = dist.new_group(backend="gloo")
    peaks = load_peaks()
    name, seg_all, off_all = make_workload(args.config, 0, args.images)
    B_all = len(off_all) - 1
    if args.strong:
        # STRONG scaling: the one batch is sharded (LPT on the N^2 + const cost model); rank r owns images `idx`
        idx = pipeline.shard_batch(off_all, world, rank)
        seg, off = pipeline.take_images(seg_all, off_all, idx)
    else:
        # weak scaling with FIXED per-GPU work: every rank processes the same synthetic batch
        idx = np.arange(B_all)
        seg, off = seg_all, off_all
    B = len(off) - 1
    ws, bs = vcnn.random_weights(0, scale=args.weight_scale)
    # `depth` batches in flight: one library context + one host thread each (pipeline.StreamedPipeline); the serial
    # and the profiled legs use the first context alone
    depth = max(1, args.inflight)
    em_kw = {}
    if args.num_init_vp is not None or args.config == 5:
        em_kw["num_init_vp"] = args.num_init_vp if args.num_init_vp is not None else 32
    sp = pipeline.StreamedPipeline(local_rank, ws, bs, depth=depth, sphere_mode=args.sphere_mode, **em_kw)
    pipe = sp.pipes[0]
    ctx = pipe.ctx

    # pinned host inputs for the end-to-end leg
    seg_pin = torch.from_numpy(seg).pin_memory()
    off_pin = torch.from_numpy(off).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        for q in sp.pipes:
            q.ctx.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def flush_l2():
        flush.zero_()
        torch.cuda.synchronize()

    # ---- resident leg: `value` (no per-kernel events inside the timed region)
    pipe.upload(seg_pin.numpy(), off_pin.numpy())
    for _ in range(args.warmup):
        pipe.run()
    # settle: further untimed warm-up steps until three in a row are within 5 % of the fastest one seen
    # (a fresh box keeps paging the image in for a while and disturbs the first steps), at most 30
    settle, best, streak = 0, float("inf"), 0
    while settle < args.settle and streak < 3:
        pipe.run()
        t = pipe.stage_ms()["total"]
        best = min(best, t)
        streak = streak + 1 if t <= 1.05 * best else 0
        settle += 1
    # ---- serial leg: ONE batch at a time on one context (the latency of a batch; per-stage device times)
    barrier()
    dev_ms, stage, step_ms = 0.0, {"sphere": 0.0, "cnn": 0.0, "em": 0.0}, []
    for _ in range(args.steps):
        flush_l2()
        pipe.run()
        ms = pipe.stage_ms()
        dev_ms += ms["total"]
        step_ms.append(ms["total"])
        for k in stage:
            stage[k] += ms[k]
    barrier()
    serial_ms = dev_ms / args.steps
    results = pipe.fetch(raw=True)
    n_ok = int(np.sum(results["status"] == 0))

    # ---- resident leg -> `value`: K steps, `depth` of them in flight (step i runs on context i % depth); device time
    # from the first context's start mark to the last context's end mark.  No global synchronisation (hence no L2
    # flush) inside the region: every step streams > 1 GB of intermediates (similarity matrices, activations)
    # through the 126 MB L2, nothing of a previous step survives in it.
    import threading
    for q in sp.pipes[1:]:
        q.upload(seg_pin.numpy(), off_pin.numpy())
        for _ in range(args.warmup):
            q.run()
    gate = threading.Barrier(depth)

    def resident_worker(q):
        k = sp.pipes.index(q)
        gate.wait()
        q.ctx.mark(0)
        for _ in range(k, args.steps, depth):
            q.run()
        q.ctx.mark(1)
        return True

    sp.each(resident_worker)                      # one untimed pass in the overlapped regime
    sampler = ClockSampler(local_rank, args.clock_period)
    sampler.start()
    barrier()
    launches0 = sum(q.ctx.launch_count() for q in sp.pipes)
    t0 = time.perf_counter()
    sp.each(resident_worker)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    used = [q for k, q in enumerate(sp.pipes) if k < args.steps]
    dev_total_ms = max(a.ctx.elapsed_ms(0, b.ctx, 1) for a in used for b in used)
    launches = sum(q.ctx.launch_count() for q in sp.pipes) - launches0

    # ---- profiled leg: the same steps again with CUDA events around every kernel launch (on the
    # library's stream) -> per-kernel times, the dominant kernel and its roofline
    psteps = max(1, min(args.steps, 5))
    ctx.profile_reset()
    ctx.em_stats(reset=True)
    ctx.em_phase_cycles(reset=True)
    ctx.profile_enable(True)
    for _ in range(psteps):
        flush_l2()
        pipe.run()
    barrier()
    ctx.profile_enable(False)
    prof = ctx.profile_read()
    em_stats = ctx.em_stats()

    # ---- end-to-end leg from pinned host buffers -> `e2e`: every step is one public-API call (H2D, path, D2H), `depth`
    # calls in flight; with several ranks the results of every step are then gathered on rank 0 (in step order, on this
    # thread).  Wall clock between two barriers: host work, copies and the gather are all inside.
    e2e_wait = [0.0]
    from concurrent.futures import ThreadPoolExecutor
    gather_pool = ThreadPoolExecutor(max_workers=1)      # ONE thread: every rank issues its gathers in step order

    def gather_step(res):
        # the path's only exchange: the per-image results of every shard end up on rank 0
        tg = time.perf_counter()
        full_ = pipeline.gather_raw(res, off_all, world, rank, dist, group=host_group)
        return full_, (time.perf_counter() - tg) * 1e3

    def e2e_steps(n_steps, seg_h, off_h, gather):
        last, gfuts = None, []
        futs = [sp.submit(seg_h, off_h, raw=True) for _ in range(min(depth, n_steps))]
        for i in range(n_steps):
            tw = time.perf_counter()
            last = futs[i % depth].result()
            e2e_wait[0] += (time.perf_counter() - tw) * 1e3
            if i + depth < n_steps:
                futs[i % depth] = sp.submit(seg_h, off_h, raw=True)
            if gather:
                gfuts.append(gather_pool.submit(gather_step, last))     # off the submit loop; completed inside the timed region
        done = [g.result() for g in gfuts]
        return last, (done[-1][0] if done else None), sum(d[1] for d in done)

    do_gather = args.strong and world > 1
    e2e_steps(max(depth, args.warmup // 2), seg_pin.numpy(), off_pin.numpy(), do_gather)
    barrier()
    e2e_wait[0] = 0.0
    t0 = time.perf_counter()
    out, full, gather_ms = e2e_steps(args.steps, seg_pin.numpy(), off_pin.numpy(), do_gather)
    wait_ms = e2e_wait[0] / args.steps
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    clocks = sampler.summary()            # sampled over both timed legs (and the profiled leg between them)
    h2d = seg.nbytes + off.nbytes
    d2h = sum(a.nbytes for a in out.values() if a is not None)
    n_ok_all = None
    if args.strong and world > 1 and rank == 0:
        n_ok_all = int(np.sum(full["status"] == 0))
        assert full["status"].shape[0] == B_all and full["vp_assoc"].shape[0] == int(off_all[-1])

    # ---- strong scaling: the one-GPU figure of the SAME batch, measured by rank 0 in this very run
    one_gpu = None
    if args.strong and world > 1:
        if rank == 0:
            sa, oa = torch.from_numpy(seg_all).pin_memory(), torch.from_numpy(off_all).pin_memory()
            e2e_steps(depth, sa.numpy(), oa.numpy(), False)
            k1 = max(depth, min(args.steps, 4))
            t1 = time.perf_counter()
            e2e_steps(k1, sa.numpy(), oa.numpy(), False)
            one_gpu = {"e2e_images_per_s": B_all * k1 / (time.perf_counter() - t1), "steps": k1}
        barrier()

    # ---- reduce over ranks: max time, total images
    t = torch.tensor([dev_total_ms / args.steps, e2e_ms, wall_ms / args.steps, serial_ms], dtype=torch.float64, device="cuda")
    tmin = t.clone()
    nimg = torch.tensor([float(B), float(n_ok)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(nimg, op=dist.ReduceOp.SUM)
    ms_step, e2e_step, wall_step, serial_step = [float(x) for x in t.tolist()]
    total_images = int(nimg[0].item())
    n_ok = int(nimg[1].item())
    if args.strong:
        assert total_images == B_all

    if rank == 0:
        # Dominant kernel and its roofline.  `roofline_all` lists every kernel above 2 % of the profiled (serial) step by
        # time.  The headline `roofline` is the largest of them that is throughput-bound by construction: em_post and em_init
        # are one-CTA-per-image state machines (dependent L2 round trips and block barriers on at most one CTA per image;
        # 64 registers, so other kernels share their SMs) -- with several batches in flight, the regime `value` is
        # measured in, they overlap with the other batches' kernels and do not bound the throughput.
        STATE_MACHINES = ("em_post", "em_init", "em_poste")
        cands = {k: v for k, v in prof.items() if k not in STATE_MACHINES} or prof
        top = max(cands.items(), key=lambda kv: kv[1]["ms"]) if cands else (None, None)
        roof = None
        n = np.diff(off).astype(np.float64)

        def roofline_of(kname, k):
            avg_ms = k["ms"] / max(k["launches"], 1)
            if kname.startswith("gemm_"):
                flops = 2.0 * CNN_MACS.get(kname, 0) * B * psteps / k["launches"]
                ach = flops / (avg_ms * 1e-3) / 1e12
                peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
                r = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak}
            else:
                # HBM-bound kernels: algorithmic bytes per launch (DESIGN.md, "Kernels")
                if kname == "em_fused":
                    # the fused superstep kernel: per image and superstep the similarity matrix once (8 N^2, the
                    # weight-matrix product) + the planes the E-step writes and POST reads (counted on the device)
                    byt = (em_stats["wmat_bytes"] + em_stats["post_bytes"] + em_stats["estep_bytes"]) / max(k["launches"], 1)
                elif kname == "em_wmat":
                    # 8 N^2 bytes of similarity matrix per per-image product (counted on the device)
                    byt = em_stats["wmat_bytes"] / max(k["launches"], 1)
                elif kname == "em_poste":
                    byt = (em_stats["post_bytes"] + em_stats["estep_bytes"]) / max(k["launches"], 1)
                elif kname == "em_post":
                    byt = em_stats["post_bytes"] / max(k["launches"], 1)
                elif kname == "em_estep":
                    byt = em_stats["estep_bytes"] / max(k["launches"], 1)
                elif kname == "em_pair":
                    byt = float(np.sum(8.0 * n * n + 32.0 * n))
                elif kname == "sphere_votes":
                    byt = float(np.sum(24.0 * n) + 4.0 * 500 * 500 * B)
                elif kname in ("lrn_pool1", "pool1"):
                    byt = B * (96 * 123 * 123 * 2 + 96 * 61 * 61 * 2.0)
                elif kname in ("lrn_pool2", "pool2"):
                    byt = B * (256 * 61 * 61 * 2 + 256 * 30 * 30 * 2.0)
                else:
                    byt = 0.0
                ach = byt / (avg_ms * 1e-3) / 1e9
                r = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": ach / peaks["hbm_gbs"]}
            r.update({"traffic": ncu_traffic(name, kname), "kernel": kname, "avg_launch_ms": avg_ms,
                      "peak_source": peaks["_source"]})
            # kernels that are not bound by either roofline the contract names: say what ncu shows instead
            note = {"em_pair": "instruction-issue bound (ncu: issue slots 67 %, FP64 pipe 35 %; ~415 instructions per ordered pair)",
                    "sphere_votes": "instruction-issue bound (ncu: issue slots 55 %, ALU 31 %, XU 27 %) + L2 integer atomics",
                    "em_post": "latency bound by construction: one CTA per image, dependent L2 round trips and block barriers",
                    "em_estep": "latency bound: one short launch per superstep (rsqrt + exp in float64 per line and hypothesis)",
                    "gemm_conv1": "HBM bound (K = 121): 204 MB operand in, 296 MB normalised bf16 out per 102 images"}.get(kname)
            if note:
                r["note"] = note
            if not kname.startswith("gemm_"):
                r["algorithmic_bytes_per_launch"] = byt
            if kname in ("em_wmat", "em_post", "em_estep") and r["traffic"] is not None:
                # `achieved` averages over every superstep of the run (late ones have few active images);
                # the ncu capture behind `traffic` is of supersteps 10-12, where all images are active
                full = {"em_wmat": float(np.sum(8.0 * n * n))}.get(kname)
                r["traffic_note"] = ("ncu capture of supersteps 10-12 (every image active)" +
                                     ("; algorithmic bytes of those launches: %.0f" % full if full else ""))
            return r

        if top[0] is not None:
            roof = roofline_of(*top)
            roof["selection"] = ("largest kernel of the profiled step by time, one-CTA-per-image state machines (em_post, "
                                 "em_init) excepted: latency-bound, they overlap with the other batches in flight")
        # the same figure for every kernel with a share of the step above 2 % (the headline `roofline` is the top one)
        tot_ms = sum(v["ms"] for v in prof.values()) or 1.0
        roof_all = [roofline_of(k, v) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]) if v["ms"] > 0.02 * tot_ms]
        for r in roof_all:
            r["share_of_step"] = prof[r["kernel"]]["ms"] / tot_ms
        kernels = {k: {"ms_per_step": v["ms"] / psteps, "launches_per_step": v["launches"] / psteps}
                   for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}
        # CNN aggregate tensor-pipe fraction
        gemm_ms = sum(v["ms"] for k, v in prof.items() if k.startswith("gemm_")) / psteps
        cnn_tflops = (2.0 * sum(CNN_MACS.values()) * B / (gemm_ms * 1e-3) / 1e12) if gemm_ms > 0 else None
        em_info = None
        if "em_fused" in prof:
            fm = prof["em_fused"]
            cyc = ctx.em_phase_cycles()
            tot = float(sum(cyc.values())) or 1.0
            em_info = {"supersteps_of_slowest_image_per_step": em_stats["supersteps"] / psteps,
                       "image_supersteps_per_step": em_stats["wmat_products"] / psteps,
                       "wmat_algorithmic_GBps_over_kernel_time": em_stats["wmat_bytes"] / (fm["ms"] * 1e-3) / 1e9,
                       "wmat_fp64_TFLOPs_over_kernel_time": em_stats["wmat_flops"] / (fm["ms"] * 1e-3) / 1e12,
                       "phase_share_of_leading_cta": {k: v / tot for k, v in cyc.items()},
                       "us_per_image_superstep_leading_cta": tot / max(em_stats["wmat_products"], 1) / (clocks["sm_mhz"] or 1965.0)}
        elif "em_wmat" in prof:
            wm = prof["em_wmat"]
            em_info = {"supersteps_per_step": em_stats["supersteps"] / psteps,
                       "wmat_products_per_step": em_stats["wmat_products"] / psteps,
                       "wmat_algorithmic_GBps": em_stats["wmat_bytes"] / (wm["ms"] * 1e-3) / 1e9,
                       "wmat_fp64_TFLOPs": em_stats["wmat_flops"] / (wm["ms"] * 1e-3) / 1e12}

        # ---- CPU baseline on a bounded sample (rank 0, N = 1 only)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            sample = min(B, args.cpu_sample)
            v, dt = time_oracle(seg, off, ws, bs, sample)
            cores = os.cpu_count() or 1
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": "%d of the %d images (evenly spaced), %.1f s; numpy+torch CPU oracle (oracle/), "
                             "BLAS/torch threads = %d" % (sample, B, dt, cores),
                   "reference_em": None if args.no_reference_em else time_reference_em(seg, off, ws, bs, 2)}

        line = {
            "metric": METRIC, "value": total_images / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
            "dtype": "f64 (sphere, EM) + bf16/f32-accumulate (CNN)",
            "data": "synthetic",
            "config": {"workload": "%s-shaped synthetic batch (BASELINE.json configs[%d])" % (name, args.config - 1),
                       "images": total_images, "images_on_rank0": B,
                       "segments_per_image_mean": float(np.mean(np.diff(off_all))),
                       "sphere_size": 500, "sphere_mode": args.sphere_mode, "cnn_weights": "random-init "
                       "(train_val.prototxt fillers x%g, seed 0)" % args.weight_scale,
                       "batches_in_flight": depth, "num_init_vp": em_kw.get("num_init_vp", 25),
                       "l2": "each step streams > 1 GB of intermediates through the 126 MB L2 (inputs larger than L2); the "
                             "serial and profiled legs also flush it between steps (256 MiB memset)",
                       "parallelism": ("ONE batch sharded over the ranks (pipeline.shard_batch: LPT on N^2 + const), no data-path "
                                       "collective, results gathered on rank 0 inside the e2e region" if args.strong else
                                       "images sharded, no collective; every rank runs the same batch (fixed per-GPU work)")},
            "e2e": {"value": total_images / (e2e_step * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_step},
            "strong_scaling": None if not (args.strong and world > 1) else {
                "one_gpu_same_batch": one_gpu,
                "speedup_e2e": (total_images / (e2e_step * 1e-3)) / one_gpu["e2e_images_per_s"] if one_gpu else None,
                "rank_time_ms": {"resident_max": ms_step, "resident_min": float(tmin[0].item()),
                                 "e2e_max": e2e_step, "e2e_min": float(tmin[1].item())},
                "gather_ms_per_step_rank0": gather_ms / args.steps, "wait_for_own_shard_ms_per_step_rank0": wait_ms,
                "images_with_vps_after_gather": n_ok_all},
            "serial": {"value": total_images / (serial_step * 1e-3), "unit": UNIT, "ms_per_step": serial_step,
                       "what": "one batch at a time on one context, L2 flushed between steps (the latency of a batch; "
                               "`stages_ms_per_step` and `step_ms` are of this leg)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "roofline_all": roof_all,
            "cpu_baseline": cpu,
            "stages_ms_per_step": {k: v / args.steps for k, v in stage.items()},
            "kernels": kernels,
            "cnn_tflops": cnn_tflops,
            "em": em_info,
            "wall_ms_per_step": wall_step,
            "step_ms": {"min": float(np.min(step_ms)), "median": float(np.median(step_ms)), "max": float(np.max(step_ms)),
                        "settle_steps": settle},
            "kernels_note": "per-kernel times from a separate profiled leg (CUDA events around every launch on the library's "
                            "stream; the pair pass then does not overlap stages 1-2 as it does in the timed legs)",
            "images_with_vps": n_ok,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, *((full, off_all) if full is not None else (out, off)))
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_RESULT_FD = None


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=None, choices=[2, 3, 4, 5],
                    help="BASELINE.json config (1-based); default 2 (YUD) on one GPU, 4 (HLW, sharded) on several")
    ap.add_argument("--strong", action="store_true", help="shard ONE batch over the ranks (default for --gpus > 1)")
    ap.add_argument("--weak", action="store_true", help="every rank runs its own copy of the batch")
    ap.add_argument("--no-reference-em", action="store_true", help="skip the reference's own EM in the CPU baseline")
    ap.add_argument("--num-init-vp", type=int, default=None,
                    help="EM hypotheses per image (default 25, vp_localisation.py:170; 32 for the stress config 5)")
    ap.add_argument("--inflight", type=int, default=4, help="batches in flight per GPU (library contexts + host threads)")
    ap.add_argument("--images", type=int, default=None, help="override the number of images per GPU")
    ap.add_argument("--sphere-mode", default="votes", choices=["votes", "curves"])
    ap.add_argument("--weight-scale", type=float, default=1.0,
                    help="multiplier on the train_val.prototxt filler std (1.0 = the prototxt's own)")
    ap.add_argument("--cpu-sample", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--settle", type=int, default=30, help="upper bound of the extra untimed settling steps after the warm-up")
    ap.add_argument("--clock-period", type=float, default=0.005, help="seconds between NVML clock samples in the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the EM result of the last timed end-to-end step as DIR/<name>.npy (float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's result (--impl ours)")
    # stdout carries the ONE JSON line and nothing else: libraries that write to file descriptor 1 (NCCL prints its
    # version banner there) are sent to stderr; emit() writes the line to the real stdout
    sys.stdout.flush()
    global _RESULT_FD
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    args.warmup = max(args.warmup, 0)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not args.weak and world > 1:
        args.strong = True
    if args.weak:
        args.strong = False
    if args.config is None:
        args.config = 4 if args.strong else 2
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3          # timing rule: at least 3 warm-up steps
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
