"""The EM's data-parallel kernels one by one on the device: every buffer em_pair, em_estep and em_wmat leave in the
workspace (vpk_em_debug_fetch) against its per-element reference (oracle/em_kernel_oracle.py), at the N where the
kernels change path (32-row chunks, 64-column slabs, 1536 / 3072: 1-, 2- and 4-CTA clusters of em_wmat) and at the
M where the W operand changes tiles and passes (MT = 1 ... 4 in the first and the second 32-row pass).  Every case
states the M its last superstep ran on.  Bit-exact claims are asserted bit for bit."""
import os

import numpy as np
import pytest

from oracle import cnn_oracle
from oracle import em_kernel_oracle as ek
from oracle import sphere_oracle as so
from vanishing_points_2017_b200 import _lib, synth
from vanishing_points_2017_b200 import vp_localisation as vl

pytestmark = pytest.mark.gpu

# given as init_vp with these settings, every hypothesis keeps the lines through it (oracle vp_scene)
FIXED_M = dict(do_iterations=False, do_merge=False, do_split=False, num_min_lines=0)
NAMES = ["lsim", "colsum", "lweight", "lvsq", "pvl", "w", "wt", "estep"]
WORST = {}


def _run(segs, offsets, init=None, init_off=None, resp=None, ctx=None, **kw):
    B = len(offsets) - 1
    lines = synth.lines_from_segments(segs)
    if resp is None:
        resp = np.stack([synth.ideal_response(init[init_off[b]:init_off[b + 1]], seed=b) for b in range(B)])
    return vl.expectation_maximisation_batch(lines, segs, offsets, resp, None, init_vp=init, init_vp_offsets=init_off,
                                             ctx=ctx, **kw), resp


def _fetch(image, ctx=None, planes=True):
    return {n: vl.em_debug_fetch(image, n, ctx) for n in (NAMES if planes else NAMES[:3])}


def _record(case, worst):
    for k, v in worst.items():
        WORST[k] = max(WORST.get(k, 0.0), v)
    print("%s worst |dev - ref| / bound: %s" % (case, {k: "%.3g" % v for k, v in worst.items()}))


def _check(case, segs, res, resp, buf, wbias=1.0, use_weights=True):
    worst, ties = ek.check_all(segs, buf, wbias=wbias, use_weights=use_weights, row_limit=1100)
    if "estep" in buf:
        worst["estep_pv"] = ek.check_estep_constants(buf["estep"], res["vp"], res["sigma"], resp)
    _record(case, worst)
    assert max(worst.values()) <= 1.0, (case, worst)
    assert len(ties) <= max(1, segs.shape[0] // 100), (case, ties)
    return worst


# (N, M): every chunk / slab / split boundary, and M spanning MT = 1 .. 4 in both passes; M > 32 with one CTA
# (513, 1536) and with clusters of 2 (1537) and 4 (3073, 6000)
CASES = [(31, 7), (32, 8), (33, 9), (63, 16), (64, 17), (65, 1), (129, 24), (200, 32), (513, 33), (1536, 64),
         (1537, 40), (3072, 25), (3073, 33), (6000, 40)]


@pytest.mark.parametrize("N,M", CASES, ids=["n%d_m%d" % c for c in CASES])
def test_kernels_at_fixed_m(N, M):
    sc = ek.vp_scene(9000 + N, N, M)
    (res,), resp = _run(sc["segments"], [0, N], sc["vps"], [0, M], **FIXED_M)
    assert res["vp"] is not None and res["vp"].shape[0] == M, "the last superstep ran on %r hypotheses" % (
        None if res["vp"] is None else res["vp"].shape[0])
    _check("N=%d M=%d" % (N, M), sc["segments"], res, resp[0], _fetch(0))


@pytest.mark.parametrize("N", [1, 2])
def test_pair_buffers_of_tiny_images(N):
    seg = synth.make_scene(40 + N, N)["segments"]
    (res,), resp = _run(seg, [0, N], np.array([[0.3, 0.2, 0.93]]), [0, 1], **FIXED_M)
    assert res["vp"] is None                      # fewer than three lines: no hypothesis survives the first count
    worst, _ = ek.check_all(seg, _fetch(0, planes=False))
    _record("N=%d" % N, worst)
    assert max(worst.values()) <= 1.0
    with pytest.raises(_lib.VpkError):
        vl.em_debug_fetch(0, "w")


@pytest.mark.parametrize("num_iter", [1, 2, 5, 11])
def test_kernels_after_truncated_runs(num_iter):
    sc = synth.make_scene(8100 + num_iter, 700, 800, 600, noise_deg=1.0)
    img = so.votes_to_image(so.sphere_votes(sc["lines"], 500))
    resp = synth.ideal_response(sc["vps"], seed=num_iter)
    res = vl.expectation_maximisation_batch(sc["lines"], sc["segments"], [0, 700], resp[None], img[None],
                                            num_iter=num_iter, split_merge_freq=2)[0]
    assert res["vp"] is not None
    _check("iter=%d M=%d" % (num_iter, res["vp"].shape[0]), sc["segments"], res, resp, _fetch(0))


@pytest.mark.parametrize("use_weights,wbias,N,M", [(False, 1.0, 300, 12), (True, 0.37, 1700, 36), (False, 1.0, 1700, 36)])
def test_weights_off_and_bias(use_weights, wbias, N, M):
    sc = ek.vp_scene(500 + N, N, M)
    (res,), resp = _run(sc["segments"], [0, N], sc["vps"], [0, M], use_weights=use_weights, wbias=wbias, **FIXED_M)
    assert res["vp"].shape[0] == M
    buf = _fetch(0, planes=True) if use_weights else {n: vl.em_debug_fetch(0, n) for n in NAMES if n != "lsim"}
    if not use_weights:
        with pytest.raises(_lib.VpkError):
            vl.em_debug_fetch(0, "lsim")
    _check("weights=%d wbias=%g N=%d M=%d" % (use_weights, wbias, N, M), sc["segments"], res, resp[0], buf, wbias,
           use_weights)


def _ragged():
    rs = np.random.RandomState(5)
    Ns = [1, 2, 31, 32, 33, 63, 64, 65, 129, 1536, 1537, 3073] + list(rs.randint(3, 400, 28))
    Ms = [1, 1, 7, 8, 9, 16, 17, 21, 33, 64, 40, 25] + list(rs.randint(1, 64, 28))
    scenes = [ek.vp_scene(700 + i, n, min(m, max(1, n // 3))) for i, (n, m) in enumerate(zip(Ns, Ms))]
    return scenes


def test_batch_equals_single_bit_for_bit():
    scenes = _ragged()
    segs = np.concatenate([s["segments"] for s in scenes])
    off = np.concatenate([[0], np.cumsum([s["segments"].shape[0] for s in scenes])]).astype(np.int32)
    init = np.concatenate([s["vps"] for s in scenes])
    ioff = np.concatenate([[0], np.cumsum([s["vps"].shape[0] for s in scenes])]).astype(np.int32)
    res, resp = _run(segs, off, init, ioff, **FIXED_M)
    batch = [_fetch(b, planes=res[b]["vp"] is not None) for b in range(len(scenes))]
    for b, s in enumerate(scenes):
        (r1,), _ = _run(s["segments"], [0, s["segments"].shape[0]], s["vps"], [0, s["vps"].shape[0]], resp=resp[b:b + 1],
                        **FIXED_M)
        one = _fetch(0, planes=r1["vp"] is not None)
        assert one.keys() == batch[b].keys()
        for n in one:
            a, c = (np.concatenate(list(one[n].values())), np.concatenate(list(batch[b][n].values()))) if n == "estep" \
                else (one[n], batch[b][n])
            assert np.array_equal(a.view(np.uint64), c.view(np.uint64)), (b, n)


def test_loop_forms_bit_identical():
    sc = ek.vp_scene(77, 1700, 40)
    out = {}
    old = os.environ.get("VPK_EM_MODE")
    try:
        for mode in ("fused", "graph", "host"):
            os.environ["VPK_EM_MODE"] = mode
            (res,), resp = _run(sc["segments"], [0, 1700], sc["vps"], [0, 40], **FIXED_M)
            assert res["vp"].shape[0] == 40
            out[mode] = _fetch(0)
    finally:
        if old is None:
            os.environ.pop("VPK_EM_MODE", None)
        else:
            os.environ["VPK_EM_MODE"] = old
    for mode in ("graph", "host"):
        for n in NAMES:
            a, b = out["fused"][n], out[mode][n]
            if n == "estep":
                a, b = np.concatenate(list(a.values())), np.concatenate(list(b.values()))
            assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), (mode, n)


def test_pipeline_pair_pass_equals_vpk_em():
    from vanishing_points_2017_b200 import pipeline
    ws, bs = cnn_oracle.random_weights(0, scale=3.0)
    pipe = pipeline.Pipeline(0, ws, bs, sphere_mode="votes")
    ns = [90, 1537, 200]
    seg = np.concatenate([synth.make_scene(4300 + i, n)["segments"] for i, n in enumerate(ns)])
    off = np.concatenate([[0], np.cumsum(ns)]).astype(np.int32)
    pipe(seg, off)
    got = [_fetch(b, pipe.ctx, planes=False) for b in range(len(ns))]
    ctx = _lib.Context(0)
    try:
        _run(seg, off, np.tile([[0.3, 0.2, 0.93]], (len(ns), 1)), np.arange(len(ns) + 1, dtype=np.int32), ctx=ctx,
             **FIXED_M)
        for b in range(len(ns)):
            want = _fetch(b, ctx, planes=False)
            for n in want:
                assert np.array_equal(got[b][n].view(np.uint64), want[n].view(np.uint64)), (b, n)
    finally:
        ctx.close()


def test_fetch_errors():
    ctx = _lib.Context(0)
    try:
        with pytest.raises(_lib.VpkError, match="workspace"):
            vl.em_debug_fetch(0, "lsim", ctx)                  # before any EM call
        sc = [ek.vp_scene(60 + i, 200, 5) for i in range(3)]
        segs = np.concatenate([s["segments"] for s in sc])
        off = np.array([0, 200, 400, 600], np.int32)
        init, ioff = np.concatenate([s["vps"] for s in sc]), np.array([0, 5, 10, 15], np.int32)
        os.environ["VPK_EM_WAVE_MB"] = "1"
        try:
            _run(segs, off, init, ioff, ctx=ctx, **FIXED_M)
        finally:
            del os.environ["VPK_EM_WAVE_MB"]
        with pytest.raises(_lib.VpkError, match="wave"):
            vl.em_debug_fetch(0, "colsum", ctx)                # the batch ran in several waves
        # image 1 is refused: more hypotheses than a slot holds
        init2 = np.concatenate([sc[0]["vps"], np.tile(sc[1]["vps"], (14, 1)), sc[2]["vps"]])
        res, _ = _run(segs, off, init2, np.array([0, 5, 75, 80], np.int32), ctx=ctx, resp=np.stack(
            [synth.ideal_response(s["vps"]) for s in sc]), **FIXED_M)
        assert res[1]["vp"] is None and res[1]["status"] == _lib.EM_CAPACITY
        assert vl.em_debug_fetch(1, "colsum", ctx).size == 200
        with pytest.raises(_lib.VpkError, match="status"):
            vl.em_debug_fetch(1, "w", ctx)
        assert vl.em_debug_fetch(0, "w", ctx).shape == (5, 200)
        with pytest.raises(_lib.VpkError, match="bad argument"):
            vl._em_fetch_raw(ctx, 0, len(NAMES))                # bad `which`
        with pytest.raises(_lib.VpkError, match="not part"):
            vl.em_debug_fetch(3, "colsum", ctx)
        small = np.empty(199)
        assert ctx.lib.vpk_em_debug_fetch(ctx.h, 0, 1, _lib.ptr(small), small.size, None) == 1   # VPK_ERR_ARG
    finally:
        ctx.close()


def test_zz_report_worst_ratios():
    """the worst |dev - ref| / bound per kernel over every case above (printed with -s)."""
    print("EM kernels, worst |dev - ref| / bound over all cases: %s" % {k: "%.3g" % v for k, v in sorted(WORST.items())})
    assert all(v <= 1.0 for v in WORST.values())
