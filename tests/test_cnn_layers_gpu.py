"""The CNN layer by layer on the device: every activation buffer of a forward (vpk_cnn_debug_fetch) against the float64
reference of that layer computed from the device's own input (oracle/cnn_layer_oracle.py states the bounds), at the
batch sizes where the code changes path, plus buffer reuse and position / chunk invariance of the results."""
import time

import numpy as np
import pytest

from oracle import cnn_layer_oracle as L, cnn_oracle
from vanishing_points_2017_b200 import _lib, cnn

pytestmark = pytest.mark.gpu

FC_BUFFERS = ("a6", "f6", "f7", "logits", "sig")
CONV_LAYERS = ["a1", "conv1", "pool1", "conv2", "pool2", "conv3", "conv4", "conv5", "pool5"]
FC_LAYERS = ["fc6", "fc7", "fc8", "sigmoid"]


@pytest.fixture(scope="module")
def images():
    return L.stress_images()


@pytest.fixture(scope="module")
def weight_sets():
    return {"stress": L.stress_weights(0), "filler3": cnn_oracle.random_weights(0, scale=3.0)}


@pytest.fixture(scope="module")
def nets(weight_sets):
    """one context (own CNN state) per weight set"""
    return {k: cnn.Net(_lib.Context(0), ws, bs) for k, (ws, bs) in weight_sets.items()}


def tiled(images, n):
    names = list(images)
    return np.stack([images[names[i % len(names)]] for i in range(n)])


def fetch(net, n, raw=True):
    return {name: net.debug_activations(name, n, raw=raw) for name in L.BUFFERS}


def as_float(a):
    return L.bits_to_float(a) if a.dtype == np.uint16 else a


def assert_padding_zero(raw):
    for name in L.CONV_BUFFERS:
        pads = raw[name][:, L.padding_mask(name)]
        assert not pads.any(), "%s: %d non-zero padding values" % (name, np.count_nonzero(pads))


def check_forward(raw, ws, bs, x, mean, rows):
    """conv layers on images `rows`, fc layers on every image; returns {layer: worst ratio} after asserting"""
    conv = {k: as_float(raw[k][rows]) for k in L.CONV_BUFFERS}
    res = L.check_all(conv, ws, bs, x[rows], mean=mean, layers=CONV_LAYERS)
    fc = {k: as_float(raw[k]) for k in FC_BUFFERS}
    res.update(L.check_all(fc, ws, bs, x, mean=mean, layers=FC_LAYERS))
    bad = {k: v for k, v in res.items() if v[1]}
    assert not bad, "layers over the bound (worst ratio, elements): %r" % bad
    return {k: round(v[0], 4) for k, v in res.items()}


CASES = [("stress", 1, False), ("stress", 3, True), ("stress", 129, False),
         ("filler3", 1, False), ("filler3", 3, True), ("filler3", 129, False)]


@pytest.mark.parametrize("wset,n,with_mean", CASES)
def test_every_layer_within_its_bound(images, weight_sets, nets, wset, n, with_mean):
    """n = 1 and 3: every image; n = 129: fc layers with split-K over two M tiles, conv layers on the first, middle and
    last image."""
    ws, bs = weight_sets[wset]
    net = nets[wset]
    mean = L.fractional_mean() if with_mean else None
    net.set_mean(mean)
    x = tiled(images, n)
    net.forward_batch(x)
    raw = fetch(net, n)
    net.set_mean(None)
    assert_padding_zero(raw)
    rows = sorted({0, n // 2, n - 1})
    print("\nworst |dev - ref| / bound, %s n=%d%s: %r" % (wset, n, " mean" if with_mean else "",
                                                         check_forward(raw, ws, bs, x, mean, rows)))


@pytest.mark.parametrize("persist", ["1", "0"])
@pytest.mark.parametrize("wset", ["stress", "filler3"])
def test_every_layer_without_split_k(images, weight_sets, nets, monkeypatch, wset, persist):
    """n = 257: the fully connected layers run without split-K (three M tiles); the convolutions through the
    persistent kernel and through the one-tile-per-CTA kernel."""
    ws, bs = weight_sets[wset]
    net = nets[wset]
    n = 257
    x = tiled(images, n)[::-1].copy()
    monkeypatch.setenv("VPK_GEMM_PERSIST", persist)
    net.forward_batch(x)
    monkeypatch.delenv("VPK_GEMM_PERSIST")
    raw = fetch(net, n)
    assert_padding_zero(raw)
    print("\nworst |dev - ref| / bound, %s n=257 persist=%s: %r" % (wset, persist,
                                                                    check_forward(raw, ws, bs, x, None, [0, 128, 256])))


def test_pixels_outside_every_conv1_window_change_nothing(images, nets):
    """Row and column 499 lie outside every conv1 window (the last covers 488..498): an image non-zero only there gives
    the zero image's activations bit for bit from c1 on; the a1 operand still carries the pixels."""
    net = nets["stress"]
    net.set_mean(None)
    net.forward_batch(np.stack([images["zeros"], images["outside"], images["edge"]]))
    raw = fetch(net, 3)
    assert raw["a1"][1].any() and not raw["a1"][0].any()
    for name in L.BUFFERS[1:]:
        assert np.array_equal(raw[name][0], raw[name][1]), name
    assert not np.array_equal(raw["c1"][0], raw["c1"][2])


def test_buffer_reuse_matches_a_fresh_context(images, weight_sets):
    """A batch after a larger one reuses the activation buffers (padding zeroed only when they grow); a batch after a
    smaller one grows them.  Both must give a fresh context's bits, with every pad ring and group-padding channel
    still zero."""
    ws, bs = weight_sets["stress"]
    rs = np.random.RandomState(7)
    nine = np.stack([rs.randint(0, 256, (500, 500)).astype(np.uint8) for _ in range(9)])
    two = np.stack([images["votes"], images["full"]])
    a = cnn.Net(_lib.Context(0), ws, bs)
    a.forward_batch(nine)
    a9 = fetch(a, 9)
    a.forward_batch(two)
    a2 = fetch(a, 2)
    b = cnn.Net(_lib.Context(0), ws, bs)
    b.forward_batch(two)
    b2 = fetch(b, 2)
    b.forward_batch(nine)
    b9 = fetch(b, 9)
    for got in (a9, a2, b2, b9):
        assert_padding_zero(got)
    for name in L.BUFFERS:
        assert np.array_equal(a2[name], b2[name]), "2 after 9: %s differs from a fresh context" % name
        assert np.array_equal(b9[name], a9[name]), "9 after 2: %s differs from a fresh context" % name
    with pytest.raises(_lib.VpkError):
        b.debug_activations("c1", 10)


def test_debug_fetch_refuses_bad_requests(weight_sets):
    ws, bs = weight_sets["filler3"]
    net = cnn.Net(_lib.Context(0), ws, bs)
    with pytest.raises(_lib.VpkError, match="no vpk_cnn_forward"):
        net.debug_activations("a1", 1)
    net.forward_batch(np.zeros((2, 500, 500), np.uint8))
    out = np.empty(400, np.float32)
    for which in (-1, 13):
        assert net.ctx.lib.vpk_cnn_debug_fetch(net.ctx.h, which, 1, _lib.ptr(out)) == 1
    assert net.ctx.lib.vpk_cnn_debug_fetch(net.ctx.h, 11, 3, _lib.ptr(out)) == 1
    assert net.ctx.lib.vpk_cnn_debug_fetch(net.ctx.h, 11, 1, _lib.ptr(out)) == 0


def test_rows_do_not_depend_on_position_or_chunk(images, weight_sets, nets):
    """n = 1030 runs as a chunk of 1024 (fully connected layers without split-K) and one of 6 (with split-K).  Each row
    must equal the same image's row of a 300-image batch (no split-K) resp. of a 6-image batch (split-K) bit for bit,
    whatever its position; the 16 distinct images must match the fp32 oracle end to end."""
    ws, bs = weight_sets["stress"]
    net = nets["stress"]
    net.set_mean(None)
    rs = np.random.RandomState(11)
    distinct = list(images.values())
    while len(distinct) < 16:                             # noise of rising density
        d = len(distinct) / 16
        distinct.append((rs.randint(0, 256, (500, 500)) * (rs.uniform(size=(500, 500)) < d)).astype(np.uint8))
    distinct = np.stack(distinct)
    ids = np.arange(1030) % 16
    t0 = time.perf_counter()
    _, big = net.forward_batch(distinct[ids], want_logits=True)
    print("\nforward of 1030 images (two chunks, incl. copies): %.3f s" % (time.perf_counter() - t0))
    ids300 = (np.arange(300) * 7 + 3) % 16
    _, mid = net.forward_batch(distinct[ids300], want_logits=True)
    ids6 = np.arange(6)[::-1]
    _, small = net.forward_batch(distinct[ids6], want_logits=True)
    for i in range(16):
        rows = big[:1024][ids[:1024] == i]
        assert (rows == rows[0]).all(), "copies of image %d differ within the 1024-image chunk" % i
        rows300 = mid[ids300 == i]
        assert (rows300 == rows300[0]).all(), "copies of image %d differ within the 300-image batch" % i
        assert np.array_equal(rows[0], rows300[0]), "image %d: 1024-image chunk vs 300-image batch" % i
    for k in range(6):
        assert np.array_equal(big[1024 + k], small[list(ids6).index(ids[1024 + k])]), "row %d vs 6-image batch" % (1024 + k)
    _, ref = cnn_oracle.forward(distinct, ws, bs)
    rel = np.max(np.abs(big[:16] - ref)) / np.max(np.abs(ref))
    assert rel < 1e-2, rel
