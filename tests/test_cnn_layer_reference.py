"""CPU checks of the per-layer CNN reference (oracle/cnn_layer_oracle.py) that tests/test_cnn_layers_gpu.py holds the
device to: the layouts round-trip, a legitimate bf16 / fp32 implementation passes every layer, every planted bug fails
the layer it is in, and the stress weights put every layer (the LRNs above all) in its working range."""
import numpy as np
import pytest

from oracle import cnn_layer_oracle as L, cnn_oracle

# the layer each planted bug is in
MUTATION_LAYER = {
    "lrn_seam": "conv2", "norm2_alpha2": "conv2", "lrn_window3": "conv1", "norm1_skip": "conv1",
    "conv1_ch95_zero": "conv1", "conv4_ch383_zero": "conv4", "fc6_nchw": "fc6", "pool5_unclipped": "pool5",
    "a1_block_row": "a1", "mean_ignored": "a1",
}


@pytest.fixture(scope="module")
def stress():
    imgs = L.stress_images()
    ws, bs = L.stress_weights(0)
    return imgs, ws, bs


@pytest.fixture(scope="module")
def pair(stress):
    """two images (dense noise, votes sphere image) through the emulated device, with the fractional mean"""
    imgs, ws, bs = stress
    x = np.stack([imgs["noise"], imgs["votes"]])
    mean = L.fractional_mean()
    return x, mean, L.emulate_device(x, ws, bs, mean=mean)


@pytest.mark.parametrize("name", L.BUFFERS)
def test_pack_unpack_round_trip(name):
    rs = np.random.RandomState(len(name))
    if name == "a1":
        img = rs.standard_normal((2, 500, 500)).astype(np.float32)
        dev = L.pack("a1", img)
        assert np.array_equal(L.unpack("a1", dev), img)
        # every 4x4 block appears at kwb = 0..3 of the rows to its left
        assert np.array_equal(dev[1, 7, 10, 16 * 3 + 4 * 2 + 1], img[1, 4 * 7 + 2, 4 * 13 + 1])
    elif name in L.LAYOUT:
        H, W, Cs, pad, C, cg, cgp = L.LAYOUT[name]
        x = rs.standard_normal((2, C, H, W)).astype(np.float32)
        dev = L.pack(name, x)
        assert dev.shape == (2, H + 2 * pad, W + 2 * pad, Cs)
        assert np.array_equal(L.unpack(name, dev), x)
        dev2 = rs.standard_normal(dev.shape).astype(np.float32)
        dev2[:, L.padding_mask(name)] = 0
        assert np.array_equal(L.pack(name, L.unpack(name, dev2)), dev2)
    else:
        return
    mask = L.padding_mask(name)
    assert np.all(dev[:, mask] == 0)
    assert np.count_nonzero(dev[:, ~mask] == 0) == 0          # and nothing else is padding


def test_group_padding_of_a2_is_where_conv2_expects_it():
    m = L.padding_mask("a2")
    assert m.shape == (65, 65, 128)
    assert m[:2].all() and m[-2:].all() and m[:, :2].all() and m[:, -2:].all()
    assert not m[2:63, 2:63, :48].any() and m[2:63, 2:63, 48:64].all()
    assert not m[2:63, 2:63, 64:112].any() and m[2:63, 2:63, 112:].all()


def test_conv1_operand_rounds_pixel_minus_mean_to_nearest_bf16():
    img = np.zeros((1, 500, 500), np.uint8)
    img[0, 0, :4] = [1, 2, 3, 255]
    mean = np.zeros((500, 500), np.float32)
    mean[0, :4] = [0.5, 2 ** -9, 3 * 2 ** -7, 0.75]
    a1 = L.conv1_operand(img, mean)
    # spacing 2^-7 in [1, 2), 2^-6 in [2, 4), 1 in [128, 256): 2 - 2^-9 -> 2; 3 - 3 * 2^-7 is a tie -> the even
    # 3 - 2^-5; 255 - 0.75 -> 254
    assert list(a1[0, 0, 0, :4]) == [0.5, 2.0, 3 - 2 ** -5, 254.0]


def test_emulated_device_passes_every_layer(stress, pair):
    imgs, ws, bs = stress
    x, mean, bufs = pair
    res = L.check_all(bufs, ws, bs, x, mean=mean)
    assert set(res) == {"a1"} | {l[0] for l in L.LAYERS}
    for layer, (ratio, bad) in res.items():
        assert bad == 0 and ratio <= 1.0, (layer, ratio, bad)


@pytest.mark.parametrize("mutation", L.MUTATIONS)
def test_every_planted_bug_fails_its_layer(stress, pair, mutation):
    imgs, ws, bs = stress
    x, mean, _ = pair
    bufs = L.emulate_device(x, ws, bs, mean=mean, mutation=mutation)
    layer = MUTATION_LAYER[mutation]
    ratio, bad = L.check_all(bufs, ws, bs, x, mean=mean, layers=[layer])[layer]
    assert bad > 0 and ratio > 4, (mutation, layer, ratio, bad)
    if mutation == "lrn_window3":
        ratio2, bad2 = L.check_layer("conv2", bufs["a2"], bufs["c2"], ws, bs)
        assert bad2 > 0 and ratio2 > 4, (ratio2, bad2)


def test_seam_mutation_moves_many_norm2_outputs_far_beyond_the_bound(stress, pair):
    imgs, ws, bs = stress
    x, mean, bufs = pair
    ref, bound = L.gemm_layer("lrn", L.unpack("a2", bufs["a2"]), ws[1], bs[1], (1, 2, 2))
    seam = L.unpack("c2", L.emulate_device(x, ws, bs, mean=mean, mutation="lrn_seam")["c2"])
    far = np.abs(seam - ref) > 4 * bound
    assert np.count_nonzero(far) >= 50, np.count_nonzero(far)
    assert not far[:, :126].any() and not far[:, 130:].any()          # and only at the channels whose window crosses


def test_stress_weights_exercise_every_layer(stress):
    imgs, ws, bs = stress
    x = np.stack(list(imgs.values()))
    sig, logits, lay = cnn_oracle.forward(x, ws, bs, return_layers=True)
    for name in ["conv1", "conv2", "conv3", "conv4", "conv5", "fc6", "fc7"]:
        active = float(np.mean(lay[name] > 0))
        assert 0.2 <= active <= 0.8, (name, active)
    for conv, norm in [("conv1", "norm1"), ("conv2", "norm2")]:
        act = lay[conv] > 0
        factor = lay[norm][act] / lay[conv][act]
        assert np.mean(factor <= 0.5) >= 0.01, (norm, np.mean(factor <= 0.5))
    bf16_max = 3.3895e38
    for v in list(lay.values()) + [logits]:
        assert np.all(np.isfinite(v)) and np.abs(v).max() < bf16_max / 1e30


def test_filler_weights_leave_the_lrn_near_one():
    """Why the stress weights exist: with the train_val.prototxt fillers (x3, as the end-to-end tests use them) the LRN
    factor stays above 0.9, so even a per-layer check would hardly see it."""
    ws, bs = cnn_oracle.random_weights(0, scale=3.0)
    x = np.stack([L.stress_images()["votes"]])
    _, _, lay = cnn_oracle.forward(x, ws, bs, return_layers=True)
    act = lay["conv1"] > 0
    assert (lay["norm1"][act] / lay["conv1"][act]).min() > 0.9
