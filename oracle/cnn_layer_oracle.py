"""ORACLE (test infrastructure, not product code) -- the CNN checked layer by layer.

Every layer of cnn/deploy.prototxt is recomputed in float64 from the DEVICE'S OWN input to that layer (the activation
buffers vpk_cnn_debug_fetch returns), so an error in one layer cannot hide behind, or be diluted by, the layers after
it.  Device layouts (include/vpk.h, VPK_CNN_BUF_*) are unpacked to NCHW here; the packers are their inverses, used by
the CPU tests and by `emulate_device`.

What is compared, and how:
  a1 (conv1 operand)  bit-exact: bf16_rn(float32(pixel) - float32(mean)) in the 4x4-block layout, 0 where X + kwb > 124.
  pool1, pool2, pool5 bit-exact: ceil-mode 3x3/2 maximum with clipped windows of the device's bf16 input.
  GEMM layers         |dev - ref| <= bound (below), ref in float64 from the device's bf16 input and the bf16 RNE-rounded
                      weights (what pack_weights_kernel stores), then bias, ReLU and, for conv1 / conv2, the LRN.
  sigmoid             |dev - ref| <= 1e-6 from the device's own logits.

The bound of a GEMM layer, per output element:

    |dev - ref| <= u_out * |ref| + (1 + u_out) * C_ACC * S,     S = sum_k |a_k w_k| + |bias|

  * u_out = 2^-8 for a bf16 output: round-to-nearest into 8 significant bits (2^-24 for fc8's float32 logits).
  * C_ACC * S is the fp32 accumulation.  The worst-case bound of recursive summation, K * 2^-24 * S, is 3.4e-3 * S at
    fc6's K = 57600 and would hide whole dropped channels.  The tensor cores add 16 products per instruction into an
    fp32 accumulator, so an output sees K/16 accumulator roundings (3600 at fc6, 400 per split), each at most
    2^-24 of the partial sum (2^-23 if the hardware truncates).  With zero-mean weights the partial sums are random
    walks, of size S / sqrt(K) rather than S, so even errors that all point the same way stay near
    (K / 16) * 2^-23 * S / sqrt(K) = 1.8e-6 * S at fc6 and less in every other layer.  C_ACC = 2^-14 = 6.1e-5 keeps a
    factor of 30 over that and is still well below every bug the CPU tests plant (the smallest, a dropped input
    channel, moves an output by about S / K_group per element of the group).
  * The LRN (conv1, conv2) acts on the fp32 pre-norm values x (not rounded to bf16 before it), with s = window sum of
    x^2, f = (1 + (alpha/5) s)^-beta and y = x f.  Its partial derivatives are
        dy_i/dx_i = f (1 - 2 beta (alpha/5) x_i^2 / (1 + (alpha/5) s))  in [(1 - 2 beta) f, f], so |.| <= f <= 1,
        dy_i/dx_j = -2 beta (alpha/5) f x_i x_j / (1 + (alpha/5) s)      (j != i in the window),
    so it is 1-Lipschitz in its own input and contracts by f, but the neighbours add a cross term; the pre-norm error
    e = C_ACC * S is therefore carried through to first order as
        E_i = f_i * (e_i + 2 beta (alpha/5) |x_i| * sum_window(|x_j| e_j) / (1 + (alpha/5) s_i))
    (the sum includes j = i, an overestimate), times 1.01 for the second-order terms (e / x is below 1e-4), plus
    2^-18 |y| for __powf (ex2.approx(y * lg2.approx(x)), a few ulp) and the fp32 window sum.  Then the bf16 rounding
    as above: bound = u_out |ref| + (1 + u_out) (1.01 E + 2^-18 |ref|).
"""
import numpy as np
import torch
import torch.nn.functional as F

ALPHA, BETA = 1e-4, 0.75                 # cnn/deploy.prototxt:34-44, 82-92 (local_size 5, k 1)
U_BF16, U_F32 = 2.0 ** -8, 2.0 ** -24
C_ACC = 2.0 ** -14
POW_REL = 2.0 ** -18
SIG_ATOL = 1e-6

# conv buffers: (H, W, stored channels, zero ring, channels, channels per group, stored channels per group)
LAYOUT = {
    "c1": (123, 123, 96, 0, 96, 96, 96),
    "a2": (61, 61, 128, 2, 96, 48, 64),
    "c2": (61, 61, 256, 0, 256, 256, 256),
    "a3": (30, 30, 256, 1, 256, 256, 256),
    "a4": (30, 30, 384, 1, 384, 384, 384),
    "a5": (30, 30, 384, 1, 384, 384, 384),
    "c5": (30, 30, 256, 0, 256, 256, 256),
    "a6": (15, 15, 256, 0, 256, 256, 256),
}
BUFFERS = ["a1", "c1", "a2", "c2", "a3", "a4", "a5", "c5", "a6", "f6", "f7", "logits", "sig"]

# layer -> (input buffer, output buffer, kind, weight index, conv stride / padding / groups)
LAYERS = [
    ("conv1", "a1", "c1", "lrn", 0, (4, 0, 1)),
    ("pool1", "c1", "a2", "pool", None, None),
    ("conv2", "a2", "c2", "lrn", 1, (1, 2, 2)),
    ("pool2", "c2", "a3", "pool", None, None),
    ("conv3", "a3", "a4", "conv", 2, (1, 1, 1)),
    ("conv4", "a4", "a5", "conv", 3, (1, 1, 2)),
    ("conv5", "a5", "c5", "conv", 4, (1, 1, 2)),
    ("pool5", "c5", "a6", "pool", None, None),
    ("fc6", "a6", "f6", "fc", 5, None),
    ("fc7", "f6", "f7", "fc", 6, None),
    ("fc8", "f7", "logits", "fc", 7, None),
    ("sigmoid", "logits", "sig", "sigmoid", None, None),
]
CONV_BUFFERS = ("a1",) + tuple(LAYOUT)       # per-image spatial buffers (the ones a test may sample images of)


def bf16(x):
    """round to bf16 (nearest, ties to even), returned as float64 numpy"""
    return torch.as_tensor(np.asarray(x, dtype=np.float32)).to(torch.bfloat16).to(torch.float64).numpy()


def bf16_bits(x):
    """float -> bf16 bit patterns (RNE), uint16"""
    t = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32)).to(torch.bfloat16)
    return t.view(torch.int16).numpy().view(np.uint16)


def bits_to_float(bits):
    return (np.asarray(bits, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32)


# ---------------------------------------------------------------------------------------------------------------
# layouts
# ---------------------------------------------------------------------------------------------------------------
def _channel_index(name):
    H, W, Cs, pad, C, cg, cgp = LAYOUT[name]
    c = np.arange(C)
    return (c // cg) * cgp + c % cg


def padding_mask(name):
    """bool (Hp, Wp, Cs) (a1: (125, 125, 64)): True where the device layout holds padding that must stay zero"""
    if name == "a1":
        m = np.zeros((125, 125, 64), dtype=bool)
        for kwb in range(1, 4):
            m[:, 125 - kwb:, 16 * kwb:16 * (kwb + 1)] = True
        return m
    H, W, Cs, pad, C, cg, cgp = LAYOUT[name]
    m = np.ones((H + 2 * pad, W + 2 * pad, Cs), dtype=bool)
    inner = np.ones((H, W, Cs), dtype=bool)
    inner[:, :, _channel_index(name)] = False
    m[pad:pad + H, pad:pad + W] = inner
    return m


def unpack(name, arr):
    """device layout (n, Hp, Wp, Cs) -> NCHW (n, C, H, W); a1 -> the (n, 500, 500) operand image; others as they are"""
    arr = np.asarray(arr)
    if name == "a1":
        n = arr.shape[0]
        blk = arr[..., :16].reshape(n, 125, 125, 4, 4)                 # (n, Y, X, dy, dx)
        return np.ascontiguousarray(blk.transpose(0, 1, 3, 2, 4).reshape(n, 500, 500))
    if name not in LAYOUT:
        return arr
    H, W, Cs, pad, C, cg, cgp = LAYOUT[name]
    x = arr[:, pad:pad + H, pad:pad + W, :][..., _channel_index(name)]
    return np.ascontiguousarray(x.transpose(0, 3, 1, 2))


def pack(name, x):
    """inverse of unpack: NCHW (or the (n, 500, 500) operand image for a1) -> device layout with zero padding"""
    x = np.asarray(x)
    n = x.shape[0]
    if name == "a1":
        blk = x.reshape(n, 125, 4, 125, 4).transpose(0, 1, 3, 2, 4).reshape(n, 125, 125, 16)
        out = np.zeros((n, 125, 125, 64), dtype=x.dtype)
        for kwb in range(4):
            out[:, :, :125 - kwb, 16 * kwb:16 * (kwb + 1)] = blk[:, :, kwb:, :]
        return out
    if name not in LAYOUT:
        return x.copy()
    H, W, Cs, pad, C, cg, cgp = LAYOUT[name]
    out = np.zeros((n, H + 2 * pad, W + 2 * pad, Cs), dtype=x.dtype)
    out[:, pad:pad + H, pad:pad + W, _channel_index(name)] = x.transpose(0, 2, 3, 1)
    return out


# ---------------------------------------------------------------------------------------------------------------
# float64 layers
# ---------------------------------------------------------------------------------------------------------------
def _t(x):
    return torch.as_tensor(np.asarray(x, dtype=np.float64))


def window_sum(t):
    """sum over the 5-channel window (zero beyond channels 0 and C-1) of an NCHW tensor"""
    p = F.pad(t, (0, 0, 0, 0, 2, 2))
    return sum(p[:, k:k + t.shape[1]] for k in range(5))


def conv1_operand(images, mean=None):
    """the exact a1 the device must hold (float32 values of bf16)"""
    x = np.asarray(images, dtype=np.float32)
    if mean is not None:
        x = x - np.asarray(mean, dtype=np.float32).reshape(500, 500)
    return pack("a1", bf16(x).astype(np.float32))


def pool(x):
    """ceil-mode 3x3/2 max pool with clipped windows (Caffe), NCHW"""
    return F.max_pool2d(_t(x), 3, 2, ceil_mode=True).numpy()


def gemm_layer(kind, x, w, b, conv=None):
    """float64 reference and bound of one GEMM layer.  x: the device's input (NCHW, or (n, K) for fc; fc6's is the
    (n, 256, 15, 15) unpacked a6, flattened here in Caffe's NCHW order), w / b: Caffe-layout float32 weights / biases
    (rounded to bf16 here, as pack_weights_kernel does).  Returns (ref, bound)."""
    xt, wt, bt = _t(x), _t(bf16(w)), _t(b)
    if conv is None:
        xt = xt.reshape(xt.shape[0], -1)
        z = xt @ wt.T + bt
        S = xt.abs() @ wt.abs().T + bt.abs()
    else:
        stride, padding, groups = conv
        z = F.conv2d(xt, wt, bt, stride=stride, padding=padding, groups=groups)
        S = F.conv2d(xt.abs(), wt.abs(), bt.abs(), stride=stride, padding=padding, groups=groups)
    e = C_ACC * S
    if kind == "fc" and w.shape[0] == 400:                                  # fc8: float32 logits, no ReLU
        return z.numpy(), (U_F32 * z.abs() + (1 + U_F32) * e).numpy()
    xr = torch.relu(z)
    if kind != "lrn":
        return xr.numpy(), (U_BF16 * xr + (1 + U_BF16) * e).numpy()
    a = ALPHA / 5
    s = window_sum(xr * xr)
    f = (1 + a * s) ** -BETA
    y = xr * f
    E = f * (e + 2 * BETA * a * xr * window_sum(xr * e) / (1 + a * s))
    return y.numpy(), (U_BF16 * y + (1 + U_BF16) * (1.01 * E + POW_REL * y)).numpy()


def sigmoid(logits):
    return 1.0 / (1.0 + np.exp(-np.asarray(logits, dtype=np.float64)))


def check_layer(layer, dev_in, dev_out, weights, biases, images=None, mean=None):
    """One layer against the float64 reference on the device's own input.  dev_in / dev_out: float arrays in device
    layout (bf16 values as float32) for the same images; for conv1, dev_in is ignored and `images` / `mean` give the
    a1 check.  Returns (worst |dev - ref| / bound, number of elements over the bound); exact layers give 0 or inf."""
    name, bin_, bout, kind, wi, conv = next(l for l in LAYERS if l[0] == layer)
    out = unpack(bout, dev_out)
    if kind == "pool":
        ref = pool(unpack(bin_, dev_in))
        bad = int(np.count_nonzero(ref != out))
        return (np.inf if bad else 0.0), bad
    if kind == "sigmoid":
        err = np.abs(np.asarray(dev_out, dtype=np.float64) - sigmoid(dev_in))
        return float(err.max() / SIG_ATOL), int(np.count_nonzero(err > SIG_ATOL))
    x = unpack(bin_, dev_in)
    if layer == "conv1":
        x = x[:, None]
    ref, bound = gemm_layer(kind, x, weights[wi], biases[wi], conv)
    with np.errstate(divide="ignore", invalid="ignore"):               # bound 0: ref 0 from an all-zero input and bias
        ratio = np.abs(out.astype(np.float64) - ref) / bound
    ratio = np.where(bound > 0, ratio, np.where(out == ref, 0.0, np.inf))
    return float(ratio.max()), int(np.count_nonzero(ratio > 1))


def check_operand(dev_a1, images, mean=None):
    """a1 bit-exact: returns the number of differing values"""
    return int(np.count_nonzero(conv1_operand(images, mean) != dev_a1))


def check_all(bufs, weights, biases, images, mean=None, layers=None):
    """every layer (or `layers`) of a forward: bufs maps buffer name -> float array in device layout (bf16 as float32),
    all for the same images; images (n, 500, 500) uint8.  Returns {layer: (worst ratio, elements over the bound)}
    with "a1" giving (0 or inf, differing values)."""
    res = {}
    if layers is None or "a1" in layers:
        bad = check_operand(bufs["a1"], images, mean)
        res["a1"] = (np.inf if bad else 0.0, bad)
    for name, bin_, bout, kind, wi, conv in LAYERS:
        if layers is not None and name not in layers:
            continue
        res[name] = check_layer(name, bufs[bin_], bufs[bout], weights, biases, images, mean)
    return res


# ---------------------------------------------------------------------------------------------------------------
# stress weights: every layer in its working range
# ---------------------------------------------------------------------------------------------------------------
SHAPES = [(96, 1, 11, 11), (256, 48, 5, 5), (384, 256, 3, 3), (384, 192, 3, 3), (256, 192, 3, 3),
          (4096, 57600), (4096, 4096), (400, 4096)]
# weight std = gain / sqrt(fan_in); bias std (absolute)
STRESS_GAIN = [1.6, 1.6, 1.5, 1.5, 1.5, 1.5, 1.5, 1.0]
STRESS_BIAS = [20.0, 20.0, 10.0, 10.0, 10.0, 10.0, 10.0, 5.0]


def stress_weights(seed=0):
    """Seeded Gaussian weights scaled so that ReLUs are active on part of every layer and the LRNs normalise hard
    (the train_val.prototxt fillers leave the LRN factor near 1 and the suite blind to it)."""
    g = torch.Generator().manual_seed(seed)
    ws, bs = [], []
    for shape, gain, bstd in zip(SHAPES, STRESS_GAIN, STRESS_BIAS):
        fan_in = int(np.prod(shape[1:]))
        ws.append((torch.randn(shape, generator=g, dtype=torch.float32) * (gain / np.sqrt(fan_in))).numpy())
        bs.append((torch.randn(shape[0], generator=g, dtype=torch.float32) * bstd).numpy())
    return ws, bs


# ---------------------------------------------------------------------------------------------------------------
# an emulated device: what a correct kernel may legitimately compute (bf16 operands, fp32 accumulation, bf16
# outputs), with optional planted bugs for the tests to reject
# ---------------------------------------------------------------------------------------------------------------
MUTATIONS = ["lrn_seam", "norm2_alpha2", "lrn_window3", "norm1_skip", "conv1_ch95_zero", "conv4_ch383_zero",
             "fc6_nchw", "pool5_unclipped", "a1_block_row", "mean_ignored"]


def _lrn32(x, alpha=ALPHA, size=5, seam=None):
    """LRN in float32; seam: the window stops at this channel (a per-group normalisation)"""
    sq = x * x
    if seam is not None:
        return torch.cat([_lrn32(x[:, :seam], alpha, size), _lrn32(x[:, seam:], alpha, size)], 1)
    h = size // 2
    p = F.pad(sq, (0, 0, 0, 0, h, h))
    s = sum(p[:, k:k + x.shape[1]] for k in range(size))
    return x * (1 + (alpha / 5) * s) ** -BETA


def _b16(t):
    return t.to(torch.bfloat16).to(torch.float32)


def emulate_device(images, weights, biases, mean=None, mutation=None):
    """All 13 buffers in device layout (float32 holding bf16 values, float32 logits / sigmoid)."""
    assert mutation is None or mutation in MUTATIONS, mutation
    m = mutation
    img = np.asarray(images, dtype=np.float32)
    if mean is not None and m != "mean_ignored":
        img = img - np.asarray(mean, dtype=np.float32).reshape(500, 500)
    if m == "a1_block_row":                                   # block row Y holds the pixels of block row Y + 1
        img = np.concatenate([img[:, 4:], np.zeros_like(img[:, :4])], 1)
    w = [_b16(torch.from_numpy(np.ascontiguousarray(a))) for a in weights]
    b = [torch.from_numpy(np.ascontiguousarray(a)) for a in biases]
    bufs = {}
    x = _b16(torch.from_numpy(np.ascontiguousarray(img)))
    bufs["a1"] = pack("a1", x.numpy())
    x = x[:, None]
    with torch.no_grad():
        x = torch.relu(F.conv2d(x, w[0], b[0], stride=4))
        if m == "conv1_ch95_zero":
            x[:, 95] = 0
        if m != "norm1_skip":
            x = _lrn32(x, size=3 if m == "lrn_window3" else 5)
        x = _b16(x)
        bufs["c1"] = pack("c1", x.numpy())
        x = F.max_pool2d(x, 3, 2, ceil_mode=True)
        bufs["a2"] = pack("a2", x.numpy())
        x = torch.relu(F.conv2d(x, w[1], b[1], padding=2, groups=2))
        x = _lrn32(x, alpha=2 * ALPHA if m == "norm2_alpha2" else ALPHA, size=3 if m == "lrn_window3" else 5,
                   seam=128 if m == "lrn_seam" else None)
        x = _b16(x)
        bufs["c2"] = pack("c2", x.numpy())
        x = F.max_pool2d(x, 3, 2, ceil_mode=True)
        bufs["a3"] = pack("a3", x.numpy())
        x = _b16(torch.relu(F.conv2d(x, w[2], b[2], padding=1)))
        bufs["a4"] = pack("a4", x.numpy())
        x = torch.relu(F.conv2d(x, w[3], b[3], padding=1, groups=2))
        if m == "conv4_ch383_zero":
            x[:, 383] = 0
        x = _b16(x)
        bufs["a5"] = pack("a5", x.numpy())
        x = _b16(torch.relu(F.conv2d(x, w[4], b[4], padding=1, groups=2)))
        bufs["c5"] = pack("c5", x.numpy())
        if m == "pool5_unclipped":
            # windows at the right / bottom edge run on into the next row (the flat NHWC index), not clipped
            n = x.shape[0]
            flat = F.pad(x.permute(0, 2, 3, 1).reshape(n, 900, 256), (0, 0, 0, 64))
            out = torch.full((n, 15, 15, 256), -np.inf)
            for dy in range(3):
                for dx in range(3):
                    yy, xx = np.meshgrid(np.arange(15) * 2 + dy, np.arange(15) * 2 + dx, indexing="ij")
                    idx = torch.as_tensor(np.minimum(yy * 30 + xx, 963).reshape(-1))
                    out = torch.maximum(out, flat[:, idx].reshape(n, 15, 15, 256))
            x = out.permute(0, 3, 1, 2).contiguous()
        else:
            x = F.max_pool2d(x, 3, 2, ceil_mode=True)
        bufs["a6"] = pack("a6", x.numpy())
        if m == "fc6_nchw":                                   # Caffe's weights applied to the NHWC order of a6
            x = x.permute(0, 2, 3, 1)
        x = _b16(torch.relu(F.linear(x.reshape(x.shape[0], -1), w[5], b[5])))
        bufs["f6"] = x.numpy()
        x = _b16(torch.relu(F.linear(x, w[6], b[6])))
        bufs["f7"] = x.numpy()
        logits = F.linear(x, w[7], b[7])
        bufs["logits"] = logits.numpy()
        bufs["sig"] = torch.sigmoid(logits).numpy()
    return bufs


# ---------------------------------------------------------------------------------------------------------------
# images
# ---------------------------------------------------------------------------------------------------------------
def stress_images():
    """name -> (500, 500) uint8: the image kinds the layer checks run on"""
    from oracle import sphere_oracle as so
    from vanishing_points_2017_b200 import synth
    rs = np.random.RandomState(2024)
    sc = synth.make_scene(5000, 150)
    imgs = {
        "votes": so.votes_to_image(so.sphere_votes(sc["lines"], 500)),
        "curves": so.curve_image(so.sphere_curve_counts(synth.make_scene(5001, 190)["lines"], 500), 0.1),
        "noise": rs.randint(0, 256, (500, 500)).astype(np.uint8),
        "zeros": np.zeros((500, 500), np.uint8),
        "full": np.full((500, 500), 255, np.uint8),
    }
    edge = np.zeros((500, 500), np.uint8)                      # only rows / columns 496..499: the last block column
    edge[496:] = rs.randint(1, 256, (4, 500))
    edge[:, 496:] = rs.randint(1, 256, (500, 4))
    imgs["edge"] = edge
    outside = np.zeros((500, 500), np.uint8)                   # only row / column 499: outside every conv1 window
    outside[499] = rs.randint(1, 256, 500)
    outside[:, 499] = rs.randint(1, 256, 500)
    imgs["outside"] = outside
    return imgs


def fractional_mean(seed=1):
    """a mean image with fractional values (0..40), for the a1 check"""
    return (np.random.RandomState(seed).uniform(0, 40, (500, 500)).astype(np.float32))
