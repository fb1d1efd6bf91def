"""Drop-in for the CNN predict glue of the reference (evaluation.py:17-38) on
the B200: init_caffe / read_mean_blob / caffe_forward with the same argument
order.  The forward pass of cnn/deploy.prototxt runs as tcgen05 implicit-GEMM
kernels behind libvpk.so's C ABI.

The trained caffemodel is an external download (reference README.md:23).  Caffe
is not needed to use it: `model_weights` may be the `.caffemodel` itself (parsed
by caffe_proto.py), a dict / .npz of Caffe-layout float32 arrays {conv1_w,
conv1_b, ..., fc8_20x20_w, fc8_20x20_b}, or None for the seeded random fillers
of train/train_val.prototxt (benchmarks and tests only: a RuntimeWarning says so).
"""
import ctypes as C
import warnings

import numpy as np

from . import _lib

LAYER_NAMES = ["conv1", "conv2", "conv3", "conv4", "conv5", "fc6", "fc7", "fc8_20x20"]
LAYER_SHAPES = [(96, 1, 11, 11), (256, 48, 5, 5), (384, 256, 3, 3), (384, 192, 3, 3), (256, 192, 3, 3),
                (4096, 57600), (4096, 4096), (400, 4096)]
# fillers of train/train_val.prototxt:83-90,139-146,194-201,228-235,262-269,304-311,344-351,384-391
FILLERS = [(0.01, 0.0), (0.01, 0.1), (0.01, 0.0), (0.01, 0.1), (0.01, 0.1), (0.005, 0.1), (0.005, 0.1), (0.01, 0.0)]


def random_weights(seed=0, scale=1.0):
    """Seeded Gaussian/constant fillers (same tensors as oracle.cnn_oracle.random_weights)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    ws, bs = [], []
    for shape, (std, bias) in zip(LAYER_SHAPES, FILLERS):
        ws.append((torch.randn(shape, generator=g, dtype=torch.float32) * (std * scale)).numpy())
        bs.append(np.full(shape[0], bias, dtype=np.float32))
    return ws, bs


class Net:
    """Handle returned by init_caffe (stands in for caffe.Net)."""

    def __init__(self, ctx, weights, biases):
        self.ctx = ctx
        self._mean_loaded = None
        self._last_chunk = 0
        self._w = [np.ascontiguousarray(w, dtype=np.float32) for w in weights]
        self._b = [np.ascontiguousarray(b, dtype=np.float32) for b in biases]
        for w, shape in zip(self._w, LAYER_SHAPES):
            if w.shape != shape:
                raise ValueError("weight blob %r, expected %r" % (w.shape, shape))
        self._load(None)

    def _load(self, mean):
        wp = (C.c_void_p * 8)(*[w.ctypes.data for w in self._w])
        bp = (C.c_void_p * 8)(*[b.ctypes.data for b in self._b])
        m = None if mean is None else np.ascontiguousarray(mean, dtype=np.float32).reshape(500, 500)
        _lib.check(self.ctx.lib.vpk_cnn_load(self.ctx.h, wp, bp, _lib.ptr(m)), "vpk_cnn_load")
        self._mean_loaded = None if mean is None else m.copy()

    def set_mean(self, mean):
        same = (mean is None and self._mean_loaded is None) or (
            mean is not None and self._mean_loaded is not None and np.array_equal(
                np.asarray(mean, dtype=np.float32).reshape(500, 500), self._mean_loaded))
        if not same:
            self._load(mean)

    def forward_batch(self, images, want_logits=False):
        images = np.ascontiguousarray(images, dtype=np.uint8).reshape(-1, 500, 500)
        n = images.shape[0]
        sig = np.empty((n, 20, 20), dtype=np.float32)
        logits = np.empty((n, 400), dtype=np.float32) if want_logits else None
        _lib.check(self.ctx.lib.vpk_cnn_forward(self.ctx.h, _lib.ptr(images), n, _lib.ptr(sig), _lib.ptr(logits)),
                   "vpk_cnn_forward")
        if n:
            self._last_chunk = (n - 1) % 1024 + 1          # vpk_cnn_forward runs the batch in chunks of 1024
        return (sig, logits) if want_logits else sig

    def debug_activations(self, which, n=None, raw=False):
        """Activation buffer `which` (a name of ACTIVATIONS) of the last chunk forward_batch ran (its last 1024 or
        fewer images), copied as the device holds it: padding rings and group padding included (layouts in
        include/vpk.h).  Returns an (n, H, W, C) array for the convolution buffers, (n, K) for f6 / f7 / logits / sig;
        bf16 buffers as float32, or as their uint16 bit patterns with raw=True.  n defaults to the whole chunk."""
        index, shape, is_bf16 = ACTIVATIONS[which]
        if n is None:
            n = self._last_chunk
        out = np.empty((n,) + shape, dtype=np.uint16 if is_bf16 else np.float32)
        _lib.check(self.ctx.lib.vpk_cnn_debug_fetch(self.ctx.h, index, int(n), _lib.ptr(out)), "vpk_cnn_debug_fetch")
        return out if raw or not is_bf16 else bf16_bits_to_float(out)


# name -> (vpk_cnn_debug_fetch index, per-image shape, bf16?)   (include/vpk.h, VPK_CNN_BUF_*)
ACTIVATIONS = {
    "a1": (0, (125, 125, 64), True), "c1": (1, (123, 123, 96), True), "a2": (2, (65, 65, 128), True),
    "c2": (3, (61, 61, 256), True), "a3": (4, (32, 32, 256), True), "a4": (5, (32, 32, 384), True),
    "a5": (6, (32, 32, 384), True), "c5": (7, (30, 30, 256), True), "a6": (8, (15, 15, 256), True),
    "f6": (9, (4096,), True), "f7": (10, (4096,), True), "logits": (11, (400,), False), "sig": (12, (400,), False),
}


def bf16_bits_to_float(bits):
    """uint16 bf16 bit patterns -> float32 (exact)."""
    return (np.asarray(bits, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32)


def init_caffe(model_def=None, model_weights=None, gpu_id=0):
    """evaluation.init_caffe(model_def, model_weights, gpu_id) (reference
    evaluation.py:17-22).  model_def is accepted for signature compatibility:
    the architecture is cnn/deploy.prototxt, compiled in."""
    ctx = _lib.default_context(gpu_id)
    ws, bs = load_weights(model_weights)
    return Net(ctx, ws, bs)


def load_weights(model_weights, allow_random=False):
    """The eight (weight, bias) blob pairs of cnn/deploy.prototxt from a .caffemodel, an .npz / dict
    of `<layer>_w` / `<layer>_b` arrays, or (None) the random fillers of train/train_val.prototxt."""
    if model_weights is None:
        if not allow_random:
            warnings.warn("no CNN weights given: using the seeded random fillers of train/train_val.prototxt -- the "
                          "response (and every vanishing point initialised from it) is meaningless; pass the "
                          "reference's weights.caffemodel", RuntimeWarning, stacklevel=3)
        return random_weights(0)
    if isinstance(model_weights, str) and not model_weights.endswith(".npz"):
        from . import caffe_proto
        layers = caffe_proto.read_caffemodel(model_weights)
        missing = [n for n in LAYER_NAMES if n not in layers or len(layers[n]) < 2]
        if missing:
            raise ValueError("%s: no weight/bias blobs for layers %s (found %s)" % (model_weights, missing, sorted(layers)))
        ws = [layers[n][0].reshape(shape) for n, shape in zip(LAYER_NAMES, LAYER_SHAPES)]
        bs = [layers[n][1].reshape(-1) for n in LAYER_NAMES]
        return ws, bs
    src = np.load(model_weights) if isinstance(model_weights, str) else model_weights
    return [src[n + "_w"] for n in LAYER_NAMES], [src[n + "_b"] for n in LAYER_NAMES]


def read_mean_blob(mean_file=None):
    """evaluation.read_mean_blob (reference evaluation.py:25-31): returns a
    (1,1,500,500) float32 array.  Accepts the reference's mean.binaryproto (BlobProto wire format, parsed
    by caffe_proto.py) or a .npy file; None = zeros."""
    if mean_file is None:
        return np.zeros((1, 1, 500, 500), dtype=np.float32)
    if str(mean_file).endswith(".npy"):
        arr = np.load(mean_file)
    else:
        from . import caffe_proto
        arr = caffe_proto.read_binaryproto(mean_file)
    return np.asarray(arr, dtype=np.float32).reshape(1, 1, 500, 500)


def caffe_forward(net, image, mean_arr):
    """evaluation.caffe_forward(net, image, mean_arr) (reference evaluation.py:34-38):
    (500,500) uint8 sphere image -> (20,20) float32 sigmoid response."""
    mean = None if mean_arr is None or not np.any(mean_arr) else mean_arr
    net.set_mean(mean)
    return net.forward_batch(image[None])[0]


def debug_gemm(a_bf16_bits, b_bf16_bits, bias=None, relu=False, bn=128, ksplit=1, ctx=None):
    ctx = ctx or _lib.default_context()
    a = np.ascontiguousarray(a_bf16_bits, dtype=np.uint16)
    b = np.ascontiguousarray(b_bf16_bits, dtype=np.uint16)
    m, k = a.shape
    n = b.shape[0]
    out = np.empty((m, n), dtype=np.float32)
    bias = None if bias is None else np.ascontiguousarray(bias, dtype=np.float32)
    _lib.check(ctx.lib.vpk_debug_gemm(ctx.h, m, n, k, _lib.ptr(a), _lib.ptr(b), _lib.ptr(bias), int(relu), int(bn),
                                      int(ksplit), _lib.ptr(out)), "vpk_debug_gemm")
    return out
