"""ORACLE (test infrastructure, not product code) -- stage 2, the CNN.

torch-CPU float32 execution of the reference's cnn/deploy.prototxt (lines
cited per layer) with Caffe semantics: cross-correlation convolutions, LRN
ACROSS_CHANNELS scale = 1 + (alpha/n) * sum x^2, ceil-mode max pooling with
clipped windows, InnerProduct over the NCHW flattening, Dropout = identity at
TEST.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference leg may import this module.

PARITY STATUS: *unpinned* against Caffe RC5 itself (not installable offline,
its weights/mean files are external downloads, reference README.md:23); the
layer shapes of SURVEY.md section 8(a) are asserted in tests/test_oracle_cnn.py.
Random-init uses the fillers of train/train_val.prototxt (deploy.prototxt has
none except on fc8, so its Caffe default would be an all-zero net).
"""
import numpy as np
import torch
import torch.nn.functional as F

# (name, Caffe blob shape, filler std, bias value): train/train_val.prototxt:83-90,
# 139-146, 194-201, 228-235, 262-269, 304-311, 344-351, 384-391
LAYERS = [
    ("conv1", (96, 1, 11, 11), 0.01, 0.0),
    ("conv2", (256, 48, 5, 5), 0.01, 0.1),
    ("conv3", (384, 256, 3, 3), 0.01, 0.0),
    ("conv4", (384, 192, 3, 3), 0.01, 0.1),
    ("conv5", (256, 192, 3, 3), 0.01, 0.1),
    ("fc6", (4096, 57600), 0.005, 0.1),
    ("fc7", (4096, 4096), 0.005, 0.1),
    ("fc8_20x20", (400, 4096), 0.01, 0.0),
]


def random_weights(seed=0, scale=1.0):
    """Gaussian/constant fillers of train_val.prototxt, float32 numpy arrays.
    `scale` multiplies every weight std (scale > 1 makes the random net less
    degenerate so the 20x20 response has real maxima)."""
    g = torch.Generator().manual_seed(seed)
    ws, bs = [], []
    for _, shape, std, bias in LAYERS:
        ws.append((torch.randn(shape, generator=g, dtype=torch.float32) * (std * scale)).numpy())
        bs.append(np.full(shape[0], bias, dtype=np.float32))
    return ws, bs


def forward(images, weights, biases, mean=None, return_layers=False):
    """images (n,500,500) uint8 -> (sigout (n,20,20) float32, logits (n,400) float32).
    evaluation.py:35: data = image - mean (raw 0..255 scale)."""
    x = torch.from_numpy(np.ascontiguousarray(images)).to(torch.float32)[:, None]
    if mean is not None:
        x = x - torch.from_numpy(np.asarray(mean, dtype=np.float32)).reshape(1, 1, 500, 500)
    w = [torch.from_numpy(a) for a in weights]
    b = [torch.from_numpy(a) for a in biases]
    layers = {}
    with torch.no_grad():
        x = F.relu(F.conv2d(x, w[0], b[0], stride=4))                              # deploy.prototxt:9-33
        layers["conv1"] = x
        x = F.local_response_norm(x, 5, alpha=1e-4, beta=0.75, k=1.0)              # :34-44
        layers["norm1"] = x
        x = F.max_pool2d(x, 3, 2, ceil_mode=True)                                  # :45-55
        layers["pool1"] = x
        x = F.relu(F.conv2d(x, w[1], b[1], padding=2, groups=2))                   # :56-81
        layers["conv2"] = x
        x = F.local_response_norm(x, 5, alpha=1e-4, beta=0.75, k=1.0)              # :82-92
        layers["norm2"] = x
        x = F.max_pool2d(x, 3, 2, ceil_mode=True)                                  # :93-103
        layers["pool2"] = x
        x = F.relu(F.conv2d(x, w[2], b[2], padding=1))                             # :104-128
        layers["conv3"] = x
        x = F.relu(F.conv2d(x, w[3], b[3], padding=1, groups=2))                   # :129-154
        layers["conv4"] = x
        x = F.relu(F.conv2d(x, w[4], b[4], padding=1, groups=2))                   # :155-180
        layers["conv5"] = x
        x = F.max_pool2d(x, 3, 2, ceil_mode=True)                                  # :181-191
        layers["pool5"] = x
        x = x.flatten(1)
        x = F.relu(F.linear(x, w[5], b[5]))                                        # :192-223 (drop6 = identity)
        layers["fc6"] = x
        x = F.relu(F.linear(x, w[6], b[6]))                                        # :224-256
        layers["fc7"] = x
        logits = F.linear(x, w[7], b[7])                                           # :257-281
        sig = torch.sigmoid(logits).reshape(-1, 20, 20)                            # :283-304
    if return_layers:
        return sig.numpy(), logits.numpy(), {k: v.numpy() for k, v in layers.items()}
    return sig.numpy(), logits.numpy()
