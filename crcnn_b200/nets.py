"""Network topologies of the reference's builder and a device-resident predict path over the C ABI.

Topologies mirror CnnBuilder::buildNetwork (CrCNN/src/cnnBuilder.cpp:108-179: Approx, WoPad and
Tiny blocks); `PlainModel` is the weights file PlainModel.h5 run through the unchanged layer API on
a 32x32 zero-bordered input (SURVEY.md section 8(a), table of topologies, and Appendix B3).
PADDED_TOPOLOGIES holds the networks whose convolutions have zero padding: `PlainModelPadded` is
PlainModel.h5 as it was trained, conv1 with padding 2 on the 28x28 image.

Network.forward mirrors Network::forward (CrCNN/src/network.cpp:22-47) without the hard-coded
re-encryption before layer 6: re-encryption needs the SECRET key and therefore belongs to the
client; `forward(first, last)` exposes the segment API for it (SURVEY.md section 8(f) row N2).
"""
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
WEIGHTS_DIR = os.path.join(os.path.dirname(_HERE), "weights")

# coeff_modulus_128(n) of SEAL 2.3.1 (SEAL/seal/util/globals.cpp:50-74 via defaultparams.h:22-26): the reference's parameter choice
# (CrCNN/src/globals.cpp:30); tests pin the same table against the compiled reference
DEFAULT_PRIMES_128 = {
    2048: [0x3fffffff000001],
    4096: [0x7fffffff380001, 0x3fffffff000001],
    8192: [0x7fffffff380001, 0x7ffffffef00001, 0x3fffffff000001, 0x3ffffffef40001],
    16384: [0x7fffffff380001, 0x7ffffffef00001, 0x7ffffffeac0001, 0x7ffffffe700001,
            0x7ffffffe600001, 0x7ffffffe4c0001, 0x3fffffff000001, 0x3ffffffef40001],
}

# layer tuples: (kind, name, args...) with the reference's constructor argument order
TOPOLOGIES = {
    # cnnBuilder.cpp:115-134
    "ApproxPlainModel": dict(input=(1, 28, 28), layers=[
        ("conv", "pool1_features.conv1", 28, 28, 1, 2, 2, 5, 5, 20),
        ("avgpool", "pool1", 12, 12, 20, 1, 1, 2, 2),
        ("bn", "pool1_features.norm1", 20, 11, 11),
        ("conv", "pool2_features.conv2", 11, 11, 20, 2, 2, 3, 3, 50),
        ("square", "act1", 50, 5, 5),
        ("avgpool", "pool2", 5, 5, 50, 1, 1, 2, 2),
        ("bn", "pool2_features.norm2", 50, 4, 4),
        ("fc", "classifier.fc3", 800, 500),
        ("fc", "classifier.fc4", 500, 10)]),
    # cnnBuilder.cpp:136-155
    "PlainModelWoPad": dict(input=(1, 28, 28), layers=[
        ("conv", "pool1_features.conv1", 28, 28, 1, 2, 2, 5, 5, 20),
        ("pool", "pool1", 12, 12, 20, 1, 1, 2, 2),
        ("bn", "pool1_features.norm1", 20, 11, 11),
        ("conv", "pool2_features.conv2", 11, 11, 20, 2, 2, 3, 3, 50),
        ("square", "act1", 50, 5, 5),
        ("pool", "pool2", 5, 5, 50, 1, 1, 2, 2),
        ("bn", "pool2_features.norm2", 50, 4, 4),
        ("fc", "classifier.fc3", 800, 500),
        ("fc", "classifier.fc4", 500, 10)]),
    # cnnBuilder.cpp:157-169
    "PlainModelTiny": dict(input=(1, 28, 28), layers=[
        ("conv", "pool1_features.conv1", 28, 28, 1, 1, 1, 5, 5, 32),
        ("avgpool", "pool1", 24, 24, 32, 2, 2, 2, 2),
        ("conv", "pool2_features.conv2", 12, 12, 32, 1, 1, 5, 5, 64),
        ("avgpool", "pool2", 8, 8, 64, 2, 2, 2, 2),
        ("fc", "classifier.fc3", 1024, 512),
        ("fc", "classifier.fc4", 512, 10)]),
    # PlainModel.h5: conv1 trained with padding=2 -> 32x32 zero-bordered input, fc3 is 1250 -> 500
    "PlainModel": dict(input=(1, 32, 32), layers=[
        ("conv", "pool1_features.conv1", 32, 32, 1, 2, 2, 5, 5, 20),
        ("avgpool", "pool1", 14, 14, 20, 1, 1, 2, 2),
        ("bn", "pool1_features.norm1", 20, 13, 13),
        ("conv", "pool2_features.conv2", 13, 13, 20, 2, 2, 3, 3, 50),
        ("square", "act1", 50, 6, 6),
        ("avgpool", "pool2", 6, 6, 50, 1, 1, 2, 2),
        ("bn", "pool2_features.norm2", 50, 5, 5),
        ("fc", "classifier.fc3", 1250, 500),
        ("fc", "classifier.fc4", 500, 10)]),
}

# Networks with zero-padded convolutions: conv tuples carry two more fields, the padding (xp, yp) (ConvolutionalLayer's padded
# constructors).  Kept apart from TOPOLOGIES, whose conv tuples have the reference's ten fields.  "weights": the .npz they read.
PADDED_TOPOLOGIES = {
    # PlainModel.h5 as trained: conv1 5x5 / 2 with padding 2 on 28x28, then the same eight layers as "PlainModel"
    "PlainModelPadded": dict(input=(1, 28, 28), weights="PlainModel", layers=[
        ("conv", "pool1_features.conv1", 28, 28, 1, 2, 2, 5, 5, 20, 2, 2)] + TOPOLOGIES["PlainModel"]["layers"][1:]),
}


def topology(model):
    """The topology dict of `model`, from TOPOLOGIES or PADDED_TOPOLOGIES."""
    return TOPOLOGIES[model] if model in TOPOLOGIES else PADDED_TOPOLOGIES[model]


def load_weights(model):
    name = PADDED_TOPOLOGIES[model]["weights"] if model in PADDED_TOPOLOGIES else model
    return dict(np.load(os.path.join(WEIGHTS_DIR, name + ".npz")))


def conv_out(layer):
    """(xo, yo) of a conv tuple, with its padding (0 for the reference's ten-field tuples)."""
    _, _, xd, yd, zd, xs, ys, xf, yf, nf = layer[:10]
    xp, yp = layer[10:12] if len(layer) > 10 else (0, 0)
    return (xd + 2 * xp - xf) // xs + 1, (yd + 2 * yp - yf) // ys + 1


def layer_terms(layer):
    """Weighted-sum terms (ciphertext x plaintext products) per image of one layer."""
    if layer[0] == "conv":
        _, _, xd, yd, zd, xs, ys, xf, yf, nf = layer[:10]
        xo, yo = conv_out(layer)
        return nf * xo * yo * zd * xf * yf
    if layer[0] == "fc":
        return layer[2] * layer[3]
    return 0


def layer_io_counts(layer):
    """(input ciphertexts, output ciphertexts) per image."""
    k = layer[0]
    if k == "conv":
        _, _, xd, yd, zd, xs, ys, xf, yf, nf = layer[:10]
        xo, yo = conv_out(layer)
        return zd * xd * yd, nf * xo * yo
    if k in ("pool", "avgpool"):
        _, _, xd, yd, zd, xs, ys, xf, yf = layer
        return zd * xd * yd, zd * ((xd - xf) // xs + 1) * ((yd - yf) // ys + 1)
    if k in ("bn", "square"):
        c = layer[2] * layer[3] * layer[4]
        return c, c
    if k == "fc":
        return layer[2], layer[3]
    raise ValueError(k)


class Network:
    """Encoded network resident on one GPU (weights as plaintext packs behind the C ABI)."""

    def __init__(self, eng, model, weights=None, evk=None, limit=None):
        """limit: optional dict {layer_name: max_outputs} to build a cropped network (used only by the
        bounded CPU-baseline sample; the GPU path always runs the full layers)."""
        self.eng, self.model = eng, model
        topo = topology(model)
        self.input_shape = topo["input"]
        self.layers = list(topo["layers"])
        w = weights if weights is not None else load_weights(model)
        self.evk = evk
        self.packs = {}
        self.params = {}   # the float32 values every pack was encoded from (what a checker re-encodes)
        for layer in self.layers:
            kind, name = layer[0], layer[1]
            if kind in ("conv", "fc"):
                self.params[name] = (w[name + ".weight"].ravel().astype(np.float32), w[name + ".bias"].ravel().astype(np.float32))
                self.packs[name] = (eng.plain_encode(w[name + ".weight"].ravel()), eng.plain_encode(w[name + ".bias"].ravel()))
            elif kind == "bn":
                # CnnBuilder::buildBatchNormLayer, cnnBuilder.cpp:89-105 (float32 arithmetic as in the reference)
                var = w[name + ".running_var"].astype(np.float32)
                invstd = (1.0 / np.sqrt(var.astype(np.float64) + 0.00001)).astype(np.float32)  # double arithmetic, float result: cnnBuilder.cpp:101
                self.params[name] = (w[name + ".running_mean"].astype(np.float32), invstd)
                self.packs[name] = (eng.plain_encode(w[name + ".running_mean"]), eng.plain_encode(invstd))
            elif kind == "avgpool":
                xf, yf = layer[7], layer[8]
                self.packs[name] = (eng.plain_encode_f64([1.0 / (xf * yf)]),)  # encode(1./(xf*yf)) on a DOUBLE: avgPoolingLayer.cpp:10-13

    def num_layers(self):
        return len(self.layers)

    def forward_layer(self, i, x, batch):
        eng, layer = self.eng, self.layers[i]
        kind, name = layer[0], layer[1]
        if kind == "conv":
            w, b = self.packs[name]
            return eng.conv(x, w, b, batch, *layer[2:])
        if kind == "fc":
            w, b = self.packs[name]
            return eng.fc(x, w, b, batch, layer[2], layer[3])
        if kind == "pool":
            return eng.pool(x, batch, *layer[2:])
        if kind == "avgpool":
            return eng.pool(x, batch, *layer[2:], scale=self.packs[name][0])
        if kind == "bn":
            m, v = self.packs[name]
            return eng.bn(x, batch, layer[2], layer[3], layer[4], m, v)
        if kind == "square":
            if self.evk is None:
                raise RuntimeError("square layer needs evaluation keys")
            return eng.square_layer(x, self.evk)
        raise ValueError(kind)

    def forward(self, x, batch=1, first=0, last=None, on_layer=None):
        """Layers [first, last) applied in order, activations staying on the device.
        on_layer(i, layer) is called after each layer has been enqueued (for event timing)."""
        last = len(self.layers) if last is None else last
        for i in range(first, last):
            y = self.forward_layer(i, x, batch)
            if i > first:
                x.free()  # intermediate activation
            x = y
            if on_layer is not None:
                on_layer(i, self.layers[i])
        return x


# ------------------------------------------------------------------------------------------------
# Output-neuron sharding (SURVEY.md section 8(e) item 3): the reference splits a layer's output
# filters / rows across std::threads (convolutionalLayer.cpp:177-187, fullyConnectedLayer.cpp:148-158);
# across GPUs the same split applies, followed by an all-gather of the layer's output ciphertexts
# before the next layer that consumes every channel.  The sharded network itself is C++
# (crcnn_b200::ShardedNetwork in cpp/crcnn_b200.hpp, driven through host.HostNetwork); these two helpers
# restate its split for the CPU tests of the gather order (tests/test_sharding_gloo.py).
# ------------------------------------------------------------------------------------------------
def shard_range(total, world, rank):
    """Contiguous, balanced split of `total` output channels/rows: the first total % world ranks get one more."""
    base, extra = divmod(total, world)
    first = rank * base + min(rank, extra)
    return first, base + (1 if rank < extra else 0)


def gather_counts(total, world, per_channel):
    """Ciphertexts each rank contributes to the all-gather of a [channels][per_channel] activation."""
    return [shard_range(total, world, r)[1] * per_channel for r in range(world)]
