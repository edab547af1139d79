"""Network::forward_dev(x, first, last) on EVERY layer range of the four topologies, with layer fusion on and off, through the C++ host
library (crcnn_b200.host.HostNetwork, the path bench.py measures).

forward_dev does not make one call per reference layer: Network::group_at (crcnn_b200.hpp) looks at the dynamic types of the layers from
i on and at where the range ends, and runs a composed group (DESIGN 4.5) -- conv + pool + batch-norm on the pooled grid, conv + pool with an
identity batch-norm, pool + batch-norm + fc + fc, fc + fc, pool + batch-norm -- or a single layer.  A range boundary that cuts a group must
give the smaller compositions on either side and the reference's bytes.  Here:

* the checked chain: with fusion off, a[i+1] = forward(a[i], i, i+1) for every layer, each step (and its output shape) against the oracle --
  whole layers where the oracle is cheap, the sampled checker (oracle/sampled.py) for conv / square / the large fc at n >= 4096;
* every range 0 <= first < last <= L: forward(a[first], first, last) == a[last] byte for byte with fusion off and on, per image as well at
  batch 2, and the kernel-class work counters of the run equal what the expected decomposition (group_at restated below) must do -- so a
  silent fall-back to layer by layer, or a group that reaches past `last`, cannot pass as "same bytes";
* the edges: first == last, invalid ranges (HostError, network still usable), and crcnn_host_forward_range on a network that has to
  re-encrypt before layer 6 (it runs forward_dev and never re-encrypts; Network::forward on the same network refuses).

Regression list (ranges that once failed; each runs in test_every_range_same_bytes_and_composed_groups and the checked chain):
* PlainModelTiny [0, 1) and every range ending at conv1: HostNetwork.forward sized its output buffer for 4096 ciphertexts per image;
  Tiny's conv1 gives 32 x 24 x 24 = 18,432 ("output buffer too small").  It now holds the network's largest activation.
"""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import util
from crcnn_b200 import nets
from oracle import sampled
from oracle.port import Oracle

# (model, n, batch); the suite's primes and T_FOR_N
CASES = [("ApproxPlainModel", 2048, 2), ("ApproxPlainModel", 4096, 2), ("PlainModelWoPad", 4096, 2), ("PlainModelTiny", 4096, 2),
         ("PlainModel", 8192, 1)]
CASE_IDS = ["Approx-n2048", "Approx-n4096", "WoPad-n4096", "Tiny-n4096", "PlainModel-n8192"]
SAMPLES = 12          # sampled outputs per large layer of the checked chain
POOL = ("pool", "avgpool")


# ---- Network::group_at restated over nets.TOPOLOGIES
def out_shape(layer, shape):
    """Per-image (z, x, y) after `layer` (the DeviceTensor shapes of crcnn_b200.hpp) from the input's `shape`."""
    kind = layer[0]
    if kind == "conv":
        _, _, xd, yd, zd, xs, ys, xf, yf, nf = layer
        return (nf, (xd - xf) // xs + 1, (yd - yf) // ys + 1)
    if kind in POOL:
        _, _, xd, yd, zd, xs, ys, xf, yf = layer
        return (zd, (xd - xf) // xs + 1, (yd - yf) // ys + 1)
    if kind == "fc":
        return (1, layer[3], 1)
    return tuple(shape)          # bn, square


def group_at(layers, i, last, fused=True):
    """(group, number of layers) that Network::group_at picks from layer i of the range [i, last); fused=False: set_fusion(False)."""
    kind = lambda k: layers[i + k][0]
    if not fused:
        return "Single", 1
    if i + 2 < last and kind(0) == "conv" and kind(1) in POOL and kind(2) == "bn":
        return "ConvPoolBn", 3
    if i + 1 < last and kind(0) == "conv" and kind(1) in POOL and tuple(layers[i + 1][2:4]) == out_shape(layers[i], None)[1:]:
        return "ConvPool", 2
    if i + 3 < last and kind(0) in POOL and kind(1) == "bn" and kind(2) == "fc" and kind(3) == "fc":
        return "PoolBnFcFc", 4
    if i + 1 < last and kind(0) == "fc" and kind(1) == "fc":
        return "FcFc", 2
    if i + 1 < last and kind(0) in POOL and kind(1) == "bn":
        return "PoolBn", 2
    return "Single", 1


def decompose(layers, first, last, fused=True):
    """[(group, first layer, number of layers)] that forward_dev(first, last) runs, in order."""
    out, i = [], first
    while i < last:
        g, k = group_at(layers, i, last, fused)
        out.append((g, i, k))
        i += k
    return out


def pool_sums(layer):
    """Window-sum terms per image of a pooling layer (pool_sum work / 2Kn)."""
    _, _, xd, yd, zd, xs, ys, xf, yf = layer
    return zd * ((xd - xf) // xs + 1) * ((yd - yf) // ys + 1) * xf * yf


def expected_work(layers, groups, batch):
    """What the kernel-class counters must show for `groups` at `batch`: weighted-sum terms (rows x columns x fan-in), window-sum terms
    and batch-norm launches.  The composed groups have their own signatures: the pooled grid sums the CONVOLUTION's input (dilated
    windows) and convolves at the combined stride, pool + bn + fc + fc sums windows and runs one out x in weighted sum with no
    batch-norm kernel, fc + fc runs one out2 x in weighted sum.  A pool + batch-norm group is only ever entered in coefficient form in
    these topologies (from the host, or after the square layer), where crcnn_pool_bn_forward runs the two layers' own kernels."""
    terms = sums = bn = 0
    for g, i, k in groups:
        ls = layers[i:i + k]
        if g in ("ConvPoolBn", "ConvPool"):
            _, _, xd, yd, zd, xs, ys, xf, yf, nf = ls[0]
            pxs, pys, pxf, pyf = ls[1][5:9]
            sums += zd * (xd - (pxf - 1) * xs) * (yd - (pyf - 1) * ys) * pxf * pyf
            _, pxo, pyo = out_shape(ls[1], None)
            terms += nf * pxo * pyo * zd * xf * yf
        elif g == "PoolBnFcFc":
            sums += pool_sums(ls[0])
            terms += ls[2][2] * ls[3][3]
        elif g == "FcFc":
            terms += ls[0][2] * ls[1][3]
        elif g == "PoolBn":
            sums += pool_sums(ls[0])
            bn += 1
        elif ls[0][0] in ("conv", "fc"):
            terms += nets.layer_terms(ls[0])
        elif ls[0][0] in POOL:
            sums += pool_sums(ls[0])
        elif ls[0][0] == "bn":
            bn += 1
    return dict(terms=terms * batch, sums=sums * batch, bn=bn)


# decompositions pinned by hand: (model, first, last) -> [(group, first layer)]
GROUP_TABLE = {
    ("ApproxPlainModel", 0, 9): [("ConvPoolBn", 0), ("Single", 3), ("Single", 4), ("PoolBnFcFc", 5)],
    ("ApproxPlainModel", 0, 2): [("ConvPool", 0)],
    ("ApproxPlainModel", 0, 3): [("ConvPoolBn", 0)],
    ("ApproxPlainModel", 0, 6): [("ConvPoolBn", 0), ("Single", 3), ("Single", 4), ("Single", 5)],
    ("ApproxPlainModel", 6, 9): [("Single", 6), ("FcFc", 7)],
    ("ApproxPlainModel", 1, 3): [("PoolBn", 1)],
    ("ApproxPlainModel", 1, 9): [("PoolBn", 1), ("Single", 3), ("Single", 4), ("PoolBnFcFc", 5)],
    ("ApproxPlainModel", 2, 9): [("Single", 2), ("Single", 3), ("Single", 4), ("PoolBnFcFc", 5)],
    ("ApproxPlainModel", 5, 8): [("PoolBn", 5), ("Single", 7)],
    ("ApproxPlainModel", 5, 9): [("PoolBnFcFc", 5)],
    ("ApproxPlainModel", 7, 9): [("FcFc", 7)],
    ("ApproxPlainModel", 8, 9): [("Single", 8)],
    ("PlainModelWoPad", 0, 9): [("ConvPoolBn", 0), ("Single", 3), ("Single", 4), ("PoolBnFcFc", 5)],
    ("PlainModelWoPad", 0, 2): [("ConvPool", 0)],
    ("PlainModelWoPad", 3, 7): [("Single", 3), ("Single", 4), ("PoolBn", 5)],
    ("PlainModelTiny", 0, 6): [("ConvPool", 0), ("ConvPool", 2), ("FcFc", 4)],
    ("PlainModelTiny", 0, 3): [("ConvPool", 0), ("Single", 2)],
    ("PlainModelTiny", 1, 5): [("Single", 1), ("ConvPool", 2), ("Single", 4)],
    ("PlainModelTiny", 3, 6): [("Single", 3), ("FcFc", 4)],
    ("PlainModel", 0, 9): [("ConvPoolBn", 0), ("Single", 3), ("Single", 4), ("PoolBnFcFc", 5)],
    ("PlainModel", 4, 9): [("Single", 4), ("PoolBnFcFc", 5)],
}


def test_group_at_restatement_table():
    """CPU: the Python restatement of Network::group_at gives the hand-written decompositions, and nothing but singles without fusion."""
    for (model, first, last), want in GROUP_TABLE.items():
        layers = nets.TOPOLOGIES[model]["layers"]
        assert [(g, i) for g, i, _ in decompose(layers, first, last)] == want, (model, first, last)
    for model, topo in nets.TOPOLOGIES.items():
        layers = topo["layers"]
        L = len(layers)
        for first in range(L):
            for last in range(first + 1, L + 1):
                groups = decompose(layers, first, last)
                assert groups[0][1] == first and sum(k for _, _, k in groups) == last - first, (model, first, last)
                assert decompose(layers, first, last, fused=False) == [("Single", i, 1) for i in range(first, last)]
    # the signatures tell the groups apart: a composed group never has its layers' work
    layers = nets.TOPOLOGIES["ApproxPlainModel"]["layers"]
    for first, last in [(0, 2), (0, 3), (5, 9), (7, 9)]:
        assert expected_work(layers, decompose(layers, first, last), 1) != expected_work(layers, decompose(layers, first, last, False), 1)


# ---- one network at a time (the host library holds one per process)
class _ParamsOnly:
    """Stands in for the engine so that nets.Network gives the float parameters (.params) without device packs."""
    plain_encode = plain_encode_f64 = staticmethod(lambda values: None)


class Case:
    def __init__(self, model, n, batch):
        self.model, self.n, self.batch = model, n, batch
        self.primes, self.t = util.PRIMES[n], util.T_FOR_N[n]
        self.K = len(self.primes)
        self.layers = nets.TOPOLOGIES[model]["layers"]
        self.L = len(self.layers)
        rng = np.random.default_rng(4000 + n + len(model))
        self.evk = util.random_evk(rng, n, self.primes)
        zd, xd, yd = nets.TOPOLOGIES[model]["input"]
        self.x = util.random_cts(rng, n, self.primes, batch * zd * xd * yd)
        self.shape0 = (zd, xd, yd)
        self.params = nets.Network(_ParamsOnly(), model).params
        self.encoded = {}
        self.chain = None
        self.net = self.eng = None
        self.build()

    def build(self, skip_reencryption=True):
        from crcnn_b200.host import HostNetwork
        from crcnn_b200.lib import Engine
        self.close()
        self.net = HostNetwork(self.n, self.primes, self.t, self.model, evk=self.evk, skip_reencryption=skip_reencryption)
        self.eng = Engine.adopt(self.net.ctx(), self.n, self.primes, self.t)
        return self.net

    def close(self):
        if self.net is not None:
            self.net.close()
            self.eng.h = None          # the context is gone: stray handles must not free into it
            self.net = self.eng = None

    def forward(self, x, first, last, shape, batch=None):
        return self.net.forward(x, batch=self.batch if batch is None else batch, first=first, last=last, shape=shape)

    def checked_chain(self):
        """(a, shapes): a[0] the input, a[i+1] = forward(a[i], i, i+1) with fusion off; computed once per network."""
        if self.chain is None:
            self.net.set_fusion(False)
            try:
                a, shapes = [self.x], [self.shape0]
                for i in range(self.L):
                    y, s = self.forward(a[i], i, i + 1, shapes[i])
                    a.append(y)
                    shapes.append(s)
            finally:
                self.net.set_fusion(True)
            self.chain = (a, shapes)
        return self.chain

    def work(self):
        """The counters since the last prof_reset, in units of 2Kn (one ring operation on both polynomials of a ciphertext)."""
        launches = {k: v[0] for k, v in self.eng.prof().items()}
        ops = {k: v[1] for k, v in self.eng.prof_work().items()}
        unit = 2.0 * self.K * self.n
        terms = ops["weighted_sum_mac"] / unit + ops["weighted_sum_tcn_i8"] / (49 * unit)
        return dict(terms=terms, sums=ops["pool_sum"] / unit, bn=launches["batch_norm"]), ops["weighted_sum_tc_i8"]


@pytest.fixture(scope="module", params=CASES, ids=CASE_IDS)
def case(request):
    c = Case(*request.param)
    yield c
    c.close()


# ---- the oracle for one layer of the chain
def _full_oracle(c, layer):
    if c.n == 2048:
        return True
    kind = layer[0]
    return kind in POOL or kind == "bn" or (kind == "fc" and layer[2] * layer[3] <= 10000)


def _encoded(c, orc, name):
    """The layer's float parameters encoded by the oracle (FractionalEncoder), once per network."""
    if name not in c.encoded:
        c.encoded[name] = tuple(orc.encode_many(v) for v in c.params[name])
    return c.encoded[name]


def oracle_layer(c, orc, i, x, pool):
    """Layer i of the reference on the host ciphertexts x ([batch * count][2][K][n+1]), image by image, each split into chunks of
    filters / rows / channels / ciphertexts (the reference's outputs are independent along these) run on the thread pool."""
    layer, kind = c.layers[i], c.layers[i][0]
    ct = x.shape[1:]
    per = len(x) // c.batch
    jobs = []
    for b in range(c.batch):
        xb = x[b * per:(b + 1) * per]
        if kind == "conv":
            _, name, xd, yd, zd, xs, ys, xf, yf, nf = layer
            W, B = _encoded(c, orc, name)
            R = zd * xf * yf
            jobs += [lambda xb=xb, k0=k0, k1=min(nf, k0 + 4): orc.conv(xb, xd, yd, zd, xs, ys, xf, yf, k1 - k0, W[k0 * R:k1 * R], B[k0:k1])
                     for k0 in range(0, nf, 4)]
        elif kind == "fc":
            _, name, in_dim, out_dim = layer
            W, B = _encoded(c, orc, name)
            step = max(1, out_dim // 16)
            jobs += [lambda xb=xb, r0=r0, r1=min(out_dim, r0 + step): orc.fc(xb, in_dim, r1 - r0, W[r0 * in_dim:r1 * in_dim], B[r0:r1])
                     for r0 in range(0, out_dim, step)]
        elif kind in POOL:
            _, name, xd, yd, zd, xs, ys, xf, yf = layer
            div = orc.encode(1.0 / (xf * yf)) if kind == "avgpool" else (None, None)     # a double: avgPoolingLayer.cpp:10-13
            jobs += [lambda xb=xb, z=z: orc.pool(xb[z * xd * yd:(z + 1) * xd * yd], xd, yd, 1, xs, ys, xf, yf, *div) for z in range(zd)]
        elif kind == "bn":
            _, name, zd, xd, yd = layer
            M, V = _encoded(c, orc, name)
            jobs += [lambda xb=xb, z=z: orc.bn(xb[z * xd * yd:(z + 1) * xd * yd], 1, xd, yd, M[z:z + 1], V[z:z + 1]) for z in range(zd)]
        else:
            step = max(1, per // 16)
            jobs += [lambda xb=xb, s=s: orc.square_layer(xb[s:s + step], *c.evk) for s in range(0, per, step)]
    return np.concatenate([np.asarray(r).reshape(-1, *ct) for r in pool.map(lambda f: f(), jobs)])


@pytest.mark.gpu
def test_checked_chain_layer_by_layer_equals_the_oracle(case):
    """Every step of the fusion-off chain, and its output shape, against the oracle: whole layers where that is cheap, the sampled
    checker (first / last / tile-boundary outputs + random ones, their input windows downloaded) for the large layers at n >= 4096."""
    c = case
    a, shapes = c.checked_chain()
    orc = Oracle(c.n, c.primes, c.t)
    rng = np.random.default_rng(c.n)
    shim = type("Layers", (), {"layers": c.layers, "params": c.params})
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as pool:
        for i, layer in enumerate(c.layers):
            assert shapes[i + 1] == out_shape(layer, shapes[i]), (i, shapes[i + 1])
            assert a[i + 1].shape == (c.batch * int(np.prod(shapes[i + 1])), 2, c.K, c.n + 1), i
            if _full_oracle(c, layer):
                want = oracle_layer(c, orc, i, a[i], pool)
                assert np.array_equal(want, a[i + 1]), "layer %d (%s) differs from the oracle" % (i, layer[1])
            else:
                x, y = c.eng.upload(a[i]), c.eng.upload(a[i + 1])
                try:
                    assert sampled.check_layer(c.eng, orc, shim, i, x, y, c.batch, rng, SAMPLES, c.evk, pool) > 0
                finally:
                    x.free()
                    y.free()
    assert shapes[-1] == (1, nets.TOPOLOGIES[c.model]["layers"][-1][3], 1)


@pytest.mark.gpu
def test_every_range_same_bytes_and_composed_groups(case):
    """For every 0 <= first < last <= L: forward(a[first], first, last) == a[last] (bytes and shape) with fusion off and on, per image as
    well at batch 2.  Which path ran, from the kernel-class counters: window-sum terms and batch-norm launches in both modes; with fusion
    on, a second run with the ternary-tap GEMM off (so that every weighted sum counts its work in the limb-split or CUDA-core classes,
    and after the first run built any composed constants) must show the weighted-sum terms of the expected decomposition."""
    c = case
    a, shapes = c.checked_chain()
    checked = 0
    for first in range(c.L):
        for last in range(first + 1, c.L + 1):
            where = (c.model, first, last)
            for fused in (False, True):
                c.net.set_fusion(fused)
                want = expected_work(c.layers, decompose(c.layers, first, last, fused), c.batch)
                c.eng.prof_reset()
                got, s = c.forward(a[first], first, last, shapes[first])
                assert s == shapes[last] and np.array_equal(got, a[last]), (where, "fused" if fused else "layer by layer")
                work, _ = c.work()
                assert (work["sums"], work["bn"]) == (want["sums"], want["bn"]), (where, fused, work, want)
                checked += 1
            c.eng.set_tensor_core_mode(0)
            try:
                c.eng.prof_reset()
                got, s = c.forward(a[first], first, last, shapes[first])
                work, tc_ops = c.work()
            finally:
                c.eng.set_tensor_core_mode(1)
            assert s == shapes[last] and np.array_equal(got, a[last]), (where, "fused, ternary-tap GEMM off")
            assert tc_ops == 0 and work == want, (where, decompose(c.layers, first, last), work, want)
            if c.batch > 1:
                pin, pout = int(np.prod(shapes[first])), int(np.prod(shapes[last]))
                for b in range(c.batch):
                    one, s = c.forward(a[first][b * pin:(b + 1) * pin], first, last, shapes[first], batch=1)
                    assert s == shapes[last] and np.array_equal(one, a[last][b * pout:(b + 1) * pout]), (where, "image", b)
    assert checked == c.L * (c.L + 1)


@pytest.mark.gpu
def test_range_edges(case):
    """first == last hands the input back unchanged (same shape); first > last, first < 0 and last > L raise HostError and leave the
    network usable."""
    from crcnn_b200.host import HostError
    c = case
    a, shapes = c.checked_chain()
    for i in range(c.L + 1):
        got, s = c.forward(a[i], i, i, shapes[i])
        assert s == shapes[i] and np.array_equal(got, a[i]), i
    for first, last in [(3, 2), (c.L, 0), (-1, 2), (0, c.L + 1), (c.L, c.L + 1)]:
        with pytest.raises(HostError):
            c.forward(a[0], first, last, shapes[0])
    got, s = c.forward(a[0], 0, c.L, shapes[0])
    assert s == shapes[-1] and np.array_equal(got, a[-1])


@pytest.mark.gpu
@pytest.mark.parametrize("case", [CASES[0]], ids=[CASE_IDS[0]], indirect=True)
def test_forward_range_runs_forward_dev_without_reencryption(case):
    """skip_reencryption unset: the reference re-encrypts before layer 6 (CrCNN/src/network.cpp:30), and Network::forward /
    forward_batch refuse to pass it with no re-encryption installed.  crcnn_host_forward_range is the segment API -- it runs
    forward_dev and never re-encrypts -- so ranges that cross layer 6, end there or start there give the chain's bytes."""
    from crcnn_b200.host import HostError
    import fv_keygen as kg
    c = case
    a, shapes = c.checked_chain()
    try:
        c.build(skip_reencryption=False)
        for first, last in [(0, 9), (0, 6), (6, 9), (4, 8), (5, 7), (6, 6)]:
            got, s = c.forward(a[first], first, last, shapes[first])
            assert s == shapes[last] and np.array_equal(got, a[last]), (first, last)
        keys = kg.generate(Oracle(c.n, c.primes, c.t), 3)
        c.net.use_keys(keys.sk, keys.pk)
        imgs = np.stack([util.synthetic_image(b) for b in range(c.batch)])
        with pytest.raises(HostError, match="re-encryption"):
            c.net.predict_values(imgs, batch=c.batch, seed=1)
        got, s = c.forward(a[0], 0, c.L, shapes[0])                      # and the segment API still runs
        assert np.array_equal(got, a[-1])
    finally:
        c.build()
