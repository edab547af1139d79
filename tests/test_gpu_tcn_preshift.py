"""Pre-shifted limb-split convolutions (CRCNN_TCN2_PRESHIFT=1, default: weights staged as W 2^(8b) mod q, seven accumulator
classes, double-buffered accumulator) against the 13-class kernel (CRCNN_TCN2_PRESHIFT=0), byte for byte.  Covered: fan-in 25
(conv1 of PlainModel.h5), 32 (the largest that takes the seven-class kernel) and 180 (conv2, which stays on the 13-class kernel);
20 outputs (registers keep the four slots of a sector), 30 and 40 (8-byte stores, two output tiles); column counts that are not
multiples of 128; all-(q-1) NTT-form slots; chunked launches, an output-channel shard and the fused convolution + pooling +
batch-norm call; n = 2048, 4096 and 8192.  One case per n is also checked against the oracle."""
import os

import numpy as np
import pytest

from util import PRIMES, T_FOR_N, random_cts
from oracle.port import Oracle

pytestmark = pytest.mark.gpu


def _engine(n, pre):
    from crcnn_b200.lib import Engine
    old = os.environ.get("CRCNN_TCN2_PRESHIFT")
    os.environ["CRCNN_TCN2_PRESHIFT"] = str(pre)   # read when the context is created
    try:
        eng = Engine(n, PRIMES[n], T_FOR_N[n])
    finally:
        if old is None:
            os.environ.pop("CRCNN_TCN2_PRESHIFT", None)
        else:
            os.environ["CRCNN_TCN2_PRESHIFT"] = old
    eng.set_tensor_core_mode(0)   # keep the ternary-tap kernel out of the way
    return eng


@pytest.fixture(scope="module", params=[2048, 4096, 8192])
def env(request):
    n = request.param
    pre, old = _engine(n, 1), _engine(n, 0)
    orc = Oracle(n, PRIMES[n], T_FOR_N[n])
    yield n, PRIMES[n], pre, old, orc, np.random.default_rng(5 * n + 1)
    pre.close()
    old.close()


def _vals(orc, rng, count, lo=-3.0, hi=3.0):
    vals = rng.uniform(lo, hi, size=count).astype(np.float32)
    return vals, orc.encode_many(vals)


def _diff(a, b):
    bad = np.argwhere(a != b)
    return "%d of %d words differ, first at %s" % (len(bad), a.size, tuple(int(v) for v in bad[0])) if len(bad) else "equal"


def _both(pre, old, fn):
    return [fn(eng) for eng in (pre, old)]


# (zd, xf, yf, nf, xd, yd, B): fan-in zd * xf * yf
SHAPES = [(1, 5, 5, 20, 11, 9, 4),    # fan-in 25, 20 outputs; 4 x 3 positions -> 96 columns
          (2, 4, 4, 30, 9, 9, 7),     # fan-in 32, 30 outputs; 3 x 3 positions -> 126 columns
          (1, 5, 5, 40, 13, 13, 4),   # fan-in 25, two output tiles; 5 x 5 positions -> 200 columns
          (20, 3, 3, 50, 7, 7, 2)]    # fan-in 180 (conv2 shape): 13-class kernel either way


@pytest.mark.parametrize("zd,xf,yf,nf,xd,yd,B", SHAPES)
def test_conv_preshift_matches_13_class(env, zd, xf, yf, nf, xd, yd, B):
    n, primes, pre, old, orc, rng = env
    xs = ys = 2
    per = zd * xd * yd
    x = random_cts(rng, n, primes, B * per)
    wv, _ = _vals(orc, rng, nf * zd * xf * yf, -40.0, 40.0)
    bv, _ = _vals(orc, rng, nf)
    got = _both(pre, old, lambda e: e.download(e.conv(e.upload(x), e.plain_encode(wv), e.plain_encode(bv), B, xd, yd, zd, xs, ys, xf, yf, nf)))
    assert np.array_equal(got[0], got[1]), _diff(got[0], got[1])
    # extreme residues: every NTT-form slot q - 1 (the largest class sums), kept in the NTT domain
    K = len(primes)
    xm = np.zeros((B * per, 2, K, n + 1), dtype=np.uint64)
    for j, q in enumerate(primes):
        xm[:, :, j, :n] = q - 1
    xm[::7, :, :, :n] = 0
    got = _both(pre, old, lambda e: e.download(e.conv(e.upload(xm, ntt_form=True), e.plain_encode(wv), e.plain_encode(bv), B, xd, yd, zd, xs, ys,
                                                      xf, yf, nf), ntt_form=True))
    assert np.array_equal(got[0], got[1]), _diff(got[0], got[1])


def test_conv_preshift_chunked_sharded_and_oracle(env):
    n, primes, pre, old, orc, rng = env
    zd, xd, yd, xs, ys, xf, yf, nf, B = 1, 9, 7, 2, 2, 5, 5, 6, 2    # fan-in 25, 3 x 2 positions
    per = zd * xd * yd
    x = random_cts(rng, n, primes, B * per)
    wv, wp = _vals(orc, rng, nf * zd * xf * yf)
    bv, bp = _vals(orc, rng, nf)
    want = np.stack([orc.conv(x[b * per:(b + 1) * per], xd, yd, zd, xs, ys, xf, yf, nf, wp, bp) for b in range(B)])
    w, b_ = pre.plain_encode(wv), pre.plain_encode(bv)
    got = pre.download(pre.conv(pre.upload(x), w, b_, B, xd, yd, zd, xs, ys, xf, yf, nf)).reshape(want.shape)
    assert np.array_equal(got, want), _diff(got, want)
    # a tiny scratch budget: 32 slots per launch
    for eng in (pre, old):
        eng.set_tensor_core_mode(0, 0, 1)
    try:
        got = _both(pre, old, lambda e: e.download(e.conv(e.upload(x), e.plain_encode(wv), e.plain_encode(bv), B, xd, yd, zd, xs, ys, xf, yf, nf)))
    finally:
        for eng in (pre, old):
            eng.set_tensor_core_mode(0, 0, 12 << 30)
    assert np.array_equal(got[0], got[1]), _diff(got[0], got[1])
    assert np.array_equal(got[0].reshape(want.shape), want)
    # output-channel shard: rows 2-4 of the pre-shifted planes
    want_s = want.reshape(B, nf, -1)[:, 2:5]
    got = _both(pre, old, lambda e: e.download(e.conv(e.upload(x), e.plain_encode(wv), e.plain_encode(bv), B, xd, yd, zd, xs, ys, xf, yf, nf,
                                                      shard=(2, 3))).reshape(want_s.shape))
    assert np.array_equal(got[0], want_s), _diff(got[0], want_s)
    assert np.array_equal(got[1], want_s), _diff(got[1], want_s)


def test_conv_pool_bn_preshift(env):
    """The fused convolution + average pooling + batch-norm call, whose folded weights the seven-class kernel takes in PlainModel."""
    n, primes, pre, old, orc, rng = env
    zd, xd, yd, xs, ys, xf, yf, nf, B = 1, 15, 15, 2, 2, 5, 5, 20, 5    # 6 x 6 conv outputs, pooled 2x2/2 -> 3 x 3: 90 columns
    x = random_cts(rng, n, primes, B * zd * xd * yd)
    wv, _ = _vals(orc, rng, nf * zd * xf * yf)
    bv, _ = _vals(orc, rng, nf)
    mv, _ = _vals(orc, rng, nf)
    iv, _ = _vals(orc, rng, nf, 0.5, 2.0)
    sv = np.array([0.25], dtype=np.float32)

    def run(e):
        return e.download(e.conv_pool_bn(e.upload(x), e.plain_encode(wv), e.plain_encode(bv), B, xd, yd, zd, xs, ys, xf, yf, nf, 2, 2, 2, 2,
                                         e.plain_encode(sv), e.plain_encode(mv), e.plain_encode(iv)))
    got = _both(pre, old, run)
    assert np.array_equal(got[0], got[1]), _diff(got[0], got[1])
