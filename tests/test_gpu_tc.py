"""Tensor-core (tcgen05 kind::i8) weighted-sum path against the CPU oracle, byte for byte.

The engine picks this path for conv / fc layers whose weights are base-3 fractional encodings with
|w| < 1/2, fan-in >= 256 and >= 32 outputs (crcnn_b200/csrc/tc_mac.cuh); the tests force it for small shapes.  Every test also checks through the
kernel-class counters that the tensor-core kernel is what actually ran (no silent fallback), and that the
CUDA-core NTT-domain kernel gives the same bytes.
"""
import numpy as np
import pytest

from util import PRIMES, T_FOR_N, random_cts
from oracle.port import Oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=[2048, 4096, 8192])
def env(request):
    from crcnn_b200.lib import Engine
    n = request.param
    primes, t = PRIMES[n], T_FOR_N[n]
    eng = Engine(n, primes, t)
    eng.set_tensor_core_mode(2, 64)   # mode 2: every eligible layer with fan-in >= 64, however few outputs
    orc = Oracle(n, primes, t)
    rng = np.random.default_rng(7 * n)
    yield n, primes, t, eng, orc, rng
    eng.close()


def _small(orc, rng, count):
    vals = rng.uniform(-0.49, 0.49, size=count).astype(np.float32)
    return vals, orc.encode_many(vals)


def _explain(got, want):
    bad = np.argwhere(got != want)
    if len(bad) == 0:
        return "equal"
    cts = sorted(set(int(b[0]) for b in bad))
    first = tuple(int(v) for v in bad[0])
    coeffs = sorted(set(int(b[-1]) for b in bad))
    return "%d mismatching words in %d of %d ciphertexts (first cts %s); first at %s: got %d want %d; coefficient range [%d, %d]" % (
        len(bad), len(cts), got.shape[0], cts[:8], first, int(got[first]), int(want[first]), coeffs[0], coeffs[-1])


def _tc_launches(eng):
    return eng.prof().get("weighted_sum_tc_i8", (0, 0.0))[0]


def test_fc_layer_on_tensor_cores(env):
    n, primes, t, eng, orc, rng = env
    in_dim, out_dim = 70, 9          # 3 K-steps of 32 (the last one partial), 3 row tiles (the last one partial)
    x = random_cts(rng, n, primes, in_dim)
    wv, wp = _small(orc, rng, in_dim * out_dim)
    bv, bp = _small(orc, rng, out_dim)
    want = orc.fc(x, in_dim, out_dim, wp, bp)
    before = _tc_launches(eng)
    got = eng.download(eng.fc(eng.upload(x), eng.plain_encode(wv), eng.plain_encode(bv), 1, in_dim, out_dim))
    assert _tc_launches(eng) == before + 1, "the tensor-core kernel did not run"
    got = got.reshape(want.shape)
    assert np.array_equal(got, want), _explain(got, want)
    # the CUDA-core NTT-domain kernel on the same inputs
    eng.set_tensor_core_mode(0)
    try:
        got2 = eng.download(eng.fc(eng.upload(x), eng.plain_encode(wv), eng.plain_encode(bv), 1, in_dim, out_dim))
    finally:
        eng.set_tensor_core_mode(2)
    assert np.array_equal(got2.reshape(want.shape), want)


def test_fc_layer_tc_batched_sharded_ntt_input(env):
    n, primes, t, eng, orc, rng = env
    in_dim, out_dim, B = 130, 6, 2   # two 128-byte K blocks
    x = random_cts(rng, n, primes, B * in_dim)
    wv, wp = _small(orc, rng, in_dim * out_dim)
    bv, bp = _small(orc, rng, out_dim)
    want = np.stack([orc.fc(x[b * in_dim:(b + 1) * in_dim], in_dim, out_dim, wp, bp) for b in range(B)])
    w, b_ = eng.plain_encode(wv), eng.plain_encode(bv)
    tx = eng.upload(x)
    eng.to_ntt(tx)                   # the path converts NTT-form activations back itself
    before = _tc_launches(eng)
    got = eng.download(eng.fc(tx, w, b_, B, in_dim, out_dim)).reshape(want.shape)
    assert _tc_launches(eng) == before + 1
    assert np.array_equal(got, want), _explain(got, want)
    want_s = want.reshape(B, out_dim, -1)[:, 1:5]
    got_s = eng.download(eng.fc(eng.upload(x), w, b_, B, in_dim, out_dim, shard=(1, 4))).reshape(want_s.shape)
    assert np.array_equal(got_s, want_s), _explain(got_s, want_s)


def test_conv_layer_on_tensor_cores(env):
    n, primes, t, eng, orc, rng = env
    xd, yd, zd, xs, ys, xf, yf, nf, B = 5, 4, 8, 2, 1, 3, 3, 5, 2   # fan-in 72, 2x2 positions
    per = zd * xd * yd
    x = random_cts(rng, n, primes, B * per)
    wv, wp = _small(orc, rng, nf * zd * xf * yf)
    bv, bp = _small(orc, rng, nf)
    want = np.stack([orc.conv(x[b * per:(b + 1) * per], xd, yd, zd, xs, ys, xf, yf, nf, wp, bp) for b in range(B)])
    w, b_ = eng.plain_encode(wv), eng.plain_encode(bv)
    before = _tc_launches(eng)
    got = eng.download(eng.conv(eng.upload(x), w, b_, B, xd, yd, zd, xs, ys, xf, yf, nf)).reshape(want.shape)
    assert _tc_launches(eng) == before + 1
    assert np.array_equal(got, want), _explain(got, want)
    # tiny scratch budget: one output position per launch
    eng.set_tensor_core_mode(2, 0, 1)
    try:
        got2 = eng.download(eng.conv(eng.upload(x), w, b_, B, xd, yd, zd, xs, ys, xf, yf, nf)).reshape(want.shape)
    finally:
        eng.set_tensor_core_mode(2, 0, 12 << 30)
    assert np.array_equal(got2, want), _explain(got2, want)
    want_s = want.reshape(B, nf, -1)[:, 2:5]
    got_s = eng.download(eng.conv(eng.upload(x), w, b_, B, xd, yd, zd, xs, ys, xf, yf, nf, shard=(2, 3))).reshape(want_s.shape)
    assert np.array_equal(got_s, want_s), _explain(got_s, want_s)


def test_weights_outside_the_tap_window_fall_back(env):
    """|w| >= 1/2 puts a digit at x^0: not representable by the 32 fractional taps, so the engine must
    take the NTT-domain kernel and still be exact."""
    n, primes, t, eng, orc, rng = env
    in_dim, out_dim = 66, 3
    x = random_cts(rng, n, primes, in_dim)
    wv = rng.uniform(-0.49, 0.49, size=in_dim * out_dim).astype(np.float32)
    wv[5] = 0.75
    wv[100] = -2.5
    wp = orc.encode_many(wv)
    bv, bp = _small(orc, rng, out_dim)
    want = orc.fc(x, in_dim, out_dim, wp, bp)
    before = _tc_launches(eng)
    got = eng.download(eng.fc(eng.upload(x), eng.plain_encode(wv), eng.plain_encode(bv), 1, in_dim, out_dim)).reshape(want.shape)
    assert _tc_launches(eng) == before
    assert np.array_equal(got, want), _explain(got, want)


def test_extreme_inputs_on_tensor_cores(env):
    """All-(q-1) inputs with all-ones / all-minus-ones digit patterns: the largest accumulator magnitudes."""
    n, primes, t, eng, orc, rng = env
    in_dim, out_dim = 96, 4
    K = len(primes)
    x = np.zeros((in_dim, 2, K, n + 1), dtype=np.uint64)
    for j, q in enumerate(primes):
        x[:, :, j, :n] = q - 1
    x[::7, :, :, :n] = 0
    wv = np.empty((out_dim, in_dim), dtype=np.float32)
    wv[0] = 0.5 - 2.0 ** -24          # digits (almost) all +1
    wv[1] = -(0.5 - 2.0 ** -24)       # all -1
    wv[2] = 0.0
    wv[3] = rng.uniform(-0.49, 0.49, size=in_dim)
    wv = wv.ravel()
    wp = orc.encode_many(wv)
    bv, bp = _small(orc, rng, out_dim)
    want = orc.fc(x, in_dim, out_dim, wp, bp)
    before = _tc_launches(eng)
    got = eng.download(eng.fc(eng.upload(x), eng.plain_encode(wv), eng.plain_encode(bv), 1, in_dim, out_dim)).reshape(want.shape)
    assert _tc_launches(eng) == before + 1
    assert np.array_equal(got, want), _explain(got, want)

