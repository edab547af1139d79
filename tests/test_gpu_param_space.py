"""Every C-ABI entry point against the CPU oracle at parameter sets beyond SEAL's defaults (tests/util.py: PARAM_SETS), byte for byte.

crcnn_ctx_create accepts n a power of two in [1024, 16384], up to 8 distinct primes of at most 60 bits and any t >= 2 below every
prime, and the kernels choose their code paths from exactly these properties: the number of byte planes (primes above 56 bits),
the folded reductions (primes of the 2^k - delta shape), whether R residues add up below 2^64, the relinearization digit count, K,
the auxiliary base size and the plain modulus.  Each case also checks through the kernel-class counters which kernel ran, so that a
silent fallback cannot make it vacuous.  Bar: np.array_equal, no tolerance.
"""
import types
import zlib

import numpy as np
import pytest

import fv_keygen as kg
from util import PARAM_SETS, random_cts, random_evk
from oracle.port import Oracle

pytestmark = pytest.mark.gpu


def _bits(primes):
    return max(int(q).bit_length() for q in primes)


@pytest.fixture(scope="module", params=list(PARAM_SETS))
def env(request):
    from crcnn_b200.lib import Engine
    name = request.param
    n, primes, t = PARAM_SETS[name]
    eng = Engine(n, primes, t)
    orc = Oracle(n, primes, t)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    bits = _bits(primes)
    yield types.SimpleNamespace(name=name, n=n, primes=[int(q) for q in primes], t=t, K=len(primes), eng=eng, orc=orc, rng=rng,
                                bits=bits, seven=bits <= 56)
    eng.close()


def _layers(e):
    """Layer cases stay at n <= 8192 (oracle time); the 16384 set covers tables, transforms, square and relinearize."""
    if e.n > 8192:
        pytest.skip("oracle time")


def _explain(got, want):
    bad = np.argwhere(got != want)
    if len(bad) == 0:
        return "equal"
    cts = sorted(set(int(b[0]) for b in bad))
    first = tuple(int(v) for v in bad[0])
    return "%d mismatching words in %d of %d ciphertexts (first cts %s); first at %s: got %d want %d" % (
        len(bad), len(cts), got.shape[0], cts[:8], first, int(got[first]), int(want[first]))


def _check(got, want, what=""):
    got = got.reshape(want.shape)
    assert np.array_equal(got, want), "%s: %s" % (what, _explain(got, want))


class _Ran:
    """Kernel classes launched inside the with-block: {class: launches}."""

    def __init__(self, eng):
        self.eng = eng

    def __enter__(self):
        self.before = {k: v[0] for k, v in self.eng.prof().items()}
        return self

    def __exit__(self, *exc):
        after = {k: v[0] for k, v in self.eng.prof().items()}
        self.counts = {k: v - self.before.get(k, 0) for k, v in after.items() if v - self.before.get(k, 0) > 0}
        return False

    def __getitem__(self, k):
        return self.counts.get(k, 0)


def _top(e, count, size=2):
    """All-(q-1) residues: the largest operands of every product and sum."""
    x = np.zeros((count, size, e.K, e.n + 1), dtype=np.uint64)
    for j, q in enumerate(e.primes):
        x[:, :, j, :e.n] = q - 1
    return x


def _vals(e, count, lo=-1.0, hi=1.0):
    v = e.rng.uniform(lo, hi, size=count).astype(np.float32)
    return v, e.orc.encode_many(v)


def _ntt(e, x):
    t = e.eng.upload(x)
    e.eng.to_ntt(t)
    return t


# ---------------------------------------------------------------------------------------------------- tables and transforms
def test_ntt_tables(env):
    e = env
    assert e.eng.S == e.orc.S
    for slot in range(e.K + e.orc.S):
        base, idx = (0, slot) if slot < e.K else (1, slot - e.K)
        for which in range(4):
            assert np.array_equal(e.eng.ntt_table(slot, which), e.orc.ntt_table(base, idx, which)), (slot, which)


def test_transforms_random_and_top_residues(env):
    e = env
    x = np.concatenate([random_cts(e.rng, e.n, e.primes, 3), _top(e, 1), np.zeros_like(_top(e, 1))])
    with _Ran(e.eng) as r:
        tx = _ntt(e, x)
    assert r["ntt_forward"] > 0
    _check(e.eng.download(tx, ntt_form=True), e.orc.ct_transform(x), "forward")
    # inverse: the forward images and all-(q-1) slot values
    for xn in (e.orc.ct_transform(x), x):
        tn = e.eng.upload(xn, ntt_form=True)
        with _Ran(e.eng) as r:
            e.eng.from_ntt(tn)
        assert r["ntt_inverse"] > 0
        _check(e.eng.download(tn), e.orc.ct_transform(xn, inverse=True), "inverse")


@pytest.mark.parametrize("op", ["mul", "add", "sub"])
def test_plain_ops_both_domains(env, op):
    e = env
    x = np.concatenate([random_cts(e.rng, e.n, e.primes, 2), _top(e, 1)])
    dense = np.zeros(e.n + 1, dtype=np.uint64)
    dense[:e.n] = e.rng.integers(0, e.t, size=e.n, dtype=np.uint64)
    plains = [e.orc.encode(0.0867)[0], e.orc.encode(-2.75)[0], dense, np.array([e.t - 1], dtype=np.uint64),
              np.array([1], dtype=np.uint64)]
    for i, plain in enumerate(plains):
        p = e.eng.plain_upload(plain)
        want = e.orc.plain_op(x, plain, op)
        tc = e.eng.upload(x)
        e.eng.plain_op(tc, p, 0, op)
        _check(e.eng.download(tc), want, "coefficient form, plain %d" % i)
        tn = _ntt(e, x)
        e.eng.plain_op(tn, p, 0, op)
        _check(e.eng.download(tn, ntt_form=True), e.orc.ct_transform(want), "NTT form, plain %d" % i)


# ---------------------------------------------------------------------------------------------------- square and relinearize
def test_square_both_domains(env):
    e = env
    x = np.concatenate([random_cts(e.rng, e.n, e.primes, 2), _top(e, 1), np.zeros_like(_top(e, 1))])
    x[0, 1] = _top(e, 1)[0, 1]          # one ciphertext with a top c1 and a random c0
    want = e.orc.square(x)
    _check(e.eng.download(e.eng.square(e.eng.upload(x))), want, "coefficient-form input")
    _check(e.eng.download(e.eng.square(_ntt(e, x))), want, "NTT-form input")


def test_relinearize_both_modes_and_square_layer(env):
    e = env
    evk, sizes, dbc = random_evk(e.rng, e.n, e.primes)
    x3 = np.concatenate([random_cts(e.rng, e.n, e.primes, 2, size=3), _top(e, 1, size=3), np.zeros_like(_top(e, 1, size=3))])
    want = e.orc.relinearize(x3, evk, sizes, dbc)
    k = e.eng.evk_upload(evk, sizes, dbc)
    word_size = e.K in (1, 2, 4, 8)        # the auxiliary-prime path has exact-size instances for these K only
    try:
        for mode in (1, 0):
            e.eng.set_relin_mode(mode)
            with _Ran(e.eng) as r:
                got = e.eng.download(e.eng.relinearize(e.eng.upload(x3, size=3), k))
            _check(got, want, "relin mode %d" % mode)
            if mode == 1 and word_size:
                assert r["relinearize_u32"] == 1 and r["relinearize"] == 0, r.counts
            else:
                assert r["relinearize"] >= 1 and r["relinearize_u32"] == 0, r.counts
    finally:
        e.eng.set_relin_mode(1)
    x = np.concatenate([random_cts(e.rng, e.n, e.primes, 2), _top(e, 1)])
    want2 = e.orc.square_layer(x, evk, sizes, dbc)
    _check(e.eng.download(e.eng.square_layer(e.eng.upload(x), k)), want2, "square_layer")
    _check(e.eng.download(e.eng.square_layer(_ntt(e, x), k)), want2, "square_layer, NTT-form input")


# ---------------------------------------------------------------------------------------------------- weighted sums
def _fc(e, x, wv, bv, in_dim, out_dim, ntt_out=False):
    return e.eng.download(e.eng.fc(e.eng.upload(x), e.eng.plain_encode(wv), e.eng.plain_encode(bv), 1, in_dim, out_dim), ntt_form=ntt_out)


def test_ternary_gemm(env):
    """The ternary-tap GEMM (tc_mac.cuh) takes weights |w| < 1/2 with fan-in >= 64 in mode 2: 8 byte planes above 56 bits.  At t = 2 the
    digit values 1 and t-1 coincide and multiply_plain lifts 1 to -1, so the engine must decline it and take another kernel."""
    e = env
    _layers(e)
    e.eng.set_tensor_core_mode(2, 64)
    try:
        in_dim, out_dim = 70, 3
        x = random_cts(e.rng, e.n, e.primes, in_dim)
        wv, wp = _vals(e, in_dim * out_dim, -0.49, 0.49)
        bv, bp = _vals(e, out_dim)
        want = e.orc.fc(x, in_dim, out_dim, wp, bp)
        with _Ran(e.eng) as r:
            got = _fc(e, x, wv, bv, in_dim, out_dim)
        _check(got, want, "fc %dx%d" % (in_dim, out_dim))
        assert r["weighted_sum_tc_i8"] == (1 if e.t >= 3 else 0), r.counts
        if not e.seven:
            assert r["weighted_sum_tcn_i8"] == 0, r.counts
        # all-(q-1) inputs against all +1 / all -1 digit patterns: the largest accumulator magnitudes
        in_dim, out_dim = 96, 4
        xm = _top(e, in_dim)
        xm[::7, :, :, :e.n] = 0
        wv = np.empty((out_dim, in_dim), dtype=np.float32)
        wv[0], wv[1], wv[2] = 0.5 - 2.0 ** -24, -(0.5 - 2.0 ** -24), 0.0
        wv[3] = e.rng.uniform(-0.49, 0.49, size=in_dim)
        wv = wv.ravel()
        bv, bp = _vals(e, out_dim)
        want = e.orc.fc(xm, in_dim, out_dim, e.orc.encode_many(wv), bp)
        with _Ran(e.eng) as r:
            got = _fc(e, xm, wv, bv, in_dim, out_dim)
        _check(got, want, "all-(q-1) fc")
        assert r["weighted_sum_tc_i8"] == (1 if e.t >= 3 else 0), r.counts
        # a convolution, NTT-form input (the path converts it back itself)
        xd, yd, zd, xs, ys, xf, yf, nf = 5, 4, 8, 2, 1, 3, 3, 2     # fan-in 72
        x = random_cts(e.rng, e.n, e.primes, zd * xd * yd)
        wv, wp = _vals(e, nf * zd * xf * yf, -0.49, 0.49)
        bv, bp = _vals(e, nf)
        want = e.orc.conv(x, xd, yd, zd, xs, ys, xf, yf, nf, wp, bp)
        with _Ran(e.eng) as r:
            got = e.eng.download(e.eng.conv(_ntt(e, x), e.eng.plain_encode(wv), e.eng.plain_encode(bv), 1, xd, yd, zd, xs, ys, xf, yf, nf))
        _check(got, want, "conv")
        assert r["weighted_sum_tc_i8"] == (1 if e.t >= 3 else 0), r.counts
    finally:
        e.eng.set_tensor_core_mode(1, 256)


@pytest.mark.parametrize("variant", [2, 3])
def test_limb_split_gemm(env, variant):
    """The NTT-domain limb-split GEMM (tcn_mac.cuh) in both kernel shapes and both reductions of the class sums: the 2^k - delta fold
    where the prime has the shape (Barrett otherwise, on its own) and the 128-bit recombination.  Above 56 bits seven byte planes cannot
    hold a residue: the engine must not take it, and the CUDA-core MAC gives the bytes."""
    e = env
    _layers(e)
    in_dim, out_dim = (40, 5) if e.K <= 2 else (24, 3)
    x = random_cts(e.rng, e.n, e.primes, in_dim)
    wv, wp = _vals(e, in_dim * out_dim, -30.0, 30.0)
    bv, bp = _vals(e, out_dim)
    want = e.orc.fc(x, in_dim, out_dim, wp, bp)
    xm = _top(e, in_dim)
    e.eng.set_tensor_core_mode(0)
    e.eng.set_limb_split_mode(variant)
    outs = {}
    try:
        for mode in (1, 0):
            e.eng.set_limb_split_reduction(mode)
            with _Ran(e.eng) as r:
                got = _fc(e, x, wv, bv, in_dim, out_dim)
            _check(got, want, "reduction %d" % mode)
            assert r["weighted_sum_tcn_i8"] == (1 if e.seven else 0), r.counts
            if not e.seven:
                assert r["weighted_sum_mac"] == 1, r.counts
            outs[mode] = e.eng.download(e.eng.fc(e.eng.upload(xm, ntt_form=True), e.eng.plain_encode(wv), e.eng.plain_encode(bv), 1,
                                                 in_dim, out_dim), ntt_form=True)
        e.eng.set_limb_split_mode(0)
        ref = e.eng.download(e.eng.fc(e.eng.upload(xm, ntt_form=True), e.eng.plain_encode(wv), e.eng.plain_encode(bv), 1, in_dim, out_dim),
                             ntt_form=True)
    finally:
        e.eng.set_limb_split_reduction(1)
        e.eng.set_limb_split_mode(1)
        e.eng.set_tensor_core_mode(1)
    # all-(q-1) NTT-form slots (the largest class sums): both reductions and the CUDA-core kernel agree
    _check(outs[0], ref, "all-(q-1), reduction 0")
    _check(outs[1], ref, "all-(q-1), reduction 1")


def test_conv_default_kernels(env):
    """A convolution with any weights through whatever the engine picks by default, coefficient- and NTT-form input."""
    e = env
    _layers(e)
    xd, yd, zd, xs, ys, xf, yf, nf = 5, 4, 2, 1, 1, 3, 2, 3
    x = random_cts(e.rng, e.n, e.primes, zd * xd * yd)
    wv, wp = _vals(e, nf * zd * xf * yf, -3.0, 3.0)
    bv, bp = _vals(e, nf)
    want = e.orc.conv(x, xd, yd, zd, xs, ys, xf, yf, nf, wp, bp)
    w, b = e.eng.plain_encode(wv), e.eng.plain_encode(bv)
    for tin, what in ((e.eng.upload(x), "coefficient"), (_ntt(e, x), "NTT")):
        with _Ran(e.eng) as r:
            got = e.eng.download(e.eng.conv(tin, w, b, 1, xd, yd, zd, xs, ys, xf, yf, nf))
        _check(got, want, what)
        assert r["weighted_sum_tcn_i8" if e.seven else "weighted_sum_mac"] == 1, r.counts


def test_cuda_core_mac(env):
    """The CUDA-core NTT-domain MAC (tensor cores off).  It reduces its 128-bit sums every 2^(128 - 2 bits(q)) terms: 256 at 60 bits,
    so fan-in 300 reduces part way through."""
    e = env
    _layers(e)
    in_dim, out_dim = (300, 2) if e.bits >= 60 else ((40, 3) if e.K <= 2 else (20, 2))
    x = random_cts(e.rng, e.n, e.primes, in_dim)
    x[::3] = _top(e, 1)
    wv, wp = _vals(e, in_dim * out_dim, -5.0, 5.0)
    bv, bp = _vals(e, out_dim)
    want = e.orc.fc(x, in_dim, out_dim, wp, bp)
    e.eng.set_tensor_core_mode(0)
    e.eng.set_limb_split_mode(0)
    try:
        for tin, what in ((e.eng.upload(x), "coefficient"), (_ntt(e, x), "NTT")):
            with _Ran(e.eng) as r:
                got = e.eng.download(e.eng.fc(tin, e.eng.plain_encode(wv), e.eng.plain_encode(bv), 1, in_dim, out_dim))
            _check(got, want, what)
            assert r["weighted_sum_mac"] == 1 and r["weighted_sum_tc_i8"] == 0 and r["weighted_sum_tcn_i8"] == 0, r.counts
    finally:
        e.eng.set_limb_split_mode(1)
        e.eng.set_tensor_core_mode(1)


# ---------------------------------------------------------------------------------------------------- pooling, batch-norm, composed layers
WINDOWS = [(5, 5, 2, 1, 1, 2, 2), (7, 6, 1, 1, 1, 5, 5)]     # xd yd zd xs ys xf yf: R = 4 and R = 25 (R q >= 2^64 above 59 bits)


@pytest.mark.parametrize("avg", [False, True])
def test_pool(env, avg):
    e = env
    _layers(e)
    for (xd, yd, zd, xs, ys, xf, yf) in WINDOWS:
        x = random_cts(e.rng, e.n, e.primes, zd * xd * yd)
        x[::2] = _top(e, 1)
        if avg:
            d, cc = e.orc.encode(1.0 / (xf * yf))
            want = e.orc.pool(x, xd, yd, zd, xs, ys, xf, yf, d, cc)
            scale = e.eng.plain_encode_f64([1.0 / (xf * yf)])
        else:
            want = e.orc.pool(x, xd, yd, zd, xs, ys, xf, yf)
            scale = None
        for tin, what in ((e.eng.upload(x), "coefficient"), (_ntt(e, x), "NTT")):
            got = e.eng.download(e.eng.pool(tin, 1, xd, yd, zd, xs, ys, xf, yf, scale=scale))
            _check(got, want, "%s form, %dx%d windows" % (what, xf, yf))


def test_bn(env):
    e = env
    _layers(e)
    zd, xd, yd = 3, 2, 2
    x = random_cts(e.rng, e.n, e.primes, zd * xd * yd)
    x[::3] = _top(e, 1)
    mv, mp = _vals(e, zd)
    for vv in (e.rng.uniform(0.5, 3, size=zd).astype(np.float32), np.array([0.25, -0.375, 7.25], dtype=np.float32)):
        want = e.orc.bn(x, zd, xd, yd, mp, e.orc.encode_many(vv))
        for tin, what in ((e.eng.upload(x), "coefficient"), (_ntt(e, x), "NTT")):
            got = e.eng.download(e.eng.bn(tin, 1, zd, xd, yd, e.eng.plain_encode(mv), e.eng.plain_encode(vv)))
            _check(got, want, "%s form, invstd %s" % (what, vv))


def test_pool_bn(env):
    e = env
    _layers(e)
    for (xd, yd, zd, xs, ys, xf, yf) in WINDOWS:
        xo, yo = (xd - xf) // xs + 1, (yd - yf) // ys + 1
        x = random_cts(e.rng, e.n, e.primes, zd * xd * yd)
        x[::2] = _top(e, 1)
        mv, mp = _vals(e, zd)
        vv, vp = _vals(e, zd, -3.0, 3.0)
        d, cc = e.orc.encode(1.0 / (xf * yf))
        for scaled in (True, False):
            pooled = e.orc.pool(x, xd, yd, zd, xs, ys, xf, yf, d, cc) if scaled else e.orc.pool(x, xd, yd, zd, xs, ys, xf, yf)
            want = e.orc.bn(pooled, zd, xo, yo, mp, vp)
            scale = e.eng.plain_encode_f64([1.0 / (xf * yf)]) if scaled else None
            for tin, what in ((e.eng.upload(x), "coefficient"), (_ntt(e, x), "NTT")):
                got = e.eng.download(e.eng.pool_bn(tin, 1, xd, yd, zd, xs, ys, xf, yf, scale, e.eng.plain_encode(mv), e.eng.plain_encode(vv)))
                _check(got, want, "%s form, %dx%d windows, scaled %s" % (what, xf, yf, scaled))


def test_conv_pool_bn(env):
    e = env
    _layers(e)
    cases = [  # xd yd zd  xs ys xf yf nf  pxs pys pxf pyf
        (8, 8, 1, 1, 1, 5, 5, 2, 2, 2, 2, 2),
        (9, 9, 1, 1, 1, 3, 3, 2, 1, 1, 5, 5),    # 5x5 pooling windows: R = 25
    ]
    for (xd, yd, zd, xs, ys, xf, yf, nf, pxs, pys, pxf, pyf) in cases:
        cxo, cyo = (xd - xf) // xs + 1, (yd - yf) // ys + 1
        pxo, pyo = (cxo - pxf) // pxs + 1, (cyo - pyf) // pys + 1
        x = random_cts(e.rng, e.n, e.primes, zd * xd * yd)
        wv, wp = _vals(e, nf * zd * xf * yf)
        bv, bp = _vals(e, nf)
        mv, mp = _vals(e, nf)
        vv, vp = _vals(e, nf, -3.0, 3.0)
        d, cc = e.orc.encode(1.0 / (pxf * pyf))
        conv = e.orc.conv(x, xd, yd, zd, xs, ys, xf, yf, nf, wp, bp).reshape(nf * cxo * cyo, *x.shape[1:])
        want = e.orc.bn(e.orc.pool(conv, cxo, cyo, nf, pxs, pys, pxf, pyf, d, cc), nf, pxo, pyo, mp, vp)
        packs = (e.eng.plain_encode_f64([1.0 / (pxf * pyf)]), e.eng.plain_encode(mv), e.eng.plain_encode(vv))
        geo = (1, xd, yd, zd, xs, ys, xf, yf, nf, pxs, pys, pxf, pyf)
        w, b = e.eng.plain_encode(wv), e.eng.plain_encode(bv)
        for tin, what in ((e.eng.upload(x), "coefficient"), (_ntt(e, x), "NTT")):
            got = e.eng.download(e.eng.conv_pool_bn(tin, w, b, *geo, *packs))
            _check(got, want, "%s form, %s" % (what, geo))


def test_fc_fc(env):
    e = env
    _layers(e)
    in_dim, mid, out = (21, 12, 3) if e.K <= 2 else (9, 6, 2)
    w1v, w1p = _vals(e, mid * in_dim)
    b1v, b1p = _vals(e, mid)
    w2v, w2p = _vals(e, out * mid)
    b2v, b2p = _vals(e, out)
    x = random_cts(e.rng, e.n, e.primes, in_dim)
    x[::4] = _top(e, 1)
    ct = x.shape[1:]
    want = e.orc.fc(e.orc.fc(x, in_dim, mid, w1p, b1p).reshape(mid, *ct), mid, out, w2p, b2p)
    packs = [e.eng.plain_encode(v) for v in (w1v, b1v, w2v, b2v)]
    for tin, what in ((e.eng.upload(x), "coefficient"), (_ntt(e, x), "NTT"), (e.eng.upload(x), "again")):
        _check(e.eng.download(e.eng.fc_fc(tin, *packs, 1, in_dim, mid, out)), want, what)


def test_pool_bn_fc_fc(env):
    e = env
    _layers(e)
    for (xd, yd, zd, pxs, pys, pxf, pyf, mid, out) in [(4, 4, 3, 1, 1, 2, 2, 8, 3), (6, 5, 1, 1, 1, 5, 5, 4, 2)]:
        pxo, pyo = (xd - pxf) // pxs + 1, (yd - pyf) // pys + 1
        in_dim = zd * pxo * pyo
        mv, mp = _vals(e, zd)
        vv, vp = _vals(e, zd, -3.0, 3.0)
        d, cc = e.orc.encode(1.0 / (pxf * pyf))
        w1v, w1p = _vals(e, mid * in_dim)
        b1v, b1p = _vals(e, mid)
        w2v, w2p = _vals(e, out * mid)
        b2v, b2p = _vals(e, out)
        x = random_cts(e.rng, e.n, e.primes, zd * xd * yd)
        x[::3] = _top(e, 1)
        ct = x.shape[1:]
        geo = (1, xd, yd, zd, pxs, pys, pxf, pyf)
        rest = [e.eng.plain_encode(mv), e.eng.plain_encode(vv)] + [e.eng.plain_encode(v) for v in (w1v, b1v, w2v, b2v)]
        for scaled in (True, False):
            pooled = e.orc.pool(x, xd, yd, zd, pxs, pys, pxf, pyf, d, cc) if scaled else e.orc.pool(x, xd, yd, zd, pxs, pys, pxf, pyf)
            y = e.orc.bn(pooled, zd, pxo, pyo, mp, vp).reshape(in_dim, *ct)
            want = e.orc.fc(e.orc.fc(y, in_dim, mid, w1p, b1p).reshape(mid, *ct), mid, out, w2p, b2p)
            scale = e.eng.plain_encode_f64([1.0 / (pxf * pyf)]) if scaled else None
            for tin, what in ((e.eng.upload(x), "coefficient"), (_ntt(e, x), "NTT")):
                got = e.eng.download(e.eng.pool_bn_fc_fc(tin, *geo, scale, *rest, mid, out))
                _check(got, want, "%s form, %dx%d windows, scaled %s" % (what, pxf, pyf, scaled))


# ---------------------------------------------------------------------------------------------------- client side
VALUES = np.array([0.0, 1.0, -1.0, 0.25, -0.3, 1.0 / 3.0, 2.8215, -0.4242, 1.5, -7.0, 12345.678, 1e-6], dtype=np.float32)


def _noise(rng, count, n):
    return np.stack([kg.ternary(rng, (count, n)), kg.clipped_normal(rng, (count, n)), kg.clipped_normal(rng, (count, n))], axis=1)


def _oracle_encrypt(orc, keys, v, noise):
    plain, cc = orc.encode(float(v))
    return orc.encrypt(plain, keys.pk, noise[0], noise[1], noise[2], coeff_count=cc)


def test_client_side(env):
    """encrypt_values with supplied noise, decrypt_values, noise_budget and reencrypt against the oracle's Encryptor / Decryptor /
    FractionalEncoder and the CPU restatement of invariant_noise_budget, on fresh ciphertexts and a convolution's output."""
    e = env
    _layers(e)
    n, orc = e.n, e.orc
    keys = kg.generate(orc, 5)
    dk = e.eng.keys_upload(keys.sk, keys.pk)
    P = len(VALUES)
    noise = _noise(e.rng, P, n)
    want = np.stack([_oracle_encrypt(orc, keys, VALUES[i], noise[i]) for i in range(P)])
    fresh = e.eng.encrypt_values(dk, VALUES, seed=1, noise=noise)
    _check(e.eng.download(fresh), want, "encrypt_values")
    x = kg.encrypt_values(keys, e.rng.uniform(-1, 1, 16).astype(np.float32), e.rng)       # 1 x 4 x 4
    conv = e.eng.conv(e.eng.upload(x), e.eng.plain_encode(e.rng.uniform(-1, 1, 4).astype(np.float32)),
                      e.eng.plain_encode(e.rng.uniform(-1, 1, 1).astype(np.float32)), 1, 4, 4, 1, 1, 1, 2, 2, 1)    # 1 x 3 x 3
    for t_ct, what in ((fresh, "fresh"), (conv, "conv")):
        cts = e.eng.download(t_ct)
        vals = np.array([np.float32(orc.decode(p)) for p in orc.decrypt(cts, keys.sk)], dtype=np.float32)
        assert np.array_equal(e.eng.decrypt_values(dk, t_ct), vals), what
        budget = kg.noise_budget(orc, cts, keys.sk)
        assert np.array_equal(e.eng.noise_budget(dk, t_ct), budget), what
        if what == "fresh" and budget.min() > 0:     # decryption is correct: the values round-trip through the encoder
            trip = np.array([np.float32(orc.decode(orc.encode(float(v))[0])) for v in VALUES], dtype=np.float32)
            assert np.array_equal(vals, trip)
        rn = _noise(e.rng, len(cts), n)
        got = e.eng.download(e.eng.reencrypt(dk, e.eng.upload(cts), seed=3, noise=rn))
        want_re = np.stack([_oracle_encrypt(orc, keys, v, rn[c]) for c, v in enumerate(vals)])
        _check(got, want_re, "reencrypt " + what)
