"""The CPU oracle against exact big-integer mathematics at the parameter sets beyond SEAL's defaults (tests/util.py: PARAM_SETS).

The oracle is the checker of every GPU parity test, and it has been compared with the compiled original only at SEAL's default
sets.  Here it is pinned, at every other set the GPU tests use, to what the operations mean, with Python integers:
  - its forward transform evaluates the negacyclic polynomial at psi^(2 bitrev(i) + 1), psi the minimal primitive 2n-th root;
  - with keys from tests/fv_keygen.py, its plain_op, conv, fc, pool and bn outputs decrypt to the same operations on the
    plaintext polynomials in Z_t[x]/(x^n + 1);
  - square_layer decrypts to m^2 where the noise budget after a square is positive, and relinearize keeps what a size-3
    ciphertext decrypts to.
No GPU."""
import zlib

import numpy as np
import pytest

import fv_keygen as kg
from util import PARAM_SETS
from oracle.port import Oracle

# one encryption and a square leave no noise budget at these sets (57-60-bit single primes with large t, the 30-bit prime)
NO_BUDGET_AFTER_SQUARE = {"P57", "P57n16384", "P60a", "U30"}
LAYER_SETS = [s for s in PARAM_SETS if PARAM_SETS[s][0] <= 8192]


def _ctx(name):
    n, primes, t = PARAM_SETS[name]
    orc = Oracle(n, primes, t)
    return orc, kg.generate(orc, 7), np.random.default_rng(zlib.crc32(name.encode()) + 1)


# ---------------------------------------------------------------------------------------------------- exact plaintext and ciphertext maths
def _Q(orc):
    Q = 1
    for q in orc.primes:
        Q *= int(q)
    return Q


def _crt(orc, limbs):
    """[K][n] residues -> list of n Python ints in [0, Q)"""
    Q = _Q(orc)
    parts = []
    for j, q in enumerate(orc.primes):
        q = int(q)
        qh = Q // q
        parts.append((qh, pow(qh % q, -1, q), q))
    return [sum(int(limbs[j][k]) * inv % q * qh for j, (qh, inv, q) in enumerate(parts)) % Q for k in range(orc.n)]


def decrypt_exact(orc, keys, ct):
    """round(t [c0 + c1 s + c2 s^2 + ...]_q / q) mod t with Python integers, any ciphertext size (coefficient form) -> list of n ints"""
    R = kg._Ring(orc)
    ct = np.ascontiguousarray(ct, dtype=np.uint64)
    parts = R.ntt(ct)
    acc, s_pow = parts[0], keys.sk
    for i in range(1, ct.shape[0]):
        acc = R.add(acc, R.mul(parts[i], s_pow))
        s_pow = R.mul(s_pow, keys.sk)
    d = _crt(orc, R.ntt(acc, inverse=True)[:, :orc.n])
    Q, t = _Q(orc), orc.t
    return [((t * v + Q // 2) // Q) % t for v in d]


def plain_poly(orc, words, cc=None):
    """plaintext words [n+1] -> list of n ints mod t"""
    p = [0] * orc.n
    for k, v in enumerate(words[:orc.n if cc is None else min(cc, orc.n)]):
        p[k] = int(v) % orc.t
    return p


def padd(t, a, b):
    return [(x + y) % t for x, y in zip(a, b)]


def psub(t, a, b):
    return [(x - y) % t for x, y in zip(a, b)]


def pmul(t, a, b):
    """negacyclic product in Z_t[x]/(x^n + 1)"""
    n = len(a)
    out = [0] * n
    nb = [(j, bj) for j, bj in enumerate(b) if bj]
    for i, ai in enumerate(a):
        if ai == 0:
            continue
        for j, bj in nb:
            k = i + j
            if k < n:
                out[k] += ai * bj
            else:
                out[k - n] -= ai * bj
    return [v % t for v in out]


def _plains(orc, cts, keys):
    return [decrypt_exact(orc, keys, c) for c in cts]


def _decrypted(orc, keys, cts):
    return [plain_poly(orc, p) for p in orc.decrypt(np.ascontiguousarray(cts).reshape(-1, 2, orc.K, orc.stride), keys.sk)]


def _assert_budget(orc, keys, cts, what):
    b = kg.noise_budget(orc, np.ascontiguousarray(cts).reshape(-1, 2, orc.K, orc.stride), keys.sk)
    assert b.min() > 0, "%s: no noise budget left (%s): the decryption check would be meaningless" % (what, b)


# ---------------------------------------------------------------------------------------------------- the forward transform
def _minimal_root(q, n):
    """SEAL's minimal primitive 2n-th root of unity mod q (smallest of all of them)"""
    m = 2 * n
    for g in range(2, 1 << 20):
        r = pow(g, (q - 1) // m, q)
        if pow(r, n, q) == q - 1:
            break
    best, r2, cur = r, r * r % q, r
    for _ in range(n - 1):
        cur = cur * r2 % q
        best = min(best, cur)
    return best


@pytest.mark.parametrize("name", list(PARAM_SETS))
def test_forward_transform_is_negacyclic_evaluation(name):
    n, primes, t = PARAM_SETS[name]
    orc = Oracle(n, primes, t)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    K = len(primes)
    x = np.zeros((1, K, n + 1), dtype=np.uint64)
    for j, q in enumerate(primes):
        x[0, j, :n] = rng.integers(0, q, size=n, dtype=np.uint64)
    x[0, :, 0] = [q - 1 for q in primes]
    xn = orc.ct_transform(x, size=1)
    logn = n.bit_length() - 1
    slots = sorted(set([0, 1, 2, n // 2, n - 2, n - 1] + [int(v) for v in rng.integers(0, n, size=40)]))
    for j, q in enumerate(primes):
        q = int(q)
        psi = _minimal_root(q, n)
        assert orc.minimal_root(0, j) == psi
        coeffs = [int(v) for v in x[0, j, :n]]
        for i in slots:
            point = pow(psi, 2 * int(format(i, "0%db" % logn)[::-1], 2) + 1, q)
            acc = 0
            for c in reversed(coeffs):
                acc = (acc * point + c) % q
            assert int(xn[0, j, i]) == acc, (name, j, i)


# ---------------------------------------------------------------------------------------------------- evaluator and layers
def _fresh(keys, rng, count, lo=-2.0, hi=2.0):
    return kg.encrypt_values(keys, rng.uniform(lo, hi, count).astype(np.float32), rng)


@pytest.mark.parametrize("name", LAYER_SETS)
def test_plain_ops_decrypt_to_plaintext_arithmetic(name):
    orc, keys, rng = _ctx(name)
    n, t = orc.n, orc.t
    x = _fresh(keys, rng, 2)
    m = _plains(orc, x, keys)
    dense = np.zeros(n + 1, dtype=np.uint64)
    # every coefficient set, but small once centred: the sum's rounding term (q mod t) m stays inside the budget at t = 2^30, q < 2^60
    dense[:n] = (rng.integers(-7, 8, size=n) % t).astype(np.uint64)
    tern = np.zeros(n + 1, dtype=np.uint64)
    tern[:n] = np.array([0, 1, t - 1], dtype=np.uint64)[rng.integers(0, 3, size=n)]   # dense but small once lifted, for the product
    enc = orc.encode(-0.6875)[0]
    for plain, ops in ((enc, ("mul", "add", "sub")), (dense, ("add", "sub")), (tern, ("mul",)),
                       (np.array([t - 1], dtype=np.uint64), ("mul", "add", "sub"))):
        p = plain_poly(orc, plain)
        for op in ops:
            out = orc.plain_op(x, plain, op)
            _assert_budget(orc, keys, out, op)
            want = [pmul(t, mi, p) if op == "mul" else (padd if op == "add" else psub)(t, mi, p) for mi in m]
            assert _decrypted(orc, keys, out) == want, (name, op, len(plain))


@pytest.mark.parametrize("name", LAYER_SETS)
def test_layers_decrypt_to_plaintext_arithmetic(name):
    orc, keys, rng = _ctx(name)
    t = orc.t
    enc = lambda v: orc.encode_many(np.asarray(v, dtype=np.float32))
    P = lambda words: plain_poly(orc, words)
    # conv: 2 channels of 3x3, 2x2 filters, 2 filters, stride 1
    xd, yd, zd, xs, ys, xf, yf, nf = 3, 3, 2, 1, 1, 2, 2, 2
    x = _fresh(keys, rng, zd * xd * yd)
    m = _plains(orc, x, keys)
    wv, bv = rng.uniform(-1, 1, nf * zd * xf * yf), rng.uniform(-1, 1, nf)
    wp, bp = enc(wv), enc(bv)
    out = orc.conv(x, xd, yd, zd, xs, ys, xf, yf, nf, wp, bp)
    _assert_budget(orc, keys, out, "conv")
    xo, yo, R = xd - xf + 1, yd - yf + 1, zd * xf * yf
    want = []
    for f in range(nf):
        for i in range(xo):
            for j in range(yo):
                acc, r = P(bp[f]), 0
                for z in range(zd):
                    for kx in range(xf):
                        for ky in range(yf):
                            acc = padd(t, acc, pmul(t, P(wp[f * R + r]), m[(z * xd + i + kx) * yd + j + ky]))
                            r += 1
                want.append(acc)
    assert _decrypted(orc, keys, out) == want, "conv"
    # fc: 5 -> 3
    in_dim, out_dim = 5, 3
    xf_ = _fresh(keys, rng, in_dim)
    mf = _plains(orc, xf_, keys)
    wp, bp = enc(rng.uniform(-1, 1, in_dim * out_dim)), enc(rng.uniform(-1, 1, out_dim))
    out = orc.fc(xf_, in_dim, out_dim, wp, bp)
    _assert_budget(orc, keys, out, "fc")
    want = []
    for o in range(out_dim):
        acc = P(bp[o])
        for i in range(in_dim):
            acc = padd(t, acc, pmul(t, P(wp[o * in_dim + i]), mf[i]))
        want.append(acc)
    assert _decrypted(orc, keys, out) == want, "fc"
    # pool: 2x2 windows of a 3x3 channel pair, as sums and scaled by an encoded 1/4; 5x5 windows
    for (pxd, pyd, pzd, pxs, pys, pxf, pyf) in ((3, 3, 2, 1, 1, 2, 2), (5, 6, 1, 1, 1, 5, 5)):
        xp = _fresh(keys, rng, pzd * pxd * pyd)
        mp = _plains(orc, xp, keys)
        pxo, pyo = (pxd - pxf) // pxs + 1, (pyd - pyf) // pys + 1
        d, cc = orc.encode(1.0 / (pxf * pyf))
        sums = []
        for z in range(pzd):
            for i in range(pxo):
                for j in range(pyo):
                    acc = [0] * orc.n
                    for kx in range(pxf):
                        for ky in range(pyf):
                            acc = padd(t, acc, mp[(z * pxd + i * pxs + kx) * pyd + j * pys + ky])
                    sums.append(acc)
        for scaled in (False, True):
            out = orc.pool(xp, pxd, pyd, pzd, pxs, pys, pxf, pyf, d, cc) if scaled else orc.pool(xp, pxd, pyd, pzd, pxs, pys, pxf, pyf)
            _assert_budget(orc, keys, out, "pool")
            want = [pmul(t, plain_poly(orc, d, cc), s) for s in sums] if scaled else sums
            assert _decrypted(orc, keys, out) == want, ("pool", pxf, scaled)
    # bn: (x - mean) * invstd per channel
    zd, xd, yd = 2, 2, 1
    xb = _fresh(keys, rng, zd * xd * yd)
    mb = _plains(orc, xb, keys)
    mean, invstd = enc(rng.uniform(-1, 1, zd)), enc([1.75, -0.3125])
    out = orc.bn(xb, zd, xd, yd, mean, invstd)
    _assert_budget(orc, keys, out, "bn")
    want = [pmul(t, P(invstd[c // (xd * yd)]), psub(t, mi, P(mean[c // (xd * yd)]))) for c, mi in enumerate(mb)]
    assert _decrypted(orc, keys, out) == want, "bn"


@pytest.mark.parametrize("name", list(PARAM_SETS))
def test_square_layer_decrypts_to_the_square(name):
    if name in NO_BUDGET_AFTER_SQUARE:
        pytest.skip("one encryption and a square leave no noise budget at these parameters")
    orc, keys, rng = _ctx(name)
    x = _fresh(keys, rng, 2, -1.5, 1.5)
    m = _plains(orc, x, keys)
    out = orc.square_layer(x, *keys.evk_triple)
    _assert_budget(orc, keys, out, "square_layer")
    assert _decrypted(orc, keys, out) == [pmul(orc.t, mi, mi) for mi in m]


@pytest.mark.parametrize("name", list(PARAM_SETS))
def test_relinearize_keeps_the_decryption(name):
    """A size-3 ciphertext (c0 - c2 s^2, c1, c2) with c2 uniform decrypts like the fresh (c0, c1); relinearize must keep that.  Where
    a square leaves budget, the square of a fresh ciphertext is checked as well."""
    orc, keys, rng = _ctx(name)
    R = kg._Ring(orc)
    x = _fresh(keys, rng, 2, -1.5, 1.5)
    m = _plains(orc, x, keys)
    x3 = np.zeros((2, 3, orc.K, orc.stride), dtype=np.uint64)
    s2 = R.mul(keys.sk, keys.sk)
    for c in range(2):
        c2 = R.uniform(rng)
        x3[c, 0] = R.add(x[c, 0], R.ntt(R.neg(R.mul(R.ntt(c2), s2)), inverse=True))
        x3[c, 1], x3[c, 2] = x[c, 1], c2
    assert [decrypt_exact(orc, keys, c) for c in x3] == m
    cases = [(x3, m)]
    if name not in NO_BUDGET_AFTER_SQUARE:
        sq = orc.square(x)
        cases.append((sq, [decrypt_exact(orc, keys, c) for c in sq]))
    for cts, want in cases:
        out = orc.relinearize(cts, *keys.evk_triple)
        _assert_budget(orc, keys, out, "relinearize")
        assert _decrypted(orc, keys, out) == want
