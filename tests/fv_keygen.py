"""TEST INFRASTRUCTURE ONLY.  Seeded key generation without SEAL, in SEAL 2.3.1's layouts, so that crcnn_keys_upload,
crcnn_evk_upload and the oracle's orc_encrypt / orc_relinearize take the keys unchanged:

  secret key      s ternary, kept in NTT form                           uint64[K][n+1]      (SecretKey::data())
  public key      (-(a s + e), a), NTT form                             uint64[2][K][n+1]   (PublicKey::data())
  evaluation keys for prime i and digit k (decomposition bit count dbc):
                  poly(2k)   = -(a s + e) + 2^(dbc k) (q/q_i) s^2       zero s^2 term in every limb j != i: q/q_i = 0 mod q_j
                  poly(2k+1) = a                                       NTT form, keys of prime i back to back, sizes[i] polys

relinearize adds sum_k digit_k(c2 (q/q_i)^-1 mod q_i) (poly(2k), poly(2k+1)) to (c0, c1), and sum_i [c2 (q/q_i)^-1]_{q_i} (q/q_i) = c2
(mod q), so c2 s^2 moves onto (c0, c1) with small noise.  The keys are inputs: every result is a function of them, and byte equality
with SEAL's KeyGenerator (another random stream) is neither possible nor needed.

Also here: encryption of values with these keys (orc_encrypt with sampled u, e0, e1), ciphertexts with a chosen noise polynomial
(`craft`) whose invariant noise budget follows in closed form (`budget_of`), and the CPU restatement of
Decryptor::invariant_noise_budget (`noise_budget`: the dot product through the oracle's transforms, the CRT compose and norm in C,
tests/fv_budget.c, compiled on first use into a temporary directory).
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

SIGMA = 3.19            # SEAL/seal/util/globals.cpp: default_noise_standard_deviation
MAX_DEV = 6.0 * SIGMA   # noise_distribution_width_multiplier = 6 (encryptionparams.h)

_u64p = C.POINTER(C.c_uint64)


def clipped_normal(rng, shape):
    """SEAL's noise: normal of standard deviation SIGMA, redrawn beyond MAX_DEV, truncated toward zero (int8)."""
    z = rng.normal(0.0, SIGMA, size=shape)
    bad = np.abs(z) > MAX_DEV
    while bad.any():
        z[bad] = rng.normal(0.0, SIGMA, size=int(bad.sum()))
        bad = np.abs(z) > MAX_DEV
    return np.trunc(z).astype(np.int8)


def ternary(rng, shape):
    return rng.integers(-1, 2, size=shape).astype(np.int8)


class Keys:
    def __init__(self, orc, sk, pk, evk, sizes, dbc, s):
        self.orc, self.sk, self.pk, self.evk, self.sizes, self.dbc, self.s = orc, sk, pk, evk, sizes, dbc, s

    @property
    def evk_triple(self):
        return self.evk, self.sizes, self.dbc


class _Ring:
    """Limb-wise arithmetic on [..., K, n+1] residue arrays through the oracle's dyadic product."""

    def __init__(self, orc):
        self.orc, self.n, self.K = orc, orc.n, orc.K
        self.q = [int(p) for p in orc.primes]

    def residues(self, small):
        """signed small integers [..., n] -> residues [..., K, n+1] (coefficient form)"""
        small = np.asarray(small, dtype=np.int64)
        out = np.zeros(small.shape[:-1] + (self.K, self.n + 1), dtype=np.uint64)
        for j, q in enumerate(self.q):
            out[..., j, :self.n] = np.where(small < 0, small + q, small).astype(np.uint64)
        return out

    def ntt(self, polys, inverse=False):
        a = np.ascontiguousarray(polys, dtype=np.uint64)
        return self.orc.ct_transform(a.reshape(-1, self.K, self.n + 1), size=1, inverse=inverse).reshape(a.shape)

    def uniform(self, rng, shape=()):
        out = np.zeros(tuple(shape) + (self.K, self.n + 1), dtype=np.uint64)
        for j, q in enumerate(self.q):
            out[..., j, :self.n] = rng.integers(0, q, size=tuple(shape) + (self.n,), dtype=np.uint64)
        return out

    def mul(self, a, b):
        a, b = np.ascontiguousarray(a, dtype=np.uint64), np.ascontiguousarray(b, dtype=np.uint64)
        out = np.zeros_like(a)
        for j, q in enumerate(self.q):
            x, y, o = (np.ascontiguousarray(v[j]) for v in (a, b, out))
            self.orc.lib.orc_dyadic_product(x.ctypes.data_as(_u64p), y.ctypes.data_as(_u64p), self.n + 1, q, o.ctypes.data_as(_u64p))
            out[j] = o
        return out

    def limb_times(self, a, j, s):
        """zero in every limb but j, which is limb j of a times the scalar s < q_j"""
        out = np.zeros_like(a)
        x, o = np.ascontiguousarray(a[j]), np.zeros(self.n + 1, dtype=np.uint64)
        self.orc.lib.orc_multiply_poly_scalar(x.ctypes.data_as(_u64p), self.n + 1, s, self.q[j], o.ctypes.data_as(_u64p))
        out[j] = o
        return out

    def add(self, a, b):
        out = np.empty_like(a)
        for j, q in enumerate(self.q):
            out[..., j, :] = (a[..., j, :] + b[..., j, :]) % np.uint64(q)
        return out

    def neg(self, a):
        out = np.empty_like(a)
        for j, q in enumerate(self.q):
            out[..., j, :] = (np.uint64(q) - a[..., j, :]) % np.uint64(q)
        out[..., :, self.n] = 0
        return out


def generate(orc, seed, dbc=16):
    """Secret, public and evaluation keys for the oracle's parameters from one seed."""
    rng = np.random.default_rng(seed)
    R = _Ring(orc)
    n, q = R.n, R.q
    s = ternary(rng, n)
    sk = R.ntt(R.residues(s))

    def rlwe():      # -(a s + e), a    (NTT form)
        a = R.uniform(rng)
        e = R.ntt(R.residues(clipped_normal(rng, n)))
        return R.neg(R.add(R.mul(a, sk), e)), a

    pk = np.stack(rlwe())
    s2 = R.mul(sk, sk)
    Q = 1
    for p in q:
        Q *= p
    parts, sizes = [], []
    for i, qi in enumerate(q):
        digits = (qi.bit_length() + dbc - 1) // dbc
        qhat = (Q // qi) % qi
        for k in range(digits):
            k0, a = rlwe()
            k0 = R.add(k0, R.limb_times(s2, i, (qhat << (dbc * k)) % qi))
            parts += [k0, a]
        sizes.append(2 * digits)
    evk = np.concatenate([p.ravel() for p in parts])
    return Keys(orc, sk, pk, evk, sizes, dbc, s)


def encrypt_plains(keys, plains, rng):
    """orc_encrypt of each (plain words, coeff_count) with u, e0, e1 sampled from rng -> [count][2][K][n+1]"""
    orc = keys.orc
    out = np.zeros((len(plains), 2, orc.K, orc.stride), dtype=np.uint64)
    for c, (p, cc) in enumerate(plains):
        u = ternary(rng, orc.n)
        e = clipped_normal(rng, (2, orc.n))
        out[c] = orc.encrypt(p, keys.pk, u, e[0], e[1], coeff_count=cc)
    return out


def encrypt_values(keys, values, rng):
    """FractionalEncoder::encode + Encryptor::encrypt of every value -> [count][2][K][n+1]"""
    orc = keys.orc
    return encrypt_plains(keys, [orc.encode(float(v)) for v in np.asarray(values, dtype=np.float32).ravel()], rng)


def modulus(orc):
    Q = 1
    for p in orc.primes:
        Q *= int(p)
    return Q


def craft(keys, X, rng, ntt_form=False):
    """Ciphertexts whose t (c0 + c1 s) mod q is the integer polynomial X ([count][n] Python ints, taken mod q): c1 uniform,
    c0 = w - c1 s with w = X t^-1 mod q.  Coefficient form, or NTT form with ntt_form.  -> [count][2][K][n+1]"""
    orc = keys.orc
    R = _Ring(orc)
    Q = modulus(orc)
    tinv = pow(orc.t, -1, Q)
    out = np.zeros((len(X), 2, orc.K, orc.stride), dtype=np.uint64)
    for c, row in enumerate(X):
        w = [(int(x) * tinv) % Q for x in row]
        wr = np.zeros((orc.K, orc.stride), dtype=np.uint64)
        for j, q in enumerate(R.q):
            wr[j, :orc.n] = np.array([v % q for v in w], dtype=np.uint64)
        c1 = R.uniform(rng)
        c0 = R.add(R.ntt(wr), R.neg(R.mul(c1, keys.sk)))
        out[c] = np.stack([c0, c1])
    return out if ntt_form else R.ntt(out, inverse=True)


def budget_of(orc, X):
    """Closed-form invariant noise budget of ciphertexts made by craft(keys, X): per row of X."""
    Q = modulus(orc)
    qbits = Q.bit_length()
    res = []
    for row in X:
        norm = 0
        for x in row:
            v = int(x) % Q
            norm = max(norm, Q - v if v >= (Q + 1) // 2 else v)
        res.append(max(0, qbits - norm.bit_length() - 1))
    return np.array(res, dtype=np.int32)


def budget_bigint(orc, cts, keys):
    """Independent restatement with Python integers: c0 + c1 s per limb from the oracle's transforms, CRT with int, centred
    infinity norm of t (c0 + c1 s) mod q.  -> int32[count]"""
    R = _Ring(orc)
    Q = modulus(orc)
    qbits = Q.bit_length()
    cts = np.ascontiguousarray(cts, dtype=np.uint64).reshape(-1, 2, orc.K, orc.stride)
    coeff = R.ntt(cts, inverse=False)              # NTT form of c0, c1 (cts are coefficient form)
    res = []
    for c in range(len(cts)):
        d = R.ntt(R.add(coeff[c, 0], R.mul(coeff[c, 1], keys.sk)), inverse=True)
        qhat = [Q // q for q in R.q]
        inv = [pow(qh % q, -1, q) for qh, q in zip(qhat, R.q)]
        norm = 0
        for k in range(orc.n):
            x = sum(int(d[j, k]) * inv[j] % q * qhat[j] for j, q in enumerate(R.q)) % Q
            x = x * orc.t % Q
            norm = max(norm, Q - x if x >= (Q + 1) // 2 else x)
        res.append(max(0, qbits - norm.bit_length() - 1))
    return np.array(res, dtype=np.int32)


_fvb = None


def _budget_lib():
    global _fvb
    if _fvb is None:
        src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fv_budget.c")
        so = os.path.join(tempfile.mkdtemp(prefix="crcnn_fv_budget_"), "libfv_budget.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-std=gnu11", "-o", so, src])
        lib = C.CDLL(so)
        lib.fvb_noise_budget.argtypes = [C.c_int, C.c_int, _u64p, C.c_uint64, _u64p, C.c_int, C.POINTER(C.c_int)]
        _fvb = lib
    return _fvb


def noise_budget(orc, cts, sk_ntt):
    """Decryptor::invariant_noise_budget of every size-2 ciphertext (coefficient form) -> int32[count]: d = c0 + c1 s per limb as
    Decryptor::decrypt forms it (NTT of c1, dyadic product with the NTT-form secret key, inverse NTT, + c0), then fv_budget.c."""
    R = _Ring(orc)
    cts = np.ascontiguousarray(cts, dtype=np.uint64).reshape(-1, 2, orc.K, orc.stride)
    c1 = R.ntt(cts[:, 1])
    sk = np.ascontiguousarray(sk_ntt, dtype=np.uint64)
    d = np.zeros_like(c1)
    for c in range(len(cts)):
        d[c] = R.mul(c1[c], sk)
    d = R.add(R.ntt(d, inverse=True), cts[:, 0])
    primes = np.array(R.q, dtype=np.uint64)
    out = np.zeros(len(cts), dtype=np.int32)
    rc = _budget_lib().fvb_noise_budget(orc.n, orc.K, primes.ctypes.data_as(_u64p), orc.t, d.ctypes.data_as(_u64p), len(cts),
                                        out.ctypes.data_as(C.POINTER(C.c_int)))
    assert rc == 0
    return out

