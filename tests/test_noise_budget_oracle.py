"""The CPU restatement of Decryptor::invariant_noise_budget (fv_keygen.noise_budget, fv_budget.c) and the seeded key generator of
tests/fv_keygen.py.

Crafted ciphertexts have a chosen t (c0 + c1 s) mod q, so their budget follows in closed form (keygen.budget_of); real encryptions
and layer outputs are checked against an independent Python big-integer restatement (keygen.budget_bigint), and, where the compiled
original exists, against SEAL's own invariant_noise_budget."""
import numpy as np
import pytest

from util import have_ref
import fv_keygen as kg
from oracle.port import DEFAULT_PRIMES_128 as PRIMES, Oracle

T_OF = {2048: 1 << 16, 4096: 1 << 20, 8192: 1 << 30, 16384: 1 << 30}


def setup(n, t=None, seed=5):
    orc = Oracle(n, PRIMES[n], T_OF[n] if t is None else t)
    return orc, kg.generate(orc, seed)


def sweep_rows(orc, rng, extra=()):
    """Noise polynomials X whose budgets cover 0 .. bits(q) - 2 (the fresh maximum and beyond), both signs of the dominant
    coefficient, noise past q/(2t) and the centring boundaries (q - 1)/2, (q + 1)/2."""
    n, Q = orc.n, kg.modulus(orc)
    rows = []
    for b in range(0, Q.bit_length() - 1):
        row = [0] * n
        mag = (1 << b) | int(rng.integers(0, 1 << min(b, 62))) if b else 1
        k = int(rng.integers(0, n))
        row[k] = mag if b % 2 else Q - mag                              # both signs
        if b >= 4:
            row[(k + 1 + int(rng.integers(0, n - 1))) % n] = int(rng.integers(-7, 8))   # a smaller coefficient that must not matter
        rows.append(row)
    for x in ((Q - 1) // 2, (Q + 1) // 2, (Q - 1) // 2 - 1, (Q + 1) // 2 + 1, Q // (2 * orc.t) * 3, Q - 1, 0):
        row = [0] * n
        row[n - 1] = x
        rows.append(row)
    return rows + list(extra)


@pytest.mark.parametrize("n", [2048, 4096, 8192, 16384])
def test_oracle_equals_closed_form_on_crafted(n):
    orc, keys = setup(n)
    rng = np.random.default_rng(n)
    X = sweep_rows(orc, rng)
    want = kg.budget_of(orc, X)
    assert set(range(0, kg.modulus(orc).bit_length() - 1)) <= set(want.tolist())
    got = kg.noise_budget(orc, kg.craft(keys, X, rng), keys.sk)
    assert np.array_equal(got, want)
    # the boundaries are exactly where the centred norm is largest: budget 0
    assert (want[-7:-3] == 0).all() and want[-1] == kg.modulus(orc).bit_length() - 1


def test_keygen_encrypt_decrypt_roundtrip():
    orc, keys = setup(4096)
    rng = np.random.default_rng(1)
    vals = np.array([0.5, -1.25, 3.0, 0.0, 17.75], dtype=np.float32)
    ct = kg.encrypt_values(keys, vals, rng)
    got = [orc.decode(p) for p in orc.decrypt(ct, keys.sk)]
    assert np.allclose(got, vals, atol=1e-6)


@pytest.mark.parametrize("n", [4096, 8192])
def test_keygen_square_relinearize(n):
    orc, keys = setup(n)
    rng = np.random.default_rng(2)
    vals = np.array([0.5, -1.25, 3.0], dtype=np.float32)
    ct = kg.encrypt_values(keys, vals, rng)
    rl = orc.relinearize(orc.square(ct), *keys.evk_triple)
    got = [orc.decode(p) for p in orc.decrypt(rl, keys.sk)]
    assert np.allclose(got, vals.astype(np.float64) ** 2, rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize("n,t,fresh", [(4096, 1 << 20, 78), (8192, 1 << 30, 176)])
def test_fresh_budget_near_seal_probe(n, t, fresh):
    """Plausibility only: SEAL's probe figures for a fresh encryption (SURVEY 8(d))."""
    orc, keys = setup(n, t)
    ct = kg.encrypt_values(keys, [1.5, -0.25], np.random.default_rng(3))
    assert np.all(np.abs(kg.noise_budget(orc, ct, keys.sk) - fresh) <= 2)


def test_oracle_equals_bigint_on_encryptions_and_layers():
    orc, keys = setup(4096)
    rng = np.random.default_rng(4)
    x = kg.encrypt_values(keys, rng.uniform(-1, 1, 16).astype(np.float32), rng)
    cases = [x]
    w, b = orc.encode_many(rng.uniform(-1, 1, 8)), orc.encode_many(rng.uniform(-1, 1, 2))
    conv = orc.conv(x, 4, 4, 1, 1, 1, 2, 2, 2, w, b)                       # 2 x 3 x 3
    cases.append(conv)
    d, cc = orc.encode(0.25)
    pool = orc.pool(conv, 3, 3, 2, 1, 1, 2, 2, d, cc)
    cases.append(pool)
    sq = orc.square_layer(pool, *keys.evk_triple)
    cases.append(sq)
    fc = orc.fc(sq, 8, 3, orc.encode_many(rng.uniform(-1, 1, 24)), orc.encode_many(rng.uniform(-1, 1, 3)))
    cases.append(fc)
    for c in cases:
        c = c.reshape(-1, 2, orc.K, orc.stride)[:3]
        assert np.array_equal(kg.noise_budget(orc, c, keys.sk), kg.budget_bigint(orc, c, keys))
    # budgets fall along the chain, and square costs the most
    mins = [int(kg.noise_budget(orc, c.reshape(-1, 2, orc.K, orc.stride), keys.sk).min()) for c in cases]
    assert mins == sorted(mins, reverse=True) and mins[2] - mins[3] > 10


@pytest.mark.skipif(not have_ref(), reason="needs the compiled original (oracle/_ref)")
def test_oracle_equals_seal_invariant_noise_budget():
    from oracle.ref import Ref
    n, t = 4096, 1 << 20
    r = Ref(n, t)
    orc = Oracle(r.n, r.primes, r.t)
    sk, _ = r.keys()
    rng = np.random.default_rng(6)
    x = r.encrypt(rng.uniform(-1, 1, 16).astype(np.float32))
    conv = r.conv(x, 4, 4, 1, 1, 1, 2, 2, 2, rng.uniform(-1, 1, 8).astype(np.float32), rng.uniform(-1, 1, 2).astype(np.float32))
    fc = r.fc(x, 16, 2, rng.uniform(-1, 1, 32).astype(np.float32), rng.uniform(-1, 1, 2).astype(np.float32))
    sq = r.square_layer(conv, 2, 3, 3)
    for c in (x, conv, fc, sq):
        c = c.reshape(-1, 2, orc.K, orc.stride)
        _, want = r.decrypt(c)
        assert np.array_equal(kg.noise_budget(orc, c, sk), want)
