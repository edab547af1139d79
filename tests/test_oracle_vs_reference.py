"""Pins the CPU oracle against the UNMODIFIED reference (SEAL 2.3.1 + CrCNN layers), byte for byte.  The evaluator and layer
cases compare with SHA-256 digests of the reference's outputs stored in tests/golden/reference_ops.json (tests/golden/
make_golden.py: case_reference_ops; the inputs are regenerated from splitmix64 seeds, tests/util.py: ref_ops).  The re-encryption
steps run against the compiled reference in oracle/_ref where it is built (oracle/Makefile.ref)."""
import json
import os

import numpy as np
import pytest

import util
from oracle import port, ref

GOLDEN = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_ops.json")))


@pytest.fixture(scope="module", params=sorted(util.REF_OPS), ids=lambda n: "n%d" % n)
def pair(request):
    n = request.param
    g = GOLDEN[str(n)]
    t, seed = util.REF_OPS[n]
    assert (g["t"], g["seed"]) == (t, seed) and g["primes"] == port.DEFAULT_PRIMES_128[n]  # coeff_modulus_128(n)
    o = port.Oracle(n, g["primes"], t)
    outs = {k: util.sha(v) for k, v in util.ref_ops("oracle", o, n, g["primes"], t, seed).items()}
    assert sorted(outs) == sorted(g["digests"])
    return n, o, outs, g["digests"]


def _same(pair, prefix):
    _, _, got, want = pair
    names = [k for k in want if k.startswith(prefix)]
    assert names
    for k in names:
        assert got[k] == want[k], k


def test_encoder(pair):
    _same(pair, "encode_")


def test_evaluator_ops(pair):
    for prefix in ("ct_ntt", "ct_intt", "plain_ntt", "multiply_plain_ntt", "plain_mul", "plain_add", "plain_sub", "add_many"):
        _same(pair, prefix)


def test_square_relinearize(pair):
    _same(pair, "square")
    _same(pair, "relinearize")


def test_layers(pair):
    for prefix in ("conv", "fc", "pool", "avgpool", "bn", "square_layer"):
        _same(pair, prefix)
    # the float32 value of 1/9 has other base-3 digits from about the 15th on and must NOT reproduce the reference's bytes
    n, o, _, want = pair
    xi = util.det_cts(util.REF_OPS[n][1] + 3, n, o.primes, 2 * 3 * 3)     # the input of util.ref_ops' layer cases
    assert util.sha(o.pool(xi, 3, 3, 2, 1, 1, 3, 3, *o.encode(float(np.float32(1.0 / 9.0))))) != want["avgpool9"]


@pytest.mark.parametrize("n,t", [(2048, 1 << 16), (4096, 1 << 20), (8192, 1 << 30)])
@pytest.mark.skipif(not ref.available(), reason="oracle/_ref not built")
def test_reencryption_steps_against_seal(n, t):
    """SURVEY 8(f) N4: the oracle's Decryptor::decrypt, FractionalEncoder::decode and Encryptor::encrypt restatements against
    SEAL's own objects -- decrypt bit for bit (fresh and used ciphertexts), decode -> float -> encode bit for bit, and an
    encryption with explicit sampled polynomials that SEAL's Decryptor opens to the same plaintext with a fresh noise budget."""
    r = ref.Ref(n, t, seed=5)
    o = port.Oracle(n, r.primes, t)
    sk, pk = r.keys()
    rng = np.random.default_rng(n)
    vals = rng.uniform(-3, 3, 6).astype(np.float32)
    cts = r.encrypt(vals)
    _, fresh_budget, plain = r.decrypt(cts, want_plain=True)
    assert np.array_equal(o.decrypt(cts, sk), plain)
    w = rng.uniform(-1, 1, 12).astype(np.float32); b = rng.uniform(-1, 1, 2).astype(np.float32)
    y = r.fc(cts, 6, 2, w, b, th=2).reshape(2, 2, r.K, r.stride)
    dec_vals, _, plain2 = r.decrypt(y, want_plain=True)
    assert np.array_equal(o.decrypt(y, sk), plain2)
    for i in range(2):
        assert o.decode(plain2[i]) == dec_vals[i]
        want_plain, want_val = r.reencode(y[i])
        enc, _ = o.encode(float(np.float32(o.decode(plain2[i]))))
        assert np.array_equal(enc, want_plain) and np.float32(o.decode(plain2[i])) == np.float32(want_val)
        u = rng.integers(-1, 2, n).astype(np.int8)
        e0 = np.clip(np.trunc(rng.normal(0, 3.19, n)), -19, 19).astype(np.int8)
        e1 = np.clip(np.trunc(rng.normal(0, 3.19, n)), -19, 19).astype(np.int8)
        ct = o.encrypt(want_plain, pk, u, e0, e1)
        _, budget, back = r.decrypt(ct[None], want_plain=True)
        assert np.array_equal(back[0], want_plain) and abs(int(budget[0]) - int(fresh_budget[0])) <= 1
