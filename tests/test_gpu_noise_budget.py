"""crcnn_noise_budget (Engine.noise_budget) on the B200: Decryptor::invariant_noise_budget, equal to the closed form of crafted
ciphertexts and to the CPU restatement (fv_keygen.noise_budget), in both domains, across scratch chunks, and after every layer of an Approx-shaped
chain run with generated keys."""
import numpy as np
import pytest

import fv_keygen as kg
from oracle.port import DEFAULT_PRIMES_128 as PRIMES, Oracle
from test_noise_budget_oracle import T_OF, sweep_rows

pytestmark = pytest.mark.gpu


def setup(n, t=None, seed=5):
    from crcnn_b200.lib import Engine
    t = T_OF[n] if t is None else t
    orc = Oracle(n, PRIMES[n], t)
    keys = kg.generate(orc, seed)
    eng = Engine(n, PRIMES[n], t)
    return orc, keys, eng, eng.keys_upload(keys.sk, keys.pk)


@pytest.mark.parametrize("n", [2048, 4096, 8192, 16384])
def test_crafted_both_domains(n):
    orc, keys, eng, dk = setup(n)
    rng = np.random.default_rng(n + 1)
    X = sweep_rows(orc, rng)
    want = kg.budget_of(orc, X)
    coeff = kg.craft(keys, X, rng)
    assert np.array_equal(kg.noise_budget(orc, coeff, keys.sk), want)
    assert np.array_equal(eng.noise_budget(dk, eng.upload(coeff)), want)
    ntt = kg.craft(keys, X, rng, ntt_form=True)
    assert np.array_equal(eng.noise_budget(dk, eng.upload(ntt, ntt_form=True)), want)
    assert eng.min_noise_budget(dk, eng.upload(coeff)) == want.min()


def test_two_chunks_minimum_in_second():
    """n = 2048: a scratch chunk holds 32,768 ciphertexts; the one low budget sits past it."""
    n = 2048
    orc, keys, eng, dk = setup(n)
    rng = np.random.default_rng(9)
    Q = kg.modulus(orc)
    X = [[0] * n for _ in range(4)]
    X[0][3], X[1][100] = 1 << 20, Q - (1 << 30)
    X[2][7] = 1 << 40                      # the minimum
    X[3][n - 1] = 5
    cts = kg.craft(keys, X, rng)
    want4 = kg.budget_of(orc, X)
    count = 32768 + 1000
    idx = np.tile([0, 1, 3], count // 3 + 1)[:count]
    idx[32768 + 517] = 2
    tiled = cts[idx]
    got = eng.noise_budget(dk, eng.upload(tiled))
    assert np.array_equal(got, want4[idx])
    assert eng.min_noise_budget(dk, eng.upload(tiled)) == want4[2] < want4[[0, 1, 3]].min()


def test_rejects_size3_and_null_keys():
    from crcnn_b200.lib import CrcnnError
    n = 4096
    orc, keys, eng, dk = setup(n)
    ct = kg.encrypt_values(keys, [0.5, 1.0], np.random.default_rng(1))
    sq = eng.square(eng.upload(ct))
    with pytest.raises(CrcnnError) as e:
        eng.noise_budget(dk, sq)
    assert e.value.code == -1
    with pytest.raises(CrcnnError) as e:
        eng.noise_budget(None, eng.upload(ct))
    assert e.value.code == -1


def test_approx_chain_every_layer_equals_oracle():
    """conv -> avg-pool -> bn -> square (generated evaluation keys) -> fc at n = 4096, t = 2^20: the device budget of every layer's
    output equals the oracle's on the downloaded activations."""
    n = 4096
    orc, keys, eng, dk = setup(n, 1 << 20)
    rng = np.random.default_rng(11)
    x = kg.encrypt_values(keys, rng.uniform(-1, 1, 36).astype(np.float32), rng)      # 1 x 6 x 6
    f = lambda k: rng.uniform(-1, 1, size=k).astype(np.float32)
    wv, bv, mv, vv, fv, fb = f(2 * 9), f(2), f(2), f(2), f(2 * 3 * 3 * 4), f(4)
    evk = eng.evk_upload(*keys.evk_triple)
    g = eng.upload(x)
    outs = []
    g = eng.conv(g, eng.plain_encode(wv), eng.plain_encode(bv), 1, 6, 6, 1, 1, 1, 3, 3, 2)     # 2 x 4 x 4
    outs.append(g)
    g = eng.pool(g, 1, 4, 4, 2, 1, 1, 2, 2, scale=eng.plain_encode_f64([0.25]))              # 2 x 3 x 3
    outs.append(g)
    g = eng.bn(g, 1, 2, 3, 3, eng.plain_encode(mv), eng.plain_encode(vv))
    outs.append(g)
    g = eng.square_layer(g, evk)
    outs.append(g)
    g = eng.fc(g, eng.plain_encode(fv), eng.plain_encode(fb), 1, 18, 4)
    outs.append(g)
    prev = None
    for o in outs:
        got = eng.noise_budget(dk, o)
        want = kg.noise_budget(orc, eng.download(o), keys.sk)
        assert np.array_equal(got, want)
        if prev is not None:
            assert got.min() <= prev
        prev = got.min()
    assert prev > 0
