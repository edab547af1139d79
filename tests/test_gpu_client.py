"""The client's two ends on the B200: crcnn_encrypt_values (FractionalEncoder::encode + Encryptor::encrypt of floats) and
crcnn_decrypt_values (Decryptor::decrypt + (float) FractionalEncoder::decode), through Engine, and Network::predict through the
host library.  Keys come from tests/fv_keygen.py, so nothing here needs the compiled original.

A value's integer part is encoded from round(v) as an int64, whose balanced base-3 digits end at coefficient 40 (3^40 / 2 > 2^63):
coefficients 41..63 of the encoder's 64 integer slots cannot be reached from any value SEAL can encode, so the largest float below
2^63 stands in for "the top integer slot".  The fractional digits reach coefficient n - 32 (the 32nd trit) for most fractions."""
import numpy as np
import pytest

import util
import fv_keygen as kg
from oracle.port import DEFAULT_PRIMES_128 as PRIMES, Oracle
from test_noise_budget_oracle import T_OF

pytestmark = pytest.mark.gpu

_f = np.float32
VALUES = np.array([0.0, 1.0, -1.0, -7.0, 2.0, 0.25, -0.3, 1.0 / 3.0, -2.0 / 3.0, 0.1, np.nextafter(_f(0.5), _f(0)), 0.5, -0.5, 1.5,
                   2.8215, -0.4242, 1e-20, -3.5e-16, 12345678.0, -3.0e9, 7.25e12, 9.0e18, -9.2e18, np.nextafter(_f(2.0 ** 63), _f(0))],
                  dtype=np.float32)


def setup(n, t=None, seed=5):
    from crcnn_b200.lib import Engine
    t = T_OF[n] if t is None else t
    orc = Oracle(n, PRIMES[n], t)
    keys = kg.generate(orc, seed)
    eng = Engine(n, PRIMES[n], t)
    return orc, keys, eng, eng.keys_upload(keys.sk, keys.pk)


def encrypt_step(n, K):
    """ciphertexts per 1 GiB chunk of the encrypting calls (engine.cu: encrypt_step)"""
    return (1 << 30) // ((K + 1) * n * 8 + 96 * 8 + 5 * n + 8)


def decrypt_step(n, K):
    """ciphertexts per 1 GiB chunk of the decrypting calls (engine.cu: decrypt_step)"""
    return (1 << 30) // ((K + 1) * n * 8)


def oracle_encrypt(orc, keys, v, noise):
    plain, cc = orc.encode(float(v))
    return orc.encrypt(plain, keys.pk, noise[0], noise[1], noise[2], coeff_count=cc)


def rows(eng, t, first, count):
    return eng.download(eng.slice(t, first, count))


def test_encoder_reaches_the_extreme_slots():
    orc = Oracle(4096, PRIMES[4096], T_OF[4096])
    enc = np.array([orc.encode(float(v))[0] for v in VALUES])
    assert enc[:, 40].any() and not enc[:, 41:64].any()
    assert enc[:, 4096 - 32].any()


@pytest.mark.parametrize("n", [2048, 4096, 8192, 16384])
def test_encrypt_host_noise_equals_oracle(n):
    orc, keys, eng, dk = setup(n)
    rng = np.random.default_rng(n)
    P = len(VALUES)
    noise = np.stack([kg.ternary(rng, (P, n)), kg.clipped_normal(rng, (P, n)), kg.clipped_normal(rng, (P, n))], axis=1)
    want = np.stack([oracle_encrypt(orc, keys, VALUES[i], noise[i]) for i in range(P)])
    if n == 8192:        # two chunks: row r is value / noise r % P, checked at both ends and across the boundary
        step = encrypt_step(n, orc.K)
        count = step + P + 5
        idx = np.arange(count) % P
        ct = eng.encrypt_values(dk, VALUES[idx], seed=1, noise=noise[idx])
        for first in (0, step - P, step, count - P):
            assert np.array_equal(rows(eng, ct, first, P), want[idx[first:first + P]]), first
    else:
        ct = eng.encrypt_values(dk, VALUES, seed=1, noise=noise)
        assert np.array_equal(eng.download(ct), want)


@pytest.mark.parametrize("n", [4096, 8192])
def test_encrypt_device_generator(n):
    orc, keys, eng, dk = setup(n)
    vals = np.concatenate([VALUES, np.random.default_rng(3).uniform(-3, 3, 40).astype(np.float32)])
    ct = eng.encrypt_values(dk, vals, seed=77)
    plain = eng.decrypt(dk, ct)
    assert np.array_equal(plain, np.array([orc.encode(float(v))[0] for v in vals]))
    got = eng.noise_budget(dk, ct)
    fresh = kg.noise_budget(orc, kg.encrypt_values(keys, vals, np.random.default_rng(4)), keys.sk)
    assert fresh.min() - 1 <= got.min() and got.max() <= fresh.max() + 1, (got, fresh)
    again = eng.download(eng.encrypt_values(dk, vals, seed=77))
    assert np.array_equal(eng.download(ct), again)
    other = eng.download(eng.encrypt_values(dk, vals, seed=78))
    assert not np.array_equal(other[:, 1], again[:, 1])
    assert all(not np.array_equal(other[i], again[i]) for i in range(len(vals)))


def expected_values(orc, keys, cts):
    return np.array([_f(orc.decode(p)) for p in orc.decrypt(cts, keys.sk)], dtype=np.float32)


def test_decrypt_values_fresh_and_layer_outputs_both_domains():
    n = 4096
    orc, keys, eng, dk = setup(n)
    rng = np.random.default_rng(11)
    fresh = kg.encrypt_values(keys, VALUES, rng)
    want = expected_values(orc, keys, fresh)
    assert np.array_equal(eng.decrypt_values(dk, eng.upload(fresh)), want)
    assert np.array_equal(eng.decrypt_values(dk, eng.upload(orc.ct_transform(fresh), ntt_form=True)), want)
    # conv -> square (generated evaluation keys): the layer outputs, in the domain the engine leaves them and in the other
    x = kg.encrypt_values(keys, rng.uniform(-1, 1, 36).astype(np.float32), rng)       # 1 x 6 x 6
    g = eng.conv(eng.upload(x), eng.plain_encode(rng.uniform(-1, 1, 18).astype(np.float32)),
                 eng.plain_encode(rng.uniform(-1, 1, 2).astype(np.float32)), 1, 6, 6, 1, 1, 1, 3, 3, 2)     # 2 x 4 x 4
    s = eng.square_layer(g, eng.evk_upload(*keys.evk_triple))
    for o in (g, s):
        want = expected_values(orc, keys, eng.download(o))
        assert np.array_equal(eng.decrypt_values(dk, o), want)
        ntt = eng.slice(o, 0, eng.count(o))
        if eng.device_ptr(ntt)[1]:
            eng.from_ntt(ntt)
        else:
            eng.to_ntt(ntt)
        assert np.array_equal(eng.decrypt_values(dk, ntt), want)


def test_decrypt_values_two_chunks_and_round_trip():
    """n = 2048: a decrypting chunk holds 32,768 ciphertexts; the tensor is made on the device and runs past it."""
    n = 2048
    orc, keys, eng, dk = setup(n)
    step = decrypt_step(n, orc.K)
    assert step == 32768
    P = len(VALUES)
    count = step + 3 * P
    idx = np.arange(count) % P
    ct = eng.encrypt_values(dk, VALUES[idx], seed=9)
    got = eng.decrypt_values(dk, ct)
    trip = np.array([_f(orc.decode(orc.encode(float(v))[0])) for v in VALUES], dtype=np.float32)
    assert np.array_equal(got, trip[idx])
    for first in (0, step - P, step + P):
        assert np.array_equal(got[first:first + P], expected_values(orc, keys, rows(eng, ct, first, P)))


@pytest.mark.parametrize("n", [4096, 8192])
def test_round_trip_every_value(n):
    orc, keys, eng, dk = setup(n)
    vals = np.concatenate([VALUES, np.random.default_rng(n).uniform(-100, 100, 200).astype(np.float32)])
    got = eng.decrypt_values(dk, eng.encrypt_values(dk, vals, seed=5))
    assert np.array_equal(got, np.array([_f(orc.decode(orc.encode(float(v))[0])) for v in vals], dtype=np.float32))


def oracle_reencrypt(orc, keys, cts, noise):
    out = []
    for c, p in enumerate(orc.decrypt(cts, keys.sk)):
        out.append(oracle_encrypt(orc, keys, _f(orc.decode(p)), noise[c]))
    return np.stack(out)


def test_reencrypt_host_noise_equals_oracle():
    """crcnn_reencrypt runs its encryption through the range function crcnn_encrypt_values shares: decrypt -> decode -> float ->
    encode -> encrypt equals the oracle's, on fresh ciphertexts and a layer output."""
    n = 4096
    orc, keys, eng, dk = setup(n)
    rng = np.random.default_rng(21)
    fresh = kg.encrypt_values(keys, VALUES, rng)
    x = kg.encrypt_values(keys, rng.uniform(-1, 1, 36).astype(np.float32), rng)
    conv = eng.download(eng.conv(eng.upload(x), eng.plain_encode(rng.uniform(-1, 1, 18).astype(np.float32)),
                                 eng.plain_encode(rng.uniform(-1, 1, 2).astype(np.float32)), 1, 6, 6, 1, 1, 1, 3, 3, 2))
    for cts in (fresh, conv):
        c = len(cts)
        noise = np.stack([kg.ternary(rng, (c, n)), kg.clipped_normal(rng, (c, n)), kg.clipped_normal(rng, (c, n))], axis=1)
        got = eng.download(eng.reencrypt(dk, eng.upload(cts), seed=3, noise=noise))
        assert np.array_equal(got, oracle_reencrypt(orc, keys, cts, noise))


def test_reencrypt_two_chunks_host_noise():
    n = 8192
    orc, keys, eng, dk = setup(n)
    rng = np.random.default_rng(22)
    P = 8
    vals = rng.uniform(-2, 2, P).astype(np.float32)
    step = encrypt_step(n, orc.K)
    count = step + P + 3
    idx = np.arange(count) % P
    src = eng.encrypt_values(dk, vals[idx], seed=40)
    noise = np.stack([kg.ternary(rng, (P, n)), kg.clipped_normal(rng, (P, n)), kg.clipped_normal(rng, (P, n))], axis=1)
    out = eng.reencrypt(dk, src, seed=41, noise=noise[idx])
    for first in (0, step - P, step, count - P):
        want = oracle_reencrypt(orc, keys, rows(eng, src, first, P), noise[idx[first:first + P]])
        assert np.array_equal(rows(eng, out, first, P), want), first


def test_errors_leave_the_context_usable():
    from crcnn_b200.lib import CrcnnError
    n = 4096
    orc, keys, eng, dk = setup(n)
    ct = eng.encrypt_values(dk, [0.5, -1.25], seed=1)
    for call in (lambda: eng.encrypt_values(None, [1.0]), lambda: eng.encrypt_values(dk, []),
                 lambda: eng.decrypt_values(None, ct), lambda: eng.decrypt_values(dk, eng.square(ct))):
        with pytest.raises(CrcnnError) as e:
            call()
        assert e.value.code == -1
    assert np.array_equal(eng.decrypt_values(dk, eng.encrypt_values(dk, [0.5, -1.25], seed=2)), np.array([0.5, -1.25], dtype=np.float32))


# ---- Network::predict through the host library
def host_case(model, n, t, batch, seed_keys=31):
    from crcnn_b200.host import HostNetwork
    from crcnn_b200.lib import Engine
    orc = Oracle(n, PRIMES[n], t)
    keys = kg.generate(orc, seed_keys)
    net = HostNetwork(n, PRIMES[n], t, model, evk=keys.evk_triple)
    net.use_keys(keys.sk, keys.pk)
    eng = Engine.adopt(net.ctx(), n, PRIMES[n], t)
    imgs = np.stack([util.synthetic_image(s, net.zd * net.xd * net.yd) for s in range(batch)])
    return orc, keys, net, eng, eng.keys_upload(keys.sk, keys.pk), imgs


def decoded_scores(orc, eng, dk, out, batch):
    return np.array([_f(orc.decode(p)) for p in eng.decrypt(dk, eng.upload(out))], dtype=np.float32).reshape(batch, -1)


@pytest.mark.parametrize("model,n,t,batch", [("PlainModelTiny", 4096, util.T_FOR_N[4096], 2), ("PlainModel", 8192, util.T_FOR_N[8192], 1)])
def test_predict_values_equals_forward_range(model, n, t, batch):
    orc, keys, net, eng, dk, imgs = host_case(model, n, t, batch)
    try:
        got = net.predict_values(imgs, batch=batch, seed=1234)          # the network's first encryption: seed 1234 itself
        x = eng.download(eng.encrypt_values(dk, imgs, seed=1234))
        out, shape = net.forward(x, batch=batch)
        assert got.shape == (batch, net.outputs)
        assert np.array_equal(got, decoded_scores(orc, eng, dk, out, batch))
    finally:
        del dk
        net.close()


def test_predict_values_budget_driven_reencryption():
    from crcnn_b200.host import OutOfBudget
    n, t = 4096, 1 << 20
    orc, keys, net, eng, dk, imgs = host_case("ApproxPlainModel", n, t, 1)
    try:
        net.use_keys(keys.sk, keys.pk, device_reencryption=True, seed=555)
        net.set_budget_threshold(1000)                 # every check before the last layer re-encrypts
        got = net.predict_values(imgs, batch=1, seed=99)
        log = net.budget_log()
        assert [re for _, _, re in log] == [True] * (len(log) - 1) + [False], log
        net.use_keys(keys.sk, keys.pk, device_reencryption=True, seed=555)      # fresh re-encryption call counter
        x = eng.download(eng.encrypt_values(dk, imgs, seed=99))
        out, _ = net.forward_adaptive(x)
        assert np.array_equal(got, decoded_scores(orc, eng, dk, out, 1))
        net.use_keys(keys.sk, keys.pk, device_reencryption=False)
        with pytest.raises(OutOfBudget) as e:
            net.predict_values(imgs, batch=1, seed=100)
        assert e.value.layer == net.budget_log()[0][0] < net.num_layers - 1
    finally:
        del dk
        net.close()
