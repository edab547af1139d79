"""Budget-driven re-encryption (Network::reencrypt_below_budget, forward_dev_adaptive) through the host library: the Approx net at
n = 4096, t = 2^20, keys from tests/fv_keygen.py.  A first adaptive run at threshold 0 locates a check j whose budget is below every
earlier one; with the threshold set to that budget the trigger layer is known in advance.

The decoded scores are not compared with a float evaluation: at these parameters the FractionalEncoder's plaintext coefficients
wrap modulo t after the square layer (t = 2^20) -- a limit of the plaintext modulus, not of the noise (tools/noise_trace.py,
DESIGN 4.6); the budget is checked directly instead."""
import numpy as np
import pytest

import util
import fv_keygen as kg
from oracle.port import DEFAULT_PRIMES_128 as PRIMES, Oracle

pytestmark = pytest.mark.gpu

N, T, SEED = 4096, 1 << 20, 1234
MODEL = "ApproxPlainModel"


@pytest.fixture(scope="module")
def env():
    from crcnn_b200.host import HostNetwork
    orc = Oracle(N, PRIMES[N], T)
    keys = kg.generate(orc, 21)
    net = HostNetwork(N, PRIMES[N], T, MODEL, evk=keys.evk_triple)
    imgs = [util.synthetic_image(s) for s in range(2)]
    rng = np.random.default_rng(5)
    x = [kg.encrypt_values(keys, im, rng) for im in imgs]
    yield orc, keys, net, imgs, x
    net.close()


def adaptive(net, x, threshold, batch=1):
    from crcnn_b200.host import OutOfBudget
    net.set_budget_threshold(threshold)
    try:
        out, _ = net.forward_adaptive(np.concatenate(x), batch=batch)
        return out, None
    except OutOfBudget as e:
        return None, e.layer


def locate_trigger(net, x, batch=1):
    """(j, b_j) of the latest check before the last layer whose budget is positive and below every earlier check"""
    adaptive(net, x, 0, batch=batch)
    log = net.budget_log()
    cands = [(lay, b) for k, (lay, b, _) in enumerate(log)
             if 0 < b < min([bb for _, bb, _ in log[:k]] or [1 << 30]) and lay < net.num_layers - 1]
    assert cands, log
    return cands[-1], log


@pytest.mark.parametrize("fusion", [True, False])
def test_adaptive_equals_fixed_point(env, fusion):
    from crcnn_b200.lib import Engine
    orc, keys, net, imgs, x = env
    net.set_fusion(fusion)
    net.use_keys(keys.sk, keys.pk, device_reencryption=True, seed=SEED)
    (j, bj), log0 = locate_trigger(net, x[:1])
    net.use_keys(keys.sk, keys.pk, device_reencryption=True, seed=SEED)     # fresh call counter: first re-encryption draws `SEED`
    got, failed = adaptive(net, x[:1], bj)
    assert failed is None
    log = net.budget_log()
    assert [(lay, re) for lay, _, re in log if re] == [(j, True)], log
    assert [lay for lay, _, _ in log] == [lay for lay, _, _ in log0][:len(log)]
    # Network::forward's fixed point at layer_before_reenc = j + 1 with the same seed: layers [0, j], crcnn_reencrypt, [j+1, L)
    mid, shape = net.forward(x[0], first=0, last=j + 1)
    eng = Engine.adopt(net.ctx(), N, PRIMES[N], T)
    dk = eng.keys_upload(keys.sk, keys.pk)
    fresh = eng.download(eng.reencrypt(dk, eng.upload(mid), seed=SEED))
    want, _ = net.forward(fresh, first=j + 1, shape=shape)
    assert np.array_equal(got, want)
    # budget left at every check after the re-encryption (the oracle agrees on the scores)
    assert all(b > 0 for _, b, _ in log) and kg.noise_budget(orc, got, keys.sk).min() == log[-1][1]
    net.set_fusion(True)


def test_without_reencryption_throws_at_trigger(env):
    orc, keys, net, imgs, x = env
    net.use_keys(keys.sk, keys.pk, device_reencryption=False)
    (j, bj), _ = locate_trigger(net, x[:1])
    got, failed = adaptive(net, x[:1], bj)
    assert got is None and failed == j
    assert net.budget_log()[-1][:2] == (j, bj)


def test_budget_zero_throws_even_with_reencryption(env):
    orc, keys, net, imgs, x = env
    net.use_keys(keys.sk, keys.pk, device_reencryption=True, seed=SEED)
    Q = kg.modulus(orc)
    row = [0] * N
    row[0] = 1 << (Q.bit_length() - 3)                  # budget 1
    crafted = x[0].copy()
    crafted[100] = kg.craft(keys, [row], np.random.default_rng(2))[0]
    assert kg.noise_budget(orc, crafted[100:101], keys.sk)[0] == 1
    got, failed = adaptive(net, [crafted], 5)
    log = net.budget_log()
    assert got is None and failed == log[-1][0] and log[-1][1] == 0
    assert not any(re for _, _, re in log)


def test_default_threshold_changes_nothing(env):
    orc, keys, net, imgs, x = env
    net.use_keys(keys.sk, keys.pk, device_reencryption=True, seed=SEED)
    got, failed = adaptive(net, x, -1, batch=2)
    want, _ = net.forward(np.concatenate(x), batch=2)
    assert failed is None and np.array_equal(got, want)
    log = net.budget_log()
    assert log and not any(re for _, _, re in log) and log[-1][0] == net.num_layers - 1


def test_batch_reencrypts_whole_tensor(env):
    orc, keys, net, imgs, x = env
    net.use_keys(keys.sk, keys.pk, device_reencryption=True, seed=SEED)
    (j, bj), _ = locate_trigger(net, x, batch=2)
    got, failed = adaptive(net, x, bj, batch=2)
    assert failed is None
    log = net.budget_log()
    assert [lay for lay, _, re in log if re] == [j]
    assert kg.noise_budget(orc, got, keys.sk).min() == log[-1][1] > 0
