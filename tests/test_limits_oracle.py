"""The closed forms and operand magnitudes tests/test_gpu_limits.py relies on, proved on the CPU oracle (no GPU).

The GPU file runs the weighted sums at the engine's capacity limits with worst-case operands taken from the public API: constant
plaintexts t - k as weights (q - k in every NTT slot) and NTT-form inputs of chosen residues.  Its expected outputs at fan-in 4096 come
from closed forms rather than from the oracle; this file checks each closed form against the oracle at small sizes, and prints how close
the chosen operands bring the accumulators to their bounds: the limb-split GEMM's s32 class sums (2^31) and the CUDA-core MAC's 128-bit
accumulator (2^128).
"""
import numpy as np
import pytest

from util import PARAM_SETS, PRIMES, T_FOR_N, acc7_even, bias_slots, class_sums, const_weight_fc_slots, slots_to_words, worst_operands
from oracle.port import Oracle

TCN_MAX_R = 4096          # tcn_mac.cuh
SETS = {2048: (PRIMES[2048], T_FOR_N[2048]), 4096: (PRIMES[4096], T_FOR_N[4096]), 8192: (PRIMES[8192], T_FOR_N[8192])}


def _const_plain(n, t, k):
    p = np.zeros(n + 1, dtype=np.uint64)
    p[0] = t - k
    return p


@pytest.mark.parametrize("name", ["n2048", "n4096", "P60a", "P60b"])
def test_constant_plaintext_weights_are_q_minus_k_in_every_slot(name):
    n, primes, t = (int(name[1:]), *SETS[int(name[1:])]) if name.startswith("n") else PARAM_SETS[name]
    orc = Oracle(n, primes, t)
    k, _ = worst_operands(primes, t)
    for kk in (1, 2, k, (t - 1) // 2):
        got = orc.plain_to_ntt(_const_plain(n, t, kk))
        for j, q in enumerate(primes):
            assert np.all(got[j, :n] == q - kk), (name, kk, j)


@pytest.mark.parametrize("n", [2048, 4096])
def test_worst_case_class_sums_stay_below_2_31(n):
    primes, t = SETS[n]
    k, xs = worst_operands(primes, t)
    for j, q in enumerate(primes):
        cs = class_sums(q - k, xs[j])
        top = TCN_MAX_R * max(cs)
        print("n=%d q=%#x: k=%d (weight %#x), slot %#x: largest class sum at fan-in %d = %d = 2^%.4f (bound 2^31, 7*R*255^2 = 2^%.4f)"
              % (n, q, k, q - k, xs[j], TCN_MAX_R, top, np.log2(top), np.log2(7 * TCN_MAX_R * 255 ** 2)))
        assert top < 2 ** 31
        # the chosen pair beats the plain all-(q-1) operands
        assert max(cs) >= max(class_sums(q - 1, q - 1))
        # and reaches at least 60% of the bound itself (k <= (t-1)/2 keeps the weight's middle bytes below 0xff at t = 2^18)
        assert top > 0.6 * 2 ** 31


@pytest.mark.parametrize("name", ["P60a", "P60b"])
def test_acc7_at_chunk_terms(name):
    """chunk_terms = 2^(128 - 2 bits(q)) = 256 for 60-bit primes: 256 products of (q-1)^2 on top of a reduced residue fill the even half
    of the split accumulator to within 2^-27 of 2^128; 257 would wrap it (what a doubled chunk_terms would do at fan-in 257 and 513)."""
    n, primes, t = PARAM_SETS[name]
    bits = max(int(q).bit_length() for q in primes)
    chunk = 1 << (128 - 2 * bits)
    assert chunk == 256
    for q in primes:
        full = acc7_even(q - 1, q - 1, chunk, carry=q - 1)
        print("%s q=%#x: even accumulator after %d terms of (q-1)^2 + (q-1) = 2^%.10f (bound 2^128); %d terms: 2^%.6f"
              % (name, q, chunk, np.log2(float(full)), chunk + 1, np.log2(float(acc7_even(q - 1, q - 1, chunk + 1)))))
        assert full < 1 << 128
        assert full > (1 << 128) - (1 << 101)
        assert acc7_even(q - 1, q - 1, chunk + 1) >= 1 << 128


@pytest.mark.parametrize("name", ["n2048", "n4096", "P60b"])
def test_fc_of_constant_weights_closed_form(name):
    """Oracle.fc on the inverse transform of NTT-form inputs equals const_weight_fc_slots: uniform operands (R w x + bias), and
    near-maximal operands that vary per (output, term, column, slot)."""
    n, primes, t = (int(name[1:]), *SETS[int(name[1:])]) if name.startswith("n") else PARAM_SETS[name]
    orc = Oracle(n, primes, t)
    rng = np.random.default_rng(len(name) * n)
    K = len(primes)
    k0, xb = worst_operands(primes, t)
    R, M, B = 7, 3, 2
    bv = rng.uniform(-3, 3, size=M).astype(np.float32)
    bp = orc.encode_many(bv)
    bias = bias_slots(orc, bp)
    for kind in ("uniform", "varied"):
        if kind == "uniform":
            k = np.full((M, R), k0, dtype=np.int64)
            d = np.zeros((B, R, 2, K, n), dtype=np.int64)
        else:
            k = np.clip(k0 - rng.integers(0, 8, size=(M, R)), 1, (t - 1) // 2)
            d = rng.integers(0, 8, size=(B, R, 2, K, n))
        want = const_weight_fc_slots(k, xb, d, primes, bias)
        if kind == "uniform":
            for j, q in enumerate(primes):
                assert np.all(want[:, :, 1, j] == (-R * k0 * xb[j]) % q)
                assert np.all(want[:, :, 0, j] == ((-R * k0 * xb[j]) % q + bias[None, :, j].astype(object)) % q)
        xs = np.stack([xb[j] - d[:, :, :, j, :] for j in range(K)], axis=3).astype(np.uint64)
        wp = np.stack([_const_plain(n, t, int(v)) for v in k.ravel()])
        for b in range(B):
            xc = orc.ct_transform(slots_to_words(xs[b]), inverse=True)
            got = orc.ct_transform(orc.fc(xc, R, M, wp, bp).reshape(M, 2, K, n + 1))
            assert np.array_equal(got[..., :n], want[b]), (name, kind, b)


@pytest.mark.parametrize("name", ["n2048", "n4096", "P60a"])
def test_sum_pool_of_all_q_minus_1_is_q_minus_R(name):
    """Window sums of all-(q-1) words are q - (R mod q) in every word, at the 64-bit bound R_max = floor((2^64 - 1) / max q) and one
    past it (where a plain 64-bit sum would wrap)."""
    n, primes, t = (int(name[1:]), *SETS[int(name[1:])]) if name.startswith("n") else PARAM_SETS[name]
    orc = Oracle(n, primes, t)
    K = len(primes)
    rmax = (2 ** 64 - 1) // max(primes)
    assert rmax == {"n2048": 1024, "n4096": 512, "P60a": 16}[name]
    for R in (rmax, rmax + 1):
        x = np.zeros((R, 2, K, n + 1), dtype=np.uint64)
        for j, q in enumerate(primes):
            x[:, :, j, :n] = q - 1
        got = orc.pool(x, 1, R, 1, 1, 1, 1, R)
        for j, q in enumerate(primes):
            assert np.all(got[..., j, :n] == q - R % q), (name, R)
        print("%s R=%d: R * (q-1) = 2^%.6f (64-bit sum %s)" % (name, R, np.log2(float(R * (max(primes) - 1))),
                                                            "fits" if R * (max(primes) - 1) < 2 ** 64 else "wraps"))
        assert (R * (max(primes) - 1) < 2 ** 64) == (R == rmax)
