"""CRT plaintext-modulus ensembles, CPU side: Garner's mixed-radix recombination of the instances' residues followed by
BalancedFractionalEncoder::decode under the product T (the two steps of reenc.cu's crt_decode), restated on Python integers and
IEEE doubles, against the oracle's decoder in an Oracle(n, primes, T).  The GPU tests (test_gpu_crt_ensemble.py) compare the
device against this restatement."""
import numpy as np
import pytest

from oracle.port import DEFAULT_PRIMES_128 as PRIMES, Oracle

N = 8192
Q_MIN = min(PRIMES[N])                  # 0x3ffffffef40001: T must stay below every coefficient prime
CRT_MODULI = {1: [1 << 30], 2: [32771, 32779], 4: [181, 191, 193, 197], 8: [5, 7, 11, 13, 17, 19, 23, 29]}   # bench.py's lists
SLOTS = list(range(64)) + list(range(N - 32, N))     # the coefficients the fractional decoder reads


def _is_prime(v):
    if v < 2:
        return False
    f = 2
    while f * f <= v:
        if v % f == 0:
            return False
        f += 1
    return True


def near_limit(M):
    """M pairwise coprime moduli whose product sits just below the smallest n = 8192 prime: M - 1 primes below the M-th root,
    then the largest integer that keeps the product below it and is coprime to them."""
    from math import gcd
    root = int(round(Q_MIN ** (1.0 / M)))
    ms, v = [], root
    while len(ms) < M - 1:
        if _is_prime(v):
            ms.append(v)
        v -= 1
    p = int(np.prod([1] + ms, dtype=object))
    last = (Q_MIN - 1) // p
    while any(gcd(last, m) != 1 for m in ms):
        last -= 1
    return ms + [last]


LISTS = [CRT_MODULI[1], CRT_MODULI[2], [1021, 1031, 1033], CRT_MODULI[4], CRT_MODULI[8]] + [near_limit(M) for M in (1, 2, 3, 4, 8)]


def product(moduli):
    T = 1
    for m in moduli:
        T *= int(m)
    return T


def garner(residues, moduli):
    """x mod prod(moduli) from x mod each modulus, by the mixed radix the kernel uses."""
    x, p = int(residues[0]), 1
    for k in range(1, len(moduli)):
        p *= int(moduli[k - 1])
        t = int(moduli[k])
        v = ((int(residues[k]) - x % t) * pow(p, -1, t)) % t
        x += v * p
    return x


def _wrap64(v):
    v &= (1 << 64) - 1
    return v - (1 << 64) if v >> 63 else v


def decode(coeffs96, T):
    """BalancedFractionalEncoder::decode under plain modulus T of the 96 slots (coefficients 0..63, then n-32..n-1), with the
    decoder's wrapping int64 integer part and its double arithmetic in the same order."""
    half = (T + 1) >> 1

    def signed(c):
        c = int(c)
        return c - T if c >= half else c
    ip = 0
    for i in range(63, -1, -1):
        ip = _wrap64(_wrap64(ip * 3) + signed(coeffs96[i]))
    frac = 0.0
    for i in range(32):
        frac = (frac + float(signed(coeffs96[64 + i]))) / 3.0
    return float(ip) - frac


def crt_decode(residue_slots, moduli):
    """float32 of the decode under T of the slots composed from residue_slots[m][96]"""
    T = product(moduli)
    return np.float32(decode([garner([residue_slots[m][j] for m in range(len(moduli))], moduli) for j in range(96)], T))


def cases(moduli, rng):
    """values[count][96] below T: random ones, then the edge coefficients 0, (T-1)/2, (T+1)/2, T-1 and integer parts that wrap int64"""
    T = product(moduli)
    rand = [[int(rng.integers(0, 1 << 62)) % T for _ in range(96)] for _ in range(6)]
    small = [[int(v) % T for v in rng.integers(0, 3, 96)] for _ in range(2)]        # digits of an ordinary encoded value
    edges = [[e] * 96 for e in (0, (T - 1) // 2, (T + 1) // 2, T - 1)]
    wrap = [[(T - 1) // 2] * 64 + [0] * 32, [(T + 1) // 2] * 64 + [(T - 1) // 2] * 32, [1] * 64 + [T - 1] * 32]
    mixed = [[[0, (T - 1) // 2, (T + 1) // 2, T - 1][(i * 7 + j) % 4] for j in range(96)] for i in range(2)]
    return rand + small + edges + wrap + mixed


def residues_of(values, moduli):
    """[M][count][96] residues of values[count][96]"""
    return [[[v % int(m) for v in row] for row in values] for m in moduli]


def test_lists_are_valid_ensembles():
    from math import gcd
    for ms in LISTS:
        assert all(m >= 2 for m in ms)
        assert all(gcd(a, b) == 1 for i, a in enumerate(ms) for b in ms[:i])
        assert product(ms) < Q_MIN
    for M in (1, 2, 3, 4, 8):
        assert product(near_limit(M)) > Q_MIN * 0.99


@pytest.mark.parametrize("moduli", LISTS, ids=lambda ms: "M%d_T%d" % (len(ms), product(ms)))
def test_garner_and_decode_match_the_oracle(moduli):
    T = product(moduli)
    orc = Oracle(N, PRIMES[N], T)
    rng = np.random.default_rng(T % (1 << 32))
    for row in cases(moduli, rng):
        res = [[v % int(m) for v in row] for m in moduli]
        composed = [garner([res[k][j] for k in range(len(moduli))], moduli) for j in range(96)]
        assert composed == row
        plain = np.zeros(N + 1, dtype=np.uint64)
        plain[SLOTS] = np.array(row, dtype=np.uint64)
        want = orc.decode(plain)
        got = decode(composed, T)
        assert got == want or (np.isnan(got) and np.isnan(want)), (got, want)
        assert np.float32(got).tobytes() == crt_decode([r for r in res], moduli).tobytes()
