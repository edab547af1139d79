"""CPU tests of the product's host logic: parameter derivation (crcnn_b200/csrc/params.cpp) against the
oracle's independently written derivation, and the C-ABI library's exports.  No GPU calls."""
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import port
from util import PARAM_SETS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SELFTEST = os.path.join(ROOT, "build", "host_selftest")


def fnv(a):
    h = 1469598103934665603
    for x in a:
        h ^= int(x)
        h = (h * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


@pytest.fixture(scope="module")
def selftest():
    if not os.path.exists(SELFTEST):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "crcnn_b200", "csrc"), "host_selftest"])
    return SELFTEST


def tcn_fold_ok(q):
    """modarith.cuh: tcn_fold_make -- the limb-split GEMM's folded reduction of its class sums applies to q = 2^k - delta"""
    k = q.bit_length()
    if k < 48 or k > 56:
        return False
    delta = (1 << k) - q
    if delta == 0 or delta >> 28:
        return False
    T = delta << (56 - k)
    if T >> 32 or T >= q:
        return False
    smax, w32 = 0x7fffffff, 0xffffffff
    La = smax * (1 + (1 << 8) + (1 << 16) + (1 << 24))
    Lb, Ha, Hb = smax * (1 + (1 << 8) + (1 << 16)), La, smax * (1 + (1 << 8))
    a, b, e = w32 * T + La, (Ha >> 32) * T + Lb + w32 * T, (Hb >> 32) * T
    if a >> 64 or b >> 64 or e >> 60:
        return False
    h1 = ((a + (b << 32) + (e << 64)) >> k) >> 32
    v, w = w32 * delta + ((1 << k) - 1) + (q - 1), h1 * delta
    if h1 >> 32 or v >> 64 or w >> 62:
        return False
    V = v + (w << 32)
    g = V >> k
    if V >> 96 or g >> 32:
        return False
    return g * delta + ((1 << k) - 1) < 2 * q


def fold128_ok(q):
    """modarith.cuh: fold128_make -- three folds through q = 2^k - delta reduce any 128-bit value"""
    k = q.bit_length()
    if k < 54 or k > 61:
        return False
    delta = (1 << k) - q
    if delta == 0 or delta >> 27:
        return False
    y = ((1 << k) - 1) + (((1 << 128) - 1) >> k) * delta
    V = ((1 << k) - 1) + (y >> k) * delta
    g = V >> k
    if y >> 112 or (y >> k) >> 64 or V >> 96 or g >> 32:
        return False
    return g * delta + ((1 << k) - 1) < 2 * q


# SEAL's default sets, then the other parameter sets of the GPU parity tests (tests/util.py: PARAM_SETS)
HOST_CASES = [pytest.param(n, t, port.DEFAULT_PRIMES_128[n], id="%d-%d" % (n, t))
              for n, t in [(2048, 1 << 16), (4096, 1 << 18), (8192, 1 << 30), (16384, 1 << 30)]]
HOST_CASES += [pytest.param(n, t, primes, id=name) for name, (n, primes, t) in PARAM_SETS.items()]


@pytest.mark.parametrize("n,t,primes", HOST_CASES)
def test_derived_constants_match_oracle(selftest, n, t, primes):
    out = subprocess.check_output([selftest, str(n), str(t)] + [str(p) for p in primes], text=True)
    lines = out.strip().splitlines()
    assert lines[-1] == "OK", out[-400:]
    o = port.Oracle(n, primes, t)
    head = lines[0].split()
    K, S = int(head[1]), int(head[5])
    assert K == len(primes) and S == o.S
    for ln in lines:
        f = ln.split()
        if f[0] == "slot":
            s = int(f[1])
            base, idx = (0, s) if s < K else (1, s - K)
            assert int(f[3]) == o.modulus(base, idx)
            assert int(f[9]) == o.minimal_root(base, idx)
            for col, which in ((11, 0), (13, 1), (15, 2), (17, 3)):
                assert int(f[col]) == fnv(o.ntt_table(base, idx, which)), (s, which)
        if f[0] == "fold":
            # the folded reduction of the limb-split GEMM applies where the prime has the 2^k - delta shape (every SEAL default prime;
            # not the U sets, whose delta is near 2^48); where it does, the selftest has compared tcn_fold_reduce with unsigned __int128
            # on 200000 class-sum vectors per prime before printing OK
            j, q = int(f[1]), int(primes[int(f[1])])
            k = q.bit_length()
            assert int(f[3]) == tcn_fold_ok(q), ln
            if tcn_fold_ok(q):
                assert int(f[7]) == (1 << k) - q and int(f[5]) == ((1 << k) - q) << (56 - k), ln
        if f[0] == "fold128":
            # reduce128_fold applies to the moduli of the 2^k - delta shape (every Bsk prime); checked against __int128 by the selftest
            s = int(f[1])
            q = o.modulus(0, s) if s < K else o.modulus(1, s - K)
            assert int(f[3]) == fold128_ok(q), ln
        if f[0] == "enc":
            want, _ = o.encode(float(f[1]))
            got = np.zeros(n + 1, dtype=np.uint64)
            for pair in f[4:]:
                i, v = pair.split(":")
                got[int(i)] = int(v)
            assert np.array_equal(got, want), f[1]


def test_bad_parameters_are_rejected(selftest):
    # not an NTT prime for n = 4096; plain modulus not below the primes
    for args in (["4096", "1024", "1000003"], ["4096", str(1 << 60), "0x7fffffff380001"], ["3000", "1024", "0x7fffffff380001"]):
        p = subprocess.run([selftest] + args, capture_output=True, text=True)
        assert p.returncode != 0 and "ERROR" in p.stdout


def test_capi_exports_every_declared_symbol():
    from crcnn_b200 import lib
    header = open(os.path.join(ROOT, "include", "crcnn_b200.h")).read()
    declared = set(re.findall(r"\b(crcnn_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 40
    L = lib.load()  # dlopen only; no CUDA call is made
    for name in declared:
        assert hasattr(L, name), name
    assert declared == {s[0] for s in lib.SYMBOLS}


def test_missing_gpu_fails_loudly():
    """On a box without a CUDA device the product refuses to run instead of falling back."""
    import ctypes as C
    from crcnn_b200 import lib
    L = lib.load()
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    q = np.array(port.DEFAULT_PRIMES_128[4096], dtype=np.uint64)
    h = C.c_void_p()
    rc = L.crcnn_ctx_create(4096, 2, q.ctypes.data_as(lib._u64p), 1 << 18, 0, C.byref(h))
    assert rc == -3 and b"no CPU fallback" in L.crcnn_last_error(None)
