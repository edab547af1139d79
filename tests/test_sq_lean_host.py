"""CPU checks behind the lean square: the n^-1-scaled lift / floor constants (params.h: mt_inv_qhat_n, fl_c, fl_T) against their
definitions and the transforms' approximate Shoup product on edge operands, for every modulus of the n = 2048 ... 16384 contexts.
host_selftest compares both with unsigned __int128 and prints one line per modulus."""
import os
import subprocess

import pytest

from util import PRIMES, T_FOR_N, ROOT

SELFTEST = os.path.join(ROOT, "build", "host_selftest")


@pytest.fixture(scope="module")
def selftest():
    if not os.path.exists(SELFTEST):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "crcnn_b200", "csrc"), "host_selftest"])
    return SELFTEST


@pytest.mark.parametrize("n", [2048, 4096, 8192, 16384])
def test_ninv_constants_and_lazy_shoup(selftest, n):
    primes = PRIMES[n]
    out = subprocess.check_output([selftest, str(n), str(T_FOR_N[n])] + [str(p) for p in primes], text=True)
    lines = out.strip().splitlines()
    assert lines[-1] == "OK", out[-400:]
    K, S = int(lines[0].split()[1]), int(lines[0].split()[5])
    ninv = [ln.split() for ln in lines if ln.startswith("ninv ")]
    shoup = [ln.split() for ln in lines if ln.startswith("shoup4 ")]
    assert [int(f[1]) for f in ninv] == list(range(K + S)) and all(f[3] == "1" for f in ninv)
    assert [int(f[1]) for f in shoup] == list(range(K + S)) and all(int(f[3]) >= 100000 for f in shoup)
