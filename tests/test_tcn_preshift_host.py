"""CPU checks behind the pre-shifted limb-split convolution (tcn_mac.cu: tcn2p_mac_kernel): for every coefficient modulus of the
n = 2048 ... 16384 contexts, the byte planes of W' = W 2^(8b) mod q recombine to W', the seven class sums give W X mod q, and
the two-fold reduction of the < 2^80 recombined value (modarith.cuh: tcn7_fold_reduce) equals unsigned __int128 arithmetic,
also for the largest class sums the kernel admits (all-(q-1) operands at fan-in 4096)."""
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
def test_preshift_planes_and_seven_class_reduction(selftest, n):
    primes = PRIMES[n]
    out = subprocess.check_output([selftest, str(n), str(T_FOR_N[n])] + [str(p) for p in primes], text=True)
    lines = out.strip().splitlines()
    assert lines[-1] == "OK", out[-400:]
    rows = [ln.split() for ln in lines if ln.startswith("fold7 ")]
    assert [int(f[1]) for f in rows] == list(range(len(primes)))
    assert all(f[3] == "1" for f in rows), "the seven-class fold does not admit every prime of the context"
    assert all(int(f[5]) == 22000 for f in rows)
