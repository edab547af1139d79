"""The lean square (CRCNN_SQ_LEAN=1, default: tensor products on the 2^k - delta fold, n^-1 folded into the BEHZ lift / floor
constants) against the previous formulation (CRCNN_SQ_LEAN=0), byte for byte, on coefficient- and NTT-form inputs; at n = 8192
and 16384 the batch spans more than one scratch chunk of crcnn_square.  One chunk of each is also checked against the oracle."""
import os

import numpy as np
import pytest

from util import PRIMES, T_FOR_N, random_cts, random_evk
from oracle.port import Oracle

pytestmark = pytest.mark.gpu

# n -> ciphertexts: crcnn_square runs chunks of 2 GiB / (5 (K+S) n 8) ciphertexts (728 at n = 8192, 192 at n = 16384)
COUNTS = {4096: 7, 8192: 760, 16384: 200}


def _engine(n, lean):
    from crcnn_b200.lib import Engine
    old = os.environ.get("CRCNN_SQ_LEAN")
    os.environ["CRCNN_SQ_LEAN"] = str(lean)   # read when the context is created
    try:
        return Engine(n, PRIMES[n], T_FOR_N[n])
    finally:
        if old is None:
            os.environ.pop("CRCNN_SQ_LEAN", None)
        else:
            os.environ["CRCNN_SQ_LEAN"] = old


@pytest.mark.parametrize("n", sorted(COUNTS))
def test_square_lean_matches_previous_form(n):
    primes = PRIMES[n]
    rng = np.random.default_rng(n + 17)
    x = random_cts(rng, n, primes, COUNTS[n])
    for j, q in enumerate(primes):   # extreme residues: every coefficient q - 1, and zero
        x[0, :, j, :n] = q - 1
        x[1, :, j, :n] = 0
    lean, old = _engine(n, 1), _engine(n, 0)
    try:
        orc = Oracle(n, primes, T_FOR_N[n])
        want3 = orc.square(x[:3])
        evk, sizes, dbc = random_evk(rng, n, primes)
        for ntt in (False, True):
            got = []
            for eng in (lean, old):
                t = eng.upload(x)
                if ntt:
                    eng.to_ntt(t)
                got.append(eng.download(eng.square(t)))
            assert np.array_equal(got[0], got[1]), ("lean and previous square differ", n, ntt)
            assert np.array_equal(got[0][:3], want3), ("square differs from the oracle", n, ntt)
            del got
        # square + relinearize as one call (crcnn_square_forward), NTT-form input as a convolution leaves it
        outs = []
        for eng in (lean, old):
            t = eng.upload(x[:4])
            eng.to_ntt(t)
            outs.append(eng.download(eng.square_layer(t, eng.evk_upload(evk, sizes, dbc))))
        assert np.array_equal(outs[0], outs[1])
        assert np.array_equal(outs[0], orc.relinearize(orc.square(x[:4]), evk, sizes, dbc))
    finally:
        lean.close()
        old.close()
