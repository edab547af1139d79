"""The lean square (tensor products on the 2^k - delta fold, n^-1 folded into the BEHZ lift / floor constants) against the oracle,
byte for byte, on coefficient- and NTT-form inputs: the extreme-residue ciphertexts, and at n = 8192 and 16384 a batch that spans
more than one scratch chunk of crcnn_square, checked on both sides of the chunk boundary.  The two input forms also agree on the
whole batch."""
import numpy as np
import pytest

from util import PRIMES, T_FOR_N, random_cts, random_evk
from oracle.port import Oracle

pytestmark = pytest.mark.gpu

# n -> ciphertexts: crcnn_square runs chunks of 2 GiB / (5 (K+S) n 8) ciphertexts (728 at n = 8192, 192 at n = 16384)
COUNTS = {4096: 7, 8192: 760, 16384: 200}
CHUNK = {8192: 728, 16384: 192}


@pytest.mark.parametrize("n", sorted(COUNTS))
def test_square_lean_matches_previous_form(n):
    from crcnn_b200.lib import Engine
    primes = PRIMES[n]
    rng = np.random.default_rng(n + 17)
    x = random_cts(rng, n, primes, COUNTS[n])
    for j, q in enumerate(primes):   # extreme residues: every coefficient q - 1, and zero
        x[0, :, j, :n] = q - 1
        x[1, :, j, :n] = 0
    # the extreme ciphertexts, one random one, the last ciphertext of the first chunk, the first of the second, and the last one
    idx = [0, 1, 2] + ([CHUNK[n] - 1, CHUNK[n], COUNTS[n] - 1] if n in CHUNK else [])
    eng = Engine(n, primes, T_FOR_N[n])
    try:
        orc = Oracle(n, primes, T_FOR_N[n])
        want = orc.square(x[idx])
        evk, sizes, dbc = random_evk(rng, n, primes)
        got = []
        for ntt in (False, True):
            t = eng.upload(x)
            if ntt:
                eng.to_ntt(t)
            got.append(eng.download(eng.square(t)))
            assert got[-1].shape[0] == COUNTS[n]
            assert np.array_equal(got[-1][idx], want), ("square differs from the oracle", n, ntt)
        # the two input forms take different lifts (an NTT-form input leaves n^-1 to the lift's constants): same bytes everywhere
        assert np.array_equal(got[0], got[1]), ("coefficient- and NTT-form inputs differ", n)
        del got
        # square + relinearize as one call (crcnn_square_forward), NTT-form input as a convolution leaves it
        t = eng.upload(x[:4])
        eng.to_ntt(t)
        got = eng.download(eng.square_layer(t, eng.evk_upload(evk, sizes, dbc)))
        assert np.array_equal(got, orc.relinearize(orc.square(x[:4]), evk, sizes, dbc))
    finally:
        eng.close()
