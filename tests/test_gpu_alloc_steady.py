"""GPU: a repeated step gives back every device block of 32 MB or more that it takes (DESIGN 3; crcnn_ctx_alloc_stats in
include/crcnn_b200.h).

PlainModel at n = 8192 through the C++ host library (HostNetwork, viewed through Engine.adopt for the allocator counters): its
activations are hundreds of MB, so every one of them goes through the context's exact-size cache.  After a warm-up with layer fusion
off and on, further identical steps -- resident forwards and the serving loop -- must be served from that cache alone: no new pool
allocation, no block that bypasses the cache, no flush, and as many cached bytes after the steps as before them."""
import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu

MODEL, N, BATCH = "PlainModel", 8192, 1


def test_repeated_steps_return_every_large_block():
    from crcnn_b200 import host
    from crcnn_b200.lib import Engine
    primes, t = util.PRIMES[N], util.T_FOR_N[N]
    rng = np.random.default_rng(32)
    net = host.HostNetwork(N, primes, t, MODEL, evk=util.random_evk(rng, N, primes))
    eng = Engine.adopt(net.ctx(), N, primes, t)
    try:
        count = BATCH * net.zd * net.xd * net.yd
        assert count * net.ct_words() * 8 >= 32 << 20
        pin, own_in = host.pinned_array(count * net.ct_words())
        _, own_out = host.pinned_array(BATCH * net.outputs * net.ct_words())
        pin[:] = util.random_cts(rng, N, primes, count).ravel()

        def step():
            net.resident_steps(own_in.ptr, BATCH, 0, 2)
            net.serve(own_in.ptr, own_out.ptr, BATCH, 2)

        for fused in (False, True):
            net.set_fusion(fused)
            step()
        before = eng.alloc_stats()
        step()
        step()
        after = eng.alloc_stats()
        for key in ("pool_mallocs", "cache_bypass", "flushes", "cached_bytes"):
            assert after[key] == before[key], (key, before, after)
        assert after["cache_hits"] > before["cache_hits"], (before, after)
    finally:
        eng.h = None          # the context belongs to the host library
        net.close()
