"""Generates the committed golden vectors from the UNMODIFIED reference (oracle/_ref: SEAL 2.3.1 +
CrCNN layer classes compiled from /root/reference).  Run in the dev container only:

    python tests/golden/make_golden.py

Every array is produced by the reference: real SEAL keys / encryptions (deterministic RNG factory,
see oracle/ref_harness/ref_api.cpp) and the reference's own layer forwards.  The tests compare the
CPU oracle (tests/test_golden.py, CPU) and the CUDA path (tests/test_gpu_golden.py, GPU) with these
bytes; nothing reads /root/reference at test time.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle.ref import Ref  # noqa: E402


def case_layers(n, t, seed, fname):
    r = Ref(n, t, seed=seed)
    rng = np.random.default_rng(seed)
    img = rng.uniform(-0.4242, 2.8215, size=2 * 3 * 3).astype(np.float32)  # 2 channels of 3x3
    x = r.encrypt(img)
    conv_w = rng.uniform(-1, 1, size=2 * 2 * 2 * 2).astype(np.float32)
    conv_b = rng.uniform(-1, 1, size=2).astype(np.float32)
    fc_w = rng.uniform(-1, 1, size=3 * 8).astype(np.float32)
    fc_b = rng.uniform(-1, 1, size=3).astype(np.float32)
    bn_mean = np.array([0.31, -0.12], dtype=np.float32)
    bn_invstd = np.array([1.7, 0.83], dtype=np.float32)
    evk, sizes, dbc = r.evk()
    conv = r.conv(x, 3, 3, 2, 1, 1, 2, 2, 2, conv_w, conv_b)          # -> 2x2x2
    pool = r.pool(x, 3, 3, 2, 1, 1, 2, 2, avg=False)                   # -> 2x2x2
    avgpool = r.pool(x, 3, 3, 2, 1, 1, 2, 2, avg=True)
    bn = r.bn(conv, 2, 2, 2, bn_mean, bn_invstd)
    sq3 = r.square(conv.reshape(-1, 2, r.K, r.n + 1)[:2])
    relin = r.relinearize(sq3)
    sq_layer = r.square_layer(bn, 2, 2, 2)
    fc = r.fc3d(sq_layer, 2, 2, 2, 3, fc_w, fc_b)
    dec, budget = r.decrypt(fc)
    np.savez_compressed(
        os.path.join(HERE, fname), n=n, t=t, primes=np.array(r.primes, dtype=np.uint64), img=img, x=x,
        conv_w=conv_w, conv_b=conv_b, fc_w=fc_w, fc_b=fc_b, bn_mean=bn_mean, bn_invstd=bn_invstd,
        evk=evk, evk_sizes=np.array(sizes, dtype=np.int32), dbc=dbc,
        conv=conv, pool=pool, avgpool=avgpool, bn=bn, sq3=sq3, relin=relin, sq_layer=sq_layer, fc=fc,
        fc_decrypted=dec, fc_budget=budget,
        # floats, as CnnBuilder passes them to FractionalEncoder::encode(double) (cnnBuilder.cpp:41)
        enc_vals=np.array([0.0867, -3.25, 0.0, 1.0, 2.8215, -0.4242], dtype=np.float32),
        enc_plain=np.stack([r.encode(float(v))[0] for v in np.array([0.0867, -3.25, 0.0, 1.0, 2.8215, -0.4242], dtype=np.float32)]),
        w0_ntt=r.plain_to_ntt(r.encode(float(conv_w[0]))[0]))
    print(fname, "fc decrypts to", dec, "budget", budget)


def case_chain_hashes():
    """Hash-pinned cases at the sizes the benchmark uses: inputs, parameters and keys are regenerated
    from splitmix64 seeds by the tests (tests/util.py); only SHA-256 digests of the reference's
    per-layer output ciphertexts are stored."""
    import json
    sys.path.insert(0, os.path.dirname(HERE))
    import util
    out = {}
    for n, t, seed in [(4096, 1 << 18, 41), (8192, 1 << 30, 83), (16384, 1 << 30, 167)]:
        r = Ref(n, t, seed=seed)
        x = util.det_cts(seed, n, r.primes, 2 * 4 * 4)
        p = util.chain_params(seed)
        evk, sizes, dbc = util.det_evk(seed, n, r.primes)
        r.set_evk(evk, sizes, dbc)  # deterministic key material instead of keygen output
        assert np.array_equal(r.evk()[0], evk)
        outs = util.run_chain(r, "ref", x, p, evk, sizes, dbc)
        out[str(n)] = dict(t=t, seed=seed, primes=[int(q) for q in r.primes], evk_sha=util.sha(evk),
                           layers=[util.sha(o) for o in outs])
        print(n, out[str(n)]["layers"][-1])
    json.dump(out, open(os.path.join(HERE, "chain_hashes.json"), "w"), indent=1)


def case_reference_ops():
    """SHA-256 digests of the reference's output of every evaluator / layer case of tests/test_oracle_vs_reference.py
    (util.ref_ops: inputs regenerated from splitmix64 seeds by the test)."""
    import json
    sys.path.insert(0, os.path.dirname(HERE))
    import util
    out = {}
    for n, (t, seed) in util.REF_OPS.items():
        r = Ref(n, t, seed=seed)
        outs = util.ref_ops("ref", r, n, r.primes, t, seed)
        out[str(n)] = dict(t=t, seed=seed, primes=[int(q) for q in r.primes], digests={k: util.sha(v) for k, v in outs.items()})
    json.dump(out, open(os.path.join(HERE, "reference_ops.json"), "w"), indent=1)


if __name__ == "__main__":
    case_layers(2048, 1 << 10, 7, "layers_n2048.npz")
    case_chain_hashes()
    case_reference_ops()
