"""CRT plaintext-modulus ensembles on the B200 (BASELINE config 4): a plain modulus T split into pairwise coprime t_1 .. t_M, one
instance per modulus, recombined on the device (crcnn_crt_*).

- the compose-and-decode kernel (crcnn_crt_decode_values) is bit-equal to the Python restatement of test_crt_decode_oracle.py;
- M contexts in one process, each with its own keys, run a chain; their decryptions recombined on the device give exactly the
  floats of one context under T running the same chain;
- CrtEnsemble::predict (collective re-encryption before layer 6, collective decryption) gives on every rank the floats of a
  single Network::predict under T: with one rank on one GPU, and with 2 and 3 ranks where the box has the GPUs;
- bad lists, mismatched ranks and the budget-driven policy are refused on every rank, without a hang."""
import os
import sys
import time

import numpy as np
import pytest
# torch before any NCCL call of the library: crcnn_b200 dlopens libnccl.so.2 and takes the copy already mapped, so torch's own NCCL
# must be the one in the process -- a system NCCL mapped first would break the later import of torch (multi-GPU tests below)
import torch  # noqa: F401

import util
import fv_keygen as kg
from oracle.port import DEFAULT_PRIMES_128 as PRIMES, Oracle
from test_crt_decode_oracle import LISTS, SLOTS, cases, crt_decode, product

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


# ---- one GPU: the kernel
@pytest.mark.parametrize("moduli", LISTS, ids=lambda ms: "M%d_T%d" % (len(ms), product(ms)))
def test_decode_values_equals_the_restatement(moduli):
    from crcnn_b200.lib import Engine
    n = 8192
    eng = Engine(n, PRIMES[n], 1 << 30)
    rng = np.random.default_rng(product(moduli) % 1000003)
    rows = cases(moduli, rng)
    plains = []
    for m in moduli:
        p = rng.integers(0, m, size=(len(rows), n + 1), dtype=np.uint64)     # coefficients the decoder never reads: anything below t
        p[:, n] = 0
        p[:, SLOTS] = np.array([[v % m for v in row] for row in rows], dtype=np.uint64)
        plains.append(p)
    got = eng.crt_decode_values(moduli, plains)
    want = np.array([crt_decode([[v % m for v in row] for m in moduli], moduli) for row in rows], dtype=np.float32)
    assert np.array_equal(_bits(got), _bits(want))
    eng.close()


@pytest.mark.parametrize("T", [1 << 30, LISTS[5][0]])
def test_one_modulus_equals_decrypt_values(T):
    from crcnn_b200.lib import Engine
    n = 8192
    orc = Oracle(n, PRIMES[n], T)
    keys = kg.generate(orc, 3)
    eng = Engine(n, PRIMES[n], T)
    dk = eng.keys_upload(keys.sk, keys.pk)
    vals = np.concatenate([np.array([0.0, -1.0, 0.5, 1.0 / 3.0, -7.25, 2.8215, 9.0e18, -9.2e18], dtype=np.float32),
                           np.random.default_rng(1).uniform(-1e4, 1e4, 60).astype(np.float32)])
    ct = eng.encrypt_values(dk, vals, seed=5)
    want = eng.decrypt_values(dk, ct)
    got = eng.crt_decode_values([T], [eng.decrypt(dk, ct)])
    assert np.array_equal(_bits(got), _bits(want))
    del dk
    eng.close()


def test_decode_values_refusals():
    from crcnn_b200.lib import Engine, CrcnnError
    n = 8192
    eng = Engine(n, PRIMES[n], 1 << 30)
    p = np.zeros((1, n + 1), dtype=np.uint64)
    for moduli in ([6, 15], [2, 3, 4], [1], [1 << 27, (1 << 27) + 1], [min(PRIMES[n])]):
        with pytest.raises(CrcnnError) as e:
            eng.crt_decode_values(moduli, [p] * len(moduli))
        assert e.value.code == -1, moduli
    bad = p.copy()
    bad[0, 3] = 32771
    with pytest.raises(CrcnnError):
        eng.crt_decode_values([32771, 32779], [bad, p])
    eng.close()


# ---- one GPU: chains in M contexts, recombined, against one context under T
def _run_chain(eng, dk, evk, chain, img, wts):
    x = eng.encrypt_values(dk, img, seed=17)
    if chain == "conv_square":
        g = eng.conv(x, eng.plain_encode(wts[0]), eng.plain_encode(wts[1]), 1, 4, 4, 1, 1, 1, 2, 2, 2)
        return eng.square_layer(g, evk)
    g = eng.conv(x, eng.plain_encode(wts[0]), eng.plain_encode(wts[1]), 1, 6, 6, 1, 1, 1, 3, 3, 2)      # 2 x 4 x 4
    g = eng.pool(g, 1, 4, 4, 2, 2, 2, 2, 2, scale=eng.plain_encode_f64([0.25]))                        # 2 x 2 x 2
    g = eng.square_layer(g, evk)
    return eng.fc(g, eng.plain_encode(wts[2]), eng.plain_encode(wts[3]), 1, 8, 3)


@pytest.mark.parametrize("chain,n,moduli", [("conv_square", 8192, [32771, 32779]), ("conv_pool_square_fc", 4096, [509, 521]),
                                            ("conv_pool_square_fc", 4096, [61, 67, 71])])
def test_instances_recombine_to_the_single_modulus_run(chain, n, moduli):
    from crcnn_b200.lib import Engine
    rng = np.random.default_rng(len(moduli) * n)
    img = rng.uniform(-0.4242, 2.8215, size=16 if chain == "conv_square" else 36).astype(np.float32)
    f = lambda k: rng.uniform(-1, 1, size=k).astype(np.float32)
    wts = [f(8), f(2)] if chain == "conv_square" else [f(18), f(2), f(24), f(3)]
    plains = []
    for i, t in enumerate(moduli):
        keys = kg.generate(Oracle(n, PRIMES[n], t), 40 + i)          # each instance its own keys
        eng = Engine(n, PRIMES[n], t)
        dk = eng.keys_upload(keys.sk, keys.pk)
        out = _run_chain(eng, dk, eng.evk_upload(*keys.evk_triple), chain, img, wts)
        assert eng.min_noise_budget(dk, out) > 0
        plains.append(eng.decrypt(dk, out))
        del dk
        eng.close()
    T = product(moduli)
    keys = kg.generate(Oracle(n, PRIMES[n], T), 60)
    eng = Engine(n, PRIMES[n], T)
    dk = eng.keys_upload(keys.sk, keys.pk)
    out = _run_chain(eng, dk, eng.evk_upload(*keys.evk_triple), chain, img, wts)
    assert eng.min_noise_budget(dk, out) > 0
    want = eng.decrypt_values(dk, out)
    got = eng.crt_decode_values(moduli, plains)
    assert np.array_equal(_bits(got), _bits(want))
    del dk
    eng.close()


# ---- CrtEnsemble through the host library
MODEL_N = {"ApproxPlainModel": 8192, "PlainModelTiny": 4096}


def _keys(n, t, seed):
    return kg.generate(Oracle(n, PRIMES[n], t), seed)


def _images(net, batch):
    return np.stack([util.synthetic_image(s, net.zd * net.xd * net.yd) for s in range(batch)])


def _single_predict(model, moduli, batch, fusion):
    """Network::predict under T = prod(moduli) with use_device_reencryption, on one GPU"""
    from crcnn_b200.host import HostNetwork
    n, T = MODEL_N[model], product(moduli)
    keys = _keys(n, T, 70)
    net = HostNetwork(n, PRIMES[n], T, model, evk=keys.evk_triple, skip_reencryption=False)
    try:
        net.set_fusion(fusion)
        net.use_keys(keys.sk, keys.pk, device_reencryption=True, seed=901)
        return net.predict_values(_images(net, batch), batch=batch, seed=77)
    finally:
        net.close()


def _ensemble_predict(model, moduli, rank, nccl_id, batch, fusion, device=0, key_seed=None):
    """CrtEnsemble::predict on this rank (its own keys unless key_seed is given); two calls, which must agree"""
    from crcnn_b200.host import HostNetwork
    n = MODEL_N[model]
    keys = _keys(n, moduli[rank], 80 + rank if key_seed is None else key_seed)
    net = HostNetwork(n, PRIMES[n], moduli[rank], model, device=device, evk=keys.evk_triple, skip_reencryption=False)
    try:
        net.set_fusion(fusion)
        net.use_keys(keys.sk, keys.pk)
        net.crt_begin(moduli, rank, nccl_id, reencrypt_seed=123)
        imgs = _images(net, batch)
        got = net.crt_predict_values(imgs, batch=batch, seed=77)
        again = net.crt_predict_values(imgs, batch=batch, seed=78)
        assert np.array_equal(_bits(got), _bits(again))
        return got
    finally:
        net.close()


@pytest.mark.parametrize("model,t,batch,fusion", [("ApproxPlainModel", 1 << 30, 1, True), ("ApproxPlainModel", 1 << 30, 3, False),
                                                  ("PlainModelTiny", 1 << 18, 2, True)])
def test_one_rank_ensemble_equals_predict(model, t, batch, fusion):
    from crcnn_b200.host import nccl_unique_id
    got = _ensemble_predict(model, [t], 0, nccl_unique_id(), batch, fusion)
    want = _single_predict(model, [t], batch, fusion)
    assert got.shape == want.shape
    assert np.array_equal(_bits(got), _bits(want))


def test_one_rank_refusals():
    from crcnn_b200.host import HostNetwork, HostError, nccl_unique_id
    n, t = 4096, 1 << 18
    keys = _keys(n, t, 5)
    net = HostNetwork(n, PRIMES[n], t, "PlainModelTiny", evk=keys.evk_triple, skip_reencryption=False)
    try:
        with pytest.raises(HostError, match="use_device_keys"):
            net.crt_begin([t], 0, nccl_unique_id(), 1)
        net.use_keys(keys.sk, keys.pk)
        for moduli, what in (([t + 1], "moduli\\[rank\\]"), ([3 << 60], "coefficient prime")):
            with pytest.raises(HostError, match=what) as e:
                net.crt_begin(moduli, 0, nccl_unique_id(), 1)
            assert "error -1" in str(e.value)
        net.set_budget_threshold(10)
        with pytest.raises(HostError, match="budget-driven"):
            net.crt_begin([t], 0, nccl_unique_id(), 1)
        net.set_budget_threshold(-1)
        net.crt_begin([t], 0, nccl_unique_id(), 1)
        net.set_budget_threshold(10)
        with pytest.raises(HostError, match="budget-driven"):
            net.crt_predict_values(_images(net, 1), batch=1, seed=3)
    finally:
        net.close()


def test_create_refuses_a_list_that_does_not_match_the_world():
    """crcnn_crt_create on a one-rank communicator: a list of two moduli is refused.  (The host library sizes its communicator from
    the list, so this mismatch can only be made through the C ABI.)"""
    import ctypes as C
    from crcnn_b200 import lib
    from crcnn_b200.host import nccl_unique_id
    n, t = 4096, 1 << 18
    eng = lib.Engine(n, PRIMES[n], t)
    comm = C.c_void_p()
    idbuf = (C.c_char * 128).from_buffer_copy(nccl_unique_id())
    eng._chk(eng.lib.crcnn_comm_create(eng.h, C.cast(idbuf, C.c_void_p), 1, 0, C.byref(comm)))
    try:
        with pytest.raises(lib.CrcnnError, match="one plain modulus per rank") as e:
            eng.crt_create(comm.value, [t, 3])
        assert e.value.code == -1
        eng.crt_create(comm.value, [t]).free()
    finally:
        eng.lib.crcnn_comm_destroy(eng.h, comm)
        eng.close()


# ---- 2 and 3 GPUs, one process per rank
def _shared_id(out_dir, rank, tag):
    from crcnn_b200.host import nccl_unique_id
    path = os.path.join(out_dir, "nccl_id_" + tag)
    if rank == 0:
        open(path + ".tmp", "wb").write(nccl_unique_id())
        os.rename(path + ".tmp", path)
    while not os.path.exists(path):
        time.sleep(0.05)
    return open(path, "rb").read()


def _worker(rank, world, out_dir, moduli):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from crcnn_b200.host import HostNetwork, HostError
    runs = {}
    for model, batch, fusion in (("ApproxPlainModel", 1, True), ("ApproxPlainModel", 3, True), ("ApproxPlainModel", 3, False),
                                 ("PlainModelTiny", 2, True)):
        tag = "%s_%d_%d" % (model, batch, fusion)
        runs[tag] = _ensemble_predict(model, moduli, rank, _shared_id(out_dir, rank, tag), batch, fusion, device=rank)
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **runs)
    # refusals: every rank must raise, none may hang
    n = 4096
    keys = _keys(n, moduli[rank], 90)
    net = HostNetwork(n, PRIMES[n], moduli[rank], "PlainModelTiny", device=rank, evk=keys.evk_triple, skip_reencryption=False)
    net.use_keys(keys.sk, keys.pk)
    other = [m for m in moduli]
    other[0] = moduli[0] + 2 if rank == 1 else moduli[0]        # rank 1 passes another list that is valid on its own
    one_bad = list(moduli) if rank != 1 else [moduli[1]] + list(moduli[1:])   # rank 1 alone refuses (non-coprime)
    cases_ = {"non_coprime": [moduli[0]] * world, "too_large": [m << 40 for m in moduli],
              "t_mismatch": list(moduli[1:]) + [moduli[0]], "one_rank_refuses": one_bad, "different_lists": other}
    refused = {}
    for tag, ms in cases_.items():
        try:
            net.crt_begin(ms, rank, _shared_id(out_dir, rank, "refuse_" + tag), 1)
            refused[tag] = "accepted"
        except HostError as e:
            refused[tag] = str(e)
    net.crt_begin(moduli, rank, _shared_id(out_dir, rank, "refuse_ok"), 1)
    net.set_budget_threshold(5)
    try:
        net.crt_predict_values(_images(net, 1), batch=1, seed=1)
        refused["budget"] = "accepted"
    except HostError as e:
        refused["budget"] = str(e)
    net.close()
    with open(os.path.join(out_dir, "refused%d.txt" % rank), "w") as f:
        for k, v in refused.items():
            f.write("%s\t%s\n" % (k, v.replace("\n", " ")))


@pytest.mark.parametrize("world,moduli", [(2, [32771, 32779]), (3, [1021, 1031, 1033])])
def test_ensemble_predict_matches_single_gpu(tmp_path, world, moduli):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    import torch.multiprocessing as mp
    procs = mp.start_processes(_worker, args=(world, str(tmp_path), moduli), nprocs=world, join=False, start_method="spawn")
    deadline = time.monotonic() + 900        # a collective that never completes fails the test instead of stalling the suite
    while not procs.join(timeout=5):
        if time.monotonic() > deadline:
            for p in procs.processes:
                p.kill()
            for p in procs.processes:
                p.join()
            pytest.fail("the ranks did not finish within 900 s")
    for model, batch, fusion in (("ApproxPlainModel", 1, True), ("ApproxPlainModel", 3, True), ("ApproxPlainModel", 3, False),
                                 ("PlainModelTiny", 2, True)):
        tag = "%s_%d_%d" % (model, batch, fusion)
        want = _single_predict(model, moduli, batch, fusion)
        for r in range(world):
            got = np.load(tmp_path / ("rank%d.npz" % r))[tag]
            assert np.array_equal(_bits(got), _bits(want)), "rank %d, %s: ensemble scores differ from the single-modulus run" % (r, tag)
            assert np.array_equal(got.argmax(axis=1), want.argmax(axis=1))
    for r in range(world):
        lines = dict(l.rstrip("\n").split("\t", 1) for l in open(tmp_path / ("refused%d.txt" % r)))
        for tag in ("non_coprime", "too_large", "t_mismatch", "one_rank_refuses", "different_lists"):
            assert "error -1" in lines[tag], (r, tag, lines[tag])
        assert "budget-driven" in lines["budget"], (r, lines["budget"])
