"""Zero-padded convolutions (crcnn_conv_forward_padded, crcnn_conv_pool_bn_forward_padded, ConvolutionalLayer's padding, the
"PlainModelPadded" topology) against the same layers on the input with a border of all-zero ciphertexts, byte for byte.

An all-zero ciphertext times any plaintext is zero, so the padded layer must give exactly the bytes the unpadded layer gives on X'
(X with the border): for every weighted-sum kernel (the index entry -1 each of their gathers reads), on the pooled grid (window sums
over the padded extent, all-padding windows included) and its fallback, for channel shards, and through the whole network built by
CnnBuilder.  The kernel-class counters show that the padded call ran the same kernels as the bordered one."""
import os
import time

import numpy as np
import pytest

import fv_keygen as kg
import util
from util import PRIMES, T_FOR_N, random_cts
from oracle.port import Oracle

pytestmark = pytest.mark.gpu

WEIGHTED = ("weighted_sum_mac", "weighted_sum_tcn_i8", "weighted_sum_tc_i8")


def border(x, batch, zd, xd, yd, xp, yp):
    """X' : X ([batch * zd * xd * yd][2][K][n+1]) with xp columns and yp rows of all-zero ciphertexts on each side."""
    a = x.reshape(batch, zd, xd, yd, *x.shape[1:])
    a = np.pad(a, [(0, 0), (0, 0), (xp, xp), (yp, yp)] + [(0, 0)] * (x.ndim - 1))
    return a.reshape(-1, *x.shape[1:])


@pytest.fixture(scope="module", params=[2048, 4096])
def env(request):
    from crcnn_b200.lib import Engine
    n = request.param
    eng = Engine(n, PRIMES[n], T_FOR_N[n])
    eng.prof_enable(True)
    yield n, eng, np.random.default_rng(90 + n)
    eng.close()


def _weighted_launches(eng):
    p = eng.prof()
    return {c: p.get(c, (0, 0.0))[0] for c in WEIGHTED}


def _run(eng, fn):
    """(output bytes, weighted-sum launches by class) of one call."""
    eng.prof_reset()
    out = eng.download(fn())
    return out, _weighted_launches(eng)


# kernel: (engine settings, weight range, [(zd, xd, yd, xs, ys, xf, yf, nf, xp, yp)])
KERNELS = {
    # fan-in <= 32: pre-shifted weights, seven-class limb-split kernel
    "tcn2p": (dict(tc=0, tcn=1), 3.0, [(1, 7, 6, 1, 1, 5, 5, 4, 2, 1), (1, 9, 8, 2, 2, 5, 5, 3, 4, 3)]),
    # the 13-class limb-split kernel: 20 channels, 3x3, padding 1
    "tcn2": (dict(tc=0, tcn=1), 3.0, [(20, 4, 5, 1, 1, 3, 3, 4, 1, 2), (20, 5, 4, 2, 2, 3, 3, 3, 2, 1)]),
    # the row-major / column-major limb-split kernels
    "tcn_mac2": (dict(tc=0, tcn=2), 3.0, [(3, 5, 6, 1, 1, 3, 3, 5, 2, 1), (2, 6, 5, 2, 2, 3, 3, 4, 1, 2)]),
    "tcn_mac3": (dict(tc=0, tcn=3), 3.0, [(3, 5, 6, 1, 1, 3, 3, 5, 2, 1), (2, 6, 5, 2, 2, 3, 3, 4, 1, 2)]),
    # ternary-tap GEMM: fan-in >= 256, >= 32 outputs, weights |w| < 1/2
    "tc_mac": (dict(tc=1, tcn=1), 0.49, [(32, 4, 3, 1, 1, 3, 3, 32, 2, 1), (32, 5, 4, 2, 2, 3, 3, 32, 1, 2)]),
    # CUDA-core NTT-domain MAC
    "mac": (dict(tc=0, tcn=0), 3.0, [(2, 5, 6, 1, 1, 3, 3, 3, 2, 1), (2, 6, 5, 2, 2, 3, 3, 2, 1, 2)]),
}
EXPECT_CLASS = {"tcn2p": "weighted_sum_tcn_i8", "tcn2": "weighted_sum_tcn_i8", "tcn_mac2": "weighted_sum_tcn_i8",
                "tcn_mac3": "weighted_sum_tcn_i8", "tc_mac": "weighted_sum_tc_i8", "mac": "weighted_sum_mac"}


@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("batch", [1, 2])
def test_padded_conv_equals_conv_on_bordered_input(env, kernel, batch):
    n, eng, rng = env
    modes, wmax, shapes = KERNELS[kernel]
    eng.set_tensor_core_mode(modes["tc"])
    eng.set_limb_split_mode(modes["tcn"])
    try:
        for zd, xd, yd, xs, ys, xf, yf, nf, xp, yp in shapes:
            R = zd * xf * yf
            w = eng.plain_encode(rng.uniform(-wmax, wmax, nf * R).astype(np.float32))
            b = eng.plain_encode(rng.uniform(-wmax, wmax, nf).astype(np.float32))
            x = random_cts(rng, n, PRIMES[n], batch * zd * xd * yd)
            xb = border(x, batch, zd, xd, yd, xp, yp)
            for ntt in (False, True):
                def upload(a):
                    t = eng.upload(a)
                    if ntt:
                        eng.to_ntt(t)
                    return t
                geo = (zd, xs, ys, xf, yf, nf)
                want, wl = _run(eng, lambda: eng.conv(upload(xb), w, b, batch, xd + 2 * xp, yd + 2 * yp, *geo))
                got, gl = _run(eng, lambda: eng.conv(upload(x), w, b, batch, xd, yd, *geo, xp=xp, yp=yp))
                where = (kernel, n, batch, ntt, (zd, xd, yd, xs, ys, xf, yf, nf, xp, yp))
                assert got.shape == want.shape and np.array_equal(got, want), where
                assert gl == wl and wl[EXPECT_CLASS[kernel]] > 0, (where, gl, wl)
            # a shard of the output channels is the matching slice of the whole layer
            k0, kc = 1, nf - 1
            part = eng.download(eng.conv(eng.upload(x), w, b, batch, xd, yd, *geo, xp=xp, yp=yp, shard=(k0, kc)))
            xo, yo = (xd + 2 * xp - xf) // xs + 1, (yd + 2 * yp - yf) // ys + 1
            whole = got.reshape(batch, nf, xo * yo, *got.shape[1:])[:, k0:k0 + kc].reshape(part.shape)
            assert np.array_equal(part, whole), where
    finally:
        eng.set_tensor_core_mode(1)
        eng.set_limb_split_mode(1)


def test_padded_conv_against_the_oracle(env):
    """Independent witness: the oracle's ConvolutionalLayer::forward on X' (n = 2048)."""
    n, eng, rng = env
    if n != 2048:
        pytest.skip("oracle witness at n = 2048")
    orc = Oracle(n, PRIMES[n], T_FOR_N[n])
    for zd, xd, yd, xs, ys, xf, yf, nf, xp, yp in [(1, 6, 5, 2, 2, 5, 5, 2, 2, 1), (2, 4, 4, 1, 1, 3, 3, 2, 2, 1), (3, 5, 4, 1, 1, 2, 3, 2, 1, 2)]:
        wv, bv = rng.uniform(-2, 2, nf * zd * xf * yf).astype(np.float32), rng.uniform(-2, 2, nf).astype(np.float32)
        x = random_cts(rng, n, PRIMES[n], zd * xd * yd)
        want = orc.conv(border(x, 1, zd, xd, yd, xp, yp), xd + 2 * xp, yd + 2 * yp, zd, xs, ys, xf, yf, nf, orc.encode_many(wv), orc.encode_many(bv))
        got = eng.download(eng.conv(eng.upload(x), eng.plain_encode(wv), eng.plain_encode(bv), 1, xd, yd, zd, xs, ys, xf, yf, nf, xp=xp, yp=yp))
        assert np.array_equal(got.reshape(want.shape), want), (zd, xd, yd, xs, ys, xf, yf, nf, xp, yp)


def _work(eng, n):
    unit = 2.0 * len(PRIMES[n]) * n
    launches = {k: v[0] for k, v in eng.prof().items()}
    ops = {k: v[1] for k, v in eng.prof_work().items()}
    terms = ops.get("weighted_sum_mac", 0) / unit + ops.get("weighted_sum_tcn_i8", 0) / (49 * unit)
    return launches.get("pool_sum", 0), terms, ops.get("pool_sum", 0) / unit


# (zd, xd, yd, xs, ys, xf, yf, nf, pxs, pys, pxf, pyf, xp, yp): the PlainModel block in small, and a stride-1 convolution whose window
# sums S reach two rows / columns into the border (all-padding windows of S)
POOLED = [(1, 8, 8, 2, 2, 5, 5, 4, 1, 1, 2, 2, 2, 2), (2, 5, 6, 1, 1, 3, 3, 3, 1, 1, 2, 2, 2, 1), (2, 6, 5, 1, 1, 3, 3, 4, 2, 2, 2, 2, 1, 2)]


@pytest.mark.parametrize("geo", POOLED)
def test_padded_conv_pool_bn_on_the_pooled_grid(env, geo):
    n, eng, rng = env
    zd, xd, yd, xs, ys, xf, yf, nf, pxs, pys, pxf, pyf, xp, yp = geo
    batch, R = 2, zd * xf * yf
    w = eng.plain_encode(rng.uniform(-2, 2, nf * R).astype(np.float32))
    b = eng.plain_encode(rng.uniform(-2, 2, nf).astype(np.float32))
    packs = (eng.plain_encode_f64([1.0 / (pxf * pyf)]), eng.plain_encode(rng.uniform(-1, 1, nf).astype(np.float32)),
             eng.plain_encode(rng.uniform(0.5, 2, nf).astype(np.float32)))
    x = random_cts(rng, n, PRIMES[n], batch * zd * xd * yd)
    xb = border(x, batch, zd, xd, yd, xp, yp)
    cxo, cyo = (xd + 2 * xp - xf) // xs + 1, (yd + 2 * yp - yf) // ys + 1
    pxo, pyo = (cxo - pxf) // pxs + 1, (cyo - pyf) // pys + 1
    pool = (pxs, pys, pxf, pyf)
    eng.prof_reset()
    got = eng.download(eng.conv_pool_bn(eng.upload(x), w, b, batch, xd, yd, zd, xs, ys, xf, yf, nf, *pool, *packs, xp=xp, yp=yp))
    launches, terms, sums = _work(eng, n)
    # the pooled grid ran: window sums over the padded extent, weighted-sum terms at the pooled positions only
    sxd, syd = xd + 2 * xp - (pxf - 1) * xs, yd + 2 * yp - (pyf - 1) * ys
    assert launches >= 1 and sums == batch * zd * sxd * syd * pxf * pyf, (launches, sums)
    assert terms == batch * nf * pxo * pyo * R, terms
    want = eng.download(eng.conv_pool_bn(eng.upload(xb), w, b, batch, xd + 2 * xp, yd + 2 * yp, zd, xs, ys, xf, yf, nf, *pool, *packs))
    assert got.shape == want.shape and np.array_equal(got, want), geo
    os.environ["CRCNN_NO_POOLED_CONV"] = "1"
    try:
        eng.prof_reset()
        fb = eng.download(eng.conv_pool_bn(eng.upload(x), w, b, batch, xd, yd, zd, xs, ys, xf, yf, nf, *pool, *packs, xp=xp, yp=yp))
        assert _work(eng, n)[1] == batch * nf * cxo * cyo * R       # the layer-by-layer fallback: every convolution position
    finally:
        del os.environ["CRCNN_NO_POOLED_CONV"]
    assert np.array_equal(fb, want), geo
    for k0, kc in [(0, 1), (1, nf - 1), (nf - 1, 1)]:
        part = eng.download(eng.conv_pool_bn(eng.upload(x), w, b, batch, xd, yd, zd, xs, ys, xf, yf, nf, *pool, *packs, shard=(k0, kc), xp=xp, yp=yp))
        whole = got.reshape(batch, nf, pxo * pyo, *got.shape[1:])[:, k0:k0 + kc].reshape(part.shape)
        assert np.array_equal(part, whole), (geo, k0, kc)


def test_bad_padding_is_refused_and_the_context_stays_usable(env):
    from crcnn_b200.lib import CrcnnError
    n, eng, rng = env
    w, b = eng.plain_encode(rng.uniform(-1, 1, 2 * 9).astype(np.float32)), eng.plain_encode([0.5, -0.5])
    x = eng.upload(random_cts(rng, n, PRIMES[n], 16))
    packs = (None, eng.plain_encode([0.1, 0.2]), eng.plain_encode([1.0, 1.5]))
    for xp, yp in [(-1, 0), (0, -1), (3, 0), (0, 3), (5, 5)]:
        with pytest.raises(CrcnnError) as e:
            eng.conv(x, w, b, 1, 4, 4, 1, 1, 1, 3, 3, 2, xp=xp, yp=yp)
        assert e.value.code == -1, (xp, yp)
        with pytest.raises(CrcnnError) as e:
            eng.conv_pool_bn(x, w, b, 1, 4, 4, 1, 1, 1, 3, 3, 2, 1, 1, 2, 2, *packs, xp=xp, yp=yp)
        assert e.value.code == -1, (xp, yp)
    ok = eng.download(eng.conv(x, w, b, 1, 4, 4, 1, 1, 1, 3, 3, 2, xp=2, yp=2))
    assert ok.shape[0] == 2 * 6 * 6


# ---- the network built by CnnBuilder: "PlainModelPadded" on 28x28 against "PlainModel" on the 32x32 zero-bordered input
N8 = 8192


def _forwards(model, x, batch, shape):
    """{(last, fused): output} of forward(0, last) for every last, with layer fusion on and off, through the host library."""
    from crcnn_b200.host import HostNetwork
    rng = np.random.default_rng(5)
    net = HostNetwork(N8, PRIMES[N8], T_FOR_N[N8], model, evk=util.random_evk(rng, N8, PRIMES[N8]))
    out = {}
    try:
        assert (net.zd, net.xd, net.yd) == shape
        for fused in (True, False):
            net.set_fusion(fused)
            for last in range(1, net.num_layers + 1):
                out[(last, fused)] = net.forward(x, batch=batch, first=0, last=last)
    finally:
        net.close()
    return out


def test_plain_model_padded_equals_plain_model_on_the_bordered_input():
    rng = np.random.default_rng(6)
    x = random_cts(rng, N8, PRIMES[N8], 28 * 28)
    got = _forwards("PlainModelPadded", x, 1, (1, 28, 28))
    want = _forwards("PlainModel", border(x, 1, 1, 28, 28, 2, 2), 1, (1, 32, 32))
    for key in want:
        (a, sa), (b, sb) = got[key], want[key]
        assert sa == sb and np.array_equal(a, b), key


def test_plain_model_padded_predict_and_noise_budget():
    """Network::predict on 28x28 images with device re-encryption before layer 6: the decoded scores equal PlainModel's on the same
    images zero-bordered (plaintext-level equality: the encryptions differ).  The first group's output has at least the noise budget
    of the bordered network's on the same ciphertexts with a zero-ciphertext border."""
    from crcnn_b200.host import HostNetwork
    from crcnn_b200.lib import Engine
    orc = Oracle(N8, PRIMES[N8], T_FOR_N[N8])
    keys = kg.generate(orc, 41)
    imgs = np.stack([util.synthetic_image(s).reshape(28, 28) for s in range(2)])
    scores, budget = {}, {}
    for model, im, pad in (("PlainModelPadded", imgs, 0), ("PlainModel", np.pad(imgs, [(0, 0), (2, 2), (2, 2)]), 2)):
        net = HostNetwork(N8, PRIMES[N8], T_FOR_N[N8], model, evk=keys.evk_triple)
        try:
            net.use_keys(keys.sk, keys.pk, device_reencryption=True, seed=7)
            scores[model] = net.predict_values(im.astype(np.float32), batch=2, seed=11)
            eng = Engine.adopt(net.ctx(), N8, PRIMES[N8], T_FOR_N[N8])
            dk = eng.keys_upload(keys.sk, keys.pk)
            x = eng.download(eng.encrypt_values(dk, imgs.astype(np.float32)[:1], seed=13))       # the same 28x28 ciphertexts
            y, _ = net.forward(border(x, 1, 1, 28, 28, pad, pad), batch=1, first=0, last=3)
            budget[model] = eng.min_noise_budget(dk, eng.upload(y))
            del dk
            eng.h = None
        finally:
            net.close()
    assert np.array_equal(scores["PlainModelPadded"], scores["PlainModel"]), scores
    assert budget["PlainModelPadded"] >= budget["PlainModel"] > 0, budget


def _sharded_worker(rank, world, out_dir, n):
    from crcnn_b200 import host
    primes, t = util.PRIMES[n], util.T_FOR_N[n]
    idfile = os.path.join(out_dir, "nccl_id")
    if rank == 0:
        open(idfile + ".tmp", "wb").write(host.nccl_unique_id())
        os.rename(idfile + ".tmp", idfile)
    while not os.path.exists(idfile):
        time.sleep(0.05)
    nccl_id = open(idfile, "rb").read()
    rng = np.random.default_rng(8)
    evk = util.random_evk(rng, n, primes)
    x = util.random_cts(rng, n, primes, 2 * 784)
    net = host.HostNetwork(n, primes, t, "PlainModelPadded", device=rank, evk=evk, world=world, rank=rank, nccl_id=nccl_id)
    got, _ = net.forward(x, batch=2)
    np.save(os.path.join(out_dir, "sharded%d.npy" % rank), got)
    net.close()
    if rank == 0:
        ref = host.HostNetwork(n, primes, t, "PlainModelPadded", device=0, evk=evk)
        np.save(os.path.join(out_dir, "single.npy"), ref.forward(x, batch=2)[0])
        ref.close()


def test_sharded_plain_model_padded_matches_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_sharded_worker, args=(2, str(tmp_path), 4096), nprocs=2, join=True)
    want = np.load(tmp_path / "single.npy")
    for r in range(2):
        assert np.array_equal(np.load(tmp_path / ("sharded%d.npy" % r)), want), r
