#!/usr/bin/env python
"""CRT plaintext-modulus ensembles (BASELINE config 4) end to end: one instance per GPU and process under bench.py's CRT_MODULI
for the GPU count, each with its own keys, running CrtEnsemble::predict (collective re-encryption before layer 6, collective
decryption) on PlainModelWoPad at n = 8192.  Reports, in one JSON object written to --out:
  - ensemble predict images/s (host clock around whole predict calls: encryption, forward, re-encryption, decryption);
  - ms of crcnn_crt_reencrypt and crcnn_crt_decrypt_values on the activations before layer 6, next to crcnn_reencrypt and
    crcnn_decrypt_values of the same instance on the same tensor (host clock around calls that end in a device synchronise);
  - each instance's minimum noise budget after the last layer, next to a single-modulus run under 2^30;
  - the card name and power limit, read in the same run.
usage: python tools/crt_time.py --gpus 1|2|4|8 [--model PlainModelWoPad] [--batch 8] [--steps 3] [--out crt_time.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card(rank):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(rank)],
                       capture_output=True, text=True)
    return q.stdout.strip()


def shared_id(out_dir, rank, tag):
    from crcnn_b200.host import nccl_unique_id
    path = os.path.join(out_dir, "nccl_id_" + tag)
    if rank == 0:
        open(path + ".tmp", "wb").write(nccl_unique_id())
        os.rename(path + ".tmp", path)
    while not os.path.exists(path):
        time.sleep(0.05)
    return open(path, "rb").read()


def timed(fn, reps, sync):
    fn()
    sync()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    sync()
    return (time.perf_counter() - t0) * 1000.0 / reps


def instance(rank, world, args, tmp):
    import ctypes as C
    import bench
    import fv_keygen as kg
    import util
    from oracle.port import Oracle
    from crcnn_b200 import lib
    from crcnn_b200.host import HostNetwork
    from crcnn_b200.lib import Engine
    n, primes = 8192, bench.PRIMES
    moduli = bench.CRT_MODULI[world]
    t = moduli[rank]
    keys = kg.generate(Oracle(n, primes, t), 500 + rank)
    net = HostNetwork(n, primes, t, args.model, device=rank, evk=keys.evk_triple, skip_reencryption=False)
    net.use_keys(keys.sk, keys.pk)
    net.crt_begin(moduli, rank, shared_id(tmp, rank, "net"), reencrypt_seed=1)
    imgs = np.stack([util.synthetic_image(s, net.zd * net.xd * net.yd) for s in range(args.batch)])
    scores = net.crt_predict_values(imgs, batch=args.batch, seed=10)
    t0 = time.perf_counter()
    for s in range(args.steps):
        net.crt_predict_values(imgs, batch=args.batch, seed=11 + s)
    predict_s = (time.perf_counter() - t0) / args.steps
    # the collective calls against one instance's own, on the activations before layer 6
    eng = Engine.adopt(net.ctx(), n, primes, t)
    dk = eng.keys_upload(keys.sk, keys.pk)
    L = lib.load()
    comm = C.c_void_p()
    idbuf = (C.c_char * 128).from_buffer_copy(shared_id(tmp, rank, "eng"))
    eng._chk(L.crcnn_comm_create(eng.h, C.cast(idbuf, C.c_void_p), world, rank, C.byref(comm)))
    crt = eng.crt_create(comm.value, moduli)
    x0 = eng.download(eng.encrypt_values(dk, imgs, seed=20))
    mid, shape = net.forward(x0, batch=args.batch, first=0, last=6)
    xm = eng.upload(mid)
    ops = {
        "crt_reencrypt_ms": timed(lambda: eng.crt_reencrypt(crt, dk, xm, seed=30).free(), 3, eng.sync),
        "reencrypt_ms": timed(lambda: eng.reencrypt(dk, xm, seed=31).free(), 3, eng.sync),
        "crt_decrypt_values_ms": timed(lambda: eng.crt_decrypt_values(crt, dk, xm), 3, eng.sync),
        "decrypt_values_ms": timed(lambda: eng.decrypt_values(dk, xm), 3, eng.sync),
        "ciphertexts": int(eng.count(xm)),
    }
    fresh = eng.download(eng.crt_reencrypt(crt, dk, xm, seed=32))
    out, _ = net.forward(fresh, batch=args.batch, first=6, shape=shape)
    budget = eng.min_noise_budget(dk, eng.upload(out))
    crt.free()
    L.crcnn_comm_destroy(eng.h, comm)
    del dk
    eng.close()
    net.close()
    res = {"rank": rank, "t": t, "card": card(rank), "predict_images_per_s": args.batch / predict_s, "predict_ms": predict_s * 1000.0,
           "min_budget_after_last_layer": budget, "scores_first_image": [float(v) for v in scores[0]], **ops}
    if rank == 0:      # the single-modulus run under 2^30 on the same card: its last-layer budget
        T = 1 << 30
        k1 = kg.generate(Oracle(n, primes, T), 600)
        one = HostNetwork(n, primes, T, args.model, device=0, evk=k1.evk_triple, skip_reencryption=False)
        e1 = Engine.adopt(one.ctx(), n, primes, T)
        d1 = e1.keys_upload(k1.sk, k1.pk)
        m1, s1 = one.forward(e1.download(e1.encrypt_values(d1, imgs, seed=40)), batch=args.batch, first=0, last=6)
        r1 = e1.download(e1.reencrypt(d1, e1.upload(m1), seed=41))
        o1, _ = one.forward(r1, batch=args.batch, first=6, shape=s1)
        res["single_2p30_min_budget_after_last_layer"] = e1.min_noise_budget(d1, e1.upload(o1))
        del d1
        e1.close()
        one.close()
    with open(os.path.join(tmp, "rank%d.json" % rank), "w") as f:
        json.dump(res, f)


def _spawned(rank, world, args, tmp):
    instance(rank, world, args, tmp)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1, choices=[1, 2, 4, 8])
    ap.add_argument("--model", default="PlainModelWoPad", choices=["PlainModelWoPad", "PlainModel"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default="crt_time.json")
    args = ap.parse_args()
    import tempfile
    import torch
    if torch.cuda.device_count() < args.gpus:
        raise SystemExit("needs %d GPUs, found %d" % (args.gpus, torch.cuda.device_count()))
    tmp = tempfile.mkdtemp(prefix="crt_time_")
    import torch.multiprocessing as mp
    mp.spawn(_spawned, args=(args.gpus, args, tmp), nprocs=args.gpus, join=True)
    ranks = [json.load(open(os.path.join(tmp, "rank%d.json" % r))) for r in range(args.gpus)]
    assert all(r["scores_first_image"] == ranks[0]["scores_first_image"] for r in ranks), "ranks decoded different scores"
    line = {"gpus": args.gpus, "model": args.model, "n": 8192, "batch": args.batch, "moduli": [r["t"] for r in ranks],
            "predict_images_per_s": ranks[0]["predict_images_per_s"], "ranks": ranks}
    with open(args.out, "w") as f:
        json.dump(line, f, indent=1)
    print(json.dumps({k: v for k, v in line.items() if k != "ranks"}))
    for r in ranks:
        print(json.dumps({k: v for k, v in r.items() if k != "scores_first_image"}))


if __name__ == "__main__":
    main()
