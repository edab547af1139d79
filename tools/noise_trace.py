"""Noise budget along the forward pass (Decryptor::invariant_noise_budget on the device, crcnn_noise_budget): our version of the
thesis's "NB" column, where the budget-driven policy re-encrypts, and what one budget check costs next to one decrypt.

For PlainModel (n = 8192, t = 2^30) at batch 1 and 8 and the Approx net (n = 4096, t = 2^20): keys and evaluation keys from
tests/fv_keygen.py, seeded synthetic images (tests/util.synthetic_image, zero border for PlainModel's 32x32 input) encrypted with the
oracle's Encryptor, the network run one reference layer at a time (fusion off) through the host library's segment API and the
minimum budget taken after each layer -- once without re-encryption and once with crcnn_reencrypt before layer 6.  Then the
budget_log of one adaptive forward at threshold 5 (fusion on and off), and CUDA-event times of one crcnn_noise_budget and one
crcnn_decrypt of the largest activation after warm-up, with the card's name and power limit.

    python tools/noise_trace.py --out profiles/r04_noise_trace.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from crcnn_b200.host import HostNetwork, OutOfBudget  # noqa: E402
from crcnn_b200.lib import Engine  # noqa: E402
import fv_keygen as kg  # noqa: E402
from oracle.port import DEFAULT_PRIMES_128 as PRIMES, Oracle  # noqa: E402
from util import synthetic_image  # noqa: E402

CONFIGS = [("PlainModel", 8192, 1 << 30, 1), ("PlainModel", 8192, 1 << 30, 8), ("ApproxPlainModel", 4096, 1 << 20, 1)]
REENC_BEFORE = 6
SEED = 77


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def images(model, batch, keys, rng):
    out = []
    for b in range(batch):
        img = synthetic_image(b).reshape(28, 28)
        if model == "PlainModel":
            img = np.pad(img, 2)
        out.append(kg.encrypt_values(keys, img.ravel(), rng))
    return np.concatenate(out)


def event_ms(eng, fn, reps):
    L = eng.lib
    a, b = C.c_void_p(), C.c_void_p()
    eng._chk(L.crcnn_event_create(eng.h, C.byref(a)))
    eng._chk(L.crcnn_event_create(eng.h, C.byref(b)))
    fn()
    eng.sync()
    eng._chk(L.crcnn_event_record(eng.h, a, None))
    for _ in range(reps):
        fn()
    eng._chk(L.crcnn_event_record(eng.h, b, None))
    eng.sync()
    ms = C.c_double()
    eng._chk(L.crcnn_event_elapsed_ms(eng.h, a, b, C.byref(ms)))
    L.crcnn_event_destroy(eng.h, a)
    L.crcnn_event_destroy(eng.h, b)
    return ms.value / reps


def trace(model, n, t, batch):
    orc = Oracle(n, PRIMES[n], t)
    keys = kg.generate(orc, SEED)
    t0 = time.time()
    x = images(model, batch, keys, np.random.default_rng(SEED))
    enc_s = time.time() - t0
    net = HostNetwork(n, PRIMES[n], t, model, evk=keys.evk_triple)
    eng = Engine.adopt(net.ctx(), n, PRIMES[n], t)
    dk = eng.keys_upload(keys.sk, keys.pk)
    res = {"model": model, "n": n, "t": t, "batch": batch, "q_bits": kg.modulus(orc).bit_length(), "layers": net.layer_names,
           "fresh_min_budget": int(eng.min_noise_budget(dk, eng.upload(x))), "encrypt_s_cpu_oracle": round(enc_s, 1)}
    net.set_fusion(False)
    largest = None
    for reenc in (False, True):
        h, shape, col = x, (net.zd, net.xd, net.yd), []
        for i in range(net.num_layers):
            if reenc and i == REENC_BEFORE:
                h = eng.download(eng.reencrypt(dk, eng.upload(h), seed=SEED))
                col.append({"layer": "reencrypt", "min_budget": int(eng.min_noise_budget(dk, eng.upload(h)))})
            h, shape = net.forward(h, batch=batch, first=i, last=i + 1, shape=shape)
            d = eng.upload(h)
            col.append({"layer": i, "name": net.layer_names[i], "ciphertexts": int(len(h)), "min_budget": int(eng.min_noise_budget(dk, d))})
            if not reenc and (largest is None or len(h) > largest[0]):
                largest = (len(h), i)
            del d
        if reenc:
            vals = [orc.decode(p) for p in orc.decrypt(h[:10], keys.sk)]
            res["scores_after_reencryption_first_image"] = vals
        res["per_layer_reencrypt_before_6" if reenc else "per_layer_no_reencryption"] = col
    # where the budget-driven policy (threshold 5, device re-encryption) re-encrypts
    for fusion in (True, False):
        net.set_fusion(fusion)
        net.use_keys(keys.sk, keys.pk, device_reencryption=True, seed=SEED)
        net.set_budget_threshold(5)
        err = None
        try:
            net.forward_adaptive(x, batch=batch)
        except OutOfBudget as e:
            err = "OutOfBudgetException at layer %d" % e.layer
        res["adaptive_threshold5_fusion_%s" % ("on" if fusion else "off")] = {
            "budget_log": [{"layer": a, "min_budget": b, "reencrypted": c} for a, b, c in net.budget_log()], "error": err}
    # cost of one budget check vs one decrypt of the largest activation (layer outputs re-run to get it on the device)
    net.set_fusion(False)
    h, shape = net.forward(x, batch=batch, first=0, last=largest[1] + 1)
    d = eng.upload(h)
    del h
    plain = np.zeros((eng.count(d), eng.stride), dtype=np.uint64)
    dec = lambda: eng._chk(eng.lib.crcnn_decrypt(eng.h, dk.ptr, d.ptr, plain.ctypes.data))   # noqa: E731
    nb = lambda: eng.min_noise_budget(dk, d)                                                    # noqa: E731
    res["timing_largest_activation"] = {"layer": largest[1], "ciphertexts": int(largest[0]),
                                        "noise_budget_ms": round(event_ms(eng, nb, 5), 3), "decrypt_ms": round(event_ms(eng, dec, 5), 3),
                                        "note": "CUDA events around the whole call, device-to-host copy of the result included (plaintexts for decrypt, ints for the budget)"}
    d.free()
    dk.free()
    eng.h = None          # the context belongs to the host library, which the next network re-initialises
    net.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--configs", default="0,1,2", help="indices into CONFIGS")
    a = ap.parse_args()
    out = {"card": card(), "configs": []}
    for k in [int(v) for v in a.configs.split(",")]:
        r = trace(*CONFIGS[k])
        out["configs"].append(r)
        print(json.dumps({key: r[key] for key in ("model", "n", "batch", "fresh_min_budget")}), flush=True)
    s = '{"card": %s, "configs": [\n%s\n]}\n' % (json.dumps(out["card"]), ",\n".join(json.dumps(c) for c in out["configs"]))   # one line per config
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)
    print(s)


if __name__ == "__main__":
    main()
