"""What zero padding saves at the request boundary: PlainModel.h5 run as "PlainModel" (32x32 input, the client encrypts and uploads the
zero border itself) against "PlainModelPadded" (28x28 input, conv1 with padding 2 inside the evaluator).

n = 8192, t = 2^30, batch 8, keys from tests/fv_keygen.py, seeded synthetic images (tests/util.synthetic_image).  For each model, on one
GPU, after a warm-up of every call:
  * crcnn_encrypt_values of the batch's images (CUDA events around the call; its bytes are the ciphertexts it produces);
  * the pinned host-to-device upload of one request (the encrypted batch);
  * the resident forward step (crcnn_host_resident_run, bench.py's kind);
  * the serving loop (crcnn_host_serve over `requests` requests, per-request completion times).
The two models alternate over `rounds` rounds (one network per process at a time: each round builds, measures and closes it).  The
card's name and power limit are read in the same run.

    python tools/pad_time.py --out profiles/r06_pad_time.json
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from crcnn_b200.host import HostNetwork, pinned_array  # noqa: E402
from crcnn_b200.lib import Engine  # noqa: E402
import fv_keygen as kg  # noqa: E402
from oracle.port import DEFAULT_PRIMES_128 as PRIMES, Oracle  # noqa: E402
from util import synthetic_image  # noqa: E402
from noise_trace import card, event_ms  # noqa: E402

N, T, BATCH, SEED = 8192, 1 << 30, 8, 77
MODELS = ("PlainModel", "PlainModelPadded")


def images(model):
    imgs = [synthetic_image(b).reshape(28, 28) for b in range(BATCH)]
    if model == "PlainModel":
        imgs = [np.pad(i, 2) for i in imgs]
    return np.stack(imgs).astype(np.float32)


def measure(model, keys, reps, requests, seeds):
    net = HostNetwork(N, PRIMES[N], T, model, evk=keys.evk_triple)
    eng = Engine.adopt(net.ctx(), N, PRIMES[N], T)
    dk = eng.keys_upload(keys.sk, keys.pk)
    imgs = images(model)
    held = []

    def enc():          # the previous output is freed first, so every call after the warm-up reuses its block
        while held:
            held.pop().free()
        held.append(eng.encrypt_values(dk, imgs, seed=next(seeds)))
    x = eng.encrypt_values(dk, imgs, seed=SEED)
    host_x = eng.download(x)
    count = imgs.size
    pin, owner = pinned_array(host_x.size)
    pin[:] = host_x.ravel()
    up = lambda: eng.upload_ptr(pin.ctypes.data, count).free()   # noqa: E731
    res = {"ciphertexts_in": int(count), "request_bytes": int(host_x.nbytes),
           "encrypt_values_ms": event_ms(eng, enc, reps), "upload_pinned_ms": event_ms(eng, up, reps)}
    held.clear()
    net.resident_begin(pin.ctypes.data, BATCH)
    net.resident_run(1)
    ms, _ = net.resident_run(reps)
    net.resident_end()
    res["forward_step_ms"] = ms / reps
    out, out_owner = pinned_array(BATCH * net.outputs * net.ct_words())
    net.serve(pin.ctypes.data, out.ctypes.data, BATCH, 2)          # warm-up of the server's buffers
    total = net.serve(pin.ctypes.data, out.ctypes.data, BATCH, requests)
    done = net.serve_times()
    res["serve_total_ms"] = total
    res["serve_ms_per_request"] = total / requests
    res["serve_completion_ms"] = [round(v, 3) for v in done]
    del dk, x, pin, owner, out, out_owner
    eng.h = None
    net.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--requests", type=int, default=8)
    a = ap.parse_args()
    keys = kg.generate(Oracle(N, PRIMES[N], T), SEED)
    seeds = iter(range(1000, 1000000))
    runs = {m: [] for m in MODELS}
    for r in range(a.rounds):
        for m in (MODELS if r % 2 == 0 else MODELS[::-1]):
            runs[m].append(measure(m, keys, a.reps, a.requests, seeds))
            print(m, "round", r, {k: v for k, v in runs[m][-1].items() if k != "serve_completion_ms"}, flush=True)
    keys_of = ("encrypt_values_ms", "upload_pinned_ms", "forward_step_ms", "serve_ms_per_request")
    summary = {m: {"request_bytes": runs[m][0]["request_bytes"], "ciphertexts_in": runs[m][0]["ciphertexts_in"],
                   **{k: {"median": round(float(np.median([x[k] for x in runs[m]])), 3),
                          "min": round(min(x[k] for x in runs[m]), 3), "max": round(max(x[k] for x in runs[m]), 3)} for k in keys_of}}
               for m in MODELS}
    res = {"card (name, power limit)": card(), "n": N, "t": T, "batch": BATCH, "reps": a.reps, "rounds": a.rounds,
           "requests": a.requests, "summary": summary, "runs": runs,
           "note": ("CUDA events on the context's stream, mean of `reps` calls after one warm-up call, per round; models alternated "
                    "(ABBA...); encrypt includes the host-to-device copy of the floats; upload = one request's ciphertexts from pinned "
                    "memory; forward_step = crcnn_host_resident_run; serve = crcnn_host_serve, completion times on the host clock")}
    s = json.dumps(res) + "\n"
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)
    print(json.dumps({"card": res["card (name, power limit)"], "summary": summary}))


if __name__ == "__main__":
    main()
