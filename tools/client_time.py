"""The client's two ends on the device: what encrypting the images (crcnn_encrypt_values) and decrypting the scores
(crcnn_decrypt_values) cost next to the forward step, and next to the ciphertext upload the end-to-end path makes per request.

PlainModel at n = 8192, t = 2^30, batch 8: keys and evaluation keys from tests/fv_keygen.py, seeded synthetic images
(tests/util.synthetic_image, zero border for the 32x32 input).  After a warm-up of every call, CUDA events on the context's stream
time crcnn_encrypt_values of the 8 images (8,192 ciphertexts), crcnn_decrypt_values of the 80 scores, HostNetwork.predict_values end
to end (encrypt, forward, decrypt), the resident forward step, and the host-to-device copy of the same 8 encrypted images from pinned
memory.  The card's name and power limit are read in the same run.

Also reported, not asserted: the decoded scores against a float64 NumPy evaluation of the same network on the same images.

    python tools/client_time.py --out profiles/r05_client_time.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from crcnn_b200 import nets  # noqa: E402
from crcnn_b200.host import HostNetwork, pinned_array  # noqa: E402
from crcnn_b200.lib import Engine  # noqa: E402
import fv_keygen as kg  # noqa: E402
from oracle.port import DEFAULT_PRIMES_128 as PRIMES, Oracle  # noqa: E402
from util import synthetic_image  # noqa: E402
from noise_trace import card, event_ms  # noqa: E402

MODEL, N, T, BATCH, SEED = "PlainModel", 8192, 1 << 30, 8, 77


def float_forward(model, img):
    """float64 evaluation of the topology on one [z][x][y] image: the layers the encrypted network computes, in their order"""
    w = {k: v.astype(np.float64) for k, v in nets.load_weights(model).items()}
    x = img.astype(np.float64)
    for layer in nets.TOPOLOGIES[model]["layers"]:
        kind, name = layer[0], layer[1]
        if kind == "conv":
            _, _, xd, yd, zd, xs, ys, xf, yf, nf = layer
            W = w[name + ".weight"].reshape(nf, zd, xf, yf)
            xo, yo = (xd - xf) // xs + 1, (yd - yf) // ys + 1
            y = np.empty((nf, xo, yo))
            for i in range(xo):
                for j in range(yo):
                    y[:, i, j] = np.tensordot(W, x[:, i * xs:i * xs + xf, j * ys:j * ys + yf], axes=3)
            x = y + w[name + ".bias"].reshape(nf, 1, 1)
        elif kind in ("avgpool", "pool"):
            _, _, xd, yd, zd, xs, ys, xf, yf = layer
            xo, yo = (xd - xf) // xs + 1, (yd - yf) // ys + 1
            y = np.zeros((zd, xo, yo))
            for a in range(xf):
                for b in range(yf):
                    y += x[:, a:a + xs * (xo - 1) + 1:xs, b:b + ys * (yo - 1) + 1:ys]
            x = y / (xf * yf) if kind == "avgpool" else y
        elif kind == "bn":
            mean, var = w[name + ".running_mean"], w[name + ".running_var"]
            x = (x - mean.reshape(-1, 1, 1)) / np.sqrt(var.reshape(-1, 1, 1) + 0.00001)
        elif kind == "square":
            x = x * x
        elif kind == "fc":
            x = w[name + ".weight"].reshape(layer[3], layer[2]) @ x.ravel() + w[name + ".bias"]
    return np.asarray(x).ravel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    orc = Oracle(N, PRIMES[N], T)
    keys = kg.generate(orc, SEED)
    net = HostNetwork(N, PRIMES[N], T, MODEL, evk=keys.evk_triple)
    net.use_keys(keys.sk, keys.pk)
    eng = Engine.adopt(net.ctx(), N, PRIMES[N], T)
    dk = eng.keys_upload(keys.sk, keys.pk)
    imgs = np.stack([np.pad(synthetic_image(b).reshape(28, 28), 2) for b in range(BATCH)]).astype(np.float32)   # [8][32][32]
    count = imgs.size
    seeds = iter(range(1000, 100000))
    held = []

    def enc():          # the previous output is freed first, so every call after the warm-up reuses its block (no allocation timed)
        while held:
            held.pop().free()
        held.append(eng.encrypt_values(dk, imgs, seed=next(seeds)))
    x = eng.encrypt_values(dk, imgs, seed=SEED)
    host_x = eng.download(x)
    out, _ = net.forward(host_x, batch=BATCH)
    scores_t = eng.upload(out)
    dec = lambda: eng.decrypt_values(dk, scores_t)           # noqa: E731
    pred = lambda: net.predict_values(imgs, batch=BATCH, seed=next(seeds))   # noqa: E731
    pin, owner = pinned_array(host_x.size)
    pin[:] = host_x.ravel()
    up = lambda: eng.upload_ptr(pin.ctypes.data, count).free()   # noqa: E731

    res = {"card (name, power limit)": card(), "model": MODEL, "n": N, "t": T, "batch": BATCH, "ciphertexts_in": count,
           "scores": int(eng.count(scores_t)), "reps": a.reps,
           "encrypt_values_ms": round(event_ms(eng, enc, a.reps), 3),
           "decrypt_values_ms": round(event_ms(eng, dec, a.reps), 3),
           "upload_ciphertexts_pinned_ms": round(event_ms(eng, up, a.reps), 3),
           "upload_bytes": int(host_x.nbytes)}
    held.clear()
    t0 = time.perf_counter()
    res["predict_values_ms"] = round(event_ms(eng, pred, a.reps), 3)
    res["predict_values_host_clock_ms"] = round((time.perf_counter() - t0) * 1e3 / (a.reps + 1), 3)
    net.resident_begin(pin.ctypes.data, BATCH)
    net.resident_run(1)
    ms, _ = net.resident_run(a.reps)
    net.resident_end()
    res["forward_step_ms"] = round(ms / a.reps, 3)
    # decoded scores vs float64 (a finding, not a check)
    dec_scores = eng.decrypt_values(dk, scores_t).reshape(BATCH, -1)
    ref = np.stack([float_forward(MODEL, imgs[b].reshape(1, 32, 32)) for b in range(BATCH)])
    res["scores_vs_float64"] = {"max_abs_diff": float(np.abs(dec_scores - ref).max()),
                                "max_abs_float64_score": float(np.abs(ref).max()),
                                "argmax_agree": int((dec_scores.argmax(1) == ref.argmax(1)).sum()), "of": BATCH}
    res["note"] = ("CUDA events around the whole call on the context's stream, mean of `reps` after one warm-up call; encrypt includes "
                   "the host-to-device copy of the floats, decrypt the device-to-host copy of the scores; predict_values = encrypt + "
                   "forward + decrypt through the host library; forward_step_ms = the resident forward of bench.py's kind; "
                   "upload = the 8 encrypted images from pinned host memory")
    del dk, scores_t, x
    eng.h = None
    net.close()
    s = json.dumps(res) + "\n"
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)
    print(s)


if __name__ == "__main__":
    main()
