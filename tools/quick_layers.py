#!/usr/bin/env python
"""Times a few layers of the bench network in seconds of box time (no torch import): per-kernel-class ms of `reps` forwards of layers
[first, last) at the bench batch, from the engine's own CUDA-event counters.  For A/B runs of kernel switches set through the environment.

  CRCNN_TCN_FOLD=0 python tools/quick_layers.py --first 0 --last 1      # conv1 only
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from crcnn_b200 import nets  # noqa: E402
from crcnn_b200.lib import Engine  # noqa: E402
import bench  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--first", type=int, default=0)
    ap.add_argument("--last", type=int, default=1)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    n, primes, t = bench.N_POLY, bench.PRIMES, bench.T_PLAIN
    eng = Engine(n, primes, t, device=0)
    rng = np.random.default_rng(5)
    evk = None
    if any(l[0] == "square" for l in nets.TOPOLOGIES[bench.MODEL]["layers"][args.first:args.last]):
        evk_words, sizes, dbc = bench.synth_evk(rng, primes, n)
        evk = eng.evk_upload(evk_words, sizes, dbc)
    net = nets.Network(eng, bench.MODEL, evk=evk)
    nin = nets.layer_io_counts(net.layers[args.first])[0]
    one = bench.synth_residues(rng, (nin, 2), primes, n)
    x0 = eng.upload(np.concatenate([one] * args.batch))

    def fwd():
        x = eng.slice(x0, 0, args.batch * nin)
        y = net.forward(x, batch=args.batch, first=args.first, last=args.last)
        x.free()
        y.free()
        eng.sync()

    fwd()
    eng.prof_enable(True)
    eng.prof_reset()
    for _ in range(args.reps):
        fwd()
    print({k: (v[0] // args.reps, round(v[1] / args.reps, 2)) for k, v in eng.prof().items() if v[0]},
          {k: os.environ[k] for k in os.environ if k.startswith("CRCNN_")})
    eng.close()


if __name__ == "__main__":
    main()
