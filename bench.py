#!/usr/bin/env python
"""Benchmark of the encrypted-forward hot path (BASELINE.json metric: encrypted MNIST images/sec,
per-layer latency in ms, roofline fraction of the dominant kernel).

One step = one forward pass of the encoded PlainModel.h5 network (n = 8192, K = 4, t = 2^30,
32x32 zero-bordered input, SURVEY.md section 8(d) config 2) over a batch of B independent
synthetic encrypted images on one GPU.  With --gpus N every rank runs its own batch (image
replicas, no data-path collective: weak scaling).

  python bench.py --gpus 1 --steps 3 --warmup 3
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...     # the reference's own CPU path on the host cores
  python bench.py --gpus 1 --steps 3 --warmup 3 --dump-outputs DIR

Prints ONE JSON line (rank 0).  `value` = images/s with inputs resident in HBM; `e2e` = the same
through the C ABI with host buffers (pinned H2D of every input ciphertext and D2H of the 10 output
ciphertexts per image inside the timed region).  The inputs are seeded: the same arguments give the
same inputs, so --dump-outputs of two builds can be compared array for array (see dump_outputs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# stdout carries exactly ONE JSON line: whatever NCCL has to say (its version banner under NCCL_DEBUG=VERSION/INFO) goes to stderr ...
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
# ... and so does anything a native library writes to file descriptor 1 directly: fd 1 points at stderr for the whole run, the JSON line
# goes to a duplicate of the original stdout (emit()).
_REAL_STDOUT = None


def _claim_stdout():
    """main() only (tools import this module for its constants and helpers and keep their stdout)."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from crcnn_b200 import nets  # noqa: E402

N_POLY = 8192
PRIMES = [0x7fffffff380001, 0x7ffffffef00001, 0x3fffffff000001, 0x3ffffffef40001]  # coeff_modulus_128(8192)
T_PLAIN = 1 << 30
MODEL = "PlainModel"
W = 8  # bytes per residue


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="images per step per GPU")
    ap.add_argument("--cpu-budget-s", type=float, default=20.0, help="CPU seconds for the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--literal-threads", action="store_true",
                    help="--impl reference: the reference's own thread constants (cnnBuilder.cpp:109; conv1 and fc4 then run on ONE thread, "
                         "the th_count > outputs quirk of convolutionalLayer.cpp:28-31,177-187) instead of one thread per core")
    ap.add_argument("--model", default=None, choices=sorted(nets.TOPOLOGIES),
                    help="network to run instead of the headline PlainModel (e.g. PlainModelTiny with --n 4096: BASELINE config 1)")
    ap.add_argument("--n", type=int, default=None, choices=[4096, 8192, 16384], help="polynomial degree (default 8192)")
    ap.add_argument("--no-shard", action="store_true", help="skip the neuron-sharded Approx forward appended to the line (key `shard`)")
    ap.add_argument("--shard-batch", type=int, default=8, help="images per batch of the sharded forward")
    ap.add_argument("--mode", default="replicas", choices=["replicas", "shard", "crt"],
                    help="replicas: every GPU runs its own image batch (default, weak scaling); shard: ONE image, the Approx "
                         "network's conv / fc layers split by output neuron across the GPUs with NCCL all-gathers of the "
                         "activation ciphertexts (BASELINE config 3, strong scaling); crt: the plaintext modulus ~2^30 split into "
                         "one CRT modulus per GPU, independent instances of the WoPad network on the same images (BASELINE config 4)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the score ciphertexts rank 0's last timed step computed (replicas and crt "
                         "modes): DIR/scores.npy holds every residue as four exact 16-bit words in float32, least significant first "
                         "(words, not values: compare exactly), DIR/scores_coeff_index.npy the coefficient positions kept")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.mode == "shard"):
        ap.error("--dump-outputs needs --impl b200 and --mode replicas or crt")
    return args


DUMP_BYTES = 60 * 10**6   # scores.npy stays below this; with the index file and headers the dump is under 64 MB
DUMP_SEED = 20240


def dump_outputs(directory, scores, budget=DUMP_BYTES, seed=DUMP_SEED):
    """Writes score ciphertexts ([batch][outputs][2][K][n+1] uint64 residues, pad word last) as exact float32 arrays:

      scores.npy              [batch][outputs][2][K][m][4]: each residue as four 16-bit words, least significant first
      scores_coeff_index.npy  [m]: the coefficient positions kept, all n of them when they fit in `budget` bytes, else a
                              fixed sample drawn with `seed`, so two runs with the same arguments keep the same positions

    A float32 holds every integer below 2^24, so the words are exact and two builds' dumps compare with np.array_equal; a
    residue that is off by one changes a word by one, which no tolerance meant for float data lets through."""
    scores = np.asarray(scores, dtype=np.uint64)
    n = scores.shape[-1] - 1
    per_coeff = scores[..., 0].size * 4 * 4
    m = min(n, budget // per_coeff)
    index = np.arange(n) if m == n else np.sort(np.random.default_rng(seed).choice(n, size=m, replace=False))
    kept = scores[..., index]
    words = np.stack([(kept >> np.uint64(16 * i)) & np.uint64(0xFFFF) for i in range(4)], axis=-1).astype(np.float32)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "scores.npy"), words)
    np.save(os.path.join(directory, "scores_coeff_index.npy"), index.astype(np.float32))


# ------------------------------------------------------------------------------------------
# synthetic workload
# ------------------------------------------------------------------------------------------
def synth_residues(rng, shape_front, primes, n, out=None):
    """Uniform canonical residues in SEAL ciphertext layout [..., K, n+1] (pad word 0): the
    distribution FV ciphertexts have; the evaluator's work is data independent."""
    K = len(primes)
    if out is None:
        out = np.zeros(tuple(shape_front) + (K, n + 1), dtype=np.uint64)
    for j, q in enumerate(primes):
        out[..., j, :n] = rng.integers(0, q, size=tuple(shape_front) + (n,), dtype=np.uint64)
    out[..., n] = 0
    return out


def synth_evk(rng, primes, n, dbc=16):
    sizes = [2 * ((int(q).bit_length() + dbc - 1) // dbc) for q in primes]
    parts = [synth_residues(rng, (s,), primes, n).ravel() for s in sizes]
    return np.concatenate(parts), sizes, dbc


def _bind_to_gpu_numa_node(torch, device):
    """Moves this process onto the CPUs of the NUMA node the GPU hangs off, so that the pinned request buffers allocated next are
    placed there (8 ranks uploading 4 GB per step share the host's memory controllers: VERDICT r1 weak #6).  Returns
    {"node", "restore"} or None when the box does not say (VMs report -1) -- then nothing changes."""
    try:
        pr = torch.cuda.get_device_properties(device)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        target = cpus & allowed
        if not target:
            return None
        os.sched_setaffinity(0, target)
        return {"node": node, "restore": allowed}
    except Exception:
        return None


# ------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
# CPU baseline: the reference's own layer classes (oracle/_ref) on a bounded sample
# ------------------------------------------------------------------------------------------
def _crop_layer(layer, cores, term_budget, ct_budget):
    """Same layer type and fan-in, reduced width/extent so the sample fits the time budget.
    Returns (cropped layer, scale) with scale = full work / sample work (work = weighted-sum terms for
    conv/fc, ciphertexts for the others; both are exactly linear in the cropped dimensions)."""
    kind = layer[0]
    if kind == "conv":
        _, name, xd, yd, zd, xs, ys, xf, yf, nf = layer
        nf2 = min(nf, cores)
        yo = (yd - yf) // ys + 1
        per_row = yo * zd * xf * yf                    # terms per filter per output row
        rows = max(1, min((xd - xf) // xs + 1, int(term_budget // per_row)))
        xd2 = (rows - 1) * xs + xf
        crop = ("conv", name, xd2, yd, zd, xs, ys, xf, yf, nf2)
        return crop, nets.layer_terms(layer) / nets.layer_terms(crop)
    if kind == "fc":
        _, name, i, o = layer
        o2 = min(o, cores)
        return ("fc", name, i, o2), o / o2
    if kind in ("pool", "avgpool"):
        _, name, xd, yd, zd, xs, ys, xf, yf = layer
        yo = (yd - yf) // ys + 1
        rows = max(1, min((xd - xf) // xs + 1, int(ct_budget // yo)))
        xd2 = (rows - 1) * xs + xf
        crop = (kind, name, xd2, yd, 1, xs, ys, xf, yf)
        return crop, nets.layer_io_counts(layer)[1] / nets.layer_io_counts(crop)[1]
    if kind == "bn":
        _, name, zd, xd, yd = layer
        xd2 = max(1, min(xd, int(ct_budget // yd)))
        return ("bn", name, 1, xd2, yd), (zd * xd * yd) / (xd2 * yd)
    if kind == "square":
        _, name, zd, xd, yd = layer
        zd2 = min(zd, cores)
        xd2 = max(1, min(xd, int(ct_budget // yd)))
        return ("square", name, zd2, xd2, yd), (zd * xd * yd) / (zd2 * xd2 * yd)
    raise ValueError(kind)


def run_reference_sample(budget_s, rng, literal_threads=False):
    """Times the UNMODIFIED reference layer classes (SEAL 2.3.1 Evaluator on the host cores) on a cropped PlainModel network and
    extrapolates linearly to the full layers.  STEADY STATE: every conv / fc layer object is built once, its first forward (which
    transforms the layer's weights to NTT form in place, convolutionalLayer.cpp:149-168, fullyConnectedLayer.cpp:129-131) is timed
    separately, and the per-image figure is a LATER forward of the same object -- what the reference pays per image
    (mainparams.cpp:84-111).  literal_threads: the reference's own thread constants (cnnBuilder.cpp:109: 40 / 50, i.e. the
    nf/th_count = 0 quirk that serialises conv1 and fc4) instead of one thread per core.
    Returns (images_per_s, cores, description, per_layer_seconds_full, extra)."""
    from oracle import ref as oref
    if not oref.available():
        return None
    cores = os.cpu_count() or 1
    r = oref.Ref(N_POLY, T_PLAIN, seed=1)
    weights = nets.load_weights(MODEL)
    layers = nets.TOPOLOGIES[MODEL]["layers"]
    LITERAL = {"pool1_features.conv1": 40, "pool2_features.conv2": 50, "act1": 50, "classifier.fc3": 40, "classifier.fc4": 50}
    # calibrate: one steady-state weighted-sum term and one generic multiply_plain, single thread
    x1 = synth_residues(rng, (2, 2), r.primes, N_POLY)
    c_term = max(r.fc_timed(x1, 2, 2, np.full(4, 0.37, np.float32), np.full(2, 0.1, np.float32), th=1, reps=1)[2] / 4, 1e-4)
    t0 = time.perf_counter()
    r.bn(x1, 1, 2, 1, [0.3], [1.7])
    c_ct = max((time.perf_counter() - t0) / 2, 1e-4)
    per_layer = budget_s / len(layers)
    total, total_first, desc, full_times, first_times = 0.0, 0.0, [], {}, {}
    for layer in layers:
        # a timed conv / fc sample costs encode + first forward + one steady forward: ~2.5x / ~7x one steady forward
        overhead = {"conv": 2.5, "fc": 7.0}.get(layer[0], 1.0)
        crop, scale = _crop_layer(layer, cores, per_layer / (c_term * overhead), per_layer / (4 * c_ct))
        kind, name = crop[0], crop[1]
        nin = nets.layer_io_counts(crop)[0]
        x = synth_residues(rng, (nin, 2), r.primes, N_POLY)
        first = None
        t0 = time.perf_counter()
        if kind == "conv":
            _, _, xd, yd, zd, xs, ys, xf, yf, nf = crop
            w = weights[name + ".weight"][:nf].ravel(); b = weights[name + ".bias"][:nf]
            # literal constants matter where th_count exceeds the layer's REAL output count: nf / th_count = 0 filters per thread and
            # the last thread takes them all (convolutionalLayer.cpp:177-187); elsewhere 40-50 threads on these cores are just oversubscribed
            serial = literal_threads and LITERAL[name] > layer[9]
            th = LITERAL[name] if serial else min(cores, nf)
            _, first, dt = r.conv_timed(x, xd, yd, zd, xs, ys, xf, yf, nf, w, b, th=th, reps=1)
        elif kind == "fc":
            _, _, i, o = crop
            serial = literal_threads and LITERAL[name] > layer[3]
            th = LITERAL[name] if serial else min(cores, o)
            _, first, dt = r.fc_timed(x, i, o, weights[name + ".weight"][:o].ravel(), weights[name + ".bias"][:o], th=th, reps=1)
        else:
            if kind in ("pool", "avgpool"):
                _, _, xd, yd, zd, xs, ys, xf, yf = crop
                r.pool(x, xd, yd, zd, xs, ys, xf, yf, avg=(kind == "avgpool"))
            elif kind == "bn":
                _, _, zd, xd, yd = crop
                var = weights[name + ".running_var"][:zd]
                r.bn(x, zd, xd, yd, weights[name + ".running_mean"][:zd], 1 / np.sqrt(var + 1e-5))
            elif kind == "square":
                _, _, zd, xd, yd = crop
                r.square_layer(x, zd, xd, yd, th=min(cores, zd))
            dt = time.perf_counter() - t0
        full_times[name] = dt * scale
        first_times[name] = (first if first is not None else dt) * scale
        total += dt * scale
        total_first += (first if first is not None else dt) * scale
        desc.append("%s x%.3g" % (name.split(".")[-1], scale))
    sample = ("reference layer classes (SEAL 2.3.1, -O3) on a cropped %s net, n=%d, %s; steady state (second forward of every layer object: "
              "weights already in NTT form); per-layer time x (full work / sample work): " % (
                  MODEL, N_POLY, "the reference's literal thread constants (cnnBuilder.cpp:109)" if literal_threads else "one thread per core") + ", ".join(desc))
    extra = {"first_image": {"value": 1.0 / total_first, "unit": "images/s",
                             "note": "the FIRST forward of every layer object, which also transforms the layer's weights to NTT form "
                                     "(a one-time cost the reference amortises over all later images; round 1 reported this figure)",
                             "per_layer_ms": {k: 1000 * v for k, v in first_times.items()}}}
    return 1.0 / total, cores, sample, full_times, extra


def main_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import ref as oref
    steps, warm = max(1, args.steps), max(0, args.warmup)
    if not oref.available():
        emit({"impl": "reference", "unavailable": "oracle/_ref/libcrcnn_ref.so was not built (needs /root/reference at build time)"})
        return
    rng = np.random.default_rng(0)
    per_step = max(3.0, 90.0 / (steps + warm))   # CPU seconds budgeted per sampled forward; the run measured 1.7x its budget (data generation, first forwards)
    vals = []
    for i in range(steps + warm):
        ips, cores, sample, full, extra = run_reference_sample(per_step, rng, literal_threads=args.literal_threads)
        if i >= warm:
            vals.append(ips)
    v = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": "encrypted MNIST images/sec", "value": v, "unit": "images/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1000.0 / v, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "PlainModel.h5 encoded net (conv-avgpool-bn-conv-square-avgpool-bn-fc-fc), n=8192, K=4, t=2^30, 32x32 zero-bordered input",
                   "note": "host CPU only; per-image time extrapolated from a bounded sample"},
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "per_layer_ms": {k: 1000 * s for k, s in full.items()},
    }
    line["cpu_baseline"].update(extra)
    emit(line)


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
def _init_dist(world, local_rank):
    import torch
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        return dist
    return None


def _barrier(dist):
    import torch
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(dist, values):
    import torch
    t = torch.tensor(values, device="cuda", dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def run_sharded(dist, rank, world, local_rank, batch, steps, warmup, rng_seed=1000):
    """BASELINE config 3 through the C++ host path: ApproxPlainModel.h5, n = 8192, conv / fc layers split by output neuron over
    `world` GPUs (crcnn_b200::ShardedNetwork, NCCL all-gathers of the activation ciphertexts on the compute stream).  Every rank
    runs the same batch; returns (on rank 0) latency per batch (max over ranks), the gather volume and a byte-equality verdict
    against the unsharded forward of the same input."""
    import hashlib
    from crcnn_b200 import host
    K, n = len(PRIMES), N_POLY
    nccl_id = None
    if world > 1:
        box = [host.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        nccl_id = box[0]
    rng = np.random.default_rng(rng_seed)          # the same images and keys on every rank
    evk = synth_evk(rng, PRIMES, n)
    net = host.HostNetwork(n, PRIMES, T_PLAIN, "ApproxPlainModel", device=local_rank, evk=evk, world=world, rank=rank, nccl_id=nccl_id)
    per_image = net.zd * net.xd * net.yd
    pin, own = host.pinned_array(batch * per_image * net.ct_words())
    synth_residues(rng, (batch * per_image, 2), PRIMES, n, out=pin.reshape(batch * per_image, 2, K, n + 1))
    _barrier(dist)
    net.resident_begin(own.ptr, batch)
    net.resident_run(max(1, warmup))
    _barrier(dist)
    ms, per_layer = net.resident_run(steps)
    _barrier(dist)
    net.resident_end()
    ms = _max_over_ranks(dist, [ms])[0] / steps
    got, _ = net.forward(pin, batch=batch)
    digest = hashlib.sha256(got.tobytes()).hexdigest()
    names = net.layer_names
    net.close()
    if dist is not None:
        digests = [None] * world
        dist.all_gather_object(digests, digest)
    else:
        digests = [digest]
    if rank != 0:
        return None
    single = host.HostNetwork(n, PRIMES, T_PLAIN, "ApproxPlainModel", device=local_rank, evk=evk)
    want, _ = single.forward(pin, batch=batch)
    ms1 = ms
    if world > 1:
        ms1 = single.resident_steps(own.ptr, batch, 1, max(1, steps))[0] / max(1, steps)
    single.set_fusion(False)                     # the same network with every reference layer as its own call
    ms1_lbl = single.resident_steps(own.ptr, batch, 1, max(1, steps))[0] / max(1, steps)
    single.close()
    equal = all(d == hashlib.sha256(want.tobytes()).hexdigest() for d in digests)
    ct_bytes = 2 * K * n * W
    # exchanged: batch-norm 1 output before conv2 (20 x 11 x 11) and batch-norm 2 output before the composed fc3*fc4 layer (800), which every
    # rank evaluates in full (10 rows) -- fc3's 500 rows and the 10 scores are no longer exchanged
    gathered = batch * (20 * 11 * 11 + 800) * ct_bytes * (world - 1) / max(1, world)
    return {"model": "ApproxPlainModel.h5, n=8192, K=4, t=2^30", "images_per_batch": batch, "gpus": world,
            "ms_per_batch": ms, "images_per_s": batch * 1000.0 / ms, "ms_per_batch_one_gpu_same_run": ms1,
            "speedup_vs_one_gpu": ms1 / ms, "ms_per_batch_one_gpu_layer_by_layer": ms1_lbl, "per_layer_ms_rank0": dict(zip(names, per_layer)),
            "all_gather_bytes_received_per_rank_per_batch": gathered,
            "bit_identical_to_unsharded_forward_on_every_rank": bool(equal),
            "host": "C++17 crcnn_b200::ShardedNetwork + crcnn_comm_all_gather (NCCL send/recv group on the compute stream, no host syncs); conv1+pool+bn: "
                    "this rank's channels of the pooled-grid layer; fc3*fc4 composed and evaluated by every rank"}


def main_shard(args, rank, world, local_rank):
    """--mode shard: the sharded forward as the headline line (strong scaling: total work fixed, latency per batch is the step)."""
    dist = _init_dist(world, local_rank)
    sampler = ClockSampler(local_rank); sampler.start()
    res = run_sharded(dist, rank, world, local_rank, args.batch, args.steps, max(3, args.warmup))
    clocks = sampler.stop()
    if rank == 0:
        emit({
            "metric": "encrypted MNIST images/sec", "value": res["images_per_s"], "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": res["ms_per_batch"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic: uniform residues in SEAL ciphertext layout; weights = ApproxPlainModel.h5",
            "config": {"workload": "ApproxPlainModel.h5 encoded net, n=8192, K=4, t=2^30, one batch of %d images, conv/fc layers sharded by output neuron" % args.batch,
                       "parallelism": "output-neuron shards x%d, NCCL all-gather of activation ciphertexts before conv2 and before the composed fc3*fc4 layer" % world},
            "shard": res, "clocks": clocks})
    if dist is not None:
        dist.destroy_process_group()


# BASELINE config 4: t ~ 2^30 as a product of pairwise coprime moduli (all coprime to every q_i, SEAL/seal/context.cpp:63-68), one per GPU
CRT_MODULI = {1: [1 << 30], 2: [32771, 32779], 4: [181, 191, 193, 197], 8: [5, 7, 11, 13, 17, 19, 23, 29]}


def main_b200(args, rank, world, local_rank):
    import torch
    from crcnn_b200 import host
    from crcnn_b200.lib import Engine

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    dist = _init_dist(world, local_rank)

    B, K, n = args.batch, len(PRIMES), N_POLY
    t_plain = T_PLAIN
    crt = None
    if args.mode == "crt":
        # one independent instance (context, keys, encoded weights) per GPU; the ranks work on the SAME images under different t_i,
        # the key holder recombines the decrypted coefficients by CRT (tests/test_gpu_crt.py checks that end to end)
        if world not in CRT_MODULI:
            raise SystemExit("--mode crt runs on 1, 2, 4 or 8 GPUs")
        moduli = CRT_MODULI[world]
        t_plain = moduli[rank]
        prod = 1
        for m in moduli:
            prod *= m
        crt = {"moduli": moduli, "product_bits": round(float(np.log2(prod)), 2)}
    rng = np.random.default_rng(1000 + (0 if crt else rank))
    evk_host = synth_evk(rng, PRIMES, n)
    # the C++17 host path: Runtime::init + CnnBuilder(h5).buildNetwork(topology) + BatchServer (crcnn_b200/cpp/)
    net = host.HostNetwork(n, PRIMES, t_plain, MODEL, device=local_rank, evk=evk_host)
    eng = Engine.adopt(net.ctx(), n, PRIMES, t_plain)     # the same context, for the profiling / probe entry points of the C ABI
    per_image = net.zd * net.xd * net.yd
    ct_words = 2 * K * (n + 1)
    in_words = B * per_image * ct_words
    numa = _bind_to_gpu_numa_node(torch, local_rank)     # pinned host buffers on the GPU's own NUMA node (first touch); affinity restored below
    pin_in, own_in = host.pinned_array(in_words)
    synth_residues(rng, (B * per_image, 2), PRIMES, n, out=pin_in.reshape(B * per_image, 2, K, n + 1))
    n_scores = net.outputs
    pin_out, own_out = host.pinned_array(B * n_scores * ct_words)
    if numa:
        os.sched_setaffinity(0, numa["restore"])
    h2d = in_words * 8
    d2h = B * n_scores * ct_words * 8
    layer_names = net.layer_names
    layers = nets.TOPOLOGIES[MODEL]["layers"]

    # ---- warm-up (also builds the resident weight forms once), then the timed device-resident steps
    _barrier(dist)                                       # NCCL sets its channels up lazily in the first collective: not inside the timed region
    net.resident_begin(own_in.ptr, B)
    net.resident_run(max(3, args.warmup))
    _barrier(dist)
    eng.prof_reset(); eng.prof_enable(True)
    last_scores = np.empty(B * n_scores * ct_words, dtype=np.uint64) if args.dump_outputs else None
    sampler = ClockSampler(local_rank); sampler.start()
    ms_total, per_layer_list = net.resident_run(args.steps, out=last_scores)
    _barrier(dist)
    clocks = sampler.stop()
    net.resident_end()
    prof = eng.prof()
    work = eng.prof_work()
    eng.prof_enable(False)
    # ---- timed: end to end through the serving loop (BatchServer) with host buffers
    mem_free = [torch.cuda.mem_get_info()[0] / 1e9]
    net.serve(own_in.ptr, own_out.ptr, B, 2)             # untimed: staging buffer and the two input tensors exist before the clock starts
    _barrier(dist)
    alloc0 = eng.alloc_stats()
    ms_e2e = net.serve(own_in.ptr, own_out.ptr, B, args.steps)
    _barrier(dist)
    if last_scores is not None and not np.array_equal(last_scores, np.asarray(pin_out)):
        raise RuntimeError("scores of the last timed resident step differ from the serving loop's scores of the same input")
    alloc1 = eng.alloc_stats()
    alloc_e2e = {k: alloc1[k] - alloc0[k] for k in ("pool_mallocs", "cache_hits", "cache_bypass", "flushes", "small_mallocs")}
    serve_done = net.serve_times()
    request_ms = [round(b - a, 1) for a, b in zip([0.0] + serve_done[:-1], serve_done)]
    mem_free.append(torch.cuda.mem_get_info()[0] / 1e9)
    # the host link by itself: one plain pinned H2D copy of a step's input (explains e2e when the link is the limit)
    host_t = torch.empty(in_words, dtype=torch.int64, pin_memory=True)
    dev_buf = torch.empty(in_words, dtype=torch.int64, device="cuda")
    ev3 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    dev_buf.copy_(host_t, non_blocking=True)
    ev3[0].record()
    dev_buf.copy_(host_t, non_blocking=True)
    ev3[1].record()
    torch.cuda.synchronize()
    h2d_gbs = h2d / ev3[0].elapsed_time(ev3[1]) / 1e6
    del dev_buf, host_t

    # ---- the same steps with every reference layer as its own call (layer fusion off): what the algebraic folds are worth, and the
    # ternary-tap GEMM of fc3 (which the composed fc3*fc4 layer replaces) measured at the headline shape
    lbl_steps = max(1, min(args.steps, 5))
    net.set_fusion(False)
    net.resident_begin(own_in.ptr, B)
    net.resident_run(3)
    _barrier(dist)
    eng.prof_reset(); eng.prof_enable(True)
    ms_lbl, per_layer_lbl = net.resident_run(lbl_steps)
    _barrier(dist)
    net.resident_end()
    prof_lbl, work_lbl = eng.prof(), eng.prof_work()
    eng.prof_enable(False)
    net.set_fusion(True)

    ms_total, ms_e2e, ms_lbl = _max_over_ranks(dist, [ms_total, ms_e2e, ms_lbl])
    images = B * args.steps * (1 if crt else world)
    value = images / (ms_total / 1000.0)
    e2e_value = images / (ms_e2e / 1000.0)
    per_layer = dict(zip(layer_names, per_layer_list))

    # ---- per-class rooflines from the engine's own work counters (crcnn_prof_get_work: algorithmic bytes and
    # operations counted at launch time, SURVEY 8(d)) and the CUDA-event time of every launch of the class
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    bf16_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    # integer pipe: 64x64->128-bit multiply-accumulates per second of a register-only loop, measured in this run
    probe_ms = eng.probe_imad(148 * 8, 256, 4096)
    probe_rate = 148 * 8 * 256 * 4096 * 8 / (probe_ms / 1000.0)
    # hard denominators, measured in this run on this device (crcnn_probe_pipe): the IMAD.WIDE issue rate (independent chains, nothing
    # else in the loop) and the kind::i8 UMMA rate with smem-resident operands and no epilogue
    eng.probe_pipe(1, 148 * 8, 256, 512); eng.probe_pipe(2, 148, 128, 256)            # warm
    wide_rate, _ = eng.probe_pipe(1, 148 * 8, 256, 4096)                               # IMAD.WIDE thread-instructions / s
    umma_rate, _ = eng.probe_pipe(2, 148, 128, 4096)                                   # int8 MACs / s
    counters = {}  # ncu counters of each class's main kernel from the committed capture of this round (tools/make_traffic.py)
    try:
        counters = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("counters", {})
    except Exception:
        pass
    traffic = {}   # measured DRAM bytes per launch of each class's main kernel, from the committed ncu capture (tools/make_traffic.py)
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = {k: v["dram_bytes_per_launch"] for k, v in tj["classes"].items()}
    except Exception:
        pass
    MAC_CLASSES = ("weighted_sum_mac", "behz_lift", "behz_floor_sk")
    BFLY_CLASSES = ("ntt_forward", "ntt_inverse", "square_tensor", "plain_expand_ntt", "relinearize")   # square_tensor: ntt_inv_tensor_kernel (3 products + 3 inverse transforms per limb)
    BFLY_MACS = 2.5  # one Harvey butterfly = 10 IMAD-pipe instructions (mulhi64 + two mullo64) = 2.5 split-accumulator MACs of 4
    # IMAD-pipe instruction slots per counted operation (an IMAD / IMAD.WIDE occupies the pipe 2 clk per warp, an IMAD.HI 4):
    # 64x64->128 MAC = 4 IMAD.WIDE; 64-bit Harvey butterfly = mulhi64 (4) + two mullo64 (3 each) = 10; 32-bit butterfly = IMAD.HI (2) + 2 IMAD = 4
    IMAD_SLOTS = {"mac": 4.0, "bfly64": 10.0, "bfly32": 4.0}
    kernel_ms, classes = {}, {}
    for name, (launches_c, ms_c) in prof.items():
        if not launches_c:
            continue
        byts, ops = work.get(name, (0.0, 0.0))
        sec = ms_c / 1000.0
        ent = {"launches_per_step": launches_c / args.steps, "ms_per_step": ms_c / args.steps,
               "share_of_step": ms_c / ms_total, "alg_gb_per_step": byts / args.steps / 1e9,
               "hbm_gbs": byts / sec / 1e9 if sec else None, "hbm_frac": byts / sec / 1e9 / hbm_peak if sec else None}
        if name == "weighted_sum_tc_i8":
            ent["int8_tops"] = 2 * ops / sec / 1e12
            ent["tensor_frac"] = ops / sec / umma_rate                       # vs the UMMA kind::i8 rate measured in this run
            ent["tensor_frac_vs_2x_bf16"] = ent["int8_tops"] / (2 * bf16_peak)   # round 1's derived denominator, kept for comparison
        elif name in MAC_CLASSES:
            ent["gmac_s"] = ops / sec / 1e9
            ent["int_pipe_frac"] = IMAD_SLOTS["mac"] * ops / sec / wide_rate
            ent["int_pipe_frac_vs_mac_chain"] = ops / sec / probe_rate
        elif name in BFLY_CLASSES:
            ent["gbutterfly_s"] = ops / sec / 1e9
            ent["int_pipe_frac"] = IMAD_SLOTS["bfly64"] * ops / sec / wide_rate
            ent["int_pipe_frac_vs_mac_chain"] = BFLY_MACS * ops / sec / probe_rate
        elif name == "relinearize_u32":
            # relinearize through 30-bit auxiliary primes (relin32.cuh): ops = 32-bit Harvey butterflies (1 IMAD.HI + 2 IMAD)
            ent["gbutterfly32_s"] = ops / sec / 1e9
            ent["int_pipe_frac"] = IMAD_SLOTS["bfly32"] * ops / sec / wide_rate
            ent["int_pipe_frac_vs_mac_chain"] = 0.75 * ops / sec / probe_rate
        if name in counters:
            ent["ncu"] = counters[name]      # pipe_tensor / pipe_fma / issue_active ... of the class's main kernel (committed capture)
        classes[name] = ent
        kernel_ms[name] = {"launches_per_step": ent["launches_per_step"], "ms_per_step": ent["ms_per_step"]}
    # the dominant KERNEL: classes that bundle several kernels (relinearize_u32: scale / digits / mac / intt / crt; weighted_sum_tcn_i8: three GEMM
    # instantiations; pool_sum: NTT-form and tap kernels) stay in `classes`, but none of their members is larger than the largest
    # single-kernel class (launch list of the same step: profiles/r02P_launches.txt)
    BUNDLES = ("relinearize_u32", "relinearize", "weighted_sum_tcn_i8", "pool_sum", "reencrypt")
    single = {k: v for k, v in classes.items() if k not in BUNDLES} or classes
    dom = max(single.items(), key=lambda kv: kv[1]["ms_per_step"])
    dname, d = dom
    avg_launch_ms = d["ms_per_step"] / d["launches_per_step"]
    if dname == "weighted_sum_tc_i8":
        roofline = {"kernel": dname, "bound": "tensor", "achieved": d["int8_tops"], "peak": 2 * umma_rate / 1e12, "unit": "TFLOP/s",
                    "frac": d["tensor_frac"],
                    "peak_source": "tcgen05.mma kind::i8 M128xN256xK32 issued back to back from shared-memory operands on all SMs, measured in "
                                   "this run (crcnn_probe_pipe which=2); achieved counts 2 ops per int8 multiply-accumulate of the unpadded GEMM",
                    "frac_vs_2x_measured_bf16": d["tensor_frac_vs_2x_bf16"]}
    else:
        roofline = {"kernel": dname, "bound": "hbm", "achieved": d["hbm_gbs"], "peak": hbm_peak, "unit": "GB/s",
                    "frac": d["hbm_frac"], "peak_source": peak_src}
        if "int_pipe_frac" in d:
            roofline["int_pipe"] = {"frac": d["int_pipe_frac"], "imad_wide_ginstr_s": wide_rate / 1e9,
                                    "note": "the binding resource of this kernel: the IMAD (FMA-heavy) pipe; frac = NECESSARY multiplier slots of the counted "
                                            "operations / the IMAD.WIDE.U32 issue rate measured in this run (slots per operation: %r); the pipe's "
                                            "actual busy share, overhead instructions included, is ncu.pipe_fmaheavy_cycles_pct" % (IMAD_SLOTS,)}
    if dname in counters:
        roofline["ncu"] = counters[dname]    # hardware counters of this kernel from the committed capture: pipe_fmaheavy_cycles_pct is the multiplier pipe's busy share
    roofline.update({"traffic": traffic.get(dname), "avg_launch_ms": avg_launch_ms, "launches_per_step": d["launches_per_step"],
                     "share_of_step": d["share_of_step"], "alg_bytes_per_launch": d["alg_gb_per_step"] * 1e9 / d["launches_per_step"],
                     "int_pipe_probe_gmac_s": probe_rate / 1e9, "imad_wide_probe_ginstr_s": wide_rate / 1e9,
                     "umma_i8_probe_tops": 2 * umma_rate / 1e12, "classes": classes})
    launches = int(sum(v[0] for v in prof.values()))
    layer_by_layer = {"value": B * lbl_steps * (1 if crt else world) / (ms_lbl / 1000.0), "unit": "images/s", "ms_per_step": ms_lbl / lbl_steps,
                      "steps": lbl_steps, "per_layer_ms": dict(zip(layer_names, per_layer_lbl)),
                      "note": "layer fusion off (crcnn_b200::Network::fuse_* = false): one C-ABI call per reference layer, same output bytes"}
    if prof_lbl.get("weighted_sum_tc_i8", (0, 0.0))[0]:
        l_c, ms_c = prof_lbl["weighted_sum_tc_i8"]
        ops = work_lbl.get("weighted_sum_tc_i8", (0.0, 0.0))[1]
        layer_by_layer["weighted_sum_tc_i8"] = {"ms_per_step": ms_c / lbl_steps, "int8_tops": 2 * ops / (ms_c / 1000.0) / 1e12,
                                                "tensor_frac": ops / (ms_c / 1000.0) / umma_rate, "ncu": counters.get("weighted_sum_tc_i8")}

    workload = ("PlainModel.h5 encoded net (conv-avgpool-bn-conv-square-avgpool-bn-fc-fc), n=8192, K=4, t=2^30, 32x32 zero-bordered input"
                if (MODEL, N_POLY) == ("PlainModel", 8192) else "%s encoded net, n=%d, K=%d, t=2^%d" % (MODEL, N_POLY, K, T_PLAIN.bit_length() - 1))
    parallelism = "image replicas x%d (no collective)" % world
    if crt:
        workload = "%s encoded net, n=%d, K=%d, plaintext modulus ~2^30 split into %d CRT moduli %r (one instance per GPU)" % (MODEL, N_POLY, K, world, crt["moduli"])
        parallelism = "CRT plaintext-modulus instances x%d: independent contexts on the same images, no collective; images/s of the ensemble" % world
    line = {
        "metric": "encrypted MNIST images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "strong" if crt else "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic: uniform residues in SEAL ciphertext layout; weights = %s.h5" % MODEL,
        "config": {"workload": workload, "images_per_step_per_gpu": B, "parallelism": parallelism,
                   "host": "C++17: crcnn_b200::CnnBuilder + Network::forward_dev (value) and BatchServer (e2e) behind libcrcnn_b200_host.so",
                   "l2": "inputs (%.1f GB per step) and weights exceed the 126 MB L2; no flush needed" % (h2d / 1e9),
                   "fusion": "default engine behaviour, same output bytes as layer by layer (checked in parity_sample): conv1+avgpool1+bn1 as one weighted sum "
                             "on the pooled grid with the scale and batch-norm folded into its weights; avgpool2+bn2 back to back; fc3+fc4 as one composed "
                             "layer W4*W3 (built on the device at the first forward); `layer_by_layer` repeats the measurement with all of it off",
                   "weights": "conv1/conv2/fc4: byte planes of the NTT-form plaintexts resident (limb-split tcgen05 kind::i8 weighted sum in the NTT domain); fc3: ternary tap matrix resident (tcgen05 kind::i8 weighted sum in the coefficient domain)"},
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps, "h2d_link_gbs": h2d_gbs,
                "link_bound_below_ms_per_step": h2d / h2d_gbs / 1e6,   # the upload of a step at this rank's measured pinned H2D rate: a forward faster than this is link-bound end to end
                "device_mem_free_gb": {"after_resident_loop": round(mem_free[0], 1), "after_e2e_loop": round(mem_free[1], 1)},
                "request_ms": request_ms, "allocator": alloc_e2e, "pinned_numa_node": numa["node"] if numa else None,
                "note": "crcnn_b200::BatchServer: pinned H2D + re-stride of request i+1 on a copy stream while request i runs; scores come back "
                        "through an asynchronous pinned download; the timed region starts before the first upload (not overlapped) and ends when the last scores have landed"},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "per_layer_ms": per_layer, "kernel_ms": kernel_ms,
        "layer_by_layer": layer_by_layer,
    }
    if crt:
        line["crt"] = crt
    # ---- the checker leg (rank 0 at N = 1 only, outside every timed region): a sampled-oracle parity check of the bench's own
    # network at the bench's own shapes, and the reference's CPU path on the host cores
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            from oracle import sampled
            from oracle.port import Oracle
            pnet = nets.Network(eng, MODEL, evk=eng.evk_upload(*evk_host))       # the same C ABI calls on the same context
            x = eng.upload_ptr(own_in.ptr, B * per_image)
            checked, y_checked = sampled.check_network(eng, Oracle(n, PRIMES, t_plain), pnet, x, B, evk_host=evk_host, samples=2, seed=7, keep_last=True)
            x.free()
            # the layer-by-layer path the checker walked and the C++ host path the bench timed (fused layers, serving loop) must agree on
            # every byte of the scores: own_out still holds the last timed request's download of the same input
            scores_checked = eng.download(y_checked)
            y_checked.free()
            assert np.array_equal(scores_checked.ravel(), np.asarray(pin_out).ravel()), "scores of the timed C++ host path differ from the layer-by-layer path the oracle checked"
            line["parity_sample"] = "ok"
            line["parity_sample_detail"] = {"ciphertexts_checked_per_layer": checked, "timed_host_path_scores_equal_checked_path": True,
                                            "how": "oracle/sampled.py: random + first/last output ciphertexts of every layer of this run's network at batch %d, "
                                                   "bit-compared with the CPU oracle evaluated on their input windows" % B}
        except AssertionError as e:
            line["parity_sample"] = "FAILED: %s" % (e,)
        except Exception as e:
            line["parity_sample"] = "not run: %r" % (e,)
        try:
            res = run_reference_sample(args.cpu_budget_s, np.random.default_rng(0))
            if res is not None:
                ips, cores, sample, full, extra = res
                line["cpu_baseline"] = {"value": ips, "unit": "images/s", "cores": cores, "kind": "reference", "sample": sample,
                                        "per_layer_ms": {k: 1000 * s for k, s in full.items()}}
                line["cpu_baseline"].update(extra)
            else:
                line["cpu_baseline"] = port_baseline(args.cpu_budget_s)
        except Exception as e:  # the baseline must never take the GPU number down with it
            line["cpu_baseline"] = {"value": None, "unit": "images/s", "cores": 0, "kind": "reference", "sample": "failed: %r" % (e,)}
    eng.close()
    net.close()
    del pin_in, pin_out, own_in, own_out
    # ---- BASELINE config 3 alongside (every N): the neuron-sharded Approx network over the same GPUs, with a byte-equality check
    # against the unsharded forward, so the scaling record carries the sharded path too
    if not crt and not args.no_shard:
        try:
            shard = run_sharded(dist, rank, world, local_rank, args.shard_batch, max(1, min(args.steps, 3)), 1)
            if rank == 0:
                line["shard"] = shard
        except Exception as e:
            if rank == 0:
                line["shard"] = {"failed": repr(e)}
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last_scores.reshape(B, n_scores, 2, K, n + 1))
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


def port_baseline(budget_s):
    """Fallback when oracle/_ref is absent: the plain-C oracle port, one thread, a few terms."""
    from oracle.port import Oracle
    o = Oracle(N_POLY, PRIMES, T_PLAIN)
    rng = np.random.default_rng(0)
    x = synth_residues(rng, (4, 2), PRIMES, N_POLY)
    w = o.encode_many(np.full(8, 0.37, np.float32)); b = o.encode_many(np.full(2, 0.1, np.float32))
    t0 = time.perf_counter()
    o.fc(x, 4, 2, w, b)
    c_term = (time.perf_counter() - t0) / 8
    terms = sum(nets.layer_terms(l) for l in nets.TOPOLOGIES[MODEL]["layers"])
    return {"value": 1.0 / (terms * c_term), "unit": "images/s", "cores": 1, "kind": "port",
            "sample": "oracle port, 8 weighted-sum terms at n=8192, scaled by the net's %d terms (pool/bn/square excluded)" % terms}


def main():
    global MODEL, N_POLY, PRIMES, T_PLAIN
    args = parse()
    _claim_stdout()
    if args.model:
        MODEL = args.model
    if args.mode == "crt" and not args.model:
        MODEL = "PlainModelWoPad"
    if args.n:
        N_POLY, PRIMES = args.n, [int(q) for q in nets.DEFAULT_PRIMES_128[args.n]]
        T_PLAIN = (1 << 18) if args.n == 4096 else (1 << 30)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        main_reference(args, rank, world)
    elif args.mode == "shard":
        main_shard(args, rank, world, local_rank)
    else:
        main_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
