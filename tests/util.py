"""Shared helpers for the tests: synthetic workloads and the two checkers (oracle port, reference)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import port as oport  # noqa: E402
from oracle import ref as oref  # noqa: E402

PRIMES = oport.DEFAULT_PRIMES_128
T_FOR_N = {2048: 1 << 16, 4096: 1 << 18, 8192: 1 << 30, 16384: 1 << 30}

# Parameter sets beyond SEAL's defaults: {name: (n, primes, t)}.  Every prime is = 1 (mod 2n).  They take the kernels' other
# branches: 56-bit primes (the full top byte plane of the limb-split GEMM), 57-60-bit primes (8 byte planes in the ternary GEMM,
# no limb-split GEMM, mode 2 of the forward transform on q, partial sums in the CUDA-core MAC, R * q >= 2^64), primes without
# the 2^k - delta shape (Barrett instead of the folds), small primes (other relinearization digit counts), K not a power of two
# (the generic BEHZ and the 64-bit relinearize), an extra auxiliary prime (L = K + 1) and odd or tiny plain moduli.
PARAM_SETS = {
    "P56": (4096, [0xfffffffff78001, 0xfffffffff70001], 1 << 18),
    "P57": (4096, [0x1fffffffffc0001], 1 << 18),
    "P57n16384": (16384, [0x1fffffffffc0001], 1 << 18),
    "P60a": (4096, [0xffffffffffe8001], 1 << 30),
    "P60b": (4096, [0xffffffffffe8001, 0xffffffffffd8001], (1 << 31) - 1),
    "U50": (4096, [0x2fffffff50001, 0x2ffffffee0001], 1 << 18),
    "U40": (2048, [0xbffffe8001], 1 << 8),
    "U30": (2048, [0x2ffd0001], 1 << 4),
    "K3": (8192, PRIMES[16384][:3], 1 << 30),
    "K5": (8192, PRIMES[16384][:5], 1 << 30),
    "K7": (8192, PRIMES[16384][:7], 1 << 30),
    "T2": (4096, PRIMES[4096], 2),
    "T3": (4096, PRIMES[4096], 3),
    "T5": (4096, PRIMES[4096], 5),
    "T32771": (4096, PRIMES[4096], 32771),
}


def have_ref():
    return oref.available()


def random_cts(rng, n, primes, count, size=2):
    """Uniform canonical residues in SEAL layout -- indistinguishable from ciphertexts for the evaluator."""
    K = len(primes)
    out = np.zeros((count, size, K, n + 1), dtype=np.uint64)
    for j, q in enumerate(primes):
        out[:, :, j, :n] = rng.integers(0, q, size=(count, size, n), dtype=np.uint64)
    return out


def random_evk(rng, n, primes, dbc=16):
    K = len(primes)
    sizes = [2 * ((int(q).bit_length() + dbc - 1) // dbc) for q in primes]
    parts = [random_cts(rng, n, primes, 1, s).ravel() for s in sizes]
    return np.concatenate(parts), sizes, dbc


def synthetic_image(seed, count=784):
    """SURVEY 8(d): i.i.d. uniform in the normalised MNIST range, seeded per image."""
    rng = np.random.default_rng(1000 + seed)
    return rng.uniform(-0.4242, 2.8215, size=count).astype(np.float32)


# ---- version-independent deterministic data (splitmix64), used by the hash-pinned golden cases
def splitmix64(start, count):
    z = (np.arange(count, dtype=np.uint64) + np.uint64(start)) * np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def det_cts(seed, n, primes, count, size=2):
    K = len(primes)
    out = np.zeros((count, size, K, n + 1), dtype=np.uint64)
    raw = splitmix64(seed * 1000003, count * size * K * n).reshape(count, size, K, n)
    for j, q in enumerate(primes):
        out[:, :, j, :n] = raw[:, :, j, :] % np.uint64(q)
    return out


def det_floats(seed, count):
    return ((splitmix64(seed * 7919 + 17, count) >> np.uint64(11)).astype(np.float64) / float(1 << 53) * 2 - 1).astype(np.float32)


def det_evk(seed, n, primes, dbc=16):
    sizes = [2 * ((int(q).bit_length() + dbc - 1) // dbc) for q in primes]
    return np.concatenate([det_cts(seed + 100 + i, n, primes, 1, s).ravel() for i, s in enumerate(sizes)]), sizes, dbc


def sha(a):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.uint64).tobytes()).hexdigest()


# the hash-pinned chain: conv(2ch 4x4 -> 3 filters 2x2, stride 1) -> avgpool 2x2/1 -> bn -> square -> fc(12 -> 4)
CHAIN = dict(xd=4, yd=4, zd=2, nf=3)


def chain_params(seed):
    return dict(conv_w=det_floats(seed + 1, 3 * 2 * 2 * 2), conv_b=det_floats(seed + 2, 3), mean=det_floats(seed + 3, 3),
                invstd=np.abs(det_floats(seed + 4, 3)) + np.float32(0.5), fc_w=det_floats(seed + 5, 4 * 12), fc_b=det_floats(seed + 6, 4))


def run_chain(backend, kind, x, p, evk, sizes, dbc):
    """Runs the chain on `backend` (kind: 'ref' | 'oracle' | 'gpu'); returns the list of per-layer outputs (numpy)."""
    outs = []
    if kind == "ref":
        r = backend
        o = r.conv(x, 4, 4, 2, 1, 1, 2, 2, 3, p["conv_w"], p["conv_b"]); outs.append(o)
        o = r.pool(o, 3, 3, 3, 1, 1, 2, 2, avg=True); outs.append(o)
        o = r.bn(o, 3, 2, 2, p["mean"], p["invstd"]); outs.append(o)
        o = r.square_layer(o, 3, 2, 2); outs.append(o)
        o = r.fc3d(o, 3, 2, 2, 4, p["fc_w"], p["fc_b"]); outs.append(o)
    elif kind == "oracle":
        r = backend
        e = r.encode_many
        d, cc = r.encode(0.25)
        o = r.conv(x, 4, 4, 2, 1, 1, 2, 2, 3, e(p["conv_w"]), e(p["conv_b"])); outs.append(o)
        o = r.pool(o, 3, 3, 3, 1, 1, 2, 2, d, cc); outs.append(o)
        o = r.bn(o, 3, 2, 2, e(p["mean"]), e(p["invstd"])); outs.append(o)
        o = r.square_layer(o, evk, sizes, dbc); outs.append(o)
        o = r.fc(o, 12, 4, e(p["fc_w"]), e(p["fc_b"])); outs.append(o)
    else:
        g = backend
        e = g.plain_encode
        t = g.conv(g.upload(x), e(p["conv_w"]), e(p["conv_b"]), 1, 4, 4, 2, 1, 1, 2, 2, 3); outs.append(g.download(t))
        t = g.pool(t, 1, 3, 3, 3, 1, 1, 2, 2, scale=e([0.25])); outs.append(g.download(t))
        t = g.bn(t, 1, 3, 2, 2, e(p["mean"]), e(p["invstd"])); outs.append(g.download(t))
        t = g.square_layer(t, g.evk_upload(evk, sizes, dbc)); outs.append(g.download(t))
        t = g.fc(t, e(p["fc_w"]), e(p["fc_b"]), 1, 12, 4); outs.append(g.download(t))
    return outs


# the evaluator and layer cases pinned on the reference (tests/test_oracle_vs_reference.py, tests/golden/reference_ops.json)
ENC_VALUES = [0.0867, -3.25, 0.0, 1.0, -1.0, 7.0, 0.25, 2.8215, -0.4242, 1 / 9.0, -17.5, 1e-9, 123456.789]
REF_OPS = {2048: (1 << 16, 2048), 4096: (1 << 18, 4096), 8192: (1 << 30, 8192)}   # n: (t, seed)


def ref_ops(kind, r, n, primes, t, seed):
    """Runs the cases on `r` (kind: 'ref' = oracle.ref.Ref, 'oracle' = oracle.port.Oracle) and returns {name: output array}.
    Inputs are splitmix64 residues, floats and evaluation keys, the same for both; the pool case `avgpool9` encodes the
    DOUBLE 1/9 as the reference does (avgPoolingLayer.cpp:10-13)."""
    out = {}
    for i, v in enumerate(ENC_VALUES + [float(v) for v in det_floats(seed, 40) * 3]):
        a, cc = r.encode(float(v))
        out["encode_%02d" % i] = np.append(a, np.uint64(cc))
    evk, sizes, dbc = det_evk(seed, n, primes)
    if kind == "ref":
        r.set_evk(evk, sizes, dbc)
    x = det_cts(seed + 1, n, primes, 5)
    xn = r.ct_transform(x)
    out["ct_ntt"], out["ct_intt"] = xn, r.ct_transform(xn, inverse=True)
    w, _ = r.encode(0.0867)
    wn = r.plain_to_ntt(w)
    out["plain_ntt"], out["multiply_plain_ntt"] = wn, r.multiply_plain_ntt(xn, wn)
    dense = np.zeros(n + 1, dtype=np.uint64)
    dense[:n] = splitmix64(seed * 31 + 5, n) % np.uint64(t)
    for j, plain in enumerate((w, dense, np.array([t - 2], dtype=np.uint64), np.array([3], dtype=np.uint64))):
        for op in ("mul", "add", "sub"):
            out["plain_%s_%d" % (op, j)] = r.plain_op(x, plain, op)
    out["add_many"] = r.add_many(x)
    s3 = r.square(det_cts(seed + 2, n, primes, 3))
    out["square"] = s3
    out["relinearize"] = r.relinearize(s3) if kind == "ref" else r.relinearize(s3, evk, sizes, dbc)
    xi = det_cts(seed + 3, n, primes, 2 * 3 * 3)
    wv, bv, wf, bf = det_floats(seed + 4, 16), det_floats(seed + 5, 2), det_floats(seed + 6, 3 * 18), det_floats(seed + 7, 3)
    mean, invstd = [0.3, -0.2], [1.7, 0.9]
    if kind == "ref":
        out["conv"] = r.conv(xi, 3, 3, 2, 1, 1, 2, 2, 2, wv, bv)
        out["fc"] = r.fc3d(xi, 2, 3, 3, 3, wf, bf)
        out["pool"] = r.pool(xi, 3, 3, 2, 1, 1, 2, 2)
        out["avgpool"] = r.pool(xi, 3, 3, 2, 1, 1, 2, 2, avg=True)
        out["avgpool9"] = r.pool(xi, 3, 3, 2, 1, 1, 3, 3, avg=True)
        out["bn"] = r.bn(xi, 2, 3, 3, mean, invstd)
        out["square_layer"] = r.square_layer(xi[:4], 1, 2, 2)
    else:
        e = r.encode_many
        out["conv"] = r.conv(xi, 3, 3, 2, 1, 1, 2, 2, 2, e(wv), e(bv))
        out["fc"] = r.fc(xi, 18, 3, e(wf), e(bf))
        out["pool"] = r.pool(xi, 3, 3, 2, 1, 1, 2, 2)
        out["avgpool"] = r.pool(xi, 3, 3, 2, 1, 1, 2, 2, *r.encode(0.25))
        out["avgpool9"] = r.pool(xi, 3, 3, 2, 1, 1, 3, 3, *r.encode(1.0 / 9.0))
        out["bn"] = r.bn(xi, 2, 3, 3, e(mean), e(invstd))
        out["square_layer"] = r.square_layer(xi[:4], evk, sizes, dbc)
    return out


# ---- worst-case operands at the weighted sums' accumulator limits (tests/test_limits_oracle.py proves these on the oracle,
# tests/test_gpu_limits.py runs them on the device)
def class_sums(w, x, planes=7):
    """One term w * x of the limb-split GEMM (tcn_mac.cuh): both split into `planes` unsigned bytes, class c = a + b collects
    byte_a(w) * byte_b(x).  Returns the 2 * planes - 1 class values; a layer of fan-in R with uniform operands sums R of them."""
    wb = [(int(w) >> (8 * a)) & 0xff for a in range(planes)]
    xb = [(int(x) >> (8 * b)) & 0xff for b in range(planes)]
    return [sum(wb[a] * xb[c - a] for a in range(max(0, c - planes + 1), min(c, planes - 1) + 1)) for c in range(2 * planes - 1)]


def ones_below(q, width=8):
    """Values below q whose low digits of `width` bits are all ones (one per digit count), and q - 1."""
    out = {int(q) - 1}
    for s in range(width, int(q).bit_length(), width):
        top = ((int(q) - 1) >> s) - 1
        if top >= 0:
            out.add((top << s) | ((1 << s) - 1))
    return sorted(out)


def worst_operands(primes, t):
    """(k, [x_j]) maximising the largest class sum: weights are the constant plaintext t - k, which lifts to q_j - k in every NTT slot
    of every prime (k <= (t - 1) / 2), slot values x_j < q_j.  k is shared by the primes (one plaintext), x_j is per prime."""
    kmax = (int(t) - 1) // 2
    ks = set(range(1, min(kmax, 255) + 1))
    for q in primes:
        ks.update(int(q) - v for v in ones_below(q) if 1 <= int(q) - v <= kmax)
    best = None
    for k in sorted(ks):
        xs, score = [], 0
        for q in primes:
            m, x = max((max(class_sums(int(q) - k, v)), v) for v in ones_below(q))
            xs.append(x)
            score += m
        if best is None or score > best[0]:
            best = (score, k, xs)
    return best[1], best[2]


def acc7_even(w, x, terms, carry=0):
    """The 128-bit `even` half of the CUDA-core MAC's split accumulator (modarith.cuh: Acc7) after `terms` products w * x on top of a
    reduced residue `carry`: sum of lo32(x) lo32(w) + hi32(x) hi32(w) 2^64.  Must stay below 2^128 for chunk_terms terms."""
    x0, x1, w0, w1 = int(x) & 0xffffffff, int(x) >> 32, int(w) & 0xffffffff, int(w) >> 32
    return int(carry) + terms * (x0 * w0 + ((x1 * w1) << 64))


def const_weight_fc_slots(k, xb, d, primes, bias=None):
    """Closed form of a fully connected layer in the NTT domain with constant-plaintext weights: weight (m, r) is q_j - k[m][r] in every
    slot, input slot (b, r, poly, j, s) is xb[j] - d[b][r][poly][j][s].  Then
        Y[b][m][poly][j][s] = sum_r (q_j - k[m][r]) (xb[j] - d[...]) = sum_r k[m][r] d[...] - xb[j] sum_r k[m][r]   (mod q_j)
    (+ bias[m][j][s] on polynomial 0).  k: [M][R] ints, d: [B][R][2][K][n] small ints.  Returns [B][M][2][K][n] uint64.
    The products k d are exact in float64 while R * max(k) * max(d) < 2^53."""
    k = np.asarray(k, dtype=np.int64)
    M, R = k.shape
    B, _, _, K, n = d.shape
    assert R * int(k.max()) * max(1, int(d.max())) < (1 << 53)
    ks = [int(v) for v in k.sum(axis=1)]
    out = np.zeros((B, M, 2, K, n), dtype=np.uint64)
    kf = k.astype(np.float64)
    for b in range(B):
        kd = (kf @ d[b].reshape(R, -1).astype(np.float64)).astype(np.int64).reshape(M, 2, K, n)
        for j, q in enumerate(primes):
            q = int(q)
            for m in range(M):
                a = int(xb[j]) * ks[m] % q
                y = (kd[m, :, j, :] % q - a) % q
                if bias is not None:
                    y[0] = (y[0] + bias[m][j].astype(np.int64)) % q
                out[b, m, :, j, :] = y.astype(np.uint64)
    return out


def slots_to_words(slots):
    """[..][K][n] slot values -> [..][K][n + 1] SEAL-layout words (the unused last word 0)."""
    out = np.zeros(slots.shape[:-1] + (slots.shape[-1] + 1,), dtype=np.uint64)
    out[..., :-1] = slots
    return out


def bias_slots(orc, bias_plain):
    """NTT slots [M][K][n] the bias of a layer adds to polynomial 0: the transform of Delta * b (add_plain on a zero ciphertext)."""
    M = len(bias_plain)
    z = np.zeros((M, 2, orc.K, orc.n + 1), dtype=np.uint64)
    out = np.zeros((M, orc.K, orc.n), dtype=np.uint64)
    for m in range(M):
        y = orc.ct_transform(orc.plain_op(z[m:m + 1], bias_plain[m], "add"))
        out[m] = y[0, 0, :, :orc.n]
    return out
