"""The weighted sums, window sums and relinearization at the size limits the engine itself declares, with worst-case operands.

Each limit is a point where a lazy accumulation must still fit its word; every case runs at the limit and one past it, checks the bytes
against the oracle or against a closed form that tests/test_limits_oracle.py proves on the oracle, and checks through the kernel-class
launch counters which kernel ran, so that a silent fallback cannot pass.
  - limb-split GEMM (tcn_mac.cuh): fan-in TCN_MAX_R = 4096 (s32 class sums 7 R 255^2 < 2^31), the column-major kernel's two K blocks
    (fan-in 256 / 257), the seven-class pre-shifted kernel (fan-in 32 / 33); fan-in 4097 must take the CUDA-core MAC;
  - ternary GEMM (tc_mac.cuh) at fan-in 4096 and 4100 with all-(+1) and all-(-1) digit rows against all-(q-1) inputs;
  - CUDA-core MAC with 60-bit primes at chunk_terms = 256 (the split 128-bit accumulator, modarith.cuh: Acc7), fan-in 256, 257, 513;
  - 64-bit window sums at sum_fits_64: R_max = floor((2^64 - 1) / max q) terms and R_max + 1, in the pooling, pooling + batch-norm,
    pooling + batch-norm + two fully connected layers, and add_many; the pooled-grid convolution at its Rp <= 64 cap and one past it;
  - relinearization at every decomposition bit count the ABI accepts: the word-size path while D <= 32 digits and dbc <= 16 (its generic
    MAC reduces between chunks of 16 digits), the 64-bit path beyond, an error beyond 63 digits.
Weights are constant plaintexts t - k (q - k in every NTT slot), inputs NTT-form slots of chosen residues: uniform ones for the largest
accumulator values, and near-maximal ones that vary per (output, term, column, slot) so that a permuted row or column shows.
"""
import os

import numpy as np
import pytest

from util import (PARAM_SETS, PRIMES, T_FOR_N, bias_slots, class_sums, const_weight_fc_slots, random_cts, random_evk,
                  slots_to_words, worst_operands)
from oracle.port import Oracle

pytestmark = pytest.mark.gpu

TCN_MAX_R = 4096


def _engine(n, primes, t):
    from crcnn_b200.lib import Engine
    return Engine(n, primes, t)


def _sets(name):
    if name.startswith("n"):
        n = int(name[1:])
        return n, PRIMES[n], T_FOR_N[n]
    return PARAM_SETS[name]


def _launches(eng, cls):
    return eng.prof().get(cls, (0, 0.0))[0]


def _counts(eng):
    return {c: _launches(eng, c) for c in ("weighted_sum_tcn_i8", "weighted_sum_tc_i8", "weighted_sum_mac", "relinearize_u32",
                                           "relinearize", "pool_sum", "batch_norm")}


def _delta(eng, before):
    now = _counts(eng)
    return {c: now[c] - before[c] for c in now}


def _const_pack(eng, t, k):
    """Weights (m, r) = the constant plaintext t - k[m][r] (lifts to q - k in every slot)."""
    k = np.asarray(k, dtype=np.int64).ravel()
    return eng.plain_upload_sparse(np.zeros(len(k), np.uint32), (t - k).astype(np.uint64), np.arange(len(k) + 1, dtype=np.uint32))


def _slot_inputs(primes, xb, d):
    """d [B][R][2][K][n] -> ciphertext words [B*R][2][K][n+1] whose NTT slots are xb[j] - d."""
    K = len(primes)
    s = np.stack([np.uint64(xb[j]) - d[:, :, :, j, :].astype(np.uint64) for j in range(K)], axis=3)
    return slots_to_words(s.reshape((-1,) + s.shape[2:]))


def _explain(got, want):
    bad = np.argwhere(got != want)
    if len(bad) == 0:
        return "equal"
    first = tuple(int(v) for v in bad[0])
    return "%d of %d words differ; first at %s: got %d want %d" % (len(bad), got.size, first, int(got[first]), int(want[first]))


# ============================================================================ limb-split GEMM
@pytest.fixture(scope="module", params=[2048, 4096])
def ls_env(request):
    n = request.param
    primes, t = PRIMES[n], T_FOR_N[n]
    eng = _engine(n, primes, t)
    eng.set_tensor_core_mode(0)      # keep the ternary-tap kernel out of the way
    eng.set_limb_split_mode(1)
    orc = Oracle(n, primes, t)
    yield n, primes, t, eng, orc, np.random.default_rng(97 * n)
    eng.close()


def _tcn_mac_bytes(K, n, R, M, ncols, preshift):
    """Work bytes the engine books for one limb-split GEMM over all K*n slots (engine.cu: run_weighted_sum_tcn): staged inputs,
    weight planes (seven blocks when pre-shifted), outputs.  Tells the seven-class kernel from the 13-class ones."""
    kpad = 32 if R <= 32 else max(128, (R + 31) // 32 * 32)
    return K * n * (7 * ncols * kpad + 7 * M * kpad * (7 if preshift else 1) + 8 * ncols * M)


# (fan-in, outputs, batch, limb-split mode): mode 1 picks the kernel by shape, 2 forces the row-major one, 3 the column-major one
# where it fits (fan-in <= 256); batch 4 with 2 outputs has 8 >= 4 x 2 columns: the shape that picks the column-major kernel by itself
LS_CASES = [(32, 2, 4, 1), (33, 2, 4, 1), (256, 2, 4, 1), (257, 2, 4, 1), (256, 3, 1, 2), (256, 3, 1, 3), (257, 3, 1, 3),
            (TCN_MAX_R, 65, 1, 1), (TCN_MAX_R + 1, 65, 1, 1)]


@pytest.mark.parametrize("R,M,B,mode", LS_CASES)
def test_limb_split_at_fan_in_limits(ls_env, R, M, B, mode):
    n, primes, t, eng, orc, rng = ls_env
    K = len(primes)
    if n == 4096 and M > 8:
        M = 2            # 65 x 4096 staged weights at n = 2048 only; n = 4096 runs the limit with one output tile
    k0, xb = worst_operands(primes, t)
    top = max(max(class_sums(q - k0, xb[j])) for j, q in enumerate(primes)) * min(R, TCN_MAX_R)
    print("n=%d R=%d: largest class sum %d = 2^%.4f (bound 2^31)" % (n, R, top, np.log2(top)))
    bv = rng.uniform(-3, 3, size=M).astype(np.float32)
    b_ = eng.plain_encode(bv)
    bias = bias_slots(orc, orc.encode_many(bv))
    tcn = R <= TCN_MAX_R
    preshift = R <= 32 and mode != 2 and (mode == 3 or 2 * B >= 4 * M)
    kinds = ["uniform"] + (["varied"] if R * K * n <= TCN_MAX_R * 2048 else [])
    for kind in kinds:
        if kind == "uniform":
            k = np.full((M, R), k0, dtype=np.int64)
            d = np.zeros((B, R, 2, K, n), dtype=np.int64)
        else:
            k = np.clip(k0 - rng.integers(0, 8, size=(M, R)), 1, (t - 1) // 2)
            d = rng.integers(0, 8, size=(B, R, 2, K, n))
        want = const_weight_fc_slots(k, xb, d, primes, bias)
        w = _const_pack(eng, t, k)
        x = eng.upload(_slot_inputs(primes, xb, d), ntt_form=True)
        del d

        def run():
            eng.prof_reset()
            eng.set_limb_split_mode(mode)
            try:
                y = eng.download(eng.fc(x, w, b_, B, R, M), ntt_form=True)
            finally:
                eng.set_limb_split_mode(1)
            return y.reshape(B, M, 2, K, n + 1)[..., :n], _counts(eng), eng.prof_work()
        got, cnt, work = run()
        assert np.array_equal(got, want), "%s: %s" % (kind, _explain(got, want))
        if tcn:
            assert cnt["weighted_sum_tcn_i8"] == 1 and cnt["weighted_sum_mac"] == 0, cnt
            assert work["weighted_sum_tcn_i8"][0] == _tcn_mac_bytes(K, n, R, M, 2 * B, preshift), (preshift, work)
        else:
            assert cnt["weighted_sum_tcn_i8"] == 0 and cnt["weighted_sum_mac"] == 1, cnt
        if R == TCN_MAX_R and kind == "uniform":
            # the 128-bit recombination + Barrett instead of the folded reduction
            eng.set_limb_split_reduction(0)
            try:
                got0, cnt0, _ = run()
            finally:
                eng.set_limb_split_reduction(1)
            assert cnt0["weighted_sum_tcn_i8"] == 1 and np.array_equal(got0, want), _explain(got0, want)
            # a small scratch budget: 512 slots per launch
            per_slot = 7 * 2 * B * R
            eng.set_tensor_core_mode(0, 0, 512 * per_slot)
            try:
                got1, cnt1, _ = run()
            finally:
                eng.set_tensor_core_mode(0, 0, 12 << 30)
            assert cnt1["weighted_sum_tcn_i8"] == K * n // 512 and np.array_equal(got1, want), (cnt1, _explain(got1, want))


def test_uniform_worst_case_is_r_w_x(ls_env):
    """The closed form at fan-in 4096 in its plainest shape: every slot of every output is R (q - k) x + bias mod q."""
    n, primes, t, eng, orc, rng = ls_env
    K = len(primes)
    k0, xb = worst_operands(primes, t)
    R, M = TCN_MAX_R, 2
    w = _const_pack(eng, t, np.full(M * R, k0))
    for j, q in enumerate(primes):
        assert np.all(eng.plain_get_ntt(w, 0)[j, :n] == q - k0)
    zero = eng.plain_upload_sparse([], [], np.zeros(M + 1, np.uint32))
    x = eng.upload(_slot_inputs(primes, xb, np.zeros((1, R, 2, K, n), np.int64)), ntt_form=True)
    before = _counts(eng)
    got = eng.download(eng.fc(x, w, zero, 1, R, M), ntt_form=True)
    assert _delta(eng, before)["weighted_sum_tcn_i8"] == 1
    for j, q in enumerate(primes):
        assert np.all(got[:, :, j, :n] == R * (q - k0) * xb[j] % q), j


def test_fc_fc_composed_at_fan_in_4096(ls_env):
    """Two fully connected layers 4096 -> 8 -> 2 as one composed layer: its weights W2 W1 are general residues at the limb-split GEMM's
    fan-in limit.  Composed, layer by layer and the closed form of the first layer followed by the oracle's second layer agree."""
    n, primes, t, eng, orc, rng = ls_env
    K = len(primes)
    R, mid, out = TCN_MAX_R, 8, 2
    k0, xb = worst_operands(primes, t)
    k = np.clip(k0 - rng.integers(0, 8, size=(mid, R)), 1, (t - 1) // 2)
    d = rng.integers(0, 8, size=(1, R, 2, K, n)) if n == 2048 else np.zeros((1, R, 2, K, n), np.int64)
    b1v, w2v, b2v = (rng.uniform(-3, 3, size=s).astype(np.float32) for s in (mid, out * mid, out))
    y1 = const_weight_fc_slots(k, xb, d, primes, bias_slots(orc, orc.encode_many(b1v)))[0]
    y1c = orc.ct_transform(slots_to_words(y1), inverse=True)
    want = orc.fc(y1c, mid, out, orc.encode_many(w2v), orc.encode_many(b2v)).reshape(out, 2, K, n + 1)
    packs = (_const_pack(eng, t, k), eng.plain_encode(b1v), eng.plain_encode(w2v), eng.plain_encode(b2v))
    x = eng.upload(_slot_inputs(primes, xb, d), ntt_form=True)
    del d

    def run():
        eng.prof_reset()
        y = eng.download(eng.fc_fc(x, *packs, 1, R, mid, out))
        return y.reshape(want.shape), _counts(eng), eng.prof_work()
    got0, _, _ = run()              # builds the composed weights (weighted sums of their own)
    got, cnt, work = run()          # steady state: the composed layer alone
    os.environ["CRCNN_NO_FC_COMPOSE"] = "1"
    try:
        got_l, cnt_l, work_l = run()
    finally:
        os.environ.pop("CRCNN_NO_FC_COMPOSE", None)
    assert np.array_equal(got0, want), _explain(got0, want)
    assert np.array_equal(got, want), _explain(got, want)
    assert np.array_equal(got_l, want), _explain(got_l, want)
    macs = lambda wk: sum(v[1] for c, v in wk.items() if c.startswith("weighted_sum"))
    assert cnt["weighted_sum_tcn_i8"] == 1 and cnt["weighted_sum_mac"] == 0, cnt
    assert cnt_l["weighted_sum_tcn_i8"] == 2, cnt_l
    assert macs(work) < macs(work_l), (work, work_l)


# ============================================================================ ternary GEMM
@pytest.fixture(scope="module")
def tc_env():
    n = 2048
    primes, t = PRIMES[n], T_FOR_N[n]
    eng = _engine(n, primes, t)
    eng.set_tensor_core_mode(2, 64)
    yield n, primes, t, eng, Oracle(n, primes, t), np.random.default_rng(4099)
    eng.close()


@pytest.mark.parametrize("R", [TCN_MAX_R, TCN_MAX_R + 4])
def test_ternary_gemm_at_large_fan_in(tc_env, R):
    """Digit rows all +1 and all -1 (+-(0.5 - 2^-24)) and random ones, 6 outputs (two 128-row tiles), against all-(q-1) coefficient inputs
    (batch item 0) and near-maximal ones that vary per word (item 1)."""
    n, primes, t, eng, orc, rng = tc_env
    K, M, B = len(primes), 6, 2
    wv = np.empty((M, R), dtype=np.float32)
    wv[0] = 0.5 - 2.0 ** -24
    wv[1] = -(0.5 - 2.0 ** -24)
    wv[2:] = rng.uniform(-0.49, 0.49, size=(M - 2, R))
    wv = wv.ravel()
    bv = rng.uniform(-0.49, 0.49, size=M).astype(np.float32)
    x = np.zeros((B * R, 2, K, n + 1), dtype=np.uint64)
    for j, q in enumerate(primes):
        x[:R, :, j, :n] = q - 1
        x[R:, :, j, :n] = q - 1 - rng.integers(0, 8, size=(R, 2, n)).astype(np.uint64)
    wp, bp = orc.encode_many(wv), orc.encode_many(bv)
    want = np.stack([orc.fc(x[b * R:(b + 1) * R], R, M, wp, bp) for b in range(B)]).reshape(B * M, 2, K, n + 1)
    before = _counts(eng)
    got = eng.download(eng.fc(eng.upload(x), eng.plain_encode(wv), eng.plain_encode(bv), B, R, M))
    cnt = _delta(eng, before)
    assert cnt["weighted_sum_tc_i8"] == 1 and cnt["weighted_sum_tcn_i8"] == 0 and cnt["weighted_sum_mac"] == 0, cnt
    assert np.array_equal(got, want), _explain(got, want)


# ============================================================================ CUDA-core MAC at chunk_terms
@pytest.fixture(scope="module", params=["P60a", "P60b"])
def p60_env(request):
    n, primes, t = PARAM_SETS[request.param]
    eng = _engine(n, primes, t)
    yield n, primes, t, eng, Oracle(n, primes, t), np.random.default_rng(len(primes) * 6000)
    eng.close()


@pytest.mark.parametrize("R", [256, 257, 513])
def test_cuda_core_mac_at_chunk_terms(p60_env, R):
    """60-bit primes: 8 byte planes, so every weighted sum takes the CUDA-core MAC, which reduces its 128-bit accumulators every
    chunk_terms = 256 terms.  W = X = q - 1 gives R mod q in every slot (plus the bias); near-maximal operands (k in [1, 8], slot values
    q - 1 - [0, 8)) follow the closed form; fan-in 257 is also compared with the oracle.  Batch 2 runs the 2 x 2 output tile, batch 1
    (one position) the 4 x 1 tile (kernels.cu: launch_mac)."""
    n, primes, t, eng, orc, rng = p60_env
    K, M = len(primes), 3
    bv = rng.uniform(-3, 3, size=M).astype(np.float32)
    b_ = eng.plain_encode(bv)
    bias = bias_slots(orc, orc.encode_many(bv))
    xb = [q - 1 for q in primes]
    for B, kind in ((2, "uniform"), (2, "varied"), (1, "uniform"), (1, "varied")):
        k = np.ones((M, R), np.int64) if kind == "uniform" else rng.integers(1, 9, size=(M, R))
        d = np.zeros((B, R, 2, K, n), np.int64) if kind == "uniform" else rng.integers(0, 8, size=(B, R, 2, K, n))
        want = const_weight_fc_slots(k, xb, d, primes, bias)
        if kind == "uniform":
            for j, q in enumerate(primes):
                assert np.all(want[:, :, 1, j] == R % q)
        xw = _slot_inputs(primes, xb, d)
        before = _counts(eng)
        got = eng.download(eng.fc(eng.upload(xw, ntt_form=True), _const_pack(eng, t, k), b_, B, R, M), ntt_form=True)
        cnt = _delta(eng, before)
        assert cnt["weighted_sum_mac"] == 1 and cnt["weighted_sum_tcn_i8"] == 0, cnt
        got = got.reshape(B, M, 2, K, n + 1)[..., :n]
        assert np.array_equal(got, want), "B=%d %s: %s" % (B, kind, _explain(got, want))
        if kind == "varied" and R == 257:
            xc = orc.ct_transform(xw[:R], inverse=True)
            wp = np.zeros((M * R, n + 1), np.uint64)
            wp[:, 0] = t - k.ravel()
            ref = orc.ct_transform(orc.fc(xc, R, M, wp, orc.encode_many(bv)).reshape(M, 2, K, n + 1))[..., :n]
            assert np.array_equal(got[0], ref), _explain(got[0], ref)


# ============================================================================ 64-bit window sums at sum_fits_64
# R_max = floor((2^64 - 1) / max q): 1024 at n = 2048, 512 at n = 4096, 16 for P60a.  Windows (xf, yf) of R_max and R_max + 1 terms.
WINDOWS = {"n2048": [(32, 32), (25, 41)], "n4096": [(16, 32), (27, 19)], "P60a": [(4, 4), (17, 1)]}


@pytest.fixture(scope="module", params=sorted(WINDOWS))
def pool_env(request):
    n, primes, t = _sets(request.param)
    eng = _engine(n, primes, t)
    yield request.param, n, primes, t, eng, Oracle(n, primes, t), np.random.default_rng(n + len(primes))
    eng.close()


def _all_max(primes, n, count):
    x = np.zeros((count, 2, len(primes), n + 1), dtype=np.uint64)
    for j, q in enumerate(primes):
        x[:, :, j, :n] = q - 1
    return x


@pytest.mark.parametrize("past", [0, 1])
def test_window_sums_at_sum_fits_64(pool_env, past):
    name, n, primes, t, eng, orc, rng = pool_env
    K = len(primes)
    xf, yf = WINDOWS[name][past]
    R, zd = xf * yf, 2
    assert (R <= (2 ** 64 - 1) // max(primes)) == (past == 0)
    x = _all_max(primes, n, zd * R)
    xc_ntt = orc.ct_transform(x, inverse=True)          # the coefficient form of NTT slots all q - 1
    geo = (1, xf, yf, zd, 1, 1, xf, yf)
    d, cc = orc.encode(1.0 / R)
    scale = eng.plain_encode_f64([1.0 / R])
    mv = rng.uniform(-3, 3, size=zd).astype(np.float32)
    vv = rng.uniform(-3, 3, size=zd).astype(np.float32)
    mp, vp = orc.encode_many(mv), orc.encode_many(vv)
    mean, invstd = eng.plain_encode(mv), eng.plain_encode(vv)
    for domain in ("coef", "ntt"):
        xin = x if domain == "coef" else xc_ntt
        up = lambda: eng.upload(x, ntt_form=(domain == "ntt"))
        # sum pooling: q - (R mod q) in every word of either domain
        before = _counts(eng)
        t_out = eng.pool(up(), *geo)
        assert _delta(eng, before)["pool_sum"] == 1
        raw = eng.download(t_out, ntt_form=(domain == "ntt"))
        for j, q in enumerate(primes):
            assert np.all(raw[:, :, j, :n] == q - R % q), (domain, j, _explain(raw[:, :, j, :n], np.full_like(raw[:, :, j, :n], q - R % q)))
        want = orc.pool(xin, xf, yf, zd, 1, 1, xf, yf).reshape(zd, 2, K, n + 1)
        assert np.array_equal(eng.download(t_out), want), domain
        # average pooling
        want_a = orc.pool(xin, xf, yf, zd, 1, 1, xf, yf, d, cc).reshape(zd, 2, K, n + 1)
        got_a = eng.download(eng.pool(up(), *geo, scale=scale))
        assert np.array_equal(got_a, want_a), (domain, _explain(got_a, want_a))
        # pooling + batch-norm: one pass for NTT-form input whose sums fit 64 bits, else the two layers
        want_b = orc.bn(want_a, zd, 1, 1, mp, vp).reshape(zd, 2, K, n + 1)
        before = _counts(eng)
        got_b = eng.download(eng.pool_bn(up(), *geo, scale, mean, invstd))
        fused = domain == "ntt" and past == 0
        assert _delta(eng, before)["batch_norm"] == (0 if fused else 1), (domain, past)
        assert np.array_equal(got_b, want_b), (domain, _explain(got_b, want_b))
    # add_many over R_max and R_max + 1 ciphertexts
    xs = x[:R]
    got = eng.download(eng.add_many(eng.upload(xs)))[0]
    assert np.array_equal(got, orc.add_many(xs))
    for j, q in enumerate(primes):
        assert np.all(got[:, j, :n] == q - R % q)


@pytest.mark.parametrize("past", [0, 1])
def test_pool_bn_fc_fc_at_sum_fits_64(pool_env, past):
    """Window sums + one composed layer while the window sums fit 64 bits (and the primes the limb-split GEMM), else pooling + batch-norm
    as two layers before the fully connected pair."""
    name, n, primes, t, eng, orc, rng = pool_env
    K = len(primes)
    xf, yf = WINDOWS[name][past]
    R, zd, mid, out = xf * yf, 2, 3, 1
    x = _all_max(primes, n, zd * R)
    x[::3, :, :, :n] -= rng.integers(0, 8, size=x[::3, :, :, :n].shape).astype(np.uint64)
    xc = orc.ct_transform(x, inverse=True)
    vals = lambda s, lo=-3.0: rng.uniform(lo, 3, size=s).astype(np.float32)
    mv, vv, w1v, b1v, w2v, b2v = vals(zd), vals(zd), vals(mid * zd), vals(mid), vals(out * mid), vals(out)
    d, cc = orc.encode(1.0 / R)
    e = orc.encode_many
    y = orc.bn(orc.pool(xc, xf, yf, zd, 1, 1, xf, yf, d, cc), zd, 1, 1, e(mv), e(vv)).reshape(zd, 2, K, n + 1)
    want = orc.fc(orc.fc(y, zd, mid, e(w1v), e(b1v)).reshape(mid, 2, K, n + 1), mid, out, e(w2v), e(b2v)).reshape(out, 2, K, n + 1)
    packs = [eng.plain_encode_f64([1.0 / R])] + [eng.plain_encode(v) for v in (mv, vv, w1v, b1v, w2v, b2v)]
    run = lambda: eng.download(eng.pool_bn_fc_fc(eng.upload(x, ntt_form=True), 1, xf, yf, zd, 1, 1, xf, yf, *packs, mid, out))
    first = run()                   # builds the composed weights (weighted sums of their own)
    assert np.array_equal(first, want), _explain(first, want)
    before = _counts(eng)
    got = run()
    cnt = _delta(eng, before)
    # fitting sums: the composed layer (limb-split primes) or the one-pass pooling + batch-norm; past the bound: the two layers
    assert cnt["batch_norm"] == past, cnt
    if max(int(q).bit_length() for q in primes) <= 56:
        assert cnt["weighted_sum_tcn_i8"] == 1 and cnt["weighted_sum_mac"] == 0, cnt
    else:
        assert cnt["weighted_sum_mac"] >= 1 and cnt["weighted_sum_tcn_i8"] == 0, cnt
    assert np.array_equal(got, want), _explain(got, want)


@pytest.mark.parametrize("rp", [(8, 8), (5, 13)])
def test_conv_pool_bn_pooled_grid_cap(pool_env, rp):
    """The pooled-grid convolution sums Rp = pxf * pyf inputs per window (Rp <= 64): 8 x 8 windows take it, 5 x 13 the layer-by-layer path
    (which compares the work of the weighted sums with and without CRCNN_NO_POOLED_CONV)."""
    name, n, primes, t, eng, orc, rng = pool_env
    K = len(primes)
    pxf, pyf = rp
    pooled_grid = pxf * pyf <= 64 and name != "P60a"     # 60-bit primes have no limb-split GEMM: layer by layer at any Rp
    xf = yf = 2
    zd, nf, pxs, pys = 1, 2, 2, 2
    xd, yd = pxf + 1, pyf + 1
    x = _all_max(primes, n, zd * xd * yd)
    x[::2, :, :, :n] -= rng.integers(0, 8, size=x[::2, :, :, :n].shape).astype(np.uint64)
    vals = lambda s: rng.uniform(-3, 3, size=s).astype(np.float32)
    wv, bv, mv, vv = vals(nf * zd * xf * yf), vals(nf), vals(nf), vals(nf)
    e = orc.encode_many
    d, cc = orc.encode(1.0 / (pxf * pyf))
    c = orc.conv(x, xd, yd, zd, 1, 1, xf, yf, nf, e(wv), e(bv)).reshape(nf * pxf * pyf, 2, K, n + 1)
    want = orc.bn(orc.pool(c, pxf, pyf, nf, pxs, pys, pxf, pyf, d, cc), nf, 1, 1, e(mv), e(vv)).reshape(nf, 2, K, n + 1)
    packs = (eng.plain_encode_f64([1.0 / (pxf * pyf)]), eng.plain_encode(mv), eng.plain_encode(vv))
    w, b_ = eng.plain_encode(wv), eng.plain_encode(bv)
    geo = (1, xd, yd, zd, 1, 1, xf, yf, nf, pxs, pys, pxf, pyf)

    def run():
        eng.prof_reset()
        y = eng.download(eng.conv_pool_bn(eng.upload(x), w, b_, *geo, *packs))
        return y.reshape(want.shape), eng.prof_work()
    got, work = run()
    os.environ["CRCNN_NO_POOLED_CONV"] = "1"
    try:
        got_l, work_l = run()
    finally:
        os.environ.pop("CRCNN_NO_POOLED_CONV", None)
    assert np.array_equal(got, want), _explain(got, want)
    assert np.array_equal(got_l, want), _explain(got_l, want)
    macs = lambda wk: sum(v[1] for c_, v in wk.items() if c_.startswith("weighted_sum"))
    assert (macs(work) < macs(work_l)) == pooled_grid, (work, work_l)


# ============================================================================ relinearize at every digit width
@pytest.fixture(scope="module", params=[2048, 4096, 8192, 16384])
def relin_env(request):
    n = request.param
    primes, t = PRIMES[n], T_FOR_N[n]
    eng = _engine(n, primes, t)
    yield n, primes, t, eng, Oracle(n, primes, t), np.random.default_rng(3 * n + 1)
    eng.close()


def _ones_digits(q, dbc):
    """The largest residue below q whose dbc-bit digits below the top one are all 2^dbc - 1."""
    s = dbc * ((int(q).bit_length() - 1) // dbc)
    if s == 0:
        return int(q) - 1
    return ((((int(q) - 1) >> s) - 1) << s) | ((1 << s) - 1)


def test_relinearize_every_digit_width(relin_env):
    """Keys with dbc = 1 .. 60 bit digits (a subset at n = 16384).  The word-size auxiliary-prime path runs when the digits fit its
    16-bit planes (dbc <= 16), K is a power of two up to 8 and the digit count D <= 32 (relin32_applicable); its register MAC takes
    D = 4K, the generic one the rest, reducing between chunks of 16 digits.  Beyond that the 64-bit path; beyond 63 digits an error.
    Operands: random keys and keys of q - 1, c2 random, q - 1, 0 and all-ones digits."""
    n, primes, t, eng, orc, rng = relin_env
    from crcnn_b200.lib import CrcnnError
    K = len(primes)
    bits = [int(q).bit_length() for q in primes]
    dbcs = range(1, 61) if n <= 8192 else [7, 8, 13, 14, 15, 16, 17, 30, 60]
    x3 = random_cts(rng, n, primes, 4, size=3)
    for j, q in enumerate(primes):
        x3[1, 2, j, :n] = q - 1
        x3[2, 2, j, :n] = 0
    seen = set()
    for dbc in dbcs:
        digits = [(b + dbc - 1) // dbc for b in bits]
        D = sum(digits)
        for j, q in enumerate(primes):
            x3[3, 2, j, :n] = _ones_digits(q, dbc)
        evk, sizes, _ = random_evk(rng, n, primes, dbc)
        evk_max = evk.reshape(-1, K, n + 1).copy()
        for j, q in enumerate(primes):
            evk_max[:, j, :n] = q - 1
        for keys in (evk, evk_max.ravel()):
            k = eng.evk_upload(keys, sizes, dbc)
            if D > 63:
                with pytest.raises(CrcnnError):
                    eng.relinearize(eng.upload(x3, size=3), k)
                seen.add("error")
                break
            want = orc.relinearize(x3, keys, sizes, dbc)
            for mode in (1, 0):
                word = mode == 1 and dbc <= 16 and K in (1, 2, 4, 8) and D <= 32
                eng.set_relin_mode(mode)
                try:
                    before = _counts(eng)
                    got = eng.download(eng.relinearize(eng.upload(x3, size=3), k))
                    cnt = _delta(eng, before)
                finally:
                    eng.set_relin_mode(1)
                assert (cnt["relinearize_u32"], cnt["relinearize"]) == ((1, 0) if word else (0, 1)), (dbc, D, mode, cnt)
                assert np.array_equal(got, want), (dbc, D, mode, _explain(got, want))
                if word:
                    seen.add("register" if D == 4 * K else ("generic, %d chunk%s" % ((D + 15) // 16, "s" if D > 16 else "")))
                else:
                    seen.add("64-bit, %s 32 digits" % ("over" if D > 32 else "up to"))
    print("n=%d: %s" % (n, sorted(seen)))
    if n == 8192:
        assert {"register", "generic, 2 chunks", "64-bit, over 32 digits", "error"} <= seen, seen

