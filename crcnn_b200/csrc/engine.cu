// C ABI implementation (include/crcnn_b200.h): contexts, device tensors, plaintext packs,
// evaluation keys, the layer forwards and the evaluator-level operations, all on top of the
// kernels in kernels.cu.  Host code only orchestrates; every arithmetic step runs on the GPU.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>
#include <unordered_map>
#include <string>
#include <vector>

#include "../../include/crcnn_b200.h"
#include "kernels.cuh"
#include "params.h"
#include "tc_mac.cuh"
#include "tcn_mac.cuh"
#include "relin32.cuh"
#include "reenc.cuh"

using namespace crcnn;

namespace {

enum KernelClass {
    KC_NTT_FWD = 0, KC_NTT_INV, KC_MAC, KC_PLAIN_EXPAND, KC_POOL, KC_BN, KC_PLAIN_OP,
    KC_BEHZ_LIFT, KC_SQ_TENSOR, KC_BEHZ_FLOOR, KC_RELIN, KC_PROBE, KC_TC_SPLIT, KC_TC_MAC, KC_TCN_SPLIT, KC_TCN_MAC, KC_RELIN32, KC_REENC, KC_COUNT
};
const char *kClassNames[KC_COUNT] = {"ntt_forward", "ntt_inverse", "weighted_sum_mac", "plain_expand_ntt", "pool_sum",
                                     "batch_norm", "plain_op", "behz_lift", "square_tensor", "behz_floor_sk",
                                     "relinearize", "imad_probe", "tc_plane_split", "weighted_sum_tc_i8", "tcn_plane_split",
                                     "weighted_sum_tcn_i8", "relinearize_u32", "reencrypt"};

thread_local std::string g_create_error;

}  // namespace

struct crcnn_tensor {
    long count;
    int size;
    int ntt;  // 0 coefficient form, 1 NTT form
    uint64_t *d;
};

static long next_plain_serial() { static long s = 0; return ++s; }   // contexts are driven by one thread each; ids only need to differ within a process

struct crcnn_plain {
    long serial = next_plain_serial();   // identity that survives address reuse (the fused constants below are keyed on it)
    long count;
    bool sparse_shape = false;       // every plaintext supported in [0,64) U [n-32,n) (FractionalEncoder output)
    std::vector<uint32_t> off, idx;  // host copy of the sparse form
    std::vector<uint64_t> val;
    uint32_t *d_off = nullptr, *d_idx = nullptr;
    uint64_t *d_val = nullptr;
    uint64_t *ntt_mul = nullptr;   // [count][K][n] NTT(lift)            (multiplicative use)
    uint64_t *ntt_mul_sh = nullptr;  // Shoup companions of ntt_mul (small packs only: pooling scale, batch-norm factors)
    uint64_t *ntt_add = nullptr;   // [count][K][n] NTT(Delta-scaled)    (additive use, NTT-form data)
    uint64_t *coef_add = nullptr;  // [count][K][n] Delta-scaled         (additive use, coefficient-form data)
    int tap_state = 0;             // 0 not examined, 1 every term is +-1 at an exponent in [0,64) U [n-32,n) (tapmul_kernel applies), -1 not
    // tensor-core form (tc_mac.cuh): ternary tap matrix [count/R * 32 (+128 pad rows)][Kpad] for fan-in R
    int tc_state = 0;              // 0 not examined, 1 eligible, -1 not (support outside x^(n-32..n-1) or digits other than +-1)
    int8_t *tc_A = nullptr;
    int tc_R = 0, tc_Kpad = 0;
    // limb-split tensor-core form (tcn_mac.cuh): byte planes of the NTT-form weights [K*n][7][count/R][Kpad]; pre-shifted
    // (tcn_pre): seven such blocks, block b holding the planes of W 2^(8b) mod q_j (block 0 is the plain staging)
    uint8_t *tcn_W = nullptr;
    int tcn_R = 0;
    bool tcn_pre = false;
    // fused average pooling + batch-norm (this pack = the batch-norm factors): C[z] = scale (.) invstd[z] with Shoup companions and
    // D[z] = mean[z] (.) invstd[z] in NTT form, valid for the (scale, mean) packs they were made from
    uint64_t *fused_C = nullptr, *fused_Csh = nullptr, *fused_D = nullptr;
    long fused_scale = 0, fused_mean = 0;   // serials of the packs the constants were made from
    // "this plaintext added add_mult times": the additive forms hold add_mult * (Delta-scaled plaintext) mod q.  A bias pack keeps the
    // derived pack the fused convolution + pooling path adds (one bias per pooled convolution output = window-size biases per sum).
    int add_mult = 1;
    bool dense_only = false;       // a derived pack that exists only in its device forms (no sparse plaintexts to expand from)
    // a convolution's weight pack keeps the packs of the pooled-grid path (crcnn_conv_pool_bn_forward): weights and bias with the pooling
    // scale and the batch-norm folded in, valid for the packs whose serials are in folded_key
    crcnn_plain *folded_w = nullptr, *folded_b = nullptr;
    long folded_key[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
};

struct crcnn_evk {
    uint64_t *d = nullptr;
    long key_off[MAXK];
    int digits[MAXK];
    int dbc;
    bool has_r32 = false;  // keys also converted for the word-size auxiliary-prime path (relin32.cuh)
    Relin32 r32;
};

struct crcnn_keys {
    uint64_t *sk = nullptr;   // [K][n]    secret key, NTT form
    uint64_t *pk = nullptr;   // [2][K][n] public key, NTT form
    ReencConsts c;
    BudgetConsts b;
};

struct crcnn_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    HostParams hp;
    DeviceParams *dP = nullptr;
    std::vector<void *> owned;  // table buffers
    int n = 0, logn = 0, K = 0, S = 0;
    int chunk_terms = 1 << 30;
    size_t weight_cache_bytes = 24ull << 30;
    int sm_count = 148;
    int tc_mode = 1;                 // 1: weighted sums with fan-in >= tc_min_fanin and >= tc_min_outputs outputs run on tcgen05 kind::i8 when the weights allow it; 2: regardless of the output count
    int tc_min_fanin = 256;
    int tc_min_outputs = 32;
    int tap_mode = 1;                // 1: avg-pool / batch-norm on coefficient-form inputs multiply in the coefficient domain (tapmul_kernel); env CRCNN_TAP
    int relin_mode = 1;              // 1: relinearize through 30-bit auxiliary primes when exact for the parameters (relin32.cuh); 0: 64-bit transforms
    int tcn_mode = 1;                // 1: weighted sums whose staged weights fit the weight cache run as the NTT-domain limb-split GEMM (tcn_mac.cuh)
    int sq_lean = 1;                 // 1 (default): square's tensor products reduce through the 2^k - delta fold when every modulus allows, and the inverse transforms feeding the BEHZ lift / floor leave n^-1 to their constants (params.h: *_n); 0: Barrett products, n^-1 in the transforms; same bytes; env CRCNN_SQ_LEAN
    int tcn_preshift = 1;            // 1 (default): convolution weights of fan-in <= 32 are staged pre-shifted and run on the seven-class kernel (tcn_mac.cu: tcn2p_mac_kernel) when 7x the planes fit the weight cache; 0: 13-class kernel; same bytes; env CRCNN_TCN2_PRESHIFT
    int tcn_fold = 1;                // 1 (default): the limb-split GEMM reduces its class sums through the 2^k - delta shape of the primes when every prime has it (modarith.cuh: tcn_fold_reduce), 0: 128-bit recombination + Barrett; same bytes; env CRCNN_TCN_FOLD
    size_t tc_scratch_bytes = 12ull << 30;
    std::string err;
    std::map<std::vector<int>, int *> index_cache;
    // Large device blocks (activations, GEMM staging, transform scratch) are recycled by exact size: a forward pass asks for the same
    // sizes step after step, and the stream-ordered allocator, although it never releases memory here, occasionally has to re-map
    // physical memory when its free list is fragmented -- a 100+ ms stall in the middle of a step (seen in pool1 of the bench network).
    // All work of a context runs on one stream, so a block freed after its last consumer was enqueued may be handed out again at once.
    std::unordered_map<void *, size_t> big_size;   // live and cached blocks >= kBigBlock
    std::multimap<size_t, void *> big_free;        // cached, by size
    size_t big_cached = 0, big_cache_cap = 64ull << 30;
    long long st_big_malloc = 0, st_big_hit = 0, st_big_bypass = 0, st_flush = 0, st_small_malloc = 0;   // crcnn_ctx_alloc_stats
    uint64_t *stage = nullptr;       // persistent H2D staging buffer of crcnn_tensor_upload_into (host layout, pad words included)
    size_t stage_bytes = 0;
    // profiling
    bool prof_on = false;
    long launches[KC_COUNT] = {0};
    double ms[KC_COUNT] = {0};
    double work_bytes[KC_COUNT] = {0};  // algorithmic (compulsory) HBM bytes enqueued per class since the last reset
    double work_ops[KC_COUNT] = {0};    // algorithmic operations (unit depends on the class, see crcnn_prof_get_work)
    struct Pending { int cls; cudaEvent_t a, b; };
    std::vector<Pending> pending;
    std::vector<cudaEvent_t> event_pool;
};

namespace {

int fail(crcnn_ctx *ctx, int code, const std::string &msg) {
    if (ctx) ctx->err = msg; else g_create_error = msg;
    return code;
}

#define CU(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e__ = (call);                                                                      \
        if (e__ != cudaSuccess) {                                                                      \
            int code__ = (e__ == cudaErrorMemoryAllocation) ? CRCNN_ERR_OUT_OF_MEMORY : CRCNN_ERR_CUDA; \
            return fail(ctx, code__, std::string(#call) + ": " + cudaGetErrorString(e__));            \
        }                                                                                              \
    } while (0)

#define REQUIRE(cond, msg) \
    do { if (!(cond)) return fail(ctx, CRCNN_ERR_INVALID_ARGUMENT, msg); } while (0)

struct ProfScope {
    crcnn_ctx *c; int cls; cudaEvent_t a = nullptr, b = nullptr;
    ProfScope(crcnn_ctx *ctx, int k, double bytes = 0, double ops = 0) : c(ctx), cls(k) {
        c->launches[cls]++;
        c->work_bytes[cls] += bytes;
        c->work_ops[cls] += ops;
        if (!c->prof_on) return;
        auto get = [&]() { cudaEvent_t e; if (!c->event_pool.empty()) { e = c->event_pool.back(); c->event_pool.pop_back(); } else cudaEventCreate(&e); return e; };
        a = get(); b = get();
        cudaEventRecord(a, c->stream);
    }
    ~ProfScope() {
        if (!a) return;
        cudaEventRecord(b, c->stream);
        c->pending.push_back({cls, a, b});
    }
};

void prof_collect(crcnn_ctx *c) {
    for (auto &p : c->pending) {
        cudaEventSynchronize(p.b);
        float t = 0;
        cudaEventElapsedTime(&t, p.a, p.b);
        c->ms[p.cls] += t;
        c->event_pool.push_back(p.a);
        c->event_pool.push_back(p.b);
    }
    c->pending.clear();
}

inline size_t poly_words(const crcnn_ctx *c) { return (size_t)c->K * c->n; }
// algorithmic work of `polys` limb-polynomials: bytes of one pass over them, butterflies of one transform each
inline double lp_bytes(const crcnn_ctx *c, double polys) { return polys * c->n * 8.0; }
inline double lp_bfly(const crcnn_ctx *c, double polys) { return polys * (c->n / 2) * c->logn; }

constexpr size_t kBigBlock = 32ull << 20;
void big_cache_flush(crcnn_ctx *ctx) {
    for (auto &kv : ctx->big_free) { ctx->big_size.erase(kv.second); cudaFreeAsync(kv.second, ctx->stream); }
    ctx->big_free.clear();
    ctx->big_cached = 0;
}
int dev_alloc(crcnn_ctx *ctx, size_t bytes, void **out) {
    *out = nullptr;
    if (bytes == 0) return CRCNN_OK;
    if (bytes >= kBigBlock) {
        auto it = ctx->big_free.find(bytes);
        if (it != ctx->big_free.end()) {
            *out = it->second;
            ctx->big_cached -= bytes;
            ctx->big_free.erase(it);
            ctx->st_big_hit++;
            return CRCNN_OK;
        }
        ctx->st_big_malloc++;
    } else {
        ctx->st_small_malloc++;
    }
    cudaError_t e = cudaMallocAsync(out, bytes, ctx->stream);
    if (e == cudaErrorMemoryAllocation && !ctx->big_free.empty()) {   // the cache holds what the allocator needs: give it back and retry
        cudaGetLastError();
        ctx->st_flush++;
        big_cache_flush(ctx);
        e = cudaMallocAsync(out, bytes, ctx->stream);
    }
    CU(e);
    if (bytes >= kBigBlock) ctx->big_size[*out] = bytes;
    return CRCNN_OK;
}
void dev_free(crcnn_ctx *ctx, void *p) {
    if (!p) return;
    auto it = ctx->big_size.find(p);
    if (it != ctx->big_size.end()) {
        if (ctx->big_cached + it->second <= ctx->big_cache_cap) {
            ctx->big_free.insert({it->second, p});
            ctx->big_cached += it->second;
            return;
        }
        ctx->big_size.erase(it);
        ctx->st_big_bypass++;
    }
    cudaFreeAsync(p, ctx->stream);
}

int new_tensor(crcnn_ctx *ctx, long count, int size, int ntt, crcnn_tensor **out) {
    auto *t = new crcnn_tensor{count, size, ntt, nullptr};
    int rc = dev_alloc(ctx, (size_t)count * size * poly_words(ctx) * 8, (void **)&t->d);
    if (rc) { delete t; return rc; }
    *out = t;
    return CRCNN_OK;
}

int ntt_inplace(crcnn_ctx *ctx, uint64_t *d, long npolys, int slot_base, int slot_count, bool inverse) {
    ProfScope ps(ctx, inverse ? KC_NTT_INV : KC_NTT_FWD, 2 * lp_bytes(ctx, npolys), lp_bfly(ctx, npolys));
    CU(launch_ntt(ctx->dP, ctx->logn, d, npolys, slot_base, slot_count, inverse, ctx->stream));
    return CRCNN_OK;
}

int ensure_domain(crcnn_ctx *ctx, crcnn_tensor *t, int want_ntt) {
    if (t->ntt == want_ntt) return CRCNN_OK;
    int rc = ntt_inplace(ctx, t->d, t->count * t->size * ctx->K, 0, ctx->K, !want_ntt);
    if (rc) return rc;
    t->ntt = want_ntt;
    return CRCNN_OK;
}

enum PlainForm { PF_NTT_MUL, PF_NTT_ADD, PF_COEF_ADD };

int expand_range(crcnn_ctx *ctx, crcnn_plain *p, long first, long count, PlainForm f, uint64_t *dst) {
    ProfScope ps(ctx, KC_PLAIN_EXPAND, lp_bytes(ctx, (double)count * ctx->K), f != PF_COEF_ADD ? lp_bfly(ctx, (double)count * ctx->K) : 0);
    CU(launch_plain_expand(ctx->dP, ctx->logn, ctx->K, p->d_off, p->d_idx, p->d_val, first, count,
                           (f == PF_NTT_MUL ? 0 : 1) | (p->sparse_shape ? 2 : 0), f != PF_COEF_ADD, dst, ctx->stream));
    return CRCNN_OK;
}

// Materialise (and keep) a dense form of the whole pack.
int ensure_form(crcnn_ctx *ctx, crcnn_plain *p, PlainForm f) {
    uint64_t **slot = f == PF_NTT_MUL ? &p->ntt_mul : (f == PF_NTT_ADD ? &p->ntt_add : &p->coef_add);
    if (*slot) return CRCNN_OK;
    if (p->dense_only) return fail(ctx, CRCNN_ERR_UNSUPPORTED, "this derived plaintext pack has no such form");
    int rc = dev_alloc(ctx, (size_t)p->count * poly_words(ctx) * 8, (void **)slot);
    if (rc) return rc;
    rc = expand_range(ctx, p, 0, p->count, f, *slot);
    if (!rc && f != PF_NTT_MUL && p->add_mult != 1)
        CU(launch_scale_small(ctx->dP, *slot, (long)((size_t)p->count * poly_words(ctx)), p->add_mult, ctx->stream));
    return rc;
}

int make_plain(crcnn_ctx *ctx, std::vector<uint32_t> &&off, std::vector<uint32_t> &&idx, std::vector<uint64_t> &&val,
               crcnn_plain **out) {
    auto *p = new crcnn_plain();
    p->count = (long)off.size() - 1;
    p->off = std::move(off); p->idx = std::move(idx); p->val = std::move(val);
    p->sparse_shape = true;
    for (uint32_t ix : p->idx)
        if (ix >= 64 && ix < (uint32_t)(ctx->n - 32)) { p->sparse_shape = false; break; }
    int rc = dev_alloc(ctx, p->off.size() * 4, (void **)&p->d_off);
    if (!rc) rc = dev_alloc(ctx, std::max<size_t>(p->idx.size(), 1) * 4, (void **)&p->d_idx);
    if (!rc) rc = dev_alloc(ctx, std::max<size_t>(p->val.size(), 1) * 8, (void **)&p->d_val);
    if (rc) { delete p; return rc; }
    CU(cudaMemcpyAsync(p->d_off, p->off.data(), p->off.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (!p->idx.empty()) {
        CU(cudaMemcpyAsync(p->d_idx, p->idx.data(), p->idx.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemcpyAsync(p->d_val, p->val.data(), p->val.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));  // host vectors are pageable; make the staging explicit
    *out = p;
    return CRCNN_OK;
}

// Shoup companions of the multiplicative NTT form (element-wise layers multiply by a per-channel constant:
// one mulhi + two mullo instead of a 128-bit Barrett reduction per residue).
int ensure_shoup(crcnn_ctx *ctx, crcnn_plain *p) {
    int rc = ensure_form(ctx, p, PF_NTT_MUL);
    if (rc || p->ntt_mul_sh) return rc;
    const size_t words = (size_t)p->count * poly_words(ctx);
    rc = dev_alloc(ctx, words * 8, (void **)&p->ntt_mul_sh);
    if (rc) return rc;
    CU(launch_shoup_companion(ctx->dP, p->ntt_mul, (long)words, p->ntt_mul_sh, ctx->stream));
    return CRCNN_OK;
}

// Per-channel constants of "pooling scale, then batch-norm" in NTT form, kept in the batch-norm factor pack:
// C[z] = scale (.) invstd[z] (with Shoup companions), D[z] = mean[z] (.) invstd[z];  x -> x (.) C[z] - D[z] (D on polynomial 0 only).
int ensure_pool_bn_consts(crcnn_ctx *ctx, crcnn_plain *scale, crcnn_plain *mean, crcnn_plain *invstd) {
    // scale == nullptr: sum pooling (PoolingLayer, the WoPad topology) -- C[z] = invstd[z]
    int rc = scale ? ensure_form(ctx, scale, PF_NTT_MUL) : CRCNN_OK;
    if (!rc) rc = ensure_form(ctx, mean, PF_NTT_ADD);
    if (!rc) rc = ensure_form(ctx, invstd, PF_NTT_MUL);
    if (rc) return rc;
    const long scale_id = scale ? scale->serial : -1;
    if (invstd->fused_C && invstd->fused_scale == scale_id && invstd->fused_mean == mean->serial) return CRCNN_OK;
    const size_t words = (size_t)invstd->count * poly_words(ctx);
    dev_free(ctx, invstd->fused_C); dev_free(ctx, invstd->fused_Csh); dev_free(ctx, invstd->fused_D);
    invstd->fused_C = invstd->fused_Csh = invstd->fused_D = nullptr;
    rc = dev_alloc(ctx, words * 8, (void **)&invstd->fused_C);
    if (!rc) rc = dev_alloc(ctx, words * 8, (void **)&invstd->fused_Csh);
    if (!rc) rc = dev_alloc(ctx, words * 8, (void **)&invstd->fused_D);
    if (rc) return rc;
    CU(launch_pool_bn_consts(ctx->dP, scale ? scale->ntt_mul : nullptr, invstd->ntt_mul, mean->ntt_add, (long)words, invstd->fused_C, invstd->fused_D, ctx->stream));
    CU(launch_shoup_companion(ctx->dP, invstd->fused_C, (long)words, invstd->fused_Csh, ctx->stream));
    invstd->fused_scale = scale_id; invstd->fused_mean = mean->serial;
    return CRCNN_OK;
}

// Device copy of an index table, cached by content key.
int get_index_table(crcnn_ctx *ctx, const std::vector<int> &key, const std::vector<int> &table, const int **out) {
    auto it = ctx->index_cache.find(key);
    if (it != ctx->index_cache.end()) { *out = it->second; return CRCNN_OK; }
    int *d = nullptr;
    CU(cudaMalloc((void **)&d, std::max<size_t>(table.size(), 1) * sizeof(int)));
    CU(cudaMemcpyAsync(d, table.data(), table.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->index_cache[key] = d;
    *out = d;
    return CRCNN_OK;
}

// The coefficient-domain multiply (tapmul_kernel) applies to this pack: FractionalEncoder digits only, primes below 2^56.
// tapmul_kernel reads value 1 as +1 and value t-1 as -1; multiply_plain lifts 1 to +1 only when 1 < (t+1)/2, that is t >= 3
// (at t = 2 both digits are the value 1 and it lifts to q-1), so t = 2 takes the NTT-domain multiply.
bool tap_eligible(crcnn_ctx *ctx, crcnn_plain *p) {
    if (p->tap_state == 0) {
        const uint64_t t = ctx->hp.d.t;
        p->tap_state = (p->sparse_shape && tcn_planes_for(ctx->hp.d) == 7 && ctx->n % 1024 == 0 && t >= 3) ? 1 : -1;
        for (size_t e = 0; e < p->val.size() && p->tap_state == 1; e++)
            if (p->val[e] != 1 && p->val[e] != t - 1) p->tap_state = -1;
        for (long i = 0; i < p->count && p->tap_state == 1; i++)
            if (p->off[i + 1] - p->off[i] > 96) p->tap_state = -1;
    }
    return p->tap_state == 1;
}

// R residues of any coefficient prime add up below 2^64
bool sum_fits_64(const crcnn_ctx *ctx, long R) {
    uint64_t maxq = 0;
    for (int j = 0; j < ctx->K; j++) maxq = std::max(maxq, ctx->hp.d.tab[j].mod.q);
    return R > 0 && (uint64_t)R <= UINT64_MAX / maxq;
}

// Layer::computeBoundaries (CrCNN/src/layer.cpp:12-26)
void boundaries(int xd, int yd, int xs, int ys, int xf, int yf, int *xl, int *yl) {
    *xl = (xf > xs) ? xd - xf + 1 : xd - xs + 1;
    *yl = (yf > ys) ? yd - yf + 1 : yd - ys + 1;
}

// Weighted-sum driver shared by conv and fc: M output channels [m_first, m_first+M) of Mall.
// Ternary tap matrix of a weight pack for fan-in R (tc_mac.cuh): built once, on the host, from the sparse form.
int ensure_tc_form(crcnn_ctx *ctx, crcnn_plain *w, int R) {
    if (w->tc_state < 0) return CRCNN_OK;
    if (w->tc_state == 1 && w->tc_R == R) return CRCNN_OK;
    const uint32_t n = (uint32_t)ctx->n;
    const uint64_t t = ctx->hp.d.t;
    // the digits are read as +1 (value 1) and -1 (value t-1), which is multiply_plain's lift only for t >= 3 (tap_eligible)
    if (t < 3) { w->tc_state = -1; return CRCNN_OK; }
    for (size_t e = 0; e < w->idx.size(); e++)
        if (w->idx[e] < n - TC_TAPS || (w->val[e] != 1 && w->val[e] != t - 1)) { w->tc_state = -1; return CRCNN_OK; }
    if (w->count % R) { w->tc_state = -1; return CRCNN_OK; }
    const long Mall = w->count / R;
    const int Kpad = ((R + 31) / 32 + 3) / 4 * TC_BK;
    const size_t rows = (size_t)Mall * TC_TAPS + TC_BM;  // one tile of zero rows so shard tiles may over-read
    std::vector<int8_t> A(rows * Kpad, 0);
    for (long wi = 0; wi < w->count; wi++) {
        const long m = wi / R, r = wi % R;
        for (uint32_t e = w->off[wi]; e < w->off[wi + 1]; e++) {
            const int tap = (int)(n - w->idx[e]);  // 1..32
            // lifted digit s = +1 (value 1) or -1 (value t-1); x^(n-tap) = -x^(-tap) flips it
            A[((size_t)m * TC_TAPS + tap - 1) * Kpad + r] = w->val[e] == 1 ? (int8_t)-1 : (int8_t)1;
        }
    }
    if (w->tc_A) { dev_free(ctx, w->tc_A); w->tc_A = nullptr; }
    int rc = dev_alloc(ctx, A.size(), (void **)&w->tc_A);
    if (rc) return rc;
    CU(cudaMemcpyAsync(w->tc_A, A.data(), A.size(), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    w->tc_state = 1; w->tc_R = R; w->tc_Kpad = Kpad;
    return CRCNN_OK;
}

// Weighted sum on the tensor cores: coefficient-domain inputs and outputs, no transform anywhere.
int run_weighted_sum_tc(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w, crcnn_plain *b, const int *d_index, int R,
                        int Npos, int Pimg, int m_first, int M, crcnn_tensor *out) {
    int rc = ensure_domain(ctx, in, 0);
    if (!rc) rc = ensure_form(ctx, b, PF_COEF_ADD);
    if (rc) return rc;
    const size_t pw = poly_words(ctx);
    TcMacArgs a{};
    a.A = w->tc_A + (size_t)m_first * TC_TAPS * w->tc_Kpad;
    a.x = in->d; a.bias = b->coef_add + (size_t)m_first * pw; a.out = out->d;
    a.M = M; a.Mpad = (M * TC_TAPS + TC_BM - 1) / TC_BM * TC_BM; a.R = R; a.Kpad = w->tc_Kpad;
    a.planes = tc_planes_for(ctx->hp.d);
    a.Pimg = Pimg; a.Mtotal = M; a.m0 = 0; a.n = ctx->n; a.K = ctx->K;
    a.npos = 1;
    const size_t per_pos = tc_b_bytes(a);
    long chunk = (long)std::max<size_t>(1, ctx->tc_scratch_bytes / per_pos);
    chunk = std::min<long>(std::min<long>(chunk, Npos), 65535 / (2 * ctx->K));
    uint8_t *scratch = nullptr;
    rc = dev_alloc(ctx, (size_t)chunk * per_pos, (void **)&scratch);
    if (rc) return rc;
    a.B = scratch;
    for (long p0 = 0; p0 < Npos && !rc; p0 += chunk) {
        a.npos = (int)std::min<long>(chunk, Npos - p0);
        a.p0 = (int)p0;
        a.in_index = d_index + p0 * R;
        cudaError_t e;
        // split: gathers npos*R ciphertexts and writes their byte planes; GEMM: reads the planes, writes the outputs;
        // ops = int8 multiply-accumulates of the unpadded problem (32 taps x planes per term and coefficient)
        const double bbytes = (double)a.npos * per_pos;
        { ProfScope ps(ctx, KC_TC_SPLIT, lp_bytes(ctx, (double)a.npos * R * 2 * ctx->K) + bbytes, 0); e = launch_tc_split(ctx->dP, a, ctx->stream); }
        if (e == cudaSuccess) {
            ProfScope ps(ctx, KC_TC_MAC, bbytes + lp_bytes(ctx, (double)a.npos * M * 2 * ctx->K),
                         (double)a.npos * 2 * ctx->K * ctx->n * a.planes * (double)M * TC_TAPS * R);
            e = launch_tc_mac(ctx->dP, a, ctx->sm_count, ctx->stream);
        }
        if (e != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, std::string("tensor-core weighted sum: ") + cudaGetErrorString(e));
    }
    dev_free(ctx, scratch);
    if (!rc) out->ntt = 0;
    return rc;
}

// Byte planes of the whole pack's NTT-form weights, staged once (tcn_mac.cuh); the dense NTT form is released afterwards.
// preshift: also the planes of W 2^(8b) mod q_j for b = 1..6 (the seven-class kernel).  A pack keeps its first staging: a
// pre-shifted one serves the 13-class kernels through its first block.
int ensure_tcn_weights(crcnn_ctx *ctx, crcnn_plain *w, int R, bool preshift) {
    if (w->tcn_W && w->tcn_R == R) return CRCNN_OK;
    int rc = ensure_form(ctx, w, PF_NTT_MUL);
    if (rc) return rc;
    if (w->tcn_W) { dev_free(ctx, w->tcn_W); w->tcn_W = nullptr; }
    const int Mall = (int)(w->count / R), Kpad = tcn_kpad(R);
    const size_t block = tcn_w_bytes(7, Mall, Kpad, ctx->K, ctx->n);
    const int blocks = preshift ? 7 : 1;
    rc = dev_alloc(ctx, block * blocks, (void **)&w->tcn_W);
    if (rc) return rc;
    const long words = (long)w->count * (long)poly_words(ctx);
    uint64_t *shifted = nullptr;
    if (preshift) {
        rc = dev_alloc(ctx, (size_t)words * 8, (void **)&shifted);
        if (rc) { dev_free(ctx, w->tcn_W); w->tcn_W = nullptr; return rc; }
    }
    uint64_t q[MAXK];
    for (int j = 0; j < ctx->K; j++) q[j] = ctx->hp.d.tab[j].mod.q;
    TcnSplitArgs s{};
    s.index = nullptr; s.item_polys = 1;
    s.R = R; s.Kpad = Kpad; s.planes = 7; s.ncols = Mall; s.slot0 = 0; s.nslots = ctx->K * ctx->n; s.n = ctx->n; s.K = ctx->K;
    for (int b = 0; b < blocks; b++) {
        if (b) CU(launch_tcn_preshift(q, w->ntt_mul, shifted, words, b, ctx->n, ctx->K, ctx->stream));
        s.src = b ? shifted : w->ntt_mul;
        s.dst = w->tcn_W + block * b;
        ProfScope ps(ctx, KC_TCN_SPLIT, lp_bytes(ctx, (double)w->count * ctx->K) + (double)block, 0);
        CU(launch_tcn_split(s, ctx->stream));
    }
    if (shifted) dev_free(ctx, shifted);
    dev_free(ctx, w->ntt_mul); w->ntt_mul = nullptr;
    if (w->ntt_mul_sh) { dev_free(ctx, w->ntt_mul_sh); w->ntt_mul_sh = nullptr; }
    w->tcn_R = R;
    w->tcn_pre = preshift;
    return CRCNN_OK;
}

// Weighted sum as the NTT-domain limb-split GEMM on the tensor cores: NTT-form inputs and outputs.
int run_weighted_sum_tcn(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w, crcnn_plain *b, const int *d_index, int R,
                         int Npos, int Pimg, int m_first, int M, crcnn_tensor *out) {
    const int Kpad = tcn_kpad(R), ncols = 2 * Npos, total = ctx->K * ctx->n;
    const int variant = ctx->tcn_mode >= 2 ? ctx->tcn_mode - 1 : 0;
    const bool want_pre = ctx->tcn_preshift && tcn_preshift_shape(R, ncols, M, variant) &&
                          7 * tcn_w_bytes(7, (int)(w->count / R), Kpad, ctx->K, ctx->n) <= ctx->weight_cache_bytes;
    int rc = ensure_domain(ctx, in, 1);
    if (!rc) rc = ensure_form(ctx, b, PF_NTT_ADD);
    if (!rc) rc = ensure_tcn_weights(ctx, w, R, want_pre);
    if (rc) return rc;
    const size_t pw = poly_words(ctx);
    const size_t per_slot = tcn_x_bytes_per_slot(7, ncols, Kpad);
    long chunk = (long)(ctx->tc_scratch_bytes / per_slot) / 32 * 32;
    chunk = std::max<long>(32, std::min<long>(chunk, total));
    uint8_t *scratch = nullptr;
    rc = dev_alloc(ctx, (size_t)chunk * per_slot, (void **)&scratch);
    if (rc) return rc;
    TcnSplitArgs s{};
    s.src = in->d; s.index = d_index; s.dst = scratch; s.item_polys = 2;
    s.R = R; s.Kpad = Kpad; s.planes = 7; s.ncols = ncols; s.n = ctx->n; s.K = ctx->K;
    TcnMacArgs a{};
    a.W = w->tcn_W; a.X = scratch; a.bias = b->ntt_add + (size_t)m_first * pw; a.out = out->d;
    a.Mall = (int)(w->count / R); a.m_first = m_first; a.M = M;
    a.R = R; a.Kpad = Kpad; a.planes = 7; a.ncols = ncols;
    a.Pimg = Pimg; a.Mtotal = M; a.m0 = 0; a.n = ctx->n; a.K = ctx->K;
    a.variant = variant;
    a.preshift = want_pre && w->tcn_pre;
    a.use_fold = ctx->tcn_fold;
    for (int j = 0; j < ctx->K; j++) a.fold[j] = tcn_fold_make(ctx->hp.d.tab[j].mod.q);
    for (long s0 = 0; s0 < total && !rc; s0 += chunk) {
        const int ns = (int)std::min<long>(chunk, total - s0);
        s.slot0 = a.slot0 = (int)s0; s.nslots = a.nslots = ns;
        const double xbytes = (double)ns * per_slot;
        cudaError_t e;
        { ProfScope ps(ctx, KC_TCN_SPLIT, (double)ncols * R * ns * 8.0 + xbytes, 0); e = launch_tcn_split(s, ctx->stream); }
        if (e == cudaSuccess) {
            // ops: int8 multiply-accumulates of the unpadded problem (49 plane pairs per residue product)
            ProfScope ps(ctx, KC_TCN_MAC, xbytes + (double)ns * 7 * M * Kpad * (a.preshift ? 7 : 1) + (double)ncols * M * ns * 8.0, (double)ns * ncols * M * R * 49.0);
            e = launch_tcn_mac(ctx->dP, a, ctx->sm_count, ctx->stream);
        }
        if (e != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, std::string("limb-split tensor-core weighted sum: ") + cudaGetErrorString(e));
    }
    dev_free(ctx, scratch);
    if (!rc) out->ntt = 1;
    return rc;
}

int run_weighted_sum(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w, crcnn_plain *b, const int *d_index, int R,
                     int Npos, int Pimg, int Mall, int m_first, int M, crcnn_tensor *out) {
    // the kernel (and with it the domain of the output) is chosen from the LAYER's output count Mall, not the shard's M: every rank of a
    // neuron-sharded layer then produces its rows in the same domain, whatever the split (63 rows on 2 ranks: 32 + 31)
    if (ctx->tc_mode && R >= ctx->tc_min_fanin && (ctx->tc_mode == 2 || Mall >= ctx->tc_min_outputs) && w->sparse_shape && tc_mac_available() == cudaSuccess) {
        int rc = ensure_tc_form(ctx, w, R);
        if (rc) return rc;
        if (w->tc_state == 1) return run_weighted_sum_tc(ctx, in, w, b, d_index, R, Npos, Pimg, m_first, M, out);
    }
    // any weights, NTT domain: the limb-split GEMM, as long as the staged weight planes fit the weight cache
    if (ctx->tcn_mode && tcn_planes_for(ctx->hp.d) == 7 && R <= TCN_MAX_R && w->count % R == 0 && tc_mac_available() == cudaSuccess &&
        (w->tcn_W || tcn_w_bytes(7, (int)(w->count / R), tcn_kpad(R), ctx->K, ctx->n) <= ctx->weight_cache_bytes))
        return run_weighted_sum_tcn(ctx, in, w, b, d_index, R, Npos, Pimg, m_first, M, out);
    int rc = ensure_domain(ctx, in, 1);
    if (rc) return rc;
    rc = ensure_form(ctx, b, PF_NTT_ADD);
    if (rc) return rc;
    MacArgs a{};
    a.x = in->d; a.in_index = d_index; a.out = out->d;
    a.R = R; a.Npos = Npos; a.Pimg = Pimg; a.Mtotal = M; a.K = ctx->K; a.n = ctx->n;
    a.chunk_terms = ctx->chunk_terms;
    const size_t pw = poly_words(ctx);
    const size_t all_bytes = (size_t)w->count * pw * 8;
    if (w->ntt_mul || all_bytes <= ctx->weight_cache_bytes) {
        rc = ensure_form(ctx, w, PF_NTT_MUL);  // first forward pays the transform, like the reference's lazy transform_kernel_to_ntt
        if (rc) return rc;
        a.w = w->ntt_mul + (size_t)m_first * R * pw;
        a.bias = b->ntt_add + (size_t)m_first * pw;
        a.M = M; a.m0 = 0;
        ProfScope ps(ctx, KC_MAC, lp_bytes(ctx, ((double)in->count + (double)M * Npos) * 2 * ctx->K + (double)M * R * ctx->K),
                     (double)M * Npos * R * 2 * ctx->K * ctx->n);
        CU(launch_mac(ctx->dP, a, ctx->stream));
        return CRCNN_OK;
    }
    // weights do not fit: expand `rows` output rows at a time into a scratch buffer
    long rows = (long)std::max<size_t>(1, ctx->weight_cache_bytes / ((size_t)R * pw * 8));
    rows = std::min<long>(rows, M);
    uint64_t *scratch = nullptr;
    rc = dev_alloc(ctx, (size_t)rows * R * pw * 8, (void **)&scratch);
    if (rc) return rc;
    for (long m0 = 0; m0 < M; m0 += rows) {
        long cur = std::min<long>(rows, M - m0);
        rc = expand_range(ctx, w, (long)(m_first + m0) * R, cur * R, PF_NTT_MUL, scratch);
        if (rc) break;
        a.w = scratch; a.bias = b->ntt_add + (size_t)(m_first + m0) * pw;
        a.M = (int)cur; a.m0 = (int)m0;
        ProfScope ps(ctx, KC_MAC, lp_bytes(ctx, ((double)in->count + (double)cur * Npos) * 2 * ctx->K + (double)cur * R * ctx->K),
                     (double)cur * Npos * R * 2 * ctx->K * ctx->n);
        cudaError_t e = launch_mac(ctx->dP, a, ctx->stream);
        if (e != cudaSuccess) { rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e)); break; }
    }
    dev_free(ctx, scratch);
    return rc;
}

// Host (SEAL layout, limb stride n+1) -> device (stride n): one contiguous H2D copy into a staging buffer, then a
// re-stride kernel, all on `s`.  Small uploads keep the single strided copy.
int upload_rows(crcnn_ctx *ctx, const uint64_t *host, size_t rows, uint64_t *dst, cudaStream_t s) {
    const size_t n = ctx->n;
    if (rows * n * 8 < (8u << 20)) {
        CU(cudaMemcpy2DAsync(dst, n * 8, host, (n + 1) * 8, n * 8, rows, cudaMemcpyHostToDevice, s));
        return CRCNN_OK;
    }
    uint64_t *stage = nullptr;
    CU(cudaMallocAsync((void **)&stage, rows * (n + 1) * 8, s));
    cudaError_t e = cudaMemcpyAsync(stage, host, rows * (n + 1) * 8, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = launch_strip_pad(stage, dst, (long)rows, (int)n, s);
    cudaFreeAsync(stage, s);
    if (e != cudaSuccess) return fail(ctx, CRCNN_ERR_CUDA, std::string("upload: ") + cudaGetErrorString(e));
    return CRCNN_OK;
}

}  // namespace

// ======================================================================================= C ABI
extern "C" {

const char *crcnn_last_error(const crcnn_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int crcnn_ctx_create(int n, int K, const uint64_t *q, uint64_t t, int device, crcnn_ctx **out) {
    crcnn_ctx *ctx = nullptr;  // errors before the context exists go to the thread-local slot
    if (!out || !q) return fail(nullptr, CRCNN_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(nullptr, CRCNN_ERR_NO_DEVICE, "no CUDA device: crcnn_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(nullptr, CRCNN_ERR_INVALID_ARGUMENT, "bad device ordinal");
    HostParams hp;
    try {
        hp = derive_params(n, K, q, t);
    } catch (const std::exception &e) {
        return fail(nullptr, CRCNN_ERR_INVALID_ARGUMENT, e.what());
    }
    CU(cudaSetDevice(device));
    auto *c = new crcnn_ctx();
    c->device = device; c->n = n; c->K = K; c->S = hp.d.S; c->logn = hp.d.logn;
    int maxbits = 0;
    for (int i = 0; i < K; i++) { int b = 0; for (uint64_t v = q[i]; v; v >>= 1) b++; maxbits = std::max(maxbits, b); }
    int spare = 128 - 2 * maxbits;
    c->chunk_terms = spare >= 30 ? (1 << 30) : (1 << spare);
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (const char *e = getenv("CRCNN_TC")) c->tc_mode = atoi(e);
    if (const char *e = getenv("CRCNN_TCN")) c->tcn_mode = atoi(e);
    if (const char *e = getenv("CRCNN_TAP")) c->tap_mode = atoi(e);
    if (const char *e = getenv("CRCNN_TCN_FOLD")) c->tcn_fold = atoi(e);
    if (const char *e = getenv("CRCNN_TCN2_PRESHIFT")) c->tcn_preshift = atoi(e);
    if (const char *e = getenv("CRCNN_SQ_LEAN")) c->sq_lean = atoi(e);
    // stream-ordered allocator: keep freed blocks cached
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    {   // the exact-size cache may hold up to 3/4 of the device: the CUDA pool would keep those pages anyway (release threshold above); a
        // request that does not fit flushes the cache and retries (dev_alloc), so the cap only bounds what shape changes can strand
        size_t fr = 0, tot = 0;
        if (cudaMemGetInfo(&fr, &tot) == cudaSuccess && tot) c->big_cache_cap = tot / 4 * 3;
    }
    // upload tables
    int slots = K + hp.d.S;
    auto up = [&](const std::vector<uint64_t> &v, const uint64_t **dst) -> cudaError_t {
        void *d = nullptr;
        cudaError_t e = cudaMalloc(&d, v.size() * 8);
        if (e != cudaSuccess) return e;
        c->owned.push_back(d);
        *dst = (const uint64_t *)d;
        return cudaMemcpy(d, v.data(), v.size() * 8, cudaMemcpyHostToDevice);
    };
    cudaError_t e = cudaSuccess;
    for (int s = 0; s < slots && e == cudaSuccess; s++) {
        // one 128-bit load per butterfly fetches the twiddle and its Shoup companion
        std::vector<uint64_t> fw(2 * (size_t)n), bw(2 * (size_t)n);
        for (int i = 0; i < n; i++) {
            fw[2 * i] = hp.w[s][i]; fw[2 * i + 1] = hp.wp[s][i];
            bw[2 * i] = hp.iwf[s][i]; bw[2 * i + 1] = hp.iwfp[s][i];
        }
        e = up(fw, &hp.d.tab[s].w);
        if (e == cudaSuccess) e = up(bw, &hp.d.tab[s].iw);
        // transposed pairs of the contiguous 4-stage pass: forward stage s of group G uses the 2^s pairs from ((n/16 + G) << s),
        // inverse stage s the 2^(3-s) pairs from (n/2 >> s) + (G << (3-s))
        const int NG = n >> 4;
        std::vector<uint64_t> fl(2 * (size_t)16 * NG, 0), bl(2 * (size_t)16 * NG, 0);
        for (int G = 0; G < NG; G++)
            for (int st = 0; st < 4; st++) {
                for (int lb = 0; lb < (1 << st); lb++) {
                    const size_t at = 2 * ((size_t)((1 << st) - 1 + lb) * NG + G), from = 2 * ((((size_t)NG + G) << st) + lb);
                    fl[at] = fw[from]; fl[at + 1] = fw[from + 1];
                }
                for (int lb = 0; lb < (1 << (3 - st)); lb++) {
                    const size_t at = 2 * ((size_t)(16 - (16 >> st) + lb) * NG + G);
                    const size_t from = 2 * ((size_t)((n >> 1) >> st) + ((size_t)G << (3 - st)) + lb);
                    bl[at] = bw[from]; bl[at + 1] = bw[from + 1];
                }
            }
        if (e == cudaSuccess) e = up(fl, &hp.d.tab[s].wl);
        if (e == cudaSuccess) e = up(bl, &hp.d.tab[s].iwl);
        hp.d.tab[s].tf = nullptr;
        if (e == cudaSuccess && s < K) e = up(hp.tf[s], &hp.d.tab[s].tf);
    }
    if (e == cudaSuccess) e = cudaMalloc((void **)&c->dP, sizeof(DeviceParams));
    if (e == cudaSuccess) e = cudaMemcpy(c->dP, &hp.d, sizeof(DeviceParams), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        std::string m = cudaGetErrorString(e);
        for (void *p : c->owned) cudaFree(p);
        if (c->dP) cudaFree(c->dP);
        delete c;
        return fail(nullptr, CRCNN_ERR_CUDA, "context setup: " + m);
    }
    c->hp = std::move(hp);
    *out = c;
    return CRCNN_OK;
}

int crcnn_ctx_destroy(crcnn_ctx *ctx) {
    if (!ctx) return CRCNN_OK;
    cudaSetDevice(ctx->device);
    big_cache_flush(ctx);
    cudaStreamSynchronize(ctx->stream);
    prof_collect(ctx);
    for (auto e : ctx->event_pool) cudaEventDestroy(e);
    for (auto &kv : ctx->index_cache) cudaFree(kv.second);
    if (ctx->stage) cudaFree(ctx->stage);
    for (void *p : ctx->owned) cudaFree(p);
    cudaFree(ctx->dP);
    delete ctx;
    return CRCNN_OK;
}

int crcnn_ctx_set_stream(crcnn_ctx *ctx, void *cuda_stream) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->stream = (cudaStream_t)cuda_stream;
    return CRCNN_OK;
}

int crcnn_ctx_sync(crcnn_ctx *ctx) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    CU(cudaStreamSynchronize(ctx->stream));
    prof_collect(ctx);
    return CRCNN_OK;
}

int crcnn_ctx_alloc_stats(crcnn_ctx *ctx, long long out[6]) {
    if (!ctx || !out) return CRCNN_ERR_INVALID_ARGUMENT;
    out[0] = ctx->st_big_malloc; out[1] = ctx->st_big_hit; out[2] = ctx->st_big_bypass; out[3] = ctx->st_flush;
    out[4] = ctx->st_small_malloc; out[5] = (long long)ctx->big_cached;
    return CRCNN_OK;
}

int crcnn_ctx_set_weight_cache_bytes(crcnn_ctx *ctx, size_t bytes) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    ctx->weight_cache_bytes = bytes;
    return CRCNN_OK;
}

int crcnn_ctx_set_tensor_core_mode(crcnn_ctx *ctx, int mode, int min_fanin, size_t scratch_bytes) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(mode >= 0 && mode <= 2, "tensor-core mode must be 0, 1 or 2");
    ctx->tc_mode = mode;
    if (min_fanin > 0) ctx->tc_min_fanin = min_fanin;
    if (scratch_bytes > 0) ctx->tc_scratch_bytes = scratch_bytes;
    return CRCNN_OK;
}

int crcnn_ctx_set_limb_split_mode(crcnn_ctx *ctx, int mode) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(mode >= 0 && mode <= 3, "limb-split mode must be 0 (off), 1 (on), 2 (row-major kernel) or 3 (column-major kernel)");
    ctx->tcn_mode = mode;
    return CRCNN_OK;
}

int crcnn_ctx_set_limb_split_reduction(crcnn_ctx *ctx, int mode) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(mode == 0 || mode == 1, "limb-split reduction must be 0 (128-bit recombination + Barrett) or 1 (folded through 2^k - delta)");
    ctx->tcn_fold = mode;
    return CRCNN_OK;
}

int crcnn_ctx_set_relin_mode(crcnn_ctx *ctx, int mode) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(mode == 0 || mode == 1, "relinearize mode must be 0 (64-bit transforms) or 1 (word-size auxiliary primes)");
    ctx->relin_mode = mode;
    return CRCNN_OK;
}

int crcnn_ctx_ntt_table(const crcnn_ctx *ctx_c, int slot, int which, uint64_t *out) {
    crcnn_ctx *ctx = const_cast<crcnn_ctx *>(ctx_c);
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(out && slot >= 0 && slot < ctx->K + ctx->S && which >= 0 && which < 4, "bad table selector");
    const auto &v = which == 0 ? ctx->hp.w[slot] : which == 1 ? ctx->hp.wp[slot] : which == 2 ? ctx->hp.iw[slot] : ctx->hp.iwp[slot];
    memcpy(out, v.data(), v.size() * 8);
    return CRCNN_OK;
}

int crcnn_ctx_bsk_count(const crcnn_ctx *ctx) { return ctx ? ctx->S : CRCNN_ERR_INVALID_ARGUMENT; }

// ---------------------------------------------------------------------------- tensors
int crcnn_tensor_upload_ex(crcnn_ctx *ctx, const uint64_t *host, long count, int size, int ntt_form, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(host && out && count >= 0 && size >= 2 && size <= 3, "bad tensor upload arguments");
    CU(cudaSetDevice(ctx->device));
    crcnn_tensor *t = nullptr;
    int rc = new_tensor(ctx, count, size, ntt_form ? 1 : 0, &t);
    if (rc) return rc;
    const size_t n = ctx->n, rows = (size_t)count * size * ctx->K;
    if (rows) {
        int rc2 = upload_rows(ctx, host, rows, t->d, ctx->stream);
        if (rc2) { crcnn_tensor_free(ctx, t); return rc2; }
    }
    (void)n;
    *out = t;
    return CRCNN_OK;
}
int crcnn_tensor_upload_on(crcnn_ctx *ctx, const uint64_t *host, long count, int size, int ntt_form, void *copy_stream,
                           crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(host && out && count >= 0 && size >= 2 && size <= 3, "bad tensor upload arguments");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t cs = (cudaStream_t)copy_stream;
    auto *t = new crcnn_tensor{count, size, ntt_form ? 1 : 0, nullptr};
    const size_t n = ctx->n, rows = (size_t)count * size * ctx->K;
    if (rows) {
        cudaError_t e = cudaMallocAsync((void **)&t->d, rows * n * 8, cs);
        if (e != cudaSuccess) { delete t; return fail(ctx, e == cudaErrorMemoryAllocation ? CRCNN_ERR_OUT_OF_MEMORY : CRCNN_ERR_CUDA, cudaGetErrorString(e)); }
        int rc2 = upload_rows(ctx, host, rows, t->d, cs);
        if (rc2) { cudaFreeAsync(t->d, cs); delete t; return rc2; }
    }
    *out = t;
    return CRCNN_OK;
}

int crcnn_tensor_upload_into(crcnn_ctx *ctx, const uint64_t *host, crcnn_tensor *t, int ntt_form, void *copy_stream) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(host && t, "null argument");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t cs = copy_stream ? (cudaStream_t)copy_stream : ctx->stream;
    const size_t n = ctx->n, rows = (size_t)t->count * t->size * ctx->K;
    const size_t need = rows * (n + 1) * 8;
    if (need > ctx->stage_bytes) {   // grows only: steady-state uploads allocate nothing
        if (ctx->stage) { CU(cudaStreamSynchronize(cs)); CU(cudaFree(ctx->stage)); ctx->stage = nullptr; ctx->stage_bytes = 0; }
        CU(cudaMalloc((void **)&ctx->stage, need));
        ctx->stage_bytes = need;
    }
    if (rows) {
        CU(cudaMemcpyAsync(ctx->stage, host, need, cudaMemcpyHostToDevice, cs));
        CU(launch_strip_pad(ctx->stage, t->d, (long)rows, (int)n, cs));
    }
    t->ntt = ntt_form ? 1 : 0;
    return CRCNN_OK;
}

int crcnn_ctx_wait_stream(crcnn_ctx *ctx, void *other_stream) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    cudaEvent_t ev;
    CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CU(cudaEventRecord(ev, (cudaStream_t)other_stream));
    CU(cudaStreamWaitEvent(ctx->stream, ev, 0));
    CU(cudaEventDestroy(ev));
    return CRCNN_OK;
}

int crcnn_tensor_upload(crcnn_ctx *ctx, const uint64_t *host, long count, int size, crcnn_tensor **out) {
    return crcnn_tensor_upload_ex(ctx, host, count, size, 0, out);
}

int crcnn_tensor_download_ex(crcnn_ctx *ctx, crcnn_tensor *t, int want_ntt, uint64_t *host) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(t && host, "null argument");
    CU(cudaSetDevice(ctx->device));
    const size_t n = ctx->n, rows = (size_t)t->count * t->size * ctx->K;
    const uint64_t *src = t->d;
    uint64_t *tmp = nullptr;
    if ((t->ntt != 0) != (want_ntt != 0)) {  // convert a copy; the tensor itself keeps its domain
        int rc = dev_alloc(ctx, rows * n * 8, (void **)&tmp);
        if (rc) return rc;
        CU(cudaMemcpyAsync(tmp, t->d, rows * n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        rc = ntt_inplace(ctx, tmp, (long)rows, 0, ctx->K, want_ntt == 0);
        if (rc) return rc;
        src = tmp;
    }
    if (rows) CU(cudaMemcpy2DAsync(host, (n + 1) * 8, src, n * 8, n * 8, rows, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    dev_free(ctx, tmp);
    for (size_t r = 0; r < rows; r++) host[r * (n + 1) + n] = 0;  // SEAL's pad word
    prof_collect(ctx);
    return CRCNN_OK;
}
int crcnn_tensor_download(crcnn_ctx *ctx, crcnn_tensor *t, uint64_t *host) { return crcnn_tensor_download_ex(ctx, t, 0, host); }

int crcnn_tensor_free(crcnn_ctx *ctx, crcnn_tensor *t) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    if (!t) return CRCNN_OK;
    dev_free(ctx, t->d);
    delete t;
    return CRCNN_OK;
}
long crcnn_tensor_count(const crcnn_tensor *t) { return t ? t->count : -1; }
int crcnn_tensor_ct_size(const crcnn_tensor *t) { return t ? t->size : -1; }

int crcnn_tensor_slice(crcnn_ctx *ctx, crcnn_tensor *t, long first, long count, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(t && out && first >= 0 && count >= 0 && first + count <= t->count, "slice out of range");
    crcnn_tensor *s = nullptr;
    int rc = new_tensor(ctx, count, t->size, t->ntt, &s);
    if (rc) return rc;
    size_t ctw = (size_t)t->size * poly_words(ctx);
    if (count) CU(cudaMemcpyAsync(s->d, t->d + first * ctw, count * ctw * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    *out = s;
    return CRCNN_OK;
}

int crcnn_tensor_device_ptr(crcnn_tensor *t, void **dev_ptr, int *ntt_form) {
    if (!t || !dev_ptr) return CRCNN_ERR_INVALID_ARGUMENT;
    *dev_ptr = t->d;
    if (ntt_form) *ntt_form = t->ntt;
    return CRCNN_OK;
}

int crcnn_tensor_wrap_alloc(crcnn_ctx *ctx, long count, int size, int ntt_form, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(out && count >= 0 && size >= 2 && size <= 3, "bad tensor shape");
    return new_tensor(ctx, count, size, ntt_form ? 1 : 0, out);
}

// ---------------------------------------------------------------------------- plaintext packs
int crcnn_plain_upload(crcnn_ctx *ctx, const uint64_t *host, long count, int coeff_count, long stride, crcnn_plain **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(host && out && count >= 0 && coeff_count >= 0 && stride >= coeff_count, "bad plaintext upload arguments");
    // SEAL rejects coeff_count > n+1, or == n+1 with a non-zero top coefficient (evaluator.cpp:1156-1159)
    REQUIRE(coeff_count <= ctx->n + 1, "plain is not valid for encryption parameters");
    std::vector<uint32_t> off(count + 1, 0), idx;
    std::vector<uint64_t> val;
    for (long i = 0; i < count; i++) {
        const uint64_t *p = host + i * stride;
        for (int c = 0; c < coeff_count; c++)
            if (p[c]) {
                REQUIRE(c < ctx->n, "plain is not valid for encryption parameters");
                REQUIRE(p[c] < ctx->hp.d.t, "plaintext coefficient not below the plain modulus");
                idx.push_back((uint32_t)c); val.push_back(p[c]);
            }
        off[i + 1] = (uint32_t)idx.size();
    }
    return make_plain(ctx, std::move(off), std::move(idx), std::move(val), out);
}

int crcnn_plain_upload_sparse(crcnn_ctx *ctx, const uint32_t *idx, const uint64_t *val, const uint32_t *offsets, long count,
                              crcnn_plain **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(offsets && out && count >= 0, "bad sparse plaintext arguments");
    std::vector<uint32_t> off(offsets, offsets + count + 1);
    size_t nnz = off[count];
    REQUIRE(nnz == 0 || (idx && val), "null sparse arrays");
    std::vector<uint32_t> vi(idx, idx + nnz);
    std::vector<uint64_t> vv(val, val + nnz);
    for (size_t e = 0; e < nnz; e++) {
        REQUIRE(vi[e] < (uint32_t)ctx->n, "plain is not valid for encryption parameters");
        REQUIRE(vv[e] < ctx->hp.d.t, "plaintext coefficient not below the plain modulus");
    }
    return make_plain(ctx, std::move(off), std::move(vi), std::move(vv), out);
}

int crcnn_plain_encode(crcnn_ctx *ctx, const float *values, long count, crcnn_plain **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(values && out && count >= 0, "bad encode arguments");
    std::vector<uint32_t> off(count + 1, 0), idx;
    std::vector<uint64_t> val;
    idx.reserve(count * 24); val.reserve(count * 24);
    for (long i = 0; i < count; i++) {
        encode_fractional_sparse((double)values[i], ctx->n, ctx->hp.d.t, idx, val);
        off[i + 1] = (uint32_t)idx.size();
    }
    return make_plain(ctx, std::move(off), std::move(idx), std::move(val), out);
}

int crcnn_plain_encode_f64(crcnn_ctx *ctx, const double *values, long count, crcnn_plain **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(values && out && count >= 0, "bad encode arguments");
    std::vector<uint32_t> off(count + 1, 0), idx;
    std::vector<uint64_t> val;
    for (long i = 0; i < count; i++) {
        encode_fractional_sparse(values[i], ctx->n, ctx->hp.d.t, idx, val);
        off[i + 1] = (uint32_t)idx.size();
    }
    return make_plain(ctx, std::move(off), std::move(idx), std::move(val), out);
}

int crcnn_plain_get(crcnn_ctx *ctx, const crcnn_plain *p, long index, uint64_t *out_words) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(p && out_words && index >= 0 && index < p->count, "plaintext index out of range");
    REQUIRE(!p->dense_only, "derived plaintext pack: no host form");
    memset(out_words, 0, (size_t)(ctx->n + 1) * 8);
    for (uint32_t e = p->off[index]; e < p->off[index + 1]; e++) out_words[p->idx[e]] = p->val[e];
    return CRCNN_OK;
}

int crcnn_plain_get_ntt(crcnn_ctx *ctx, crcnn_plain *p, long index, uint64_t *out_words) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(p && out_words && index >= 0 && index < p->count, "plaintext index out of range");
    REQUIRE(!p->dense_only, "derived plaintext pack: no host form");
    uint64_t *tmp = nullptr;
    int rc = dev_alloc(ctx, poly_words(ctx) * 8, (void **)&tmp);
    if (rc) return rc;
    rc = expand_range(ctx, p, index, 1, PF_NTT_MUL, tmp);
    if (rc) return rc;
    const size_t n = ctx->n;
    CU(cudaMemcpy2DAsync(out_words, (n + 1) * 8, tmp, n * 8, n * 8, ctx->K, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    dev_free(ctx, tmp);
    for (int j = 0; j < ctx->K; j++) out_words[j * (n + 1) + n] = 0;
    return CRCNN_OK;
}

int crcnn_plain_free(crcnn_ctx *ctx, crcnn_plain *p) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    if (!p) return CRCNN_OK;
    dev_free(ctx, p->d_off); dev_free(ctx, p->d_idx); dev_free(ctx, p->d_val);
    dev_free(ctx, p->ntt_mul); dev_free(ctx, p->ntt_mul_sh); dev_free(ctx, p->ntt_add); dev_free(ctx, p->coef_add); dev_free(ctx, p->tc_A); dev_free(ctx, p->tcn_W);
    dev_free(ctx, p->fused_C); dev_free(ctx, p->fused_Csh); dev_free(ctx, p->fused_D);
    if (p->folded_w) crcnn_plain_free(ctx, p->folded_w);
    if (p->folded_b) crcnn_plain_free(ctx, p->folded_b);
    delete p;
    return CRCNN_OK;
}
long crcnn_plain_count(const crcnn_plain *p) { return p ? p->count : -1; }

// ---------------------------------------------------------------------------- evaluation keys
int crcnn_evk_upload(crcnn_ctx *ctx, const uint64_t *host, int dbc, const int *sizes, crcnn_evk **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(host && sizes && out && dbc >= 1 && dbc <= 60, "bad evaluation key arguments");
    CU(cudaSetDevice(ctx->device));
    auto *k = new crcnn_evk();
    k->dbc = dbc;
    long polys = 0;
    const size_t pw = poly_words(ctx);
    for (int i = 0; i < MAXK; i++) { k->key_off[i] = 0; k->digits[i] = 0; }
    for (int i = 0; i < ctx->K; i++) {
        if (sizes[i] < 2 || (sizes[i] & 1)) { delete k; return fail(ctx, CRCNN_ERR_INVALID_ARGUMENT, "evaluation key sizes must be even and >= 2"); }
        k->key_off[i] = polys * (long)pw;
        k->digits[i] = sizes[i] / 2;
        polys += sizes[i];
    }
    int rc = dev_alloc(ctx, (size_t)polys * pw * 8, (void **)&k->d);
    if (rc) { delete k; return rc; }
    const size_t n = ctx->n, rows = (size_t)polys * ctx->K;
    CU(cudaMemcpy2DAsync(k->d, n * 8, host, (n + 1) * 8, n * 8, rows, cudaMemcpyHostToDevice, ctx->stream));
    CU(launch_canonicalize(ctx->dP, k->d, (long)(rows * n), ctx->stream));
    {
        uint64_t q[MAXK];
        for (int i = 0; i < ctx->K; i++) q[i] = ctx->hp.d.tab[i].mod.q;
        if (relin32_applicable(ctx->n, ctx->K, q, k->digits, dbc, k->r32.c)) {
            cudaError_t e = relin32_build(ctx->dP, ctx->logn, ctx->K, q, k->d, k->key_off, polys, k->r32, ctx->stream);
            if (e != cudaSuccess) { relin32_free(k->r32); dev_free(ctx, k->d); delete k; return fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e)); }
            k->has_r32 = true;
        }
    }
    *out = k;
    return CRCNN_OK;
}
int crcnn_evk_free(crcnn_ctx *ctx, crcnn_evk *k) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    if (!k) return CRCNN_OK;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    relin32_free(k->r32);
    dev_free(ctx, k->d);
    delete k;
    return CRCNN_OK;
}

// ---------------------------------------------------------------------------- layers
int crcnn_conv_forward_shard(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w, crcnn_plain *b, int batch, int xd, int yd,
                             int zd, int xs, int ys, int xf, int yf, int nf, int k0, int kc, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(in && w && b && out, "null argument");
    REQUIRE(batch > 0 && xd > 0 && yd > 0 && zd > 0 && xs > 0 && ys > 0 && xf > 0 && yf > 0 && nf > 0 && xf <= xd && yf <= yd,
            "bad convolution geometry");
    REQUIRE(k0 >= 0 && kc >= 0 && k0 + kc <= nf, "bad output-channel shard");
    REQUIRE(in->size == 2 && in->count == (long)batch * zd * xd * yd, "input tensor does not match the layer geometry");
    const int R = zd * xf * yf;
    REQUIRE(w->count == (long)nf * R && b->count == nf, "kernel/bias count does not match the layer geometry");  // convolutionalLayer.cpp:57-59
    CU(cudaSetDevice(ctx->device));
    const int xo = (xd - xf) / xs + 1, yo = (yd - yf) / ys + 1;  // convolutionalLayer.cpp:24
    int xl, yl;
    boundaries(xd, yd, xs, ys, xf, yf, &xl, &yl);
    if ((xl + xs - 1) / xs != xo || (yl + ys - 1) / ys != yo)
        return fail(ctx, CRCNN_ERR_UNSUPPORTED, "stride larger than the filter leaves outputs the reference never computes");
    const int P = xo * yo, Npos = batch * P, nin = zd * xd * yd;
    std::vector<int> key = {1, batch, xd, yd, zd, xs, ys, xf, yf};
    const int *d_index = nullptr;
    if (ctx->index_cache.find(key) == ctx->index_cache.end()) {
        std::vector<int> table((size_t)Npos * R);
        for (int bi = 0; bi < batch; bi++)
            for (int i = 0; i < xo; i++)
                for (int j = 0; j < yo; j++) {
                    int *row = &table[((size_t)bi * P + i * yo + j) * R];
                    int r = 0;
                    for (int z = 0; z < zd; z++)
                        for (int kx = 0; kx < xf; kx++)
                            for (int ky = 0; ky < yf; ky++) row[r++] = bi * nin + (z * xd + i * xs + kx) * yd + j * ys + ky;
                }
        int rc = get_index_table(ctx, key, table, &d_index);
        if (rc) return rc;
    } else {
        d_index = ctx->index_cache[key];
    }
    crcnn_tensor *o = nullptr;
    int rc = new_tensor(ctx, (long)batch * kc * P, 2, 1, &o);
    if (rc) return rc;
    rc = run_weighted_sum(ctx, in, w, b, d_index, R, Npos, P, nf, k0, kc, o);
    if (rc) { crcnn_tensor_free(ctx, o); return rc; }
    *out = o;
    return CRCNN_OK;
}

int crcnn_conv_forward(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w, crcnn_plain *b, int batch, int xd, int yd, int zd,
                       int xs, int ys, int xf, int yf, int nf, crcnn_tensor **out) {
    return crcnn_conv_forward_shard(ctx, in, w, b, batch, xd, yd, zd, xs, ys, xf, yf, nf, 0, nf, out);
}

int crcnn_fc_forward_shard(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w, crcnn_plain *b, int batch, int in_dim,
                           int out_dim, int o0, int oc, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(in && w && b && out, "null argument");
    REQUIRE(batch > 0 && in_dim > 0 && out_dim > 0, "bad fully-connected geometry");
    REQUIRE(o0 >= 0 && oc >= 0 && o0 + oc <= out_dim, "bad output-row shard");
    REQUIRE(in->size == 2 && in->count == (long)batch * in_dim, "input tensor does not match the layer geometry");
    REQUIRE(w->count == (long)out_dim * in_dim && b->count == out_dim, "weight/bias count does not match the layer geometry");
    CU(cudaSetDevice(ctx->device));
    std::vector<int> key = {2, batch, in_dim};
    const int *d_index = nullptr;
    if (ctx->index_cache.find(key) == ctx->index_cache.end()) {
        std::vector<int> table((size_t)batch * in_dim);
        for (size_t i = 0; i < table.size(); i++) table[i] = (int)i;
        int rc = get_index_table(ctx, key, table, &d_index);
        if (rc) return rc;
    } else {
        d_index = ctx->index_cache[key];
    }
    crcnn_tensor *o = nullptr;
    int rc = new_tensor(ctx, (long)batch * oc, 2, 1, &o);
    if (rc) return rc;
    rc = run_weighted_sum(ctx, in, w, b, d_index, in_dim, batch, 1, out_dim, o0, oc, o);
    if (rc) { crcnn_tensor_free(ctx, o); return rc; }
    *out = o;
    return CRCNN_OK;
}

int crcnn_fc_forward(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w, crcnn_plain *b, int batch, int in_dim, int out_dim,
                     crcnn_tensor **out) {
    return crcnn_fc_forward_shard(ctx, in, w, b, batch, in_dim, out_dim, 0, out_dim, out);
}

// Two FullyConnectedLayers with nothing between them (fc3 -> fc4 of every reference topology, cnnBuilder.cpp:121-122, 132-133, 153-154):
//     fc2(fc1(x)) = W2 (W1 x + Delta b1) + Delta b2 = (W2 W1) x + (W2 Delta b1 + Delta b2)          over Z_q[x]/(x^n+1),
// so the pair is ONE weighted sum with the composed weights W = W2 W1 (out_dim x in_dim ring elements) and bias B = W2 Delta b1 +
// Delta b2.  Both are computed once per network, on the device, by this engine's own weighted-sum kernels: column pairs (r, r+1) of
// W1's NTT form play the two polynomials of a "ciphertext", fc2 applied to them yields the matching columns of W.  The composed
// layer has out_dim x in_dim terms instead of mid_dim x (in_dim + out_dim) -- 50x fewer for PlainModel -- and produces the canonical residues
// of the same ring elements, hence the reference's bytes.  The composed weights are general residues: limb-split GEMM only.
// With C / D (per input channel, `per_channel` inputs each; ensure_pool_bn_consts) the layer in front of fc1 -- x = P (.) C_c - D_c, the pooling
// scale and batch-norm applied to window sums P -- goes into the composed constants as well: W[k,r] (.)= C_c(r), B_k -= sum_r W[k,r] (.) D_c(r).
static int compose_fc(crcnn_ctx *ctx, crcnn_plain *w1, crcnn_plain *b1, crcnn_plain *w2, crcnn_plain *b2, int in_dim, int mid_dim, int out_dim,
                      const uint64_t *C = nullptr, const uint64_t *D = nullptr, int per_channel = 1) {
    const size_t pw = poly_words(ctx);
    const int saved_tc = ctx->tc_mode;
    const bool saved_prof = ctx->prof_on;
    ctx->tc_mode = 0;           // NTT-domain kernels only: the "ciphertexts" below are NTT-form plaintexts
    ctx->prof_on = false;       // build-time work is not part of any step's profile
    crcnn_plain *zero = nullptr, *W = nullptr, *B = nullptr;
    crcnn_tensor *T = nullptr, *O = nullptr;
    uint64_t *dense = nullptr;
    int rc = CRCNN_OK;
    auto done = [&](int code) {
        if (T) crcnn_tensor_free(ctx, T);
        if (O) crcnn_tensor_free(ctx, O);
        if (zero) crcnn_plain_free(ctx, zero);
        dev_free(ctx, dense);
        if (code) { if (W) crcnn_plain_free(ctx, W); if (B) crcnn_plain_free(ctx, B); }
        ctx->tc_mode = saved_tc; ctx->prof_on = saved_prof;
        return code;
    };
    rc = make_plain(ctx, std::vector<uint32_t>((size_t)out_dim + 1, 0), {}, {}, &zero);
    if (rc) return done(rc);
    rc = dev_alloc(ctx, (size_t)out_dim * in_dim * pw * 8, (void **)&dense);
    if (rc) return done(rc);
    // column pairs per pass: the staged columns of W1 (mid_dim pseudo-ciphertexts per pair) stay below ~8 GB
    const int pairs_all = (in_dim + 1) / 2;
    int Bc = (int)std::max<size_t>(1, std::min<size_t>((size_t)pairs_all, (8ull << 30) / ((size_t)mid_dim * 2 * pw * 8)));
    if (const char *e = getenv("CRCNN_FC_COMPOSE_PAIRS")) Bc = std::max(1, std::min(Bc, atoi(e)));   // tests: several passes on small layers
    std::vector<int> table((size_t)Bc * mid_dim);
    for (int bi = 0; bi < Bc; bi++)
        for (int o = 0; o < mid_dim; o++) table[(size_t)bi * mid_dim + o] = o * Bc + bi;
    const int *d_index = nullptr;
    rc = get_index_table(ctx, {5, Bc, mid_dim}, table, &d_index);
    if (rc) return done(rc);
    rc = new_tensor(ctx, (long)mid_dim * Bc, 2, 1, &T);
    if (!rc) rc = new_tensor(ctx, (long)Bc * out_dim, 2, 1, &O);
    if (rc) return done(rc);
    CU(cudaMemsetAsync(T->d, 0, (size_t)T->count * 2 * pw * 8, ctx->stream));
    for (int r0 = 0; r0 < in_dim && !rc; r0 += 2 * Bc) {
        const int cols = std::min(2 * Bc, in_dim - r0);
        for (int o = 0; o < mid_dim && !rc; o++)
            rc = expand_range(ctx, w1, (long)o * in_dim + r0, cols, PF_NTT_MUL, T->d + (size_t)o * Bc * 2 * pw);
        if (rc) break;
        rc = run_weighted_sum(ctx, T, w2, zero, d_index, mid_dim, Bc, 1, out_dim, 0, out_dim, O);
        if (rc) break;
        // O[b][k] = (W[k][r0+2b], W[k][r0+2b+1])  ->  dense[k][r]
        for (int bi = 0; 2 * bi < cols; bi++) {
            const int polys = std::min(2, cols - 2 * bi);
            cudaError_t e = cudaMemcpy2DAsync(dense + ((size_t)r0 + 2 * bi) * pw, (size_t)in_dim * pw * 8, O->d + (size_t)bi * out_dim * 2 * pw,
                                              2 * pw * 8, (size_t)polys * pw * 8, out_dim, cudaMemcpyDeviceToDevice, ctx->stream);
            if (e != cudaSuccess) { rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e)); break; }
        }
    }
    if (rc) return done(rc);
    W = new crcnn_plain();
    W->count = (long)out_dim * in_dim; W->dense_only = true; W->sparse_shape = false; W->tc_state = -1; W->tap_state = -1;
    W->ntt_mul = dense; dense = nullptr;
    // bias: fc2 applied to the Delta-scaled b1 (polynomial 0 of one pseudo-ciphertext per middle neuron), plus Delta b2
    rc = ensure_form(ctx, b1, PF_NTT_ADD);
    if (rc) return done(rc);
    crcnn_tensor_free(ctx, T); T = nullptr;
    crcnn_tensor_free(ctx, O); O = nullptr;
    rc = new_tensor(ctx, mid_dim, 2, 1, &T);
    if (!rc) rc = new_tensor(ctx, out_dim, 2, 1, &O);
    if (rc) return done(rc);
    CU(cudaMemsetAsync(T->d, 0, (size_t)mid_dim * 2 * pw * 8, ctx->stream));
    CU(cudaMemcpy2DAsync(T->d, 2 * pw * 8, b1->ntt_add, pw * 8, pw * 8, mid_dim, cudaMemcpyDeviceToDevice, ctx->stream));
    std::vector<int> ident(mid_dim);
    for (int o = 0; o < mid_dim; o++) ident[o] = o;
    rc = get_index_table(ctx, {2, 1, mid_dim}, ident, &d_index);
    if (!rc) rc = run_weighted_sum(ctx, T, w2, b2, d_index, mid_dim, 1, 1, out_dim, 0, out_dim, O);
    if (rc) return done(rc);
    B = new crcnn_plain();
    B->count = out_dim; B->dense_only = true; B->sparse_shape = false; B->tc_state = -1; B->tap_state = -1;
    rc = dev_alloc(ctx, (size_t)out_dim * pw * 8, (void **)&B->ntt_add);
    if (rc) return done(rc);
    CU(cudaMemcpy2DAsync(B->ntt_add, pw * 8, O->d, 2 * pw * 8, pw * 8, out_dim, cudaMemcpyDeviceToDevice, ctx->stream));
    if (C) CU(launch_fold_fc_input_affine(ctx->dP, W->ntt_mul, out_dim, in_dim, (long)pw, per_channel, C, D, B->ntt_add, ctx->stream));
    rc = ensure_tcn_weights(ctx, W, in_dim, false);   // byte planes of the composed weights; releases the dense form
    if (rc) return done(rc);
    w1->folded_w = W; w1->folded_b = B;
    return done(CRCNN_OK);
}

int crcnn_fc_fc_forward(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w1, crcnn_plain *b1, crcnn_plain *w2, crcnn_plain *b2, int batch,
                        int in_dim, int mid_dim, int out_dim, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(in && w1 && b1 && w2 && b2 && out, "null argument");
    REQUIRE(batch > 0 && in_dim > 0 && mid_dim > 0 && out_dim > 0, "bad fully-connected geometry");
    REQUIRE(in->size == 2 && in->count == (long)batch * in_dim, "input tensor does not match the layer geometry");
    REQUIRE(w1->count == (long)mid_dim * in_dim && b1->count == mid_dim && w2->count == (long)out_dim * mid_dim && b2->count == out_dim,
            "weight/bias count does not match the layer geometry");
    CU(cudaSetDevice(ctx->device));
    // worth it when the composed layer is the smaller one, and possible when its byte planes fit the weight cache
    const bool composed = (double)out_dim * in_dim < (double)mid_dim * (in_dim + out_dim) && !w1->dense_only && !w2->dense_only &&
                          ctx->tcn_mode && tcn_planes_for(ctx->hp.d) == 7 && in_dim <= TCN_MAX_R && mid_dim <= TCN_MAX_R &&
                          tc_mac_available() == cudaSuccess && tcn_w_bytes(7, out_dim, tcn_kpad(in_dim), ctx->K, ctx->n) <= ctx->weight_cache_bytes &&
                          !getenv("CRCNN_NO_FC_COMPOSE");
    if (!composed) {
        crcnn_tensor *mid = nullptr;
        int rc = crcnn_fc_forward(ctx, in, w1, b1, batch, in_dim, mid_dim, &mid);
        if (rc) return rc;
        rc = crcnn_fc_forward(ctx, mid, w2, b2, batch, mid_dim, out_dim, out);
        crcnn_tensor_free(ctx, mid);
        return rc;
    }
    const long key[9] = {b1->serial, w2->serial, b2->serial, (long)mid_dim, (long)out_dim, 0, 0, 0, 0};
    if (!w1->folded_w || memcmp(key, w1->folded_key, sizeof(key)) != 0) {
        if (w1->folded_w) { crcnn_plain_free(ctx, w1->folded_w); w1->folded_w = nullptr; }
        if (w1->folded_b) { crcnn_plain_free(ctx, w1->folded_b); w1->folded_b = nullptr; }
        int rc = compose_fc(ctx, w1, b1, w2, b2, in_dim, mid_dim, out_dim);
        if (rc) return rc;
        memcpy(w1->folded_key, key, sizeof(key));
    }
    return crcnn_fc_forward(ctx, in, w1->folded_w, w1->folded_b, batch, in_dim, out_dim, out);
}

// AvgPoolingLayer -> BatchNormLayer -> FullyConnectedLayer -> FullyConnectedLayer (layers 5-8 of the reference's nine-layer networks,
// cnnBuilder.cpp:118-122): the window sums of the input, then ONE composed fully connected layer that carries the pooling scale, the
// batch-norm and both weight matrices (compose_fc with the per-channel constants).  Same bytes as the four calls.
int crcnn_pool_bn_fc_fc_forward(crcnn_ctx *ctx, crcnn_tensor *in, int batch, int xd, int yd, int zd, int pxs, int pys, int pxf, int pyf,
                                crcnn_plain *scale, crcnn_plain *mean, crcnn_plain *invstd, crcnn_plain *w1, crcnn_plain *b1,
                                crcnn_plain *w2, crcnn_plain *b2, int mid_dim, int out_dim, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(in && mean && invstd && w1 && b1 && w2 && b2 && out, "null argument");      // scale == NULL: PoolingLayer
    REQUIRE(batch > 0 && xd > 0 && yd > 0 && zd > 0 && pxs > 0 && pys > 0 && pxf > 0 && pyf > 0 && pxf <= xd && pyf <= yd, "bad pooling geometry");
    REQUIRE(mid_dim > 0 && out_dim > 0, "bad fully-connected geometry");
    const int pxo = (xd - pxf) / pxs + 1, pyo = (yd - pyf) / pys + 1, Rp = pxf * pyf;
    const int in_dim = zd * pxo * pyo;
    REQUIRE(in->size == 2 && in->count == (long)batch * zd * xd * yd, "input tensor does not match the layer geometry");
    REQUIRE((!scale || scale->count >= 1) && mean->count == zd && invstd->count == zd, "mean/var count does not match the channel count");
    REQUIRE(w1->count == (long)mid_dim * in_dim && b1->count == mid_dim && w2->count == (long)out_dim * mid_dim && b2->count == out_dim,
            "weight/bias count does not match the layer geometry");
    CU(cudaSetDevice(ctx->device));
    const bool composed = pxs <= pxf && pys <= pyf && sum_fits_64(ctx, Rp) &&
                          (double)out_dim * in_dim < (double)mid_dim * (in_dim + out_dim) && !w1->dense_only && !w2->dense_only &&
                          ctx->tcn_mode && tcn_planes_for(ctx->hp.d) == 7 && in_dim <= TCN_MAX_R && mid_dim <= TCN_MAX_R &&
                          tc_mac_available() == cudaSuccess && tcn_w_bytes(7, out_dim, tcn_kpad(in_dim), ctx->K, ctx->n) <= ctx->weight_cache_bytes &&
                          !getenv("CRCNN_NO_FC_COMPOSE");
    if (!composed) {
        crcnn_tensor *mid = nullptr;
        int rc = crcnn_pool_bn_forward(ctx, in, batch, xd, yd, zd, pxs, pys, pxf, pyf, scale, mean, invstd, &mid);
        if (rc) return rc;
        rc = crcnn_fc_fc_forward(ctx, mid, w1, b1, w2, b2, batch, in_dim, mid_dim, out_dim, out);
        crcnn_tensor_free(ctx, mid);
        return rc;
    }
    int rc = ensure_pool_bn_consts(ctx, scale, mean, invstd);
    if (rc) return rc;
    const long key[9] = {b1->serial, w2->serial, b2->serial, (long)mid_dim, (long)out_dim, scale ? scale->serial : -1, mean->serial, invstd->serial, (long)(pxo * pyo)};
    if (!w1->folded_w || memcmp(key, w1->folded_key, sizeof(key)) != 0) {
        if (w1->folded_w) { crcnn_plain_free(ctx, w1->folded_w); w1->folded_w = nullptr; }
        if (w1->folded_b) { crcnn_plain_free(ctx, w1->folded_b); w1->folded_b = nullptr; }
        rc = compose_fc(ctx, w1, b1, w2, b2, in_dim, mid_dim, out_dim, invstd->fused_C, invstd->fused_D, pxo * pyo);
        if (rc) return rc;
        memcpy(w1->folded_key, key, sizeof(key));
    }
    // window sums (no scale), in the input's domain: the pooling layer's own index table
    crcnn_tensor *sums = nullptr;
    rc = crcnn_pool_forward(ctx, in, batch, xd, yd, zd, pxs, pys, pxf, pyf, nullptr, &sums);
    if (rc) return rc;
    rc = crcnn_fc_forward(ctx, sums, w1->folded_w, w1->folded_b, batch, in_dim, out_dim, out);
    crcnn_tensor_free(ctx, sums);
    return rc;
}

int crcnn_pool_forward(crcnn_ctx *ctx, crcnn_tensor *in, int batch, int xd, int yd, int zd, int xs, int ys, int xf, int yf,
                       crcnn_plain *scale, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(in && out, "null argument");
    REQUIRE(batch > 0 && xd > 0 && yd > 0 && zd > 0 && xs > 0 && ys > 0 && xf > 0 && yf > 0 && xf <= xd && yf <= yd, "bad pooling geometry");
    REQUIRE(in->size == 2 && in->count == (long)batch * zd * xd * yd, "input tensor does not match the layer geometry");
    REQUIRE(!scale || scale->count >= 1, "empty scale pack");
    CU(cudaSetDevice(ctx->device));
    const int xo = (xd - xf) / xs + 1, yo = (yd - yf) / ys + 1;  // poolingLayer.cpp:18
    int xl, yl;
    boundaries(xd, yd, xs, ys, xf, yf, &xl, &yl);
    if ((xl + xs - 1) / xs != xo || (yl + ys - 1) / ys != yo)
        return fail(ctx, CRCNN_ERR_UNSUPPORTED, "stride larger than the window leaves outputs the reference never computes");
    const int R = xf * yf, Nout = batch * zd * xo * yo;
    std::vector<int> key = {3, batch, xd, yd, zd, xs, ys, xf, yf};
    const int *d_index = nullptr;
    if (ctx->index_cache.find(key) == ctx->index_cache.end()) {
        std::vector<int> table((size_t)Nout * R);
        size_t o = 0;
        for (int bz = 0; bz < batch * zd; bz++)
            for (int i = 0; i < xo; i++)
                for (int j = 0; j < yo; j++)
                    for (int kx = 0; kx < xf; kx++)
                        for (int ky = 0; ky < yf; ky++) table[o++] = (bz * xd + i * xs + kx) * yd + j * ys + ky;
        int rc = get_index_table(ctx, key, table, &d_index);
        if (rc) return rc;
    } else {
        d_index = ctx->index_cache[key];
    }
    int rc = CRCNN_OK;
    if (scale && !in->ntt && ctx->tap_mode && tap_eligible(ctx, scale) && sum_fits_64(ctx, R)) {
        // coefficient-form input (after the square activation): stay there, no transform in either direction
        crcnn_tensor *o = nullptr;
        rc = new_tensor(ctx, Nout, 2, 0, &o);
        if (rc) return rc;
        TapMulArgs a{};
        a.in = in->d; a.in_index = d_index; a.R = R; a.sub = nullptr;
        a.t_off = scale->d_off; a.t_idx = scale->d_idx; a.t_val = scale->d_val; a.per_channel = 1; a.channels = 1;
        a.out = o->d; a.nout = Nout;
        ProfScope ps(ctx, KC_POOL, lp_bytes(ctx, ((double)in->count + Nout) * 2 * ctx->K), (double)Nout * R * 2 * ctx->K * ctx->n);
        cudaError_t e = launch_tapmul(ctx->dP, ctx->n, ctx->K, a, ctx->stream);
        if (e != cudaSuccess) { crcnn_tensor_free(ctx, o); return fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e)); }
        *out = o;
        return CRCNN_OK;
    }
    if (scale) {
        rc = ensure_domain(ctx, in, 1);
        if (!rc) rc = ensure_shoup(ctx, scale);
        if (rc) return rc;
    }
    crcnn_tensor *o = nullptr;
    rc = new_tensor(ctx, Nout, 2, in->ntt, &o);
    if (rc) return rc;
    {
        ProfScope ps(ctx, KC_POOL, lp_bytes(ctx, ((double)in->count + Nout) * 2 * ctx->K), (double)Nout * R * 2 * ctx->K * ctx->n);
        cudaError_t e = launch_pool(ctx->dP, ctx->n, ctx->K, in->d, d_index, Nout, R, scale ? scale->ntt_mul : nullptr,
                                    scale ? scale->ntt_mul_sh : nullptr, sum_fits_64(ctx, R), o->d, ctx->stream);
        if (e != cudaSuccess) { crcnn_tensor_free(ctx, o); return fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e)); }
    }
    *out = o;
    return CRCNN_OK;
}

/* Replaces AvgPoolingLayer::forward immediately followed by BatchNormLayer::forward (CrCNN/src/avgPoolingLayer.cpp:16-45,
 * batchNormLayer.cpp:29-40) in ONE pass when the activations are in NTT form: out = (window sum) * (scale (.) invstd_z) - mean_z (.) invstd_z.
 * Same canonical residues (ring arithmetic mod q_j), one read of the inputs and one write instead of two of each.  Coefficient-form
 * activations (after the square layer) take the two coefficient-domain kernels in sequence. */
int crcnn_pool_bn_forward(crcnn_ctx *ctx, crcnn_tensor *in, int batch, int xd, int yd, int zd, int xs, int ys, int xf, int yf,
                          crcnn_plain *scale, crcnn_plain *mean, crcnn_plain *invstd, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(in && mean && invstd && out, "null argument");      // scale == NULL: PoolingLayer (window sum without a factor)
    REQUIRE((!scale || scale->count >= 1) && mean->count == zd && invstd->count == zd, "mean/var count does not match the channel count");
    const int xo = (xd - xf) / xs + 1, yo = (yd - yf) / ys + 1;
    const int R = xf * yf;
    if (!in->ntt || !sum_fits_64(ctx, R)) {      // not the fused kernel's case: the two layers one after the other
        crcnn_tensor *mid = nullptr;
        int rc = crcnn_pool_forward(ctx, in, batch, xd, yd, zd, xs, ys, xf, yf, scale, &mid);
        if (rc) return rc;
        rc = crcnn_bn_forward(ctx, mid, batch, zd, xo, yo, mean, invstd, out);
        crcnn_tensor_free(ctx, mid);
        return rc;
    }
    // geometry checks and the window index table are those of the pooling layer: run it on an empty batch? no -- build the table here
    REQUIRE(batch > 0 && xd > 0 && yd > 0 && zd > 0 && xs > 0 && ys > 0 && xf > 0 && yf > 0 && xf <= xd && yf <= yd, "bad pooling geometry");
    REQUIRE(in->size == 2 && in->count == (long)batch * zd * xd * yd, "input tensor does not match the layer geometry");
    CU(cudaSetDevice(ctx->device));
    int xl, yl;
    boundaries(xd, yd, xs, ys, xf, yf, &xl, &yl);
    if ((xl + xs - 1) / xs != xo || (yl + ys - 1) / ys != yo)
        return fail(ctx, CRCNN_ERR_UNSUPPORTED, "stride larger than the window leaves outputs the reference never computes");
    const int Nout = batch * zd * xo * yo;
    std::vector<int> key = {3, batch, xd, yd, zd, xs, ys, xf, yf};
    const int *d_index = nullptr;
    if (ctx->index_cache.find(key) == ctx->index_cache.end()) {
        std::vector<int> table((size_t)Nout * R);
        size_t o = 0;
        for (int bz = 0; bz < batch * zd; bz++)
            for (int i = 0; i < xo; i++)
                for (int j = 0; j < yo; j++)
                    for (int kx = 0; kx < xf; kx++)
                        for (int ky = 0; ky < yf; ky++) table[o++] = (bz * xd + i * xs + kx) * yd + j * ys + ky;
        int rc = get_index_table(ctx, key, table, &d_index);
        if (rc) return rc;
    } else {
        d_index = ctx->index_cache[key];
    }
    int rc = ensure_pool_bn_consts(ctx, scale, mean, invstd);
    if (rc) return rc;
    crcnn_tensor *o = nullptr;
    rc = new_tensor(ctx, Nout, 2, 1, &o);
    if (rc) return rc;
    {
        ProfScope ps(ctx, KC_POOL, lp_bytes(ctx, ((double)in->count + Nout) * 2 * ctx->K), (double)Nout * (R + 1) * 2 * ctx->K * ctx->n);
        cudaError_t e = launch_pool(ctx->dP, ctx->n, ctx->K, in->d, d_index, Nout, R, invstd->fused_C, invstd->fused_Csh, true, o->d, ctx->stream,
                                    xo * yo, zd, invstd->fused_D);
        if (e != cudaSuccess) { crcnn_tensor_free(ctx, o); return fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e)); }
    }
    *out = o;
    return CRCNN_OK;
}

// Convolution -> average pooling -> batch-norm as the reference's nine-layer blocks chain them (cnnBuilder.cpp:109-134), computed on
// the POOLED grid.  Every one of these layers is linear (affine) over Z_q[x]/(x^n+1), so with cs / ps the convolution / pooling strides
//     sum_{(a,b) in window} conv(X)[k, i*ps+a, j*ps+b]  =  sum_r W[k,r] * S[z_r, i*ps*cs + kx_r, j*ps*cs + ky_r]  +  |window| * B_k,
//     S[z,u,v] = sum_{(a,b) in window} X[z, u + a*cs, v + b*cs]             (one dilated window sum of the layer's INPUT),
// i.e. the convolution at stride ps*cs over the window sums of its input with the bias added |window| times, and the pooling scale and
// batch-norm  y -> y (.) C_k - D_k  (ensure_pool_bn_consts) go into the convolution's own constants:
//     W'[k,r] = W[k,r] (.) C_k,      B'_k = |window| * B_k (.) C_k - D_k        (NTT domain, computed once per network).
// One weighted sum with (pooled positions / convolution positions) of the columns replaces three layers and two full-size
// intermediates; the residues are the canonical ones of the same ring elements, hence the reference's bytes.
int crcnn_conv_pool_bn_forward_shard(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w, crcnn_plain *b, int batch, int xd, int yd, int zd,
                                     int xs, int ys, int xf, int yf, int nf, int pxs, int pys, int pxf, int pyf, crcnn_plain *scale,
                                     crcnn_plain *mean, crcnn_plain *invstd, int k0, int kc, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(k0 >= 0 && kc >= 0 && k0 + kc <= nf, "bad output-channel shard");
    REQUIRE(in && w && b && mean && invstd && out, "null argument");      // scale == NULL: PoolingLayer (window sum without a factor)
    REQUIRE(batch > 0 && xd > 0 && yd > 0 && zd > 0 && xs > 0 && ys > 0 && xf > 0 && yf > 0 && nf > 0 && xf <= xd && yf <= yd,
            "bad convolution geometry");
    const int cxo = (xd - xf) / xs + 1, cyo = (yd - yf) / ys + 1;          // convolution output (convolutionalLayer.cpp:24)
    REQUIRE(pxs > 0 && pys > 0 && pxf > 0 && pyf > 0 && pxf <= cxo && pyf <= cyo, "bad pooling geometry");
    const int pxo = (cxo - pxf) / pxs + 1, pyo = (cyo - pyf) / pys + 1;    // pooled output (poolingLayer.cpp:18)
    const int Rp = pxf * pyf, R = zd * xf * yf;
    REQUIRE(in->size == 2 && in->count == (long)batch * zd * xd * yd, "input tensor does not match the layer geometry");
    REQUIRE(w->count == (long)nf * R && b->count == nf, "kernel/bias count does not match the layer geometry");
    REQUIRE((!scale || scale->count >= 1) && mean->count == nf && invstd->count == nf, "mean/var count does not match the channel count");
    CU(cudaSetDevice(ctx->device));
    // the pooled grid needs: strides that leave no output the reference skips (computeBoundaries), window sums below 2^64, and the
    // limb-split weighted sum (any NTT-form weights) with the folded weight planes resident
    const bool pooled_grid = pxs <= pxf && pys <= pyf && xs <= xf && ys <= yf && pxs * xs <= xf && pys * ys <= yf && Rp <= 64 && sum_fits_64(ctx, Rp) &&
                             ctx->tcn_mode && tcn_planes_for(ctx->hp.d) == 7 && R <= TCN_MAX_R && tc_mac_available() == cudaSuccess &&
                             tcn_w_bytes(7, nf, tcn_kpad(R), ctx->K, ctx->n) <= ctx->weight_cache_bytes && !getenv("CRCNN_NO_POOLED_CONV");
    if (!pooled_grid) {   // the three layers one after the other (the last two in one pass when the activations are in NTT form)
        if (k0 != 0 || kc != nf)    // a channel shard of the layer-by-layer path is the caller's: conv shard, then pool and batch-norm on its channels
            return fail(ctx, CRCNN_ERR_UNSUPPORTED, "channel shards of conv + pool + batch-norm need the pooled-grid path");
        crcnn_tensor *mid = nullptr;
        int rc = crcnn_conv_forward(ctx, in, w, b, batch, xd, yd, zd, xs, ys, xf, yf, nf, &mid);
        if (rc) return rc;
        rc = crcnn_pool_bn_forward(ctx, mid, batch, cxo, cyo, nf, pxs, pys, pxf, pyf, scale, mean, invstd, out);
        crcnn_tensor_free(ctx, mid);
        return rc;
    }
    int rc = ensure_pool_bn_consts(ctx, scale, mean, invstd);
    if (rc) return rc;
    const long key[9] = {b->serial, scale ? scale->serial : -1, mean->serial, invstd->serial, (long)Rp, 0, 0, 0, 0};
    if (!w->folded_w || memcmp(key, w->folded_key, sizeof(key)) != 0) {
        if (w->folded_w) { crcnn_plain_free(ctx, w->folded_w); w->folded_w = nullptr; }
        if (w->folded_b) { crcnn_plain_free(ctx, w->folded_b); w->folded_b = nullptr; }
        const size_t pw = poly_words(ctx);
        // W' : the NTT form of W, row m*R + r times C[m]; staged as byte planes right away (the dense form is released by the staging)
        rc = make_plain(ctx, std::vector<uint32_t>(w->off), std::vector<uint32_t>(w->idx), std::vector<uint64_t>(w->val), &w->folded_w);
        if (rc) return rc;
        w->folded_w->sparse_shape = false;   // never the ternary-tap path: these weights are general residues
        w->folded_w->tc_state = -1; w->folded_w->tap_state = -1;
        rc = ensure_form(ctx, w->folded_w, PF_NTT_MUL);
        if (rc) return rc;
        CU(launch_fold_affine(ctx->dP, w->folded_w->ntt_mul, (long)nf * R, (long)pw, R, invstd->fused_C, nullptr, ctx->stream));
        // staged as byte planes by the first weighted sum below, which knows the shape (pre-shifted or not); it releases the dense form
        // B' : |window| * (Delta-scaled bias) in NTT form, times C[m], minus D[m]
        rc = make_plain(ctx, std::vector<uint32_t>(b->off), std::vector<uint32_t>(b->idx), std::vector<uint64_t>(b->val), &w->folded_b);
        if (rc) return rc;
        w->folded_b->add_mult = Rp;
        rc = ensure_form(ctx, w->folded_b, PF_NTT_ADD);
        if (rc) return rc;
        CU(launch_fold_affine(ctx->dP, w->folded_b->ntt_add, (long)nf, (long)pw, 1, invstd->fused_C, invstd->fused_D, ctx->stream));
        memcpy(w->folded_key, key, sizeof(key));
    }
    // S: dilated window sums of the input, (zd, sxd, syd) per image, in the input's domain
    const int sxd = xd - (pxf - 1) * xs, syd = yd - (pyf - 1) * ys;
    const int Nsum = batch * zd * sxd * syd;
    std::vector<int> skey = {4, batch, xd, yd, zd, xs, ys, pxf, pyf};
    const int *d_index = nullptr;
    if (ctx->index_cache.find(skey) == ctx->index_cache.end()) {
        std::vector<int> table((size_t)Nsum * Rp);
        size_t o = 0;
        for (int bz = 0; bz < batch * zd; bz++)
            for (int u = 0; u < sxd; u++)
                for (int v = 0; v < syd; v++)
                    for (int a = 0; a < pxf; a++)
                        for (int c = 0; c < pyf; c++) table[o++] = (bz * xd + u + a * xs) * yd + v + c * ys;
        rc = get_index_table(ctx, skey, table, &d_index);
        if (rc) return rc;
    } else {
        d_index = ctx->index_cache[skey];
    }
    crcnn_tensor *sums = nullptr, *pooled = nullptr;
    rc = new_tensor(ctx, Nsum, 2, in->ntt, &sums);
    if (rc) return rc;
    {
        ProfScope ps(ctx, KC_POOL, lp_bytes(ctx, ((double)in->count + Nsum) * 2 * ctx->K), (double)Nsum * Rp * 2 * ctx->K * ctx->n);
        cudaError_t e = launch_pool(ctx->dP, ctx->n, ctx->K, in->d, d_index, Nsum, Rp, nullptr, nullptr, true, sums->d, ctx->stream);
        if (e != cudaSuccess) { crcnn_tensor_free(ctx, sums); return fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e)); }
    }
    rc = crcnn_conv_forward_shard(ctx, sums, w->folded_w, w->folded_b, batch, sxd, syd, zd, pxs * xs, pys * ys, xf, yf, nf, k0, kc, &pooled);
    crcnn_tensor_free(ctx, sums);
    if (rc) return rc;
    if (pooled->count != (long)batch * kc * pxo * pyo || !pooled->ntt) {
        crcnn_tensor_free(ctx, pooled);
        return fail(ctx, CRCNN_ERR_UNSUPPORTED, "pooled-grid convolution produced an unexpected shape");
    }
    *out = pooled;
    return CRCNN_OK;
}

int crcnn_conv_pool_bn_forward(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w, crcnn_plain *b, int batch, int xd, int yd, int zd,
                               int xs, int ys, int xf, int yf, int nf, int pxs, int pys, int pxf, int pyf, crcnn_plain *scale,
                               crcnn_plain *mean, crcnn_plain *invstd, crcnn_tensor **out) {
    return crcnn_conv_pool_bn_forward_shard(ctx, in, w, b, batch, xd, yd, zd, xs, ys, xf, yf, nf, pxs, pys, pxf, pyf, scale, mean, invstd, 0, nf, out);
}

int crcnn_bn_forward(crcnn_ctx *ctx, crcnn_tensor *in, int batch, int zd, int xd, int yd, crcnn_plain *mean,
                     crcnn_plain *invstd, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(in && mean && invstd && out, "null argument");
    REQUIRE(batch > 0 && zd > 0 && xd > 0 && yd > 0, "bad batch-norm geometry");
    REQUIRE(in->size == 2 && in->count == (long)batch * zd * xd * yd, "input tensor does not match the layer geometry");
    REQUIRE(mean->count == zd && invstd->count == zd, "mean/var count does not match the channel count");
    CU(cudaSetDevice(ctx->device));
    if (!in->ntt && ctx->tap_mode && tap_eligible(ctx, invstd)) {
        int rc = ensure_form(ctx, mean, PF_COEF_ADD);
        if (rc) return rc;
        crcnn_tensor *o = nullptr;
        rc = new_tensor(ctx, in->count, 2, 0, &o);
        if (rc) return rc;
        TapMulArgs a{};
        a.in = in->d; a.in_index = nullptr; a.R = 1; a.sub = mean->coef_add;
        a.t_off = invstd->d_off; a.t_idx = invstd->d_idx; a.t_val = invstd->d_val; a.per_channel = xd * yd; a.channels = zd;
        a.out = o->d; a.nout = in->count;
        ProfScope ps(ctx, KC_BN, lp_bytes(ctx, (double)in->count * 4 * ctx->K), (double)in->count * 2 * ctx->K * ctx->n);
        cudaError_t e = launch_tapmul(ctx->dP, ctx->n, ctx->K, a, ctx->stream);
        if (e != cudaSuccess) { crcnn_tensor_free(ctx, o); return fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e)); }
        *out = o;
        return CRCNN_OK;
    }
    int rc = ensure_domain(ctx, in, 1);
    if (!rc) rc = ensure_form(ctx, mean, PF_NTT_ADD);
    if (!rc) rc = ensure_shoup(ctx, invstd);
    if (rc) return rc;
    crcnn_tensor *o = nullptr;
    rc = new_tensor(ctx, in->count, 2, 1, &o);
    if (rc) return rc;
    {
        ProfScope ps(ctx, KC_BN, lp_bytes(ctx, (double)in->count * 4 * ctx->K), (double)in->count * 2 * ctx->K * ctx->n);
        cudaError_t e = launch_bn(ctx->dP, ctx->n, ctx->K, in->d, in->count, xd * yd, zd, mean->ntt_add, invstd->ntt_mul, invstd->ntt_mul_sh, o->d, ctx->stream);
        if (e != cudaSuccess) { crcnn_tensor_free(ctx, o); return fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e)); }
    }
    *out = o;
    return CRCNN_OK;
}

int crcnn_square(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_tensor **out3) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(in && out3, "null argument");
    REQUIRE(in->size == 2, "square expects size-2 ciphertexts");
    CU(cudaSetDevice(ctx->device));
    // An NTT-form input (the usual case: the convolution before the activation leaves NTT form) keeps its transformed q
    // limbs: the base conversion works on an inverse-transformed COPY, and only the Bsk limbs are transformed again.
    const bool have_ntt = in->ntt != 0;
    // lean: the tensor stage leaves n^-1 to the floor's constants (and reduces on the fold where it applies); so does the INTT copy
    // to the lift's -- not a coefficient-form input, whose q limbs the lift copies into ext unscaled
    const bool lean = ctx->sq_lean != 0, fold = lean && behz_fold_ok(ctx->hp.d), copy_ninv = !(lean && have_ntt);
    crcnn_tensor *o = nullptr;
    int rc = new_tensor(ctx, in->count, 3, 0, &o);
    if (rc) return rc;
    const int KS = ctx->K + ctx->S;
    const size_t n = ctx->n, pw = poly_words(ctx);
    // bound the scratch: chunks of at most `step` ciphertexts
    const long step = std::max<long>(1, std::min<long>(in->count, (long)((2ull << 30) / (5 * (size_t)KS * n * 8))));
    uint64_t *ext = nullptr, *prod = nullptr, *coef = nullptr;
    rc = dev_alloc(ctx, (size_t)step * 2 * KS * n * 8, (void **)&ext);
    if (!rc) rc = dev_alloc(ctx, (size_t)step * 3 * KS * n * 8, (void **)&prod);
    if (!rc && have_ntt) rc = dev_alloc(ctx, (size_t)step * 2 * pw * 8, (void **)&coef);
    if (rc) { crcnn_tensor_free(ctx, o); return rc; }
    for (long c0 = 0; c0 < in->count && !rc; c0 += step) {
        const long cur = std::min<long>(step, in->count - c0);
        const uint64_t *src = in->d + c0 * 2 * pw;
        cudaError_t e = cudaSuccess;
        if (have_ntt) {
            ProfScope ps(ctx, KC_NTT_INV, 2 * lp_bytes(ctx, (double)cur * 2 * ctx->K), lp_bfly(ctx, (double)cur * 2 * ctx->K));
            e = launch_ntt_grouped(ctx->dP, ctx->logn, coef, cur * 2 * ctx->K, 0, ctx->K, true, ctx->K, 0, ctx->stream, src,  // out of place
                                   nullptr, 1, 1, copy_ninv);
        }
        if (e == cudaSuccess) { ProfScope ps(ctx, KC_BEHZ_LIFT, lp_bytes(ctx, (double)cur * 2 * (ctx->K + (have_ntt ? ctx->S : KS))), (double)cur * 2 * n * ctx->S * (ctx->K + 1)); e = launch_behz_lift(ctx->hp.d, ctx->n, have_ntt ? coef : src, have_ntt ? src : nullptr, cur, ext, ctx->stream, copy_ninv); }
        if (e == cudaSuccess) {
            if (have_ntt) {   // Bsk limbs only
                ProfScope ps(ctx, KC_NTT_FWD, 2 * lp_bytes(ctx, (double)cur * 2 * ctx->S), lp_bfly(ctx, (double)cur * 2 * ctx->S));
                e = launch_ntt_grouped(ctx->dP, ctx->logn, ext, cur * 2 * ctx->S, ctx->K, ctx->S, false, KS, ctx->K, ctx->stream);
            } else {
                ProfScope ps(ctx, KC_NTT_FWD, 2 * lp_bytes(ctx, (double)cur * 2 * KS), lp_bfly(ctx, (double)cur * 2 * KS));
                e = launch_ntt(ctx->dP, ctx->logn, ext, cur * 2 * KS, 0, KS, false, ctx->stream);
            }
        }
        if (e == cudaSuccess) {
            // tensor products formed while the inverse transform loads its polynomial (bytes: 2 inputs + 3 outputs per limb)
            ProfScope ps(ctx, KC_SQ_TENSOR, lp_bytes(ctx, (double)cur * 5 * KS), lp_bfly(ctx, (double)cur * 3 * KS));
            e = launch_ntt_inv_tensor(ctx->dP, ctx->logn, ext, have_ntt ? src : nullptr, cur, KS, prod, fold, !lean, ctx->stream);
        }
        if (e == cudaSuccess) { ProfScope ps(ctx, KC_BEHZ_FLOOR, lp_bytes(ctx, (double)cur * 3 * (KS + ctx->K)),
                                                     (double)cur * 3 * n * (ctx->S * (ctx->K + 1) + ctx->S + ctx->K * ctx->S)); e = launch_behz_floor(ctx->hp.d, ctx->n, prod, cur, o->d + c0 * 3 * pw, ctx->stream, !lean); }
        if (e != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e));
    }
    dev_free(ctx, coef);
    dev_free(ctx, ext); dev_free(ctx, prod);
    if (rc) { crcnn_tensor_free(ctx, o); return rc; }
    *out3 = o;
    return CRCNN_OK;
}

int crcnn_relinearize(crcnn_ctx *ctx, crcnn_tensor *in3, crcnn_evk *evk, crcnn_tensor **out2) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(in3 && evk && out2, "null argument");
    REQUIRE(in3->size == 3, "relinearize expects size-3 ciphertexts");
    int total_digits = 0;
    for (int i = 0; i < ctx->K; i++) {
        int bits = 0; for (uint64_t v = ctx->hp.d.tab[i].mod.q; v; v >>= 1) bits++;
        REQUIRE(evk->digits[i] * evk->dbc >= bits, "not enough evaluation keys");
        total_digits += evk->digits[i];
    }
    REQUIRE(total_digits <= 63, "too many key digits for 128-bit lazy accumulation");  // evaluator.cpp:972-976
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_domain(ctx, in3, 0);
    if (rc) return rc;
    crcnn_tensor *o = nullptr;
    rc = new_tensor(ctx, in3->count, 2, 0, &o);
    if (rc) return rc;
    const size_t pw = poly_words(ctx);
    if (evk->has_r32 && ctx->relin_mode == 1) {
        // word-size auxiliary-prime path: D*S3 forward + 2K*S3 inverse 32-bit transforms per ciphertext
        const Relin32Consts &c = evk->r32.c;
        const size_t per_ct = relin32_scratch_bytes(ctx->n, ctx->K, c);
        const long step = std::max<long>(1, std::min<long>(std::min<long>(in3->count, 200000), (long)((2ull << 30) / per_ct)));
        void *scratch = nullptr;
        rc = dev_alloc(ctx, (size_t)step * per_ct, &scratch);
        if (rc) { crcnn_tensor_free(ctx, o); return rc; }
        for (long c0 = 0; c0 < in3->count && !rc; c0 += step) {
            const long cnt = std::min<long>(step, in3->count - c0);
            // work: bytes = in (3 polys) + out (2 polys) per ciphertext; operations = 32-bit butterflies
            ProfScope ps(ctx, KC_RELIN32, lp_bytes(ctx, (double)cnt * 5 * ctx->K),
                         lp_bfly(ctx, (double)cnt * (c.D + 2 * ctx->K) * c.S3));
            cudaError_t e = relin32_run(ctx->dP, ctx->logn, ctx->K, evk->r32, in3->d + c0 * 3 * pw, o->d + c0 * 2 * pw, cnt, scratch, ctx->stream);
            if (e != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e));
        }
        dev_free(ctx, scratch);
        if (rc) { crcnn_tensor_free(ctx, o); return rc; }
        *out2 = o;
        return CRCNN_OK;
    }
    RelinArgs a{};
    a.evk = evk->d; a.dbc = evk->dbc;
    for (int i = 0; i < MAXK; i++) { a.key_off[i] = evk->key_off[i]; a.digits[i] = evk->digits[i]; }
    // scratch per ciphertext: scaled c2 (K polys) + digit NTTs (D*K polys) + accumulators (2K polys);
    // chunked so it stays near 2 GB
    const size_t per_ct = (size_t)(1 + total_digits + 2) * pw * 8;
    const long step = std::max<long>(1, std::min<long>(in3->count, (long)((2ull << 30) / per_ct)));
    uint64_t *scratch = nullptr;
    rc = dev_alloc(ctx, (size_t)step * per_ct, (void **)&scratch);
    if (rc) { crcnn_tensor_free(ctx, o); return rc; }
    a.dsc = scratch;
    a.dig = scratch + (size_t)step * pw;
    a.acc = a.dig + (size_t)step * total_digits * pw;
    for (long c0 = 0; c0 < in3->count && !rc; c0 += step) {
        a.count = std::min<long>(step, in3->count - c0);
        a.in3 = in3->d + c0 * 3 * pw;
        a.out = o->d + c0 * 2 * pw;
        cudaError_t e;
        { ProfScope ps(ctx, KC_RELIN, lp_bytes(ctx, (double)a.count * 3 * ctx->K), lp_bfly(ctx, (double)a.count * total_digits * ctx->K)); e = launch_relin(ctx->dP, ctx->logn, ctx->K, a, ctx->stream); }
        if (e == cudaSuccess) {
            // inverse transform of the key products, written straight to the output with "+ (c0, c1)" fused into the last pass
            ProfScope ps(ctx, KC_NTT_INV, 2 * lp_bytes(ctx, (double)a.count * 2 * ctx->K) + lp_bytes(ctx, (double)a.count * 2 * ctx->K), lp_bfly(ctx, (double)a.count * 2 * ctx->K));
            e = launch_ntt_grouped(ctx->dP, ctx->logn, a.out, a.count * 2 * ctx->K, 0, ctx->K, true, ctx->K, 0, ctx->stream, a.acc, a.in3,
                                   2 * ctx->K, 3 * ctx->K);
        }
        if (e != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e));
    }
    dev_free(ctx, scratch);
    if (rc) { crcnn_tensor_free(ctx, o); return rc; }
    *out2 = o;
    return CRCNN_OK;
}

int crcnn_square_forward(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_evk *evk, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    crcnn_tensor *t3 = nullptr;
    int rc = crcnn_square(ctx, in, &t3);
    if (rc) return rc;
    rc = crcnn_relinearize(ctx, t3, evk, out);
    crcnn_tensor_free(ctx, t3);
    return rc;
}

// ---------------------------------------------------------------------------- evaluator-level ops
int crcnn_transform_to_ntt(crcnn_ctx *ctx, crcnn_tensor *t) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(t, "null argument");
    REQUIRE(!t->ntt, "tensor is already in NTT form");
    CU(cudaSetDevice(ctx->device));
    return ensure_domain(ctx, t, 1);
}
int crcnn_transform_from_ntt(crcnn_ctx *ctx, crcnn_tensor *t) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(t, "null argument");
    REQUIRE(t->ntt, "tensor is not in NTT form");
    CU(cudaSetDevice(ctx->device));
    return ensure_domain(ctx, t, 0);
}

int crcnn_plain_op(crcnn_ctx *ctx, crcnn_tensor *t, crcnn_plain *p, long index, int op) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(t && p && index >= 0 && index < p->count && op >= 0 && op <= 2, "bad plain_op arguments");
    CU(cudaSetDevice(ctx->device));
    int rc;
    const uint64_t *pl, *pl_sh = nullptr;
    if (op == 0) {
        rc = ensure_domain(ctx, t, 1);
        if (!rc) rc = ensure_shoup(ctx, p);
        if (rc) return rc;
        pl = p->ntt_mul + index * poly_words(ctx);
        pl_sh = p->ntt_mul_sh + index * poly_words(ctx);
    } else {
        rc = ensure_form(ctx, p, t->ntt ? PF_NTT_ADD : PF_COEF_ADD);
        if (rc) return rc;
        pl = (t->ntt ? p->ntt_add : p->coef_add) + index * poly_words(ctx);
    }
    ProfScope ps(ctx, KC_PLAIN_OP, lp_bytes(ctx, (double)t->count * (op == 0 ? t->size : 1) * 2 * ctx->K), (double)t->count * (op == 0 ? t->size : 1) * ctx->K * ctx->n);
    CU(launch_plain_op(ctx->dP, ctx->n, ctx->K, t->d, t->count, t->size, pl, pl_sh, op, ctx->stream));
    return CRCNN_OK;
}

int crcnn_add_many(crcnn_ctx *ctx, crcnn_tensor *t, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(t && out, "null argument");
    REQUIRE(t->count >= 1, "encrypteds cannot be empty");  // evaluator.cpp:298-301
    REQUIRE(t->size == 2, "add_many is implemented for size-2 ciphertexts");
    CU(cudaSetDevice(ctx->device));
    // sum of ciphertexts [first, first + count) of `src` in groups of `g` -> `nout` ciphertexts at dst (identity index table, cached)
    auto pass = [&](const uint64_t *src, long first, int nout, int g, uint64_t *dst) -> int {
        std::vector<int> key = {4, (int)first, nout, g};
        const int *d_index = nullptr;
        auto it = ctx->index_cache.find(key);
        if (it == ctx->index_cache.end()) {
            std::vector<int> table((size_t)nout * g);
            for (size_t i = 0; i < table.size(); i++) table[i] = (int)(first + (long)i);
            int rc = get_index_table(ctx, key, table, &d_index);
            if (rc) return rc;
        } else d_index = it->second;
        ProfScope ps(ctx, KC_POOL, lp_bytes(ctx, ((double)nout * g + nout) * 2 * ctx->K), (double)nout * g * 2 * ctx->K * ctx->n);
        CU(launch_pool(ctx->dP, ctx->n, ctx->K, src, d_index, nout, g, nullptr, nullptr, sum_fits_64(ctx, g), dst, ctx->stream));
        return CRCNN_OK;
    };
    crcnn_tensor *o = nullptr;
    int rc = new_tensor(ctx, 1, 2, t->ntt, &o);
    if (rc) return rc;
    if (t->count <= 128) {
        rc = pass(t->d, 0, 1, (int)t->count, o->d);
    } else {
        // ONE output ciphertext keeps 2K CTAs busy: reduce in two levels -- groups of ~sqrt(count) summed in parallel (every input read
        // once, in full coalesced rows), then the canonical partial sums.  Modular addition is associative: same residues as the
        // reference's serial add_many (evaluator.cpp:296-308).
        int g = 1;
        while ((long)g * g < t->count) g++;
        const long full = t->count / g, tail = t->count % g, groups = full + (tail ? 1 : 0);
        crcnn_tensor *part = nullptr;
        rc = new_tensor(ctx, groups, 2, t->ntt, &part);
        if (!rc) rc = pass(t->d, 0, (int)full, g, part->d);
        if (!rc && tail) rc = pass(t->d, full * g, 1, (int)tail, part->d + full * 2 * poly_words(ctx));
        if (!rc) rc = pass(part->d, 0, 1, (int)groups, o->d);
        crcnn_tensor_free(ctx, part);
    }
    if (rc) { crcnn_tensor_free(ctx, o); return rc; }
    *out = o;
    return CRCNN_OK;
}

// ---------------------------------------------------------------------------- measurement
int crcnn_prof_enable(crcnn_ctx *ctx, int on) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    ctx->prof_on = on != 0;
    return CRCNN_OK;
}
int crcnn_prof_reset(crcnn_ctx *ctx) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    prof_collect(ctx);
    for (int i = 0; i < KC_COUNT; i++) { ctx->launches[i] = 0; ctx->ms[i] = 0; ctx->work_bytes[i] = 0; ctx->work_ops[i] = 0; }
    return CRCNN_OK;
}
int crcnn_prof_count(crcnn_ctx *ctx) { return ctx ? (int)KC_COUNT : (int)CRCNN_ERR_INVALID_ARGUMENT; }
int crcnn_prof_get(crcnn_ctx *ctx, int cls, char *name, long *launches, double *ms) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(cls >= 0 && cls < KC_COUNT, "bad kernel class");
    prof_collect(ctx);
    if (name) { strncpy(name, kClassNames[cls], 31); name[31] = 0; }
    if (launches) *launches = ctx->launches[cls];
    if (ms) *ms = ctx->ms[cls];
    return CRCNN_OK;
}

int crcnn_prof_get_work(crcnn_ctx *ctx, int cls, double *bytes, double *ops) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(cls >= 0 && cls < KC_COUNT, "bad kernel class");
    if (bytes) *bytes = ctx->work_bytes[cls];
    if (ops) *ops = ctx->work_ops[cls];
    return CRCNN_OK;
}

int crcnn_probe_pipe(crcnn_ctx *ctx, int which, int blocks, int threads, int iters, double *ms, double *ops) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(which >= 0 && which <= 4 && blocks > 0 && threads > 0 && threads <= 1024 && iters > 0 && ms, "bad probe arguments");
    CU(cudaSetDevice(ctx->device));
    uint64_t *sink = nullptr;
    int rc = dev_alloc(ctx, 8, (void **)&sink);
    if (rc) return rc;
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    ctx->launches[KC_PROBE]++;
    double work = 0;
    CU(cudaEventRecord(a, ctx->stream));
    if (which == 0) { CU(launch_imad_probe(blocks, threads, iters, sink, ctx->stream)); work = (double)blocks * threads * iters * 8.0; }
    else if (which == 1) { CU(launch_imad_wide_probe(blocks, threads, iters, sink, ctx->stream)); work = (double)blocks * threads * iters * 16.0; }
    else CU(launch_umma_i8_probe(blocks, iters, which - 2, &work, ctx->stream));
    CU(cudaEventRecord(b, ctx->stream));
    CU(cudaEventSynchronize(b));
    float t = 0;
    cudaEventElapsedTime(&t, a, b);
    *ms = t;
    if (ops) *ops = work;
    cudaEventDestroy(a); cudaEventDestroy(b);
    dev_free(ctx, sink);
    return CRCNN_OK;
}
int crcnn_probe_imad(crcnn_ctx *ctx, int blocks, int threads, int iters, double *ms) {
    return crcnn_probe_pipe(ctx, 0, blocks, threads, iters, ms, nullptr);
}

// ---------------------------------------------------------------------------------------- host support
// What a C++17 serving loop needs besides the layer calls, without linking the CUDA runtime itself: page-locked staging
// memory, a copy stream, events to time on the device and to order the two streams.
int crcnn_pinned_alloc(size_t bytes, void **out) {
    if (!out) return CRCNN_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, bytes, cudaHostAllocDefault);
    if (e != cudaSuccess) { g_create_error = std::string("cudaHostAlloc: ") + cudaGetErrorString(e); return e == cudaErrorMemoryAllocation ? CRCNN_ERR_OUT_OF_MEMORY : CRCNN_ERR_CUDA; }
    return CRCNN_OK;
}
int crcnn_pinned_free(void *p) { return (!p || cudaFreeHost(p) == cudaSuccess) ? CRCNN_OK : CRCNN_ERR_CUDA; }

int crcnn_stream_create(crcnn_ctx *ctx, void **stream) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(stream, "null argument");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t s;
    CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    *stream = s;
    return CRCNN_OK;
}
int crcnn_stream_destroy(crcnn_ctx *ctx, void *stream) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    if (stream) CU(cudaStreamDestroy((cudaStream_t)stream));
    return CRCNN_OK;
}
int crcnn_event_create(crcnn_ctx *ctx, void **event) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(event, "null argument");
    CU(cudaSetDevice(ctx->device));
    cudaEvent_t e;
    CU(cudaEventCreate(&e));
    *event = e;
    return CRCNN_OK;
}
int crcnn_event_record(crcnn_ctx *ctx, void *event, void *stream) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(event, "null argument");
    CU(cudaEventRecord((cudaEvent_t)event, stream ? (cudaStream_t)stream : ctx->stream));
    return CRCNN_OK;
}
int crcnn_stream_wait_event(crcnn_ctx *ctx, void *stream, void *event) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(event, "null argument");
    CU(cudaStreamWaitEvent(stream ? (cudaStream_t)stream : ctx->stream, (cudaEvent_t)event, 0));
    return CRCNN_OK;
}
int crcnn_event_elapsed_ms(crcnn_ctx *ctx, void *first, void *second, double *ms) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(first && second && ms, "null argument");
    CU(cudaEventSynchronize((cudaEvent_t)second));
    float t = 0;
    CU(cudaEventElapsedTime(&t, (cudaEvent_t)first, (cudaEvent_t)second));
    *ms = t;
    return CRCNN_OK;
}
int crcnn_event_destroy(crcnn_ctx *ctx, void *event) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    if (event) CU(cudaEventDestroy((cudaEvent_t)event));
    return CRCNN_OK;
}
/* Non-blocking download: enqueues the device->host copy of t (coefficient form) on the context's stream; host_words must be pinned
 * and is complete once an event recorded afterwards has fired (or after crcnn_ctx_sync).  The pad words are written too. */
int crcnn_tensor_download_async(crcnn_ctx *ctx, crcnn_tensor *t, uint64_t *host) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(t && host, "null argument");
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_domain(ctx, t, 0);
    if (rc) return rc;
    const size_t n = ctx->n, rows = (size_t)t->count * t->size * ctx->K;
    if (!rows) return CRCNN_OK;
    // re-pad on the device (pad word = 0), then ONE contiguous copy: a strided cudaMemcpy2D reaches a tenth of the link rate
    uint64_t *padded = nullptr;
    rc = dev_alloc(ctx, rows * (n + 1) * 8, (void **)&padded);
    if (rc) return rc;
    CU(cudaMemsetAsync(padded, 0, rows * (n + 1) * 8, ctx->stream));
    CU(cudaMemcpy2DAsync(padded, (n + 1) * 8, t->d, n * 8, n * 8, rows, cudaMemcpyDeviceToDevice, ctx->stream));
    CU(cudaMemcpyAsync(host, padded, rows * (n + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    dev_free(ctx, padded);
    return CRCNN_OK;
}

// ---------------------------------------------------------------------------------------- NCCL all-gather of ciphertexts
// Output-neuron sharding (SURVEY 8(e) item 3; the reference's thread split, CrCNN/src/convolutionalLayer.cpp:177-187,
// fullyConnectedLayer.cpp:148-158, taken across GPUs): every rank computes a contiguous range of a layer's output channels /
// rows; before a layer that consumes all channels the ranks exchange their ciphertexts over NVLink.  The exchange is one NCCL
// group of point-to-point sends and receives (an all-gather with per-rank counts) enqueued on the context's stream: no host
// synchronisation, no staging copy -- each rank's block lands at its final offset of the gathered tensor.  NCCL is loaded at run
// time (dlopen of libnccl.so.2: the copy torch has already mapped when there is one, else the system's), so the library has no
// link-time dependency and single-GPU users never touch it.
namespace {
struct NcclId128 { char b[128]; };   // ncclUniqueId is passed BY VALUE (nccl.h: struct { char internal[128]; })
struct NcclApi {
    void *lib = nullptr;
    int (*GetUniqueId)(void *) = nullptr;
    int (*CommInitRank)(void **, int, NcclId128, int) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*Send)(const void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    std::string why;
};
NcclApi &nccl() {
    static NcclApi api = [] {
        NcclApi a;
        const char *names[] = {getenv("CRCNN_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char *nm : names) {
            if (!nm || !*nm) continue;
            a.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (a.lib) break;
        }
        if (!a.lib) { a.why = std::string("libnccl.so.2 not found (set CRCNN_NCCL_LIB): ") + (dlerror() ? dlerror() : ""); return a; }
        auto sym = [&](const char *n) { void *p = dlsym(a.lib, n); if (!p) a.why = std::string("missing NCCL symbol ") + n; return p; };
        a.GetUniqueId = (decltype(a.GetUniqueId))sym("ncclGetUniqueId");
        a.CommInitRank = (decltype(a.CommInitRank))sym("ncclCommInitRank");
        a.CommDestroy = (decltype(a.CommDestroy))sym("ncclCommDestroy");
        a.GroupStart = (decltype(a.GroupStart))sym("ncclGroupStart");
        a.GroupEnd = (decltype(a.GroupEnd))sym("ncclGroupEnd");
        a.Send = (decltype(a.Send))sym("ncclSend");
        a.Recv = (decltype(a.Recv))sym("ncclRecv");
        a.GetErrorString = (decltype(a.GetErrorString))sym("ncclGetErrorString");
        return a;
    }();
    return api;
}
constexpr int kNcclUint64 = 5;   // ncclUint64 (nccl.h: ncclDataType_t)
}  // namespace

struct crcnn_comm {
    void *comm = nullptr;
    int world = 1, rank = 0;
};

#define NCCLCHECK(call)                                                                                              \
    do {                                                                                                             \
        int r__ = (call);                                                                                            \
        if (r__ != 0) return fail(ctx, CRCNN_ERR_CUDA, std::string(#call) + ": " + (nccl().GetErrorString ? nccl().GetErrorString(r__) : "NCCL error")); \
    } while (0)

int crcnn_comm_unique_id(void *id128) {
    crcnn_ctx *ctx = nullptr;
    if (!id128) return CRCNN_ERR_INVALID_ARGUMENT;
    if (!nccl().why.empty()) return fail(nullptr, CRCNN_ERR_UNSUPPORTED, nccl().why);
    NCCLCHECK(nccl().GetUniqueId(id128));
    return CRCNN_OK;
}
int crcnn_comm_create(crcnn_ctx *ctx, const void *id128, int world, int rank, crcnn_comm **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(id128 && out && world >= 1 && rank >= 0 && rank < world, "bad communicator arguments");
    if (!nccl().why.empty()) return fail(ctx, CRCNN_ERR_UNSUPPORTED, nccl().why);
    CU(cudaSetDevice(ctx->device));
    NcclId128 id;
    std::memcpy(id.b, id128, 128);
    auto *c = new crcnn_comm;
    c->world = world; c->rank = rank;
    int r = nccl().CommInitRank(&c->comm, world, id, rank);
    if (r != 0) { delete c; return fail(ctx, CRCNN_ERR_CUDA, std::string("ncclCommInitRank: ") + nccl().GetErrorString(r)); }
    *out = c;
    return CRCNN_OK;
}
int crcnn_comm_destroy(crcnn_ctx *ctx, crcnn_comm *c) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    if (!c) return CRCNN_OK;
    CU(cudaStreamSynchronize(ctx->stream));
    if (c->comm) nccl().CommDestroy(c->comm);
    delete c;
    return CRCNN_OK;
}
int crcnn_comm_all_gather(crcnn_ctx *ctx, crcnn_comm *c, crcnn_tensor *local, int batch, const long *counts, int want_ntt_form,
                          crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(c && local && counts && out && batch > 0, "null argument");
    long total = 0, before = 0;
    for (int r = 0; r < c->world; r++) { REQUIRE(counts[r] >= 0, "negative shard size"); if (r < c->rank) before += counts[r]; total += counts[r]; }
    REQUIRE(local->count == (long)batch * counts[c->rank], "local tensor does not hold batch x counts[rank] ciphertexts");
    CU(cudaSetDevice(ctx->device));
    // the gathered tensor carries ONE domain flag: with want_ntt_form >= 0 every rank first brings its block into that domain; with -1 the
    // blocks are exchanged as they are (all ranks of a sharded layer produce the same domain: the kernel is chosen from the layer's
    // total output count, run_weighted_sum, and pooling / batch-norm / square map a domain to a domain)
    int rc = want_ntt_form >= 0 ? ensure_domain(ctx, local, want_ntt_form ? 1 : 0) : CRCNN_OK;
    if (rc) return rc;
    crcnn_tensor *full = nullptr;
    rc = new_tensor(ctx, (long)batch * total, local->size, local->ntt, &full);
    if (rc) return rc;
    const size_t ctw = (size_t)local->size * poly_words(ctx);
    // image b of the gathered tensor = [rank 0's ciphertexts of b | rank 1's | ...]
    if (c->world > 1) NCCLCHECK(nccl().GroupStart());
    for (int b = 0; b < batch; b++) {
        const uint64_t *mine = local->d + (size_t)b * counts[c->rank] * ctw;
        long off = 0;
        for (int r = 0; r < c->world; r++) {
            uint64_t *dst = full->d + ((size_t)b * total + off) * ctw;
            if (r == c->rank) {
                if (counts[r]) CU(cudaMemcpyAsync(dst, mine, (size_t)counts[r] * ctw * 8, cudaMemcpyDeviceToDevice, ctx->stream));
            } else {
                if (counts[c->rank]) NCCLCHECK(nccl().Send(mine, (size_t)counts[c->rank] * ctw, kNcclUint64, r, c->comm, ctx->stream));
                if (counts[r]) NCCLCHECK(nccl().Recv(dst, (size_t)counts[r] * ctw, kNcclUint64, r, c->comm, ctx->stream));
            }
            off += counts[r];
        }
    }
    if (c->world > 1) NCCLCHECK(nccl().GroupEnd());
    (void)before;
    *out = full;
    return CRCNN_OK;
}

// ---------------------------------------------------------------------------------------- re-encryption (SURVEY 8(f) N4)
int crcnn_keys_upload(crcnn_ctx *ctx, const uint64_t *secret_key_ntt, const uint64_t *public_key_ntt, crcnn_keys **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(secret_key_ntt && public_key_ntt && out, "null argument");
    REQUIRE(ctx->hp.d.t >= 2 && REENC_GAMMA % ctx->hp.d.t != 0, "plain modulus not usable with the decryptor's gamma");
    CU(cudaSetDevice(ctx->device));
    auto *k = new crcnn_keys;
    k->c = make_reenc_consts(ctx->hp.d);
    k->b = make_budget_consts(ctx->hp.d);
    const size_t pw = poly_words(ctx);
    int rc = dev_alloc(ctx, pw * 8, (void **)&k->sk);
    if (!rc) rc = dev_alloc(ctx, 2 * pw * 8, (void **)&k->pk);
    if (!rc) rc = upload_rows(ctx, secret_key_ntt, (size_t)ctx->K, k->sk, ctx->stream);
    if (!rc) rc = upload_rows(ctx, public_key_ntt, (size_t)2 * ctx->K, k->pk, ctx->stream);
    if (!rc) { cudaError_t e = cudaStreamSynchronize(ctx->stream); if (e != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e)); }
    if (rc) { dev_free(ctx, k->sk); dev_free(ctx, k->pk); delete k; return rc; }
    *out = k;
    return CRCNN_OK;
}
int crcnn_keys_free(crcnn_ctx *ctx, crcnn_keys *k) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    if (!k) return CRCNN_OK;
    const size_t pw = poly_words(ctx);
    if (k->sk) cudaMemsetAsync(k->sk, 0, pw * 8, ctx->stream);      // do not leave key material in freed device memory
    dev_free(ctx, k->sk); dev_free(ctx, k->pk);
    delete k;
    return CRCNN_OK;
}

namespace {
// c0 + c1 s of ciphertexts [first, first+count) of t into scratch (count*K*n words), coefficient form -- except that for a
// coefficient-form t the "+ c0" is left to the consumer, which gets *c0 = the ciphertexts (null when c0 is already in scratch)
int dec_dot_range(crcnn_ctx *ctx, crcnn_keys *k, crcnn_tensor *t, long first, long count, uint64_t *scratch, const uint64_t **c0) {
    const size_t pw = poly_words(ctx);
    const uint64_t *ct = t->d + first * 2 * pw;
    if (!t->ntt) {
        // copy the c1 polynomials and transform them (decryptor.cpp:153-158)
        CU(cudaMemcpy2DAsync(scratch, pw * 8, ct + pw, 2 * pw * 8, pw * 8, count, cudaMemcpyDeviceToDevice, ctx->stream));
        CU(launch_ntt(ctx->dP, ctx->logn, scratch, count * ctx->K, 0, ctx->K, false, ctx->stream));
    }
    CU(launch_dec_dot(k->c, ct, t->ntt, k->sk, scratch, count, ctx->stream));
    CU(launch_ntt(ctx->dP, ctx->logn, scratch, count * ctx->K, 0, ctx->K, true, ctx->stream));
    *c0 = t->ntt ? nullptr : ct;
    return CRCNN_OK;
}

// plaintext polynomials [count][n] of ciphertexts [first, first+count) of t (Decryptor::decrypt); scratch = count*K*n words
int decrypt_range(crcnn_ctx *ctx, crcnn_keys *k, crcnn_tensor *t, long first, long count, uint64_t *scratch, uint64_t *plain) {
    ProfScope ps(ctx, KC_REENC, lp_bytes(ctx, (double)count * 2 * ctx->K) + (double)count * ctx->n * 8, lp_bfly(ctx, (double)count * 2 * ctx->K));
    const uint64_t *c0 = nullptr;
    int rc = dec_dot_range(ctx, k, t, first, count, scratch, &c0);
    if (rc) return rc;
    CU(launch_dec_scale(k->c, c0, scratch, plain, count, ctx->stream));
    return CRCNN_OK;
}

// noise bit lengths of ciphertexts [first, first+count) of t, atomically maximised into bits[count] (Decryptor::invariant_noise_budget)
int noise_bits_range(crcnn_ctx *ctx, crcnn_keys *k, crcnn_tensor *t, long first, long count, uint64_t *scratch, int *bits) {
    ProfScope ps(ctx, KC_REENC, lp_bytes(ctx, (double)count * 2 * ctx->K) + (double)count * 4, lp_bfly(ctx, (double)count * 2 * ctx->K));
    const uint64_t *c0 = nullptr;
    int rc = dec_dot_range(ctx, k, t, first, count, scratch, &c0);
    if (rc) return rc;
    CU(launch_noise_bits(k->b, c0, scratch, bits, count, ctx->stream));
    return CRCNN_OK;
}

// ciphertexts per chunk of the decrypting calls: a dot-product scratch (K*n words) and a plaintext (n words) each, 1 GiB in all
long decrypt_step(const crcnn_ctx *ctx, long count) {
    return std::max<long>(1, std::min<long>(count, (long)((1ull << 30) / ((size_t)(ctx->K + 1) * ctx->n * 8))));
}

// ciphertexts per chunk of the encrypting calls, 1 GiB in all: K*n words (dot product / u), n words (plaintext), 96 slots,
// 2n + 3n noise bytes, a float
long encrypt_step(const crcnn_ctx *ctx, long count) {
    const size_t n = ctx->n, per_ct = (size_t)(ctx->K + 1) * n * 8 + REENC_SLOTS * 8 + 5 * n + 8;
    return std::max<long>(1, std::min<long>(count, (long)((1ull << 30) / per_ct)));
}

// Encryptor::encrypt (SEAL/seal/encryptor.cpp:95-200) of the plaintexts slots[count][96] into dst[count][2][K][n], coefficient form.
// u, e0, e1 of ciphertext r come from (seed, first + r, coefficient) or, with host_noise (this range's int8 rows [count][3][n]),
// are copied through `given`.  U: count*K*n words, e: count*2*n bytes of scratch.
cudaError_t encrypt_range(crcnn_ctx *ctx, crcnn_keys *k, const uint64_t *slots, uint64_t seed, long first, double noise_standard_deviation,
                          const int8_t *host_noise, int8_t *given, uint64_t *U, int8_t *e, uint64_t *dst, long count) {
    const int K = ctx->K;
    const double sigma = noise_standard_deviation > 0 ? noise_standard_deviation : 3.19;   // SEAL/seal/util/globals.cpp: default_noise_standard_deviation
    const double max_dev = 6.0 * sigma;                                                   // noise_distribution_width_multiplier = 6 (encryptionparams.h:204-211)
    cudaError_t er = cudaSuccess;
    if (host_noise) er = cudaMemcpyAsync(given, host_noise, (size_t)count * 3 * ctx->n, cudaMemcpyHostToDevice, ctx->stream);
    if (er == cudaSuccess) er = launch_enc_sample(k->c, seed, first, sigma, max_dev, host_noise ? given : nullptr, U, e, count, ctx->stream);
    if (er == cudaSuccess) er = launch_ntt(ctx->dP, ctx->logn, U, count * K, 0, K, false, ctx->stream);
    if (er == cudaSuccess) er = launch_enc_mul(k->c, U, k->pk, dst, count, ctx->stream);
    if (er == cudaSuccess) er = launch_ntt(ctx->dP, ctx->logn, dst, count * 2 * K, 0, K, true, ctx->stream);
    if (er == cudaSuccess) er = launch_enc_finish(k->c, slots, e, dst, count, ctx->stream);
    return er;
}
}  // namespace

int crcnn_decrypt(crcnn_ctx *ctx, crcnn_keys *k, crcnn_tensor *t, uint64_t *host_plain) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(k && t && host_plain, "null argument");
    REQUIRE(t->size == 2, "decrypt is implemented for size-2 ciphertexts");
    CU(cudaSetDevice(ctx->device));
    const size_t n = ctx->n;
    const long step = decrypt_step(ctx, t->count);
    uint64_t *scratch = nullptr, *plain = nullptr;
    int rc = dev_alloc(ctx, (size_t)step * ctx->K * n * 8, (void **)&scratch);
    if (!rc) rc = dev_alloc(ctx, (size_t)step * n * 8, (void **)&plain);
    for (long c0 = 0; c0 < t->count && !rc; c0 += step) {
        const long cnt = std::min<long>(step, t->count - c0);
        rc = decrypt_range(ctx, k, t, c0, cnt, scratch, plain);
        if (!rc) {
            cudaError_t e = cudaMemcpy2DAsync(host_plain + c0 * (n + 1), (n + 1) * 8, plain, n * 8, n * 8, cnt, cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e));
            for (long r = 0; r < cnt; r++) host_plain[(c0 + r) * (n + 1) + n] = 0;
        }
    }
    dev_free(ctx, scratch); dev_free(ctx, plain);
    return rc;
}

int crcnn_noise_budget(crcnn_ctx *ctx, crcnn_keys *k, crcnn_tensor *t, int *host_budgets, int *min_budget) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(k && t, "null argument");
    REQUIRE(t->size == 2, "the noise budget is implemented for size-2 ciphertexts");
    REQUIRE(t->count > 0, "empty tensor");
    CU(cudaSetDevice(ctx->device));
    const size_t n = ctx->n;
    const long step = decrypt_step(ctx, t->count);
    uint64_t *scratch = nullptr;
    int *bits = nullptr;
    int rc = dev_alloc(ctx, (size_t)step * ctx->K * n * 8, (void **)&scratch);
    if (!rc) rc = dev_alloc(ctx, (size_t)t->count * sizeof(int), (void **)&bits);
    if (!rc) { cudaError_t e = cudaMemsetAsync(bits, 0, (size_t)t->count * sizeof(int), ctx->stream); if (e != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e)); }
    for (long c0 = 0; c0 < t->count && !rc; c0 += step)
        rc = noise_bits_range(ctx, k, t, c0, std::min<long>(step, t->count - c0), scratch, bits + c0);
    std::vector<int> hb;
    if (!rc) {
        hb.resize((size_t)t->count);
        cudaError_t e = cudaMemcpyAsync(hb.data(), bits, hb.size() * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(e));
    }
    dev_free(ctx, scratch); dev_free(ctx, bits);
    if (rc) return rc;
    int mn = k->b.q_bits;
    for (long i = 0; i < t->count; i++) {
        const int b = std::max(0, k->b.q_bits - hb[(size_t)i] - 1);     // the -1 accounts for scaling the invariant noise by 2
        if (host_budgets) host_budgets[i] = b;
        mn = std::min(mn, b);
    }
    if (min_budget) *min_budget = mn;
    return CRCNN_OK;
}

int crcnn_reencrypt(crcnn_ctx *ctx, crcnn_keys *k, crcnn_tensor *in, uint64_t seed, double noise_standard_deviation,
                    const int8_t *host_noise, crcnn_tensor **out, uint64_t *host_reencoded, float *host_values) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(k && in && out, "null argument");
    REQUIRE(in->size == 2, "re-encryption is implemented for size-2 ciphertexts");
    CU(cudaSetDevice(ctx->device));
    const size_t n = ctx->n, pw = poly_words(ctx);
    const int K = ctx->K;
    crcnn_tensor *o = nullptr;
    int rc = new_tensor(ctx, in->count, 2, 0, &o);
    if (rc) return rc;
    const long step = encrypt_step(ctx, in->count);
    uint64_t *scratch = nullptr, *plain = nullptr, *slots = nullptr;
    int8_t *e = nullptr, *given = nullptr;
    float *vals = nullptr;
    rc = dev_alloc(ctx, (size_t)step * K * n * 8, (void **)&scratch);
    if (!rc) rc = dev_alloc(ctx, (size_t)step * n * 8, (void **)&plain);
    if (!rc) rc = dev_alloc(ctx, (size_t)step * REENC_SLOTS * 8, (void **)&slots);
    if (!rc) rc = dev_alloc(ctx, (size_t)step * 2 * n, (void **)&e);
    if (!rc && host_noise) rc = dev_alloc(ctx, (size_t)step * 3 * n, (void **)&given);
    if (!rc && host_values) rc = dev_alloc(ctx, (size_t)step * 4, (void **)&vals);
    for (long c0 = 0; c0 < in->count && !rc; c0 += step) {
        const long cnt = std::min<long>(step, in->count - c0);
        rc = decrypt_range(ctx, k, in, c0, cnt, scratch, plain);
        if (rc) break;
        uint64_t *dst = o->d + c0 * 2 * pw;
        cudaError_t er = cudaSuccess;
        {
            ProfScope ps(ctx, KC_REENC, lp_bytes(ctx, (double)cnt * 2 * K), lp_bfly(ctx, (double)cnt * 3 * K));
            er = launch_reencode(k->c, plain, slots, vals, cnt, ctx->stream);
            if (er == cudaSuccess)
                er = encrypt_range(ctx, k, slots, seed, c0, noise_standard_deviation, host_noise ? host_noise + c0 * 3 * n : nullptr, given, scratch, e,
                                   dst, cnt);
        }
        if (er == cudaSuccess && host_reencoded) {     // the re-encoded plaintexts, n+1 words each (parity checks)
            std::vector<uint64_t> hs((size_t)cnt * REENC_SLOTS);
            er = cudaMemcpyAsync(hs.data(), slots, hs.size() * 8, cudaMemcpyDeviceToHost, ctx->stream);
            if (er == cudaSuccess) er = cudaStreamSynchronize(ctx->stream);
            for (long r = 0; r < cnt && er == cudaSuccess; r++) {
                uint64_t *p = host_reencoded + (c0 + r) * (n + 1);
                memset(p, 0, (n + 1) * 8);
                memcpy(p, hs.data() + r * REENC_SLOTS, 64 * 8);
                memcpy(p + n - 32, hs.data() + r * REENC_SLOTS + 64, 32 * 8);
            }
        }
        if (er == cudaSuccess && host_values) {
            er = cudaMemcpyAsync(host_values + c0, vals, (size_t)cnt * 4, cudaMemcpyDeviceToHost, ctx->stream);
            if (er == cudaSuccess) er = cudaStreamSynchronize(ctx->stream);
        }
        if (er != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, std::string("re-encryption: ") + cudaGetErrorString(er));
    }
    if (host_noise && !rc) { cudaError_t er = cudaStreamSynchronize(ctx->stream); if (er != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(er)); }
    dev_free(ctx, scratch); dev_free(ctx, plain); dev_free(ctx, slots); dev_free(ctx, e); dev_free(ctx, given); dev_free(ctx, vals);
    if (rc) { crcnn_tensor_free(ctx, o); return rc; }
    *out = o;
    return CRCNN_OK;
}

int crcnn_encrypt_values(crcnn_ctx *ctx, crcnn_keys *k, const float *host_values, long count, uint64_t seed, double noise_standard_deviation,
                         const int8_t *host_noise, crcnn_tensor **out) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(k && host_values && out, "null argument");
    REQUIRE(count > 0, "no values to encrypt");
    CU(cudaSetDevice(ctx->device));
    const size_t n = ctx->n, pw = poly_words(ctx);
    const int K = ctx->K;
    crcnn_tensor *o = nullptr;
    int rc = new_tensor(ctx, count, 2, 0, &o);
    if (rc) return rc;
    const long step = encrypt_step(ctx, count);
    uint64_t *U = nullptr, *slots = nullptr;
    int8_t *e = nullptr, *given = nullptr;
    float *vals = nullptr;
    rc = dev_alloc(ctx, (size_t)step * K * n * 8, (void **)&U);
    if (!rc) rc = dev_alloc(ctx, (size_t)step * REENC_SLOTS * 8, (void **)&slots);
    if (!rc) rc = dev_alloc(ctx, (size_t)step * 2 * n, (void **)&e);
    if (!rc && host_noise) rc = dev_alloc(ctx, (size_t)step * 3 * n, (void **)&given);
    if (!rc) rc = dev_alloc(ctx, (size_t)count * 4, (void **)&vals);
    if (!rc) { cudaError_t er = cudaMemcpyAsync(vals, host_values, (size_t)count * 4, cudaMemcpyHostToDevice, ctx->stream); if (er != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(er)); }
    for (long c0 = 0; c0 < count && !rc; c0 += step) {
        const long cnt = std::min<long>(step, count - c0);
        cudaError_t er;
        {
            ProfScope ps(ctx, KC_REENC, lp_bytes(ctx, (double)cnt * 2 * K), lp_bfly(ctx, (double)cnt * 3 * K));
            er = launch_encode_values(k->c, vals + c0, slots, cnt, ctx->stream);
            if (er == cudaSuccess)
                er = encrypt_range(ctx, k, slots, seed, c0, noise_standard_deviation, host_noise ? host_noise + c0 * 3 * n : nullptr, given, U, e,
                                   o->d + c0 * 2 * pw, cnt);
        }
        if (er != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, std::string("encryption: ") + cudaGetErrorString(er));
    }
    // the host buffers must stay untouched until their copies have run
    if (!rc) { cudaError_t er = cudaStreamSynchronize(ctx->stream); if (er != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(er)); }
    dev_free(ctx, U); dev_free(ctx, slots); dev_free(ctx, e); dev_free(ctx, given); dev_free(ctx, vals);
    if (rc) { crcnn_tensor_free(ctx, o); return rc; }
    *out = o;
    return CRCNN_OK;
}

int crcnn_decrypt_values(crcnn_ctx *ctx, crcnn_keys *k, crcnn_tensor *t, float *host_values) {
    if (!ctx) return CRCNN_ERR_INVALID_ARGUMENT;
    REQUIRE(k && t && host_values, "null argument");
    REQUIRE(t->size == 2, "decrypt is implemented for size-2 ciphertexts");
    REQUIRE(t->count > 0, "empty tensor");
    CU(cudaSetDevice(ctx->device));
    const size_t n = ctx->n;
    const long step = decrypt_step(ctx, t->count);
    uint64_t *scratch = nullptr, *plain = nullptr;
    float *vals = nullptr;
    int rc = dev_alloc(ctx, (size_t)step * ctx->K * n * 8, (void **)&scratch);
    if (!rc) rc = dev_alloc(ctx, (size_t)step * n * 8, (void **)&plain);
    if (!rc) rc = dev_alloc(ctx, (size_t)t->count * 4, (void **)&vals);
    for (long c0 = 0; c0 < t->count && !rc; c0 += step) {
        const long cnt = std::min<long>(step, t->count - c0);
        rc = decrypt_range(ctx, k, t, c0, cnt, scratch, plain);
        if (!rc) {
            ProfScope ps(ctx, KC_REENC, (double)cnt * n * 8 + (double)cnt * 4, 0);
            cudaError_t er = launch_decode_values(k->c, plain, vals + c0, cnt, ctx->stream);
            if (er != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(er));
        }
    }
    if (!rc) {
        cudaError_t er = cudaMemcpyAsync(host_values, vals, (size_t)t->count * 4, cudaMemcpyDeviceToHost, ctx->stream);
        if (er == cudaSuccess) er = cudaStreamSynchronize(ctx->stream);
        if (er != cudaSuccess) rc = fail(ctx, CRCNN_ERR_CUDA, cudaGetErrorString(er));
    }
    dev_free(ctx, scratch); dev_free(ctx, plain); dev_free(ctx, vals);
    return rc;
}

}  // extern "C"
