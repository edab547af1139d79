// Device kernels of the encrypted-forward hot path (sm_100a).  See kernels.cuh for the contracts.
#include "kernels.cuh"
#include "devcfg.cuh"
#include "ntt.cuh"
#include <cstdlib>
#include <cstring>

namespace crcnn {

// =====================================================================================
// NTT / inverse NTT of dense limb-polynomials
// =====================================================================================
template <int LOGN>
__global__ void __launch_bounds__(NttPlan<LOGN>::THREADS, NttPlan<LOGN>::MIN_CTAS)
ntt_fwd_kernel(uint64_t *__restrict__ data, const DeviceParams *__restrict__ P, int slot_base, int slot_count, int group_polys,
               int group_off) {
    extern __shared__ uint64_t sm[];
    const long p = blockIdx.x;
    const NttTable tb = P->tab[slot_base + (int)(p % slot_count)];
    // polynomial p is the (p % slot_count)-th of a group of slot_count transformed polynomials inside a record of group_polys
    uint64_t *poly = data + ((p / slot_count) * group_polys + group_off + p % slot_count) * (1L << LOGN);
    ntt_forward_to_smem<LOGN>(sm, poly, tb);
    smem_store_poly_canonical<LOGN>(sm, poly, tb.mod);
}

template <int LOGN, bool NINV>
__global__ void __launch_bounds__(NttPlan<LOGN>::THREADS, NttPlan<LOGN>::MIN_CTAS)
ntt_inv_kernel(uint64_t *__restrict__ data, const DeviceParams *__restrict__ P, int slot_base, int slot_count, int group_polys,
               int group_off, const uint64_t *__restrict__ src, const uint64_t *__restrict__ addend, int add_group, int add_stride) {
    extern __shared__ uint64_t sm[];
    const long p = blockIdx.x;
    const NttTable tb = P->tab[slot_base + (int)(p % slot_count)];
    const long off = ((p / slot_count) * group_polys + group_off + p % slot_count) * (1L << LOGN);
    uint64_t *poly = data + off;
    smem_load_poly<LOGN>(sm, src ? src + off : poly);   // src: out-of-place transform (same indexing), data is only written
    __syncthreads();
    // addend (relinearize): polynomial p adds polynomial (p / add_group) * add_stride + p % add_group of `addend`
    ntt_inverse_from_smem<LOGN, NINV>(sm, poly, tb, addend ? addend + ((p / add_group) * add_stride + p % add_group) * (1L << LOGN) : nullptr);
}

// Reductions of the BEHZ kernels.  FOLD: the three-fold reduction through the 2^k - delta shape every SEAL modulus on this path has
// (coefficient primes, the 61-bit Bsk primes and m_sk; modarith.cuh: reduce128_fold, host-checked against unsigned __int128 in
// host_selftest.cpp); its constants are derived from q on the spot (5 instructions).  The launcher takes it only when
// fold128_make(q).ok holds for EVERY modulus of the context (caller-supplied primes of another shape get the generic 128-bit
// Barrett step); env CRCNN_BEHZ_FOLD=0 forces Barrett.  Measured on B200 (profiles/r02a_first.txt): behz_lift 9.0 -> 7.8 ms,
// behz_floor 21.2 -> 18.0 ms per step of the bench network; both give the canonical residue, i.e. the same bytes.
template <bool FOLD>
__device__ __forceinline__ uint64_t behz_reduce(U128 z, const Mod &m) {
    if constexpr (FOLD) {
        Fold128 f;
        const int k = 64 - __clzll((long long)m.q);
        f.q = m.q; f.delta = (uint32_t)((1ull << k) - m.q); f.sh = (uint32_t)(k - 32); f.mask = (1u << (k - 32)) - 1; f.ok = 1;
        return reduce128_fold(z, f);
    } else {
        return barrett128(z, m);
    }
}
template <bool FOLD>
__device__ __forceinline__ uint64_t behz_mulmod(uint64_t a, uint64_t b, const Mod &m) { return behz_reduce<FOLD>(mul128(a, b), m); }

// Tensor square fused into the inverse transform (evaluator.cpp:783-848): the CTA of output limb-polynomial (ct, k, j)
// forms c0*c0 (k = 0), 2*c0*c1 (k = 1) or c1*c1 (k = 2) mod the j-th prime of q U Bsk while loading, then inverse-transforms it.
// Saves the write and re-read of the 3(K+S) product polynomials of every ciphertext.
// FOLD: products reduced by behz_reduce<true> (three folds through 2^k - delta, 6 IMAD.WIDE) instead of barrett128 (~18 multiplier
// instructions); a square takes 3 32x32 partial products instead of 4.  NINV = false: the output is left multiplied by n (the
// floor kernel's constants carry n^-1, params.h: fl_c_n / fl_T_n).  Every variant stores the same canonical residues up to that factor.
template <int LOGN, bool FOLD, bool NINV>
__global__ void __launch_bounds__(NttPlan<LOGN>::THREADS, NttPlan<LOGN>::MIN_CTAS)
ntt_inv_tensor_kernel(const DeviceParams *__restrict__ P, const uint64_t *__restrict__ ext, const uint64_t *__restrict__ qntt, int KS,
                      uint64_t *__restrict__ prod) {
    extern __shared__ uint64_t sm[];
    constexpr int N = 1 << LOGN;
    const long b = blockIdx.x;  // (ct * 3 + k) * KS + j
    const int j = (int)(b % KS);
    const int k = (int)((b / KS) % 3);
    const long ct = b / (3L * KS);
    const NttTable tb = P->tab[j];
    const uint64_t *c0 = ext + ((ct * 2) * KS + j) * N, *c1 = c0 + (long)KS * N;
    if (qntt && j < P->K) {  // q limbs straight from the NTT-form input tensor [ct][2][K][n]
        c0 = qntt + ((ct * 2) * P->K + j) * N;
        c1 = c0 + (long)P->K * N;
    }
    if (k == 1) {
#pragma unroll 8
        for (int i = threadIdx.x; i < N; i += NttPlan<LOGN>::THREADS) {
            if (FOLD) {
                U128 z = mul128(__ldg(c0 + i), __ldg(c1 + i));   // < 2^122: doubling cannot wrap
                z.hi = (z.hi << 1) | (z.lo >> 63);
                z.lo <<= 1;
                sm[ntt_pad(i)] = behz_reduce<true>(z, tb.mod);
            } else {
                const uint64_t ab = mulmod(__ldg(c0 + i), __ldg(c1 + i), tb.mod);
                sm[ntt_pad(i)] = addmod(ab, ab, tb.mod.q);
            }
        }
    } else {
        const uint64_t *c = k == 0 ? c0 : c1;
#pragma unroll 8
        for (int i = threadIdx.x; i < N; i += NttPlan<LOGN>::THREADS) {
            const uint64_t a = __ldg(c + i);
            sm[ntt_pad(i)] = FOLD ? behz_reduce<true>(sqr128(a), tb.mod) : mulmod(a, a, tb.mod);
        }
    }
    __syncthreads();
    ntt_inverse_from_smem<LOGN, NINV>(sm, prod + b * N, tb);
}

template <int LOGN, bool FOLD, bool NINV>
static cudaError_t launch_ntt_inv_tensor_t(const DeviceParams *P, const uint64_t *ext, const uint64_t *qntt, long count, int KS, uint64_t *prod,
                                           cudaStream_t stream) {
    using Pl = NttPlan<LOGN>;
    const size_t smem = Pl::SMEM_WORDS * sizeof(uint64_t);
    auto kf = ntt_inv_tensor_kernel<LOGN, FOLD, NINV>;
    static DeviceOnce once;
    if (once.first()) {
        cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(kf, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    }
    kf<<<(unsigned)(count * 3 * KS), Pl::THREADS, smem, stream>>>(P, ext, qntt, KS, prod);
    return cudaGetLastError();
}

template <int LOGN>
static cudaError_t launch_ntt_inv_tensor_l(const DeviceParams *P, const uint64_t *ext, const uint64_t *qntt, long count, int KS, uint64_t *prod,
                                           bool fold, bool ninv, cudaStream_t stream) {
    if (!ninv) return fold ? launch_ntt_inv_tensor_t<LOGN, true, false>(P, ext, qntt, count, KS, prod, stream)
                           : launch_ntt_inv_tensor_t<LOGN, false, false>(P, ext, qntt, count, KS, prod, stream);
    if (fold) return cudaErrorInvalidValue;   // not instantiated: the folded products come only with the n^-1-free output
    return launch_ntt_inv_tensor_t<LOGN, false, true>(P, ext, qntt, count, KS, prod, stream);
}

cudaError_t launch_ntt_inv_tensor(const DeviceParams *P, int logn, const uint64_t *ext, const uint64_t *qntt, long count, int KS, uint64_t *prod,
                                  bool fold, bool ninv, cudaStream_t stream) {
    if (count <= 0) return cudaSuccess;
    switch (logn) {
        case 10: return launch_ntt_inv_tensor_l<10>(P, ext, qntt, count, KS, prod, fold, ninv, stream);
        case 11: return launch_ntt_inv_tensor_l<11>(P, ext, qntt, count, KS, prod, fold, ninv, stream);
        case 12: return launch_ntt_inv_tensor_l<12>(P, ext, qntt, count, KS, prod, fold, ninv, stream);
        case 13: return launch_ntt_inv_tensor_l<13>(P, ext, qntt, count, KS, prod, fold, ninv, stream);
        case 14: return launch_ntt_inv_tensor_l<14>(P, ext, qntt, count, KS, prod, fold, ninv, stream);
        default: return cudaErrorInvalidValue;
    }
}

template <int LOGN>
static cudaError_t launch_ntt_t(const DeviceParams *P, uint64_t *data, long npolys, int slot_base, int slot_count,
                                bool inverse, int group_polys, int group_off, const uint64_t *src, const uint64_t *addend,
                                int add_group, int add_stride, bool ninv, cudaStream_t stream) {
    using Pl = NttPlan<LOGN>;
    size_t smem = Pl::SMEM_WORDS * sizeof(uint64_t);
    auto kf = ntt_fwd_kernel<LOGN>;
    auto ki = ntt_inv_kernel<LOGN, true>;
    auto kn = ntt_inv_kernel<LOGN, false>;
    static DeviceOnce once;
    if (once.first()) {
        cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(ki, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(kn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        // without this the driver sizes the carve-out for ONE resident CTA (seen in ncu: occupancy limit 1)
        cudaFuncSetAttribute(kf, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaFuncSetAttribute(ki, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaFuncSetAttribute(kn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    }
    if (npolys <= 0) return cudaSuccess;
    if ((src || addend || !ninv) && !inverse) return cudaErrorInvalidValue;
    if (inverse) (ninv ? ki : kn)<<<(unsigned)npolys, Pl::THREADS, smem, stream>>>(data, P, slot_base, slot_count, group_polys, group_off, src, addend, add_group, add_stride);
    else kf<<<(unsigned)npolys, Pl::THREADS, smem, stream>>>(data, P, slot_base, slot_count, group_polys, group_off);
    return cudaGetLastError();
}

cudaError_t launch_ntt_grouped(const DeviceParams *P, int logn, uint64_t *data, long npolys, int slot_base, int slot_count,
                               bool inverse, int group_polys, int group_off, cudaStream_t stream, const uint64_t *src,
                               const uint64_t *addend, int add_group, int add_stride, bool ninv) {
    switch (logn) {
        case 10: return launch_ntt_t<10>(P, data, npolys, slot_base, slot_count, inverse, group_polys, group_off, src, addend, add_group, add_stride, ninv, stream);
        case 11: return launch_ntt_t<11>(P, data, npolys, slot_base, slot_count, inverse, group_polys, group_off, src, addend, add_group, add_stride, ninv, stream);
        case 12: return launch_ntt_t<12>(P, data, npolys, slot_base, slot_count, inverse, group_polys, group_off, src, addend, add_group, add_stride, ninv, stream);
        case 13: return launch_ntt_t<13>(P, data, npolys, slot_base, slot_count, inverse, group_polys, group_off, src, addend, add_group, add_stride, ninv, stream);
        case 14: return launch_ntt_t<14>(P, data, npolys, slot_base, slot_count, inverse, group_polys, group_off, src, addend, add_group, add_stride, ninv, stream);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_ntt(const DeviceParams *P, int logn, uint64_t *data, long npolys, int slot_base, int slot_count,
                       bool inverse, cudaStream_t stream) {
    return launch_ntt_grouped(P, logn, data, npolys, slot_base, slot_count, inverse, slot_count, 0, stream);
}

// =====================================================================================
// plaintext expansion: sparse (index, value<t) -> dense residues, optionally NTT form
// =====================================================================================
template <int LOGN>
__global__ void __launch_bounds__(NttPlan<LOGN>::THREADS, NttPlan<LOGN>::MIN_CTAS)
plain_expand_kernel(const DeviceParams *__restrict__ P, int K, const uint32_t *__restrict__ offsets,
                    const uint32_t *__restrict__ idx, const uint64_t *__restrict__ val, long first, int mode,
                    int to_ntt, uint64_t *__restrict__ out) {
    extern __shared__ uint64_t sm[];
    constexpr int N = 1 << LOGN;
    const long b = blockIdx.x;
    const long pi = b / K;
    const int j = (int)(b % K);
    const NttTable tb = P->tab[j];
    const uint64_t half = P->half;
    const int sparse_shape = (mode >> 1) & 1;  // bit 1: every plaintext of the pack has the FractionalEncoder shape
    mode &= 1;                                 // bit 0: 0 lifted (multiplicative), 1 Delta-scaled (additive)
    for (int i = threadIdx.x; i < NttPlan<LOGN>::SMEM_WORDS; i += blockDim.x) sm[i] = 0;
    __syncthreads();
    const uint32_t lo = offsets[first + pi], hi = offsets[first + pi + 1];
    auto residue = [&](uint64_t c) -> uint64_t {
        if (mode == 0) return c >= half ? c + P->lift_inc[j] : c;  // evaluator.cpp:1475-1484
        U128 z = mul128(P->delta[j], c);                            // evaluator.cpp:1171-1190
        if (c >= half) add128_64(z, P->rho[j]);
        return barrett128(z, tb.mod);
    };
    uint64_t *dst = out + b * N;
    if (to_ntt && sparse_shape) {
        // FractionalEncoder-shaped plaintext (support in [0,64) U [n-32,n)): the first SKIP stages of
        // the Cooley-Tukey transform only copy the low part into every block and scale the top part by a
        // per-block constant (params.cpp, tf tables), so the blocks are written directly and the
        // schedule resumes at the first dense pass.
        constexpr int SKIP = sparse_skip_stages(LOGN);
        constexpr int NB = 1 << SKIP, M = N >> SKIP;
        const uint32_t cnt = (hi - lo) * NB;
        for (uint32_t w = threadIdx.x; w < cnt; w += blockDim.x) {
            const uint32_t e = lo + w / NB, blk = w % NB;
            const int ix = (int)idx[e];
            uint64_t v = residue(val[e]);
            if (ix < 64) {
                sm[ntt_pad((int)blk * M + ix)] = v;
            } else {
                sm[ntt_pad((int)blk * M + M - (N - ix))] = mulmod(v, __ldg(tb.tf + blk), tb.mod);
            }
        }
        __syncthreads();
        ntt_forward_in_smem<LOGN, NttPlan<LOGN>::skip_passes()>(sm, tb);
        smem_store_poly_canonical<LOGN>(sm, dst, tb.mod);
        return;
    }
    for (uint32_t e = lo + threadIdx.x; e < hi; e += blockDim.x) sm[ntt_pad((int)idx[e])] = residue(val[e]);
    __syncthreads();
    if (to_ntt) {
        ntt_forward_in_smem<LOGN>(sm, tb);
        smem_store_poly_canonical<LOGN>(sm, dst, tb.mod);
    } else {
        for (int i = threadIdx.x; i < N; i += blockDim.x) dst[i] = sm[ntt_pad(i)];
    }
}

template <int LOGN>
static cudaError_t launch_plain_expand_t(const DeviceParams *P, int K, const uint32_t *offsets, const uint32_t *idx,
                                         const uint64_t *val, long first, long count, int mode, bool to_ntt,
                                         uint64_t *out, cudaStream_t stream) {
    using Pl = NttPlan<LOGN>;
    size_t smem = Pl::SMEM_WORDS * sizeof(uint64_t);
    auto k = plain_expand_kernel<LOGN>;
    static DeviceOnce once;
    if (once.first()) {
        cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    }
    if (count <= 0) return cudaSuccess;
    k<<<(unsigned)(count * K), Pl::THREADS, smem, stream>>>(P, K, offsets, idx, val, first, mode, to_ntt ? 1 : 0, out);
    return cudaGetLastError();
}

cudaError_t launch_plain_expand(const DeviceParams *P, int logn, int K, const uint32_t *offsets, const uint32_t *idx,
                                const uint64_t *val, long first, long count, int mode, bool to_ntt, uint64_t *out,
                                cudaStream_t stream) {
    switch (logn) {
        case 10: return launch_plain_expand_t<10>(P, K, offsets, idx, val, first, count, mode, to_ntt, out, stream);
        case 11: return launch_plain_expand_t<11>(P, K, offsets, idx, val, first, count, mode, to_ntt, out, stream);
        case 12: return launch_plain_expand_t<12>(P, K, offsets, idx, val, first, count, mode, to_ntt, out, stream);
        case 13: return launch_plain_expand_t<13>(P, K, offsets, idx, val, first, count, mode, to_ntt, out, stream);
        case 14: return launch_plain_expand_t<14>(P, K, offsets, idx, val, first, count, mode, to_ntt, out, stream);
        default: return cudaErrorInvalidValue;
    }
}

// =====================================================================================
// fused weighted sum: out[m][p] = sum_r x[in_index[p][r]] (.) w[m][r]  (+ bias[m] on poly 0)
// One thread owns one residue column (limb j, coefficient c) of a TM x TN tile of outputs and
// keeps 2*TM*TN 128-bit accumulators in registers; Barrett happens once per output (or once per
// chunk_terms when the fan-in could overflow 128 bits).  Grid: x = output tiles (fastest, so the
// CTAs resident together share one narrow coefficient slice of every input and weight -> L2 reuse),
// y = coefficient slices of 128 residues.
// =====================================================================================
constexpr int MAC_THREADS = 128;

template <int TM, int TN>
__global__ void __launch_bounds__(MAC_THREADS, (TM * TN <= 4) ? 4 : 2)
mac_kernel(const DeviceParams *__restrict__ P, MacArgs a) {
    extern __shared__ int s_idx[];  // [TN][R]
    const int n = a.n, K = a.K, R = a.R;
    const int slices_per_limb = n / MAC_THREADS;
    const int j = blockIdx.y / slices_per_limb;
    const int c = (blockIdx.y % slices_per_limb) * MAC_THREADS + threadIdx.x;
    const int tiles_m = (a.M + TM - 1) / TM;
    // position tiles fastest: CTAs that stream the same weight rows (fc: 164 GB of them) run back to back
    // and hit L2 instead of re-reading HBM once per position tile
    const int tiles_n = (a.Npos + TN - 1) / TN;
    const int tn = blockIdx.x % tiles_n, tm = blockIdx.x / tiles_n;
    (void)tiles_m;
    const int m_base = tm * TM, p_base = tn * TN;
    const Mod mod = P->tab[j].mod;
    const long limb_off = (long)j * n + c;
    const long poly_words = (long)K * n;

    for (int i = threadIdx.x; i < TN * R; i += MAC_THREADS) {
        int t = i / R, r = i - t * R;
        int p = min(p_base + t, a.Npos - 1);
        s_idx[i] = a.in_index[(long)p * R + r];
    }
    __syncthreads();

    Acc7 acc[TM][TN][2];
#pragma unroll
    for (int m = 0; m < TM; m++)
#pragma unroll
        for (int t = 0; t < TN; t++) { acc[m][t][0] = acc7_zero(); acc[m][t][1] = acc7_zero(); }

    // byte-addressed streams: weight row m advances by one plaintext per term; inputs are gathered
    // with one 32x32+64 multiply-add per load (ciphertext index x ciphertext stride + base)
    const unsigned w_step = (unsigned)(poly_words * 8), ct_step = (unsigned)(2 * poly_words * 8);
    const char *wptr[TM];
#pragma unroll
    for (int m = 0; m < TM; m++)
        wptr[m] = reinterpret_cast<const char *>(a.w + (long)min(m_base + m, a.M - 1) * R * poly_words + limb_off);
    const char *x0 = reinterpret_cast<const char *>(a.x + limb_off);
    const char *x1 = x0 + w_step;

    for (int r0 = 0; r0 < R; r0 += a.chunk_terms) {
        const int r1 = min(R, r0 + a.chunk_terms);
#pragma unroll 2
        for (int r = r0; r < r1; r++) {
            uint64_t W[TM], X[TN][2];
#pragma unroll
            for (int m = 0; m < TM; m++) { W[m] = __ldg(reinterpret_cast<const uint64_t *>(wptr[m])); wptr[m] += w_step; }
#pragma unroll
            for (int t = 0; t < TN; t++) {
                const unsigned long long off = (unsigned long long)(unsigned)s_idx[t * R + r] * ct_step;
                X[t][0] = __ldg(reinterpret_cast<const uint64_t *>(x0 + off));
                X[t][1] = __ldg(reinterpret_cast<const uint64_t *>(x1 + off));
            }
#pragma unroll
            for (int m = 0; m < TM; m++)
#pragma unroll
                for (int t = 0; t < TN; t++) {
                    mac7(acc[m][t][0], X[t][0], W[m]);
                    mac7(acc[m][t][1], X[t][1], W[m]);
                }
        }
        if (r1 < R) {
#pragma unroll
            for (int m = 0; m < TM; m++)
#pragma unroll
                for (int t = 0; t < TN; t++) {
                    acc[m][t][0] = acc7_from(barrett128(acc7_value(acc[m][t][0]), mod));
                    acc[m][t][1] = acc7_from(barrett128(acc7_value(acc[m][t][1]), mod));
                }
        }
    }

#pragma unroll
    for (int m = 0; m < TM; m++) {
        if (m_base + m >= a.M) continue;
#pragma unroll
        for (int t = 0; t < TN; t++) {
            const int p = p_base + t;
            if (p >= a.Npos) continue;
            uint64_t v0 = barrett128(acc7_value(acc[m][t][0]), mod), v1 = barrett128(acc7_value(acc[m][t][1]), mod);
            if (a.bias) v0 = addmod(v0, __ldg(a.bias + (long)(m_base + m) * poly_words + limb_off), mod.q);
            long oct = (long)(p / a.Pimg) * ((long)a.Mtotal * a.Pimg) + (long)(a.m0 + m_base + m) * a.Pimg + p % a.Pimg;
            uint64_t *op = a.out + oct * 2 * poly_words + limb_off;
            op[0] = v0;
            op[poly_words] = v1;
        }
    }
}

template <int TM, int TN>
static cudaError_t launch_mac_t(const DeviceParams *P, const MacArgs &a, cudaStream_t stream) {
    dim3 grid(((a.M + TM - 1) / TM) * ((a.Npos + TN - 1) / TN), a.K * (a.n / MAC_THREADS));
    size_t smem = (size_t)TN * a.R * sizeof(int);
    auto k = mac_kernel<TM, TN>;
    if (smem > 48 * 1024) cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k<<<grid, MAC_THREADS, smem, stream>>>(P, a);
    return cudaGetLastError();
}

cudaError_t launch_mac(const DeviceParams *P, const MacArgs &a, cudaStream_t stream) {
    if (a.M <= 0 || a.Npos <= 0) return cudaSuccess;
    // tile override for tuning sweeps: CRCNN_MAC_TILE=<TM><TN>, e.g. 22
    static const int forced = [] { const char *e = getenv("CRCNN_MAC_TILE"); return e ? atoi(e) : 0; }();
    switch (forced) {
        case 42: return launch_mac_t<4, 2>(P, a, stream);
        case 22: return launch_mac_t<2, 2>(P, a, stream);
        case 24: return launch_mac_t<2, 4>(P, a, stream);
        case 41: return launch_mac_t<4, 1>(P, a, stream);
        case 21: return launch_mac_t<2, 1>(P, a, stream);
        case 81: return launch_mac_t<8, 1>(P, a, stream);
        case 12: return launch_mac_t<1, 2>(P, a, stream);
        case 14: return launch_mac_t<1, 4>(P, a, stream);
        default: break;
    }
    if (a.Npos == 1) return launch_mac_t<4, 1>(P, a, stream);
    return launch_mac_t<2, 2>(P, a, stream);
}

// =====================================================================================
// pooling (window sums, optional NTT-domain scale)
// =====================================================================================
// grid.x = 1 KB... (word chunk of 512 residues) fastest, then the output ciphertext: the CTAs resident together work on a
// handful of neighbouring outputs, so overlapping windows (2x2 stride 1 reads every input 4 times) are served by L2.
// SMALL: R * max(q) < 2^64, the window sum fits 64 bits.  scale_sh = Shoup companions of `scale` (floor(s * 2^64 / q)).
// One CTA = 512 * EW_PER consecutive residues of one output ciphertext (inside one limb: it divides n), a thread owns
// EW_PER groups of two residues, 512 words apart, with all its loads issued before the arithmetic.
constexpr int EW_PER = 4;

template <bool SMALL>
__global__ void __launch_bounds__(256)
pool_kernel(const DeviceParams *__restrict__ P, const uint64_t *__restrict__ in, const int *__restrict__ in_index,
            int R, const uint64_t *__restrict__ scale, const uint64_t *__restrict__ scale_sh, uint64_t *__restrict__ out,
            int chunks, int per, int per_channel, int channels, const uint64_t *__restrict__ sub) {
    const int n = P->n, K = P->K;
    const long ctw = 2L * K * n;
    const long o = blockIdx.x / chunks;
    if (channels > 0) {
        // fused average pooling + batch-norm (NTT form): out = (sum of the window) * C_z - D_z, C_z = scale (.) invstd_z, D_z = mean_z (.)
        // invstd_z precomputed per channel z -- ((sum * s) - m) * v = sum * (s v) - m v mod q, the same canonical residues as
        // AvgPoolingLayer::forward followed by BatchNormLayer::forward (avgPoolingLayer.cpp:16-45, batchNormLayer.cpp:29-40)
        const long z = (o / per_channel) % channels;
        scale += z * (long)K * n;
        scale_sh += z * (long)K * n;
        sub += z * (long)K * n;
    }
    const long word0 = (long)(blockIdx.x % chunks) * (512L * per) + 2 * threadIdx.x;  // within the ciphertext
    const int j = (int)((word0 / n) % K);
    const Mod mod = P->tab[j].mod;
    const long lw0 = (long)j * n + word0 % n;
    ulonglong2 res[EW_PER];
    if (SMALL) {
#pragma unroll
        for (int k = 0; k < EW_PER; k++) res[k] = make_ulonglong2(0, 0);
        for (int r = 0; r < R; r++) {
            const uint64_t *src = in + (long)__ldg(in_index + o * R + r) * ctw + word0;
#pragma unroll
            for (int k = 0; k < EW_PER; k++)
                if (k < per) {
                    const ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2 *>(src + 512 * k));
                    res[k].x += v.x;
                    res[k].y += v.y;
                }
        }
    } else {
#pragma unroll
        for (int k = 0; k < EW_PER; k++) {
            if (k >= per) continue;
            U128 s0{0, 0}, s1{0, 0};
            for (int r = 0; r < R; r++) {
                const ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2 *>(in + (long)__ldg(in_index + o * R + r) * ctw + word0 + 512 * k));
                add128_64(s0, v.x);
                add128_64(s1, v.y);
            }
            res[k].x = barrett128(s0, mod);
            res[k].y = barrett128(s1, mod);
        }
    }
#pragma unroll
    for (int k = 0; k < EW_PER; k++) {
        if (k >= per) continue;
        ulonglong2 v = res[k];
        if (scale) {
            const ulonglong2 sc = __ldg(reinterpret_cast<const ulonglong2 *>(scale + lw0 + 512 * k));
            const ulonglong2 sh = __ldg(reinterpret_cast<const ulonglong2 *>(scale_sh + lw0 + 512 * k));
            v.x = mulshoup_lazy(v.x, sc.x, sh.x, mod.q);   // reduces any 64-bit sum
            v.y = mulshoup_lazy(v.y, sc.y, sh.y, mod.q);
            v.x = v.x >= mod.q ? v.x - mod.q : v.x;
            v.y = v.y >= mod.q ? v.y - mod.q : v.y;
            if (channels > 0 && word0 < (long)K * n) {     // polynomial 0 only: sub_plain touches c0 (evaluator.cpp:1218-1240)
                const ulonglong2 d = __ldg(reinterpret_cast<const ulonglong2 *>(sub + lw0 + 512 * k));
                v.x = submod(v.x, d.x, mod.q);
                v.y = submod(v.y, d.y, mod.q);
            }
        } else if (SMALL) {
            v.x = reduce64(v.x, mod);
            v.y = reduce64(v.y, mod);
        }
        *reinterpret_cast<ulonglong2 *>(out + o * ctw + word0 + 512 * k) = v;
    }
}

// =====================================================================================
// batch-norm and evaluator-level plaintext ops
// =====================================================================================
// invstd_sh = Shoup companions of invstd: the product is one mulhi + two mullo instead of a 128-bit Barrett,
// which leaves the kernel bound by HBM instead of by the integer pipe.
__global__ void __launch_bounds__(256)
bn_kernel(const DeviceParams *__restrict__ P, const uint64_t *__restrict__ in, int per_channel, int channels,
          const uint64_t *__restrict__ mean, const uint64_t *__restrict__ invstd, const uint64_t *__restrict__ invstd_sh,
          uint64_t *__restrict__ out, int chunks, int per) {
    const int n = P->n, K = P->K;
    const long pw = (long)K * n, ctw = 2 * pw;
    const long ct = blockIdx.x / chunks;
    const long word0 = (long)(blockIdx.x % chunks) * (512L * per) + 2 * threadIdx.x;  // two adjacent residues per group
    const int poly = (int)(word0 / pw);
    const long lw0 = word0 - poly * pw;  // j*n + c
    const int j = (int)(lw0 / n);
    const int z = (int)((ct / per_channel) % channels);
    const uint64_t q = P->tab[j].mod.q;
    const uint64_t *src = in + ct * ctw + word0, *mp = mean + z * pw + lw0, *vp = invstd + z * pw + lw0, *sp = invstd_sh + z * pw + lw0;
    ulonglong2 x[EW_PER], m[EW_PER], v[EW_PER], vs[EW_PER];
#pragma unroll
    for (int k = 0; k < EW_PER; k++)
        if (k < per) {
            x[k] = __ldg(reinterpret_cast<const ulonglong2 *>(src + 512 * k));
            v[k] = __ldg(reinterpret_cast<const ulonglong2 *>(vp + 512 * k));
            vs[k] = __ldg(reinterpret_cast<const ulonglong2 *>(sp + 512 * k));
            if (poly == 0) m[k] = __ldg(reinterpret_cast<const ulonglong2 *>(mp + 512 * k));
        }
#pragma unroll
    for (int k = 0; k < EW_PER; k++)
        if (k < per) {
            ulonglong2 y = x[k];
            if (poly == 0) {
                y.x = submod(y.x, m[k].x, q);
                y.y = submod(y.y, m[k].y, q);
            }
            y.x = mulshoup_lazy(y.x, v[k].x, vs[k].x, q);
            y.y = mulshoup_lazy(y.y, v[k].y, vs[k].y, q);
            y.x = y.x >= q ? y.x - q : y.x;
            y.y = y.y >= q ? y.y - q : y.y;
            *reinterpret_cast<ulonglong2 *>(out + ct * ctw + word0 + 512 * k) = y;
        }
}

// =====================================================================================
// multiply_plain in the COEFFICIENT domain for FractionalEncoder plaintexts (pooling scale, batch-norm factor).
// Such a plaintext is sum_e s_e x^(i_e) with s_e = +-1 (values 1 / t-1, lifted to +-1 mod every q_j by
// Evaluator::transform_to_ntt, evaluator.cpp:1465-1486) and at most 96 terms (64 integer, 32 fraction digits), so
//       (X * w)[c] = sum_e s_e * X~[c - i_e],     X~ = X extended negacyclically (X~[c +- n] = -X[c]),
// a few dozen additions per residue instead of a forward transform, a pointwise product and an inverse transform.
// Fused in front of it: the window sum of a pooling layer (in_index, R) and the mean subtraction of batch-norm
// (sub: Delta-scaled mean, polynomial 0 only).  One CTA = 256 consecutive coefficients of one output limb-polynomial;
// needs q < 2^56 (96 residues add up below 2^63).
// =====================================================================================
constexpr int TAP_CT = 1024;   // coefficients per CTA (4 consecutive ones per thread)

__global__ void __launch_bounds__(256, 5)
tapmul_kernel(const DeviceParams *__restrict__ P, TapMulArgs a) {
    __shared__ __align__(16) uint64_t sm[64 + TAP_CT + 32];
    __shared__ short t_delta[96];          // positive terms first, then the negative ones
    __shared__ int t_count[2];
    const int n = P->n, K = P->K;
    const int chunks = n / TAP_CT;
    long b = blockIdx.x;
    const int c0 = (int)(b % chunks) * TAP_CT; b /= chunks;
    const int j = (int)(b % K); b /= K;
    const int poly = (int)(b & 1);
    const long o = b >> 1;
    const int z = a.channels > 1 ? (int)((o / a.per_channel) % a.channels) : 0;
    const Mod mod = P->tab[j].mod;
    const long pw = (long)K * n, ctw = 2 * pw;
    const uint32_t lo = a.t_off[z], hi = a.t_off[z + 1];
    const int ntaps = (int)(hi - lo);
    if (threadIdx.x < 32) {
        // low index: X~[c - ix] with sign s; high index ix = n - tap: x^ix = -x^(-tap), X~[c + tap] with sign -s.
        // One warp sorts the terms by sign with ballots (at most 96 terms = 3 rounds).
        int npos = 0, nneg = 0;
        for (int e0 = 0; e0 < ntaps; e0 += 32) {
            const int e = e0 + threadIdx.x;
            int ix = 0, sgn = 0;
            if (e < ntaps) {
                ix = (int)a.t_idx[lo + e];
                const int s1 = a.t_val[lo + e] == 1 ? 1 : -1;
                sgn = ix < 64 ? s1 : -s1;
            }
            const unsigned mp = __ballot_sync(0xffffffffu, sgn > 0), mn = __ballot_sync(0xffffffffu, sgn < 0);
            const unsigned below = (1u << threadIdx.x) - 1;
            const short delta = (short)(ix < 64 ? -ix : n - ix);
            if (sgn > 0) t_delta[npos + __popc(mp & below)] = delta;
            npos += __popc(mp);
            (void)mn;
            nneg += __popc(mn);
        }
        // negatives go after all positives: second pass now that npos is known
        int k = 0;
        for (int e0 = 0; e0 < ntaps; e0 += 32) {
            const int e = e0 + threadIdx.x;
            int ix = 0, sgn = 0;
            if (e < ntaps) {
                ix = (int)a.t_idx[lo + e];
                const int s1 = a.t_val[lo + e] == 1 ? 1 : -1;
                sgn = ix < 64 ? s1 : -s1;
            }
            const unsigned mn = __ballot_sync(0xffffffffu, sgn < 0);
            const unsigned below = (1u << threadIdx.x) - 1;
            if (sgn < 0) t_delta[npos + k + __popc(mn & below)] = (short)(ix < 64 ? -ix : n - ix);
            k += __popc(mn);
        }
        if (threadIdx.x == 0) { t_count[0] = npos; t_count[1] = nneg; }
    }
    const uint64_t *subp = (a.sub && poly == 0) ? a.sub + (long)z * pw + (long)j * n : nullptr;
    // Load phase: the limb-polynomial of every window input is resolved ONCE per CTA (s_src), then every thread moves pairs of
    // residues with 128-bit loads -- the per-element index load and 64-bit address product of the first version were a third of the
    // kernel's instructions (ncu r02E: 10.6 k warp instructions per CTA, 70 % issue-active).
    __shared__ const uint64_t *s_src[16];
    const int R = a.in_index ? a.R : 1;
    if (threadIdx.x >= 32 && threadIdx.x < 32 + (R < 16 ? R : 16)) {
        const int r = threadIdx.x - 32;
        const long ct = a.in_index ? (long)__ldg(a.in_index + o * a.R + r) : o;
        s_src[r] = a.in + ct * ctw + (long)poly * pw + (long)j * n;
    }
    __syncthreads();
    constexpr int PAIRS = (64 + TAP_CT + 32) / 2, ITER = (PAIRS + 255) / 256;
    auto finish = [&](int i2, ulonglong2 v, bool summed) {
        int cc = c0 - 64 + 2 * i2;
        const bool wrapped = cc < 0 || cc >= n;
        cc = cc < 0 ? cc + n : (cc >= n ? cc - n : cc);
        if (summed) { v.x = reduce64(v.x, mod); v.y = reduce64(v.y, mod); }
        if (subp) {
            const ulonglong2 m2 = __ldg(reinterpret_cast<const ulonglong2 *>(subp + cc));
            v.x = submod(v.x, m2.x, mod.q); v.y = submod(v.y, m2.y, mod.q);
        }
        if (wrapped) { v.x = negmod(v.x, mod.q); v.y = negmod(v.y, mod.q); }
        *reinterpret_cast<ulonglong2 *>(sm + 2 * i2) = v;
    };
    auto wrap_cc = [&](int i2) { int cc = c0 - 64 + 2 * i2; return cc < 0 ? cc + n : (cc >= n ? cc - n : cc); };   // even: a pair wraps together
    if (R == 4 || R == 1) {
        // all loads of a thread (ITER pairs x R inputs) are issued before the first use: the kernel waits on DRAM latency otherwise
        // (in batches of two pairs per thread: 32 registers of loads in flight keep the kernel at five CTAs per SM)
#pragma unroll
        for (int it0 = 0; it0 < ITER; it0 += 2) {
            ulonglong2 w[2][4];
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int i2 = threadIdx.x + (it0 + u) * 256;
                if (it0 + u < ITER && i2 < PAIRS) {
                    const int cc = wrap_cc(i2);
#pragma unroll
                    for (int r = 0; r < 4; r++)
                        if (r < R) w[u][r] = __ldg(reinterpret_cast<const ulonglong2 *>(s_src[r] + cc));
                }
            }
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int i2 = threadIdx.x + (it0 + u) * 256;
                if (it0 + u < ITER && i2 < PAIRS) {
                    ulonglong2 v = w[u][0];
                    if (R == 4) { v.x += w[u][1].x + w[u][2].x + w[u][3].x; v.y += w[u][1].y + w[u][2].y + w[u][3].y; }
                    finish(i2, v, R > 1);
                }
            }
        }
    } else {
        for (int i2 = threadIdx.x; i2 < PAIRS; i2 += 256) {
            const int cc = wrap_cc(i2);
            ulonglong2 v = make_ulonglong2(0, 0);
            for (int r = 0; r < R; r++) {
                const uint64_t *src = R <= 16 ? s_src[r] + cc
                                              : a.in + (long)__ldg(a.in_index + o * a.R + r) * ctw + (long)poly * pw + (long)j * n + cc;
                const ulonglong2 x2 = __ldg(reinterpret_cast<const ulonglong2 *>(src));
                v.x += x2.x; v.y += x2.y;
            }
            finish(i2, v, true);
        }
    }
    __syncthreads();
    const int npos = t_count[0], nneg = t_count[1];
    // thread t owns coefficients t, t + 256, t + 512, t + 768 of the CTA's 1024: every shared-memory access of a warp
    // touches 32 consecutive words (conflict free for any tap offset)
    const uint64_t *base = sm + 64 + threadIdx.x;
    uint64_t pos[4] = {0, 0, 0, 0}, neg[4] = {0, 0, 0, 0};
    for (int e = 0; e < npos; e++) {
        const uint64_t *v = base + t_delta[e];
#pragma unroll
        for (int k = 0; k < 4; k++) pos[k] += v[256 * k];
    }
    for (int e = npos; e < npos + nneg; e++) {
        const uint64_t *v = base + t_delta[e];
#pragma unroll
        for (int k = 0; k < 4; k++) neg[k] += v[256 * k];
    }
    const uint64_t off = (uint64_t)nneg * mod.q;
    uint64_t *op = a.out + o * ctw + (long)poly * pw + (long)j * n + c0 + threadIdx.x;
#pragma unroll
    for (int k = 0; k < 4; k++) op[256 * k] = reduce64(pos[k] + off - neg[k], mod);
}

cudaError_t launch_tapmul(const DeviceParams *P, int n, int K, const TapMulArgs &a, cudaStream_t stream) {
    if (a.nout <= 0) return cudaSuccess;
    const long blocks = a.nout * 2 * K * (n / TAP_CT);
    if (n % TAP_CT || blocks > 0x7fffffffL) return cudaErrorInvalidValue;
    tapmul_kernel<<<(unsigned)blocks, 256, 0, stream>>>(P, a);
    return cudaGetLastError();
}

// Shoup companions floor(v * 2^64 / q) of canonical residues v (data = [..][K][n]); runs once per plaintext pack.
__global__ void __launch_bounds__(256)
shoup_companion_kernel(const DeviceParams *__restrict__ P, const uint64_t *__restrict__ data, long words, uint64_t *__restrict__ out) {
    const long w = (long)blockIdx.x * 256 + threadIdx.x;
    if (w >= words) return;
    const uint64_t q = P->tab[(w / P->n) % P->K].mod.q;
    out[w] = (uint64_t)((((unsigned __int128)__ldg(data + w)) << 64) / q);
}

cudaError_t launch_shoup_companion(const DeviceParams *P, const uint64_t *data, long words, uint64_t *out, cudaStream_t stream) {
    if (words <= 0) return cudaSuccess;
    shoup_companion_kernel<<<(unsigned)((words + 255) / 256), 256, 0, stream>>>(P, data, words, out);
    return cudaGetLastError();
}

// data[w] = times * data[w] mod q (times small): the additive form of a plaintext that is added `times` times.  Once per pack.
__global__ void __launch_bounds__(256)
scale_small_kernel(const DeviceParams *__restrict__ P, uint64_t *__restrict__ data, long words, int times) {
    const long w = (long)blockIdx.x * 256 + threadIdx.x;
    if (w >= words) return;
    const uint64_t q = P->tab[(w / P->n) % P->K].mod.q;
    const uint64_t v = data[w];
    uint64_t acc = 0;
    for (int i = 0; i < times; i++) acc = addmod(acc, v, q);
    data[w] = acc;
}

// data[row][K][n] = data[row] (.) C[row / group] - D[row / group] (D may be null; pointwise mod q_j): folds per-channel constants into
// the NTT forms of a convolution's weights (group = fan-in) and bias (group = 1).  Once per network.
__global__ void __launch_bounds__(256)
fold_affine_kernel(const DeviceParams *__restrict__ P, uint64_t *__restrict__ data, long rows, int group, const uint64_t *__restrict__ C,
                   const uint64_t *__restrict__ D) {
    const long pw = (long)P->K * P->n;
    const long w = (long)blockIdx.x * 256 + threadIdx.x;
    if (w >= rows * pw) return;
    const long row = w / pw, lw = w - row * pw;
    const Mod mod = P->tab[lw / P->n].mod;
    const long cw = (row / group) * pw + lw;
    uint64_t v = mulmod(data[w], __ldg(C + cw), mod);
    if (D) v = submod(v, __ldg(D + cw), mod.q);
    data[w] = v;
}

cudaError_t launch_fold_affine(const DeviceParams *P, uint64_t *data, long rows, long poly_words, int group, const uint64_t *C,
                               const uint64_t *D, cudaStream_t stream) {
    if (rows <= 0) return cudaSuccess;
    fold_affine_kernel<<<(unsigned)((rows * poly_words + 255) / 256), 256, 0, stream>>>(P, data, rows, group, C, D);
    return cudaGetLastError();
}

// Composed fully connected layer behind a per-channel affine map x = P (.) C_c - D_c (pooling scale + batch-norm, NTT domain):
// Bias[k] -= sum_r W[k][r] (.) D[r / per_channel],  then  W[k][r] (.)= C[r / per_channel].  One thread per (k, residue slot).  Once per network.
__global__ void __launch_bounds__(256)
fold_fc_input_affine_kernel(const DeviceParams *__restrict__ P, uint64_t *__restrict__ W, int out_dim, int in_dim, int per_channel,
                            const uint64_t *__restrict__ C, const uint64_t *__restrict__ D, uint64_t *__restrict__ Bias) {
    const long pw = (long)P->K * P->n;
    const long id = (long)blockIdx.x * 256 + threadIdx.x;
    if (id >= (long)out_dim * pw) return;
    const long k = id / pw, lw = id - k * pw;
    const Mod mod = P->tab[lw / P->n].mod;
    uint64_t acc = Bias[k * pw + lw];
    for (int r = 0; r < in_dim; r++) {
        const long cw = (long)(r / per_channel) * pw + lw;
        uint64_t *wp = W + ((long)k * in_dim + r) * pw + lw;
        const uint64_t w = *wp;
        acc = submod(acc, mulmod(w, __ldg(D + cw), mod), mod.q);
        *wp = mulmod(w, __ldg(C + cw), mod);
    }
    Bias[k * pw + lw] = acc;
}

cudaError_t launch_fold_fc_input_affine(const DeviceParams *P, uint64_t *W, int out_dim, int in_dim, long poly_words, int per_channel,
                                        const uint64_t *C, const uint64_t *D, uint64_t *Bias, cudaStream_t stream) {
    if (out_dim <= 0 || in_dim <= 0) return cudaSuccess;
    fold_fc_input_affine_kernel<<<(unsigned)((out_dim * poly_words + 255) / 256), 256, 0, stream>>>(P, W, out_dim, in_dim, per_channel, C, D, Bias);
    return cudaGetLastError();
}

cudaError_t launch_scale_small(const DeviceParams *P, uint64_t *data, long words, int times, cudaStream_t stream) {
    if (words <= 0) return cudaSuccess;
    scale_small_kernel<<<(unsigned)((words + 255) / 256), 256, 0, stream>>>(P, data, words, times);
    return cudaGetLastError();
}

// Four consecutive residues per thread (two 128-bit loads and stores); additive ops touch polynomial 0 only, and only those words
// are launched.  HBM-bound: 2 x 8 bytes per residue of the ciphertext, the plaintext operand (K*n words, shared by every
// ciphertext of the launch) comes from L2.
__global__ void __launch_bounds__(256)
plain_op_kernel(const DeviceParams *__restrict__ P, uint64_t *__restrict__ data, int size, const uint64_t *__restrict__ pl,
                const uint64_t *__restrict__ pl_sh, int op) {
    const int n = P->n, K = P->K;
    const long pw = (long)K * n, ctw = size * pw, active = op == 0 ? ctw : pw;
    const long ct = blockIdx.x;
    const long word = ((long)blockIdx.y * 256 + threadIdx.x) * 4;
    if (word >= active) return;
    const long lw = word % pw;
    const int j = (int)(lw / n);
    const Mod mod = P->tab[j].mod;
    ulonglong2 *x = reinterpret_cast<ulonglong2 *>(data + ct * ctw + word);
    const ulonglong2 *w = reinterpret_cast<const ulonglong2 *>(pl + lw);
    ulonglong2 a = x[0], b = x[1];
    const ulonglong2 wa = __ldg(w), wb = __ldg(w + 1);
    if (op == 0) {
        // the plaintext is a constant of the launch: Shoup companions (floor(w 2^64 / q)) make each product 1 mulhi + 2 mullo and one
        // conditional subtraction instead of a 128-bit Barrett step -- the same canonical residue
        const ulonglong2 *ws = reinterpret_cast<const ulonglong2 *>(pl_sh + lw);
        const ulonglong2 sa = __ldg(ws), sb = __ldg(ws + 1);
        uint64_t r;
        r = mulshoup_lazy(a.x, wa.x, sa.x, mod.q); a.x = r >= mod.q ? r - mod.q : r;
        r = mulshoup_lazy(a.y, wa.y, sa.y, mod.q); a.y = r >= mod.q ? r - mod.q : r;
        r = mulshoup_lazy(b.x, wb.x, sb.x, mod.q); b.x = r >= mod.q ? r - mod.q : r;
        r = mulshoup_lazy(b.y, wb.y, sb.y, mod.q); b.y = r >= mod.q ? r - mod.q : r;
    }
    else if (op == 1) { a.x = addmod(a.x, wa.x, mod.q); a.y = addmod(a.y, wa.y, mod.q); b.x = addmod(b.x, wb.x, mod.q); b.y = addmod(b.y, wb.y, mod.q); }
    else { a.x = submod(a.x, wa.x, mod.q); a.y = submod(a.y, wa.y, mod.q); b.x = submod(b.x, wb.x, mod.q); b.y = submod(b.y, wb.y, mod.q); }
    x[0] = a; x[1] = b;
}

// =====================================================================================
// BEHZ square pieces
// =====================================================================================
// q -> Bsk U {m_tilde} fast conversion followed by the Montgomery-style q-overflow removal
// (baseconverter.cpp:663-742 then :581-622), one thread per coefficient.  With
// y_i = x_i * m_tilde*(q/q_i)^-1 mod q_i and r = -(sum_i y_i (q/q_i)) * q^-1 mod 2^32 (not centred), the
// output residue mod p_k is ((sum_i y_i (q/q_i) + q r) * m_tilde^-1) mod p_k; the constant factors are
// folded (lift_a, lift_b) so each residue is one lazy 128-bit sum and one Barrett reduction.
// KT/ST > 0: K and S are compile-time (loops unroll exactly, every constant is an immediate constant-bank operand
// because the parameter block is passed by value); KT == 0: any K <= MAXK, S <= MAXS at run time.
template <int KT, int ST, bool FOLD>
__global__ void __launch_bounds__(128)
behz_lift_kernel(const __grid_constant__ DeviceParams P, const uint64_t *__restrict__ in, const uint64_t *__restrict__ in_ntt,
                 uint64_t *__restrict__ ext) {
    const int n = P.n, K = KT ? KT : P.K, S = KT ? ST : P.S;
    constexpr int KB = KT ? KT : MAXK, SB = KT ? ST : MAXS;
    const int per = n / 128;
    const long poly = blockIdx.x / per;  // ct*2 + p
    const int c = (blockIdx.x % per) * 128 + threadIdx.x;
    const uint64_t *src = in + poly * K * n + c;
    uint64_t *dst = ext + poly * (K + S) * n + c;
    uint64_t y[KB];
    uint32_t zmt = 0;
#pragma unroll
    for (int i = 0; i < KB; i++) {
        if (i < K) {
            uint64_t x = __ldg(src + (long)i * n);
            // the q limbs of ext are transformed next; when the caller already holds them transformed (in_ntt) the tensor
            // stage reads them from there and nothing is written here
            if (!in_ntt) dst[(long)i * n] = x;
            y[i] = behz_mulmod<FOLD>(x, P.mt_inv_qhat[i], P.tab[i].mod);
            zmt += (uint32_t)y[i] * (uint32_t)P.qhat_mod_mt[i];  // arithmetic mod m_tilde = 2^32
        }
    }
    const uint32_t r = zmt * (uint32_t)P.neg_inv_q_mod_mt;  // (-(z * q^-1)) mod 2^32, in [0, 2^32)
#pragma unroll
    for (int k = 0; k < SB; k++) {
        if (k < S) {
            Acc7 acc = acc7_zero();
#pragma unroll
            for (int i = 0; i < KB; i++)
                if (i < K) mac7(acc, y[i], P.lift_a[k][i]);
            mac7(acc, (uint64_t)r, P.lift_b[k]);
            dst[(long)(K + k) * n] = behz_reduce<FOLD>(acc7_value(acc), P.tab[K + k].mod);
        }
    }
}

// multiply by t, fast_floor (q U Bsk -> Bsk), fastbconv_sk (Bsk -> q)
// (evaluator.cpp:852-883, baseconverter.cpp:624-661, :448-579), one thread per coefficient.  Constant
// factors are folded (fl_c, fl_T, fl_N, fl_P in params.h) so that every residue the reference computes
// in several reduced steps is one lazy sum + one Barrett here:
//   u_i   = x_i * t (q/q_i)^-1                       mod q_i
//   f_k   = (x_k t - sum_i u_i (q/q_i)) q^-1          mod p_k      (fast_floor)
//   g_k   = f_k (M/m_k)^-1                            mod m_k, k < L
//   alpha = (sum_k g_k (M/m_k) - f_sk) M^-1           mod m_sk, centred
//   out_j = sum_k g_k (M/m_k) - alpha M               mod q_j      (fastbconv_sk)
template <int KT, int ST, bool FOLD>
__global__ void __launch_bounds__(128)
behz_floor_kernel(const __grid_constant__ DeviceParams P, const uint64_t *__restrict__ prod, uint64_t *__restrict__ out) {
    const int n = P.n, K = KT ? KT : P.K, S = KT ? ST : P.S, L = S - 1;
    constexpr int KB = KT ? KT : MAXK, SB = KT ? ST : MAXS;
    const int per = n / 128;
    const long poly = blockIdx.x / per;  // ct*3 + p
    const int c = (blockIdx.x % per) * 128 + threadIdx.x;
    const uint64_t *src = prod + poly * (K + S) * n + c;
    uint64_t *dst = out + poly * K * n + c;
    uint64_t u[KB], g[SB];
#pragma unroll
    for (int i = 0; i < KB; i++)
        if (i < K) u[i] = behz_mulmod<FOLD>(__ldg(src + (long)i * n), P.fl_c[i], P.tab[i].mod);
    uint64_t f_sk = 0;
#pragma unroll
    for (int k = 0; k < SB; k++)
        if (k < S) {
            Acc7 acc = acc7_zero();
            mac7(acc, __ldg(src + (long)(K + k) * n), P.fl_T[k]);
#pragma unroll
            for (int i = 0; i < KB; i++)
                if (i < K) mac7(acc, u[i], P.fl_N[k][i]);
            uint64_t v = behz_reduce<FOLD>(acc7_value(acc), P.tab[K + k].mod);
            if (k < L) g[k] = v; else f_sk = v;
        }
    const Mod msk = P.tab[K + L].mod;
    Acc7 acc = acc7_zero();
#pragma unroll
    for (int i = 0; i < SB; i++)
        if (i < L) mac7(acc, g[i], P.fl_P[i]);
    mac7(acc, msk.q - f_sk, P.inv_M_mod_msk);
    const uint64_t alpha = behz_reduce<FOLD>(acc7_value(acc), msk);
    const bool centered_neg = alpha > (msk.q >> 1);  // baseconverter.cpp:547-577
    const uint64_t alpha_mag = centered_neg ? msk.q - alpha : alpha;
#pragma unroll
    for (int j = 0; j < KB; j++)
        if (j < K) {
            Acc7 e = acc7_zero();
#pragma unroll
            for (int i = 0; i < SB; i++)
                if (i < L) mac7(e, g[i], P.Mhat_mod_q[j][i]);
            mac7(e, alpha_mag, centered_neg ? P.M_mod_q[j] : P.neg_M_mod_q[j]);
            dst[(long)j * n] = behz_reduce<FOLD>(acc7_value(e), P.tab[j].mod);
        }
}

// relinearize 3 -> 2 (evaluator.cpp:934-1069), staged so every transform runs in the tuned NTT
// kernel and nothing is recomputed:
//   1. scale:   d_i = c2_i * (q/q_i)^-1 mod q_i                          (:984-985)
//   2. digits:  for every (prime i, digit k, prime j): forward NTT mod q_j of the 16-bit digit
//               polynomial (d_i >> 16k) & 0xffff, built on the fly while loading   (:997-1011)
//   3. mac:     acc_p[j] = sum_(i,k) D_(i,k,j) (.) key_(i,k,p)[j], 128-bit lazy, one Barrett   (:1015-1046)
//   4. inverse NTT of acc (generic kernel), 5. out_p = c_p + acc_p                 (:1047-1068)
// =====================================================================================
__global__ void __launch_bounds__(256)
relin_scale_kernel(const DeviceParams *__restrict__ P, const uint64_t *__restrict__ in3, uint64_t *__restrict__ dsc) {
    const int n = P->n, K = P->K;
    const long pw = (long)K * n;
    const long ct = blockIdx.x;
    const long lw = (long)blockIdx.y * 256 + threadIdx.x;  // i*n + e
    const int i = (int)(lw / n);
    dsc[ct * pw + lw] = mulmod(__ldg(in3 + (ct * 3 + 2) * pw + lw), P->inv_qhat[i], P->tab[i].mod);
}

// crcnn_relinearize admits up to 63 digits (the 128-bit lazy sum of relin_mac_kernel, evaluator.cpp:972-976): keys of 1-bit
// digits over a 54-bit prime, or 4-bit digits over four 55-bit primes, have more than 32
constexpr int RELIN_MAXD = 64;
struct DigitMap {
    int D;                             // total digits = sum_i digits_i
    unsigned char prime[RELIN_MAXD];   // digit d belongs to prime i
    unsigned char shift[RELIN_MAXD];   // and is (d_i >> shift) & mask
};

template <int LOGN>
__global__ void __launch_bounds__(NttPlan<LOGN>::THREADS, NttPlan<LOGN>::MIN_CTAS)
ntt_fwd_digits_kernel(const DeviceParams *__restrict__ P, const uint64_t *__restrict__ dsc, DigitMap map, uint64_t mask,
                      uint64_t *__restrict__ dig) {
    extern __shared__ uint64_t sm[];
    constexpr int N = 1 << LOGN;
    const int K = P->K;
    const long b = blockIdx.x;  // (ct, digit, j)
    const int j = (int)(b % K);
    const int d = (int)((b / K) % map.D);
    const long ct = b / ((long)K * map.D);
    const NttTable tb = P->tab[j];
    const uint64_t *src = dsc + (ct * K + map.prime[d]) * N;
    const int shift = map.shift[d];
    for (int e = threadIdx.x; e < N; e += blockDim.x) sm[ntt_pad(e)] = (__ldg(src + e) >> shift) & mask;
    __syncthreads();
    ntt_forward_in_smem<LOGN>(sm, tb);
    smem_store_poly_canonical<LOGN>(sm, dig + b * N, tb.mod);
}

__global__ void __launch_bounds__(256)
relin_mac_kernel(const DeviceParams *__restrict__ P, const uint64_t *__restrict__ dig, const uint64_t *__restrict__ evk,
                 RelinArgs a, DigitMap map, uint64_t *__restrict__ acc_out) {
    const int n = P->n, K = P->K;
    const long pw = (long)K * n;
    const long ct = blockIdx.x;
    const long lw = (long)blockIdx.y * 256 + threadIdx.x;  // j*n + e
    const int j = (int)(lw / n);
    Acc7 acc0 = acc7_zero(), acc1 = acc7_zero();
    const uint64_t *dp = dig + ct * map.D * pw + lw;
    for (int d = 0; d < map.D; d++) {
        const int i = map.prime[d], k = map.shift[d] / a.dbc;
        const uint64_t *key = evk + a.key_off[i] + (long)(2 * k) * pw + lw;
        const uint64_t dv = __ldg(dp + (long)d * pw);
        mac7(acc0, dv, __ldg(key));
        mac7(acc1, dv, __ldg(key + pw));
    }
    const Mod mod = P->tab[j].mod;
    acc_out[(ct * 2) * pw + lw] = barrett128(acc7_value(acc0), mod);
    acc_out[(ct * 2 + 1) * pw + lw] = barrett128(acc7_value(acc1), mod);
}

__global__ void __launch_bounds__(256)
relin_add_kernel(const DeviceParams *__restrict__ P, const uint64_t *__restrict__ in3, const uint64_t *__restrict__ acc,
                 uint64_t *__restrict__ out) {
    const int n = P->n, K = P->K;
    const long pw = (long)K * n;
    const long ct = blockIdx.x;
    const long w = (long)blockIdx.y * 256 + threadIdx.x;  // p*pw + j*n + e, p in {0,1}
    const uint64_t q = P->tab[(w % pw) / n].mod.q;
    out[ct * 2 * pw + w] = addmod(__ldg(in3 + ct * 3 * pw + w), __ldg(acc + ct * 2 * pw + w), q);
}

template <int LOGN>
static cudaError_t launch_digits_t(const DeviceParams *P, int K, const uint64_t *dsc, const DigitMap &map, uint64_t mask,
                                   long count, uint64_t *dig, cudaStream_t stream) {
    using Pl = NttPlan<LOGN>;
    size_t smem = Pl::SMEM_WORDS * sizeof(uint64_t);
    auto k = ntt_fwd_digits_kernel<LOGN>;
    static DeviceOnce once;
    if (once.first()) {
        cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    }
    k<<<(unsigned)(count * map.D * K), Pl::THREADS, smem, stream>>>(P, dsc, map, mask, dig);
    return cudaGetLastError();
}

// Stages 1-3 of the relinearisation for a.count ciphertexts; the caller runs the inverse NTT on
// a.acc (count*2*K polynomials) and then launch_relin_finish.
cudaError_t launch_relin(const DeviceParams *P, int logn, int K, const RelinArgs &a, cudaStream_t stream) {
    if (a.count <= 0) return cudaSuccess;
    const int n = 1 << logn;
    DigitMap map{};
    for (int i = 0; i < K; i++)
        for (int k = 0; k < a.digits[i]; k++) {
            if (map.D >= RELIN_MAXD) return cudaErrorInvalidValue;
            map.prime[map.D] = (unsigned char)i;
            map.shift[map.D] = (unsigned char)(k * a.dbc);
            map.D++;
        }
    const uint64_t mask = (1ULL << a.dbc) - 1;
    dim3 g1((unsigned)a.count, (unsigned)((long)K * n / 256));
    relin_scale_kernel<<<g1, 256, 0, stream>>>(P, a.in3, a.dsc);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    switch (logn) {
        case 10: e = launch_digits_t<10>(P, K, a.dsc, map, mask, a.count, a.dig, stream); break;
        case 11: e = launch_digits_t<11>(P, K, a.dsc, map, mask, a.count, a.dig, stream); break;
        case 12: e = launch_digits_t<12>(P, K, a.dsc, map, mask, a.count, a.dig, stream); break;
        case 13: e = launch_digits_t<13>(P, K, a.dsc, map, mask, a.count, a.dig, stream); break;
        case 14: e = launch_digits_t<14>(P, K, a.dsc, map, mask, a.count, a.dig, stream); break;
        default: return cudaErrorInvalidValue;
    }
    if (e != cudaSuccess) return e;
    relin_mac_kernel<<<g1, 256, 0, stream>>>(P, a.dig, a.evk, a, map, a.acc);
    return cudaGetLastError();
}

cudaError_t launch_relin_finish(const DeviceParams *P, int n, int K, const RelinArgs &a, cudaStream_t stream) {
    if (a.count <= 0) return cudaSuccess;
    dim3 g((unsigned)a.count, (unsigned)(2L * K * n / 256));
    relin_add_kernel<<<g, 256, 0, stream>>>(P, a.in3, a.acc, a.out);
    return cudaGetLastError();
}

// =====================================================================================
// simple launch wrappers
// =====================================================================================
// groups of 512 residues a CTA of the element-wise kernels covers: the largest of 4, 2, 1 that keeps a CTA inside one limb
static int ew_per(int n) { return n % (512 * 4) == 0 ? 4 : (n % (512 * 2) == 0 ? 2 : 1); }

cudaError_t launch_pool(const DeviceParams *P, int n, int K, const uint64_t *in, const int *in_index, int Nout,
                           int R, const uint64_t *scale_ntt, const uint64_t *scale_shoup, bool sum_fits_64, uint64_t *out,
                           cudaStream_t stream, int per_channel, int channels, const uint64_t *sub) {
    if (Nout <= 0) return cudaSuccess;
    const int per = ew_per(n), chunks = (int)(2L * K * n / (512 * per));
    const unsigned grid = (unsigned)((long)Nout * chunks);
    if (sum_fits_64) pool_kernel<true><<<grid, 256, 0, stream>>>(P, in, in_index, R, scale_ntt, scale_shoup, out, chunks, per, per_channel, channels, sub);
    else pool_kernel<false><<<grid, 256, 0, stream>>>(P, in, in_index, R, scale_ntt, scale_shoup, out, chunks, per, per_channel, channels, sub);
    return cudaGetLastError();
}

// C[z] = S (.) V[z], D[z] = M[z] (.) V[z] (pointwise mod q_j): the per-channel constants of the fused pooling + batch-norm
__global__ void __launch_bounds__(256)
pool_bn_consts_kernel(const DeviceParams *__restrict__ P, const uint64_t *__restrict__ S, const uint64_t *__restrict__ V,
                      const uint64_t *__restrict__ M, long words, uint64_t *__restrict__ C, uint64_t *__restrict__ D) {
    const long w = (long)blockIdx.x * 256 + threadIdx.x;
    if (w >= words) return;
    const long pw = (long)P->K * P->n, lw = w % pw;
    const Mod mod = P->tab[lw / P->n].mod;
    const uint64_t v = __ldg(V + w);
    C[w] = S ? mulmod(__ldg(S + lw), v, mod) : v;      // no pooling factor (sum pooling): C = V
    D[w] = mulmod(__ldg(M + w), v, mod);
}
cudaError_t launch_pool_bn_consts(const DeviceParams *P, const uint64_t *S, const uint64_t *V, const uint64_t *M, long words,
                                  uint64_t *C, uint64_t *D, cudaStream_t stream) {
    if (words <= 0) return cudaSuccess;
    pool_bn_consts_kernel<<<(unsigned)((words + 255) / 256), 256, 0, stream>>>(P, S, V, M, words, C, D);
    return cudaGetLastError();
}

cudaError_t launch_bn(const DeviceParams *P, int n, int K, const uint64_t *in, long count, int per_channel,
                         int channels, const uint64_t *mean_ntt, const uint64_t *invstd_ntt, const uint64_t *invstd_shoup,
                         uint64_t *out, cudaStream_t stream) {
    if (count <= 0) return cudaSuccess;
    const int per = ew_per(n), chunks = (int)(2L * K * n / (512 * per));
    const unsigned grid = (unsigned)(count * chunks);
    bn_kernel<<<grid, 256, 0, stream>>>(P, in, per_channel, channels, mean_ntt, invstd_ntt, invstd_shoup, out, chunks, per);
    return cudaGetLastError();
}

cudaError_t launch_plain_op(const DeviceParams *P, int n, int K, uint64_t *data, long count, int size,
                               const uint64_t *pl, const uint64_t *pl_sh, int op, cudaStream_t stream) {
    if (count <= 0) return cudaSuccess;
    const long active = (long)(op == 0 ? size : 1) * K * n;     // additive ops: polynomial 0 only
    dim3 grid((unsigned)count, (unsigned)((active / 4 + 255) / 256));
    plain_op_kernel<<<grid, 256, 0, stream>>>(P, data, size, pl, pl_sh, op);
    return cudaGetLastError();
}

// K and S pairs of SEAL's default parameter sets get exact-size kernels (n = 4096: 2/3, 8192: 4/5, 16384: 8/9)
#define CRCNN_BEHZ_DISPATCH(KERNEL, GRID, ...)                                                                  \
    do {                                                                                                       \
        if (behz_fold_ok(hp)) {                                                                                \
            if (hp.K == 2 && hp.S == 3) KERNEL<2, 3, true><<<GRID, 128, 0, stream>>>(hp, __VA_ARGS__);          \
            else if (hp.K == 4 && hp.S == 5) KERNEL<4, 5, true><<<GRID, 128, 0, stream>>>(hp, __VA_ARGS__);     \
            else if (hp.K == 8 && hp.S == 9) KERNEL<8, 9, true><<<GRID, 128, 0, stream>>>(hp, __VA_ARGS__);     \
            else KERNEL<0, 0, true><<<GRID, 128, 0, stream>>>(hp, __VA_ARGS__);                                 \
        } else {                                                                                               \
            if (hp.K == 2 && hp.S == 3) KERNEL<2, 3, false><<<GRID, 128, 0, stream>>>(hp, __VA_ARGS__);         \
            else if (hp.K == 4 && hp.S == 5) KERNEL<4, 5, false><<<GRID, 128, 0, stream>>>(hp, __VA_ARGS__);    \
            else if (hp.K == 8 && hp.S == 9) KERNEL<8, 9, false><<<GRID, 128, 0, stream>>>(hp, __VA_ARGS__);    \
            else KERNEL<0, 0, false><<<GRID, 128, 0, stream>>>(hp, __VA_ARGS__);                                \
        }                                                                                                      \
    } while (0)

// every modulus the BEHZ kernels reduce by (coefficient primes, Bsk primes incl. m_sk) has the 2^k - delta shape reduce128_fold needs
bool behz_fold_ok(const DeviceParams &hp) {
    static const int env = [] { const char *e = getenv("CRCNN_BEHZ_FOLD"); return e ? atoi(e) : 1; }();
    if (!env) return false;
    for (int i = 0; i < hp.K + hp.S; i++)
        if (!fold128_make(hp.tab[i].mod.q).ok) return false;
    return true;
}

// The kernels take the parameter block by value, so an input left multiplied by n (ninv_in = false) is served by a copy of
// the block whose first-step constants carry n^-1 -- the kernels themselves do not change.
cudaError_t launch_behz_lift(const DeviceParams &P, int n, const uint64_t *in, const uint64_t *in_ntt, long count, uint64_t *ext,
                                cudaStream_t stream, bool ninv_in) {
    if (count <= 0) return cudaSuccess;
    if (!ninv_in && !in_ntt) return cudaErrorInvalidValue;   // the copied q limbs would carry the factor n
    DeviceParams scaled;
    if (!ninv_in) {
        scaled = P;
        std::memcpy(scaled.mt_inv_qhat, P.mt_inv_qhat_n, sizeof scaled.mt_inv_qhat);
    }
    const DeviceParams &hp = ninv_in ? P : scaled;
    const unsigned grid = (unsigned)(count * 2 * (n / 128));
    CRCNN_BEHZ_DISPATCH(behz_lift_kernel, grid, in, in_ntt, ext);
    return cudaGetLastError();
}

cudaError_t launch_behz_floor(const DeviceParams &P, int n, const uint64_t *prod, long count, uint64_t *out,
                                 cudaStream_t stream, bool ninv_in) {
    if (count <= 0) return cudaSuccess;
    DeviceParams scaled;
    if (!ninv_in) {
        scaled = P;
        std::memcpy(scaled.fl_c, P.fl_c_n, sizeof scaled.fl_c);
        std::memcpy(scaled.fl_T, P.fl_T_n, sizeof scaled.fl_T);
    }
    const DeviceParams &hp = ninv_in ? P : scaled;
    const unsigned grid = (unsigned)(count * 3 * (n / 128));
    CRCNN_BEHZ_DISPATCH(behz_floor_kernel, grid, prod, out);
    return cudaGetLastError();
}

// Reduce lazily stored residues (< 4q, as SEAL keeps the "second" evaluation-key polys,
// keygenerator.cpp:238-247) to canonical form once at upload.
__global__ void __launch_bounds__(256)
canonicalize_kernel(const DeviceParams *__restrict__ P, uint64_t *__restrict__ data, long words) {
    const long w = (long)blockIdx.x * 256 + threadIdx.x;
    if (w >= words) return;
    const int n = P->n, K = P->K;
    const uint64_t q = P->tab[(w / n) % K].mod.q;
    uint64_t v = data[w];
    v = v >= 2 * q ? v - 2 * q : v;
    data[w] = v >= q ? v - q : v;
}

cudaError_t launch_canonicalize(const DeviceParams *P, uint64_t *data, long words, cudaStream_t stream) {
    if (words <= 0) return cudaSuccess;
    canonicalize_kernel<<<(unsigned)((words + 255) / 256), 256, 0, stream>>>(P, data, words);
    return cudaGetLastError();
}

// =====================================================================================
// SEAL host layout <-> device layout: a limb-polynomial is n+1 words on the host (trailing pad word),
// n words on the device.  Uploads arrive as ONE contiguous copy (a strided cudaMemcpy2D from pinned memory
// reaches only a fraction of the PCIe rate) and are re-strided here; rows start 8-byte aligned only.
// =====================================================================================
__global__ void __launch_bounds__(256)
strip_pad_kernel(const uint64_t *__restrict__ src, uint64_t *__restrict__ dst, int n) {
    const long row = blockIdx.x;
    const uint64_t *s = src + row * (n + 1);
    uint64_t *d = dst + row * n;
    for (int i = threadIdx.x; i < n; i += 256) d[i] = __ldg(s + i);
}

cudaError_t launch_strip_pad(const uint64_t *src_padded, uint64_t *dst, long rows, int n, cudaStream_t stream) {
    if (rows <= 0) return cudaSuccess;
    strip_pad_kernel<<<(unsigned)rows, 256, 0, stream>>>(src_padded, dst, n);
    return cudaGetLastError();
}

// =====================================================================================
// integer-pipe probe: 8 independent 64x64->128 multiply-accumulate chains per thread
// =====================================================================================
__global__ void imad_probe_kernel(int iters, uint64_t *sink) {
    uint64_t a = 0x9E3779B97F4A7C15ULL * (threadIdx.x + 1), b = 0xD1B54A32D192ED03ULL + blockIdx.x;
    Acc7 acc[8];
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i] = acc7_from((uint64_t)i);
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 8; i++) mac7(acc[i], a + i, b);
        a += acc[0].a3;
        b ^= acc[7].a0;
    }
    uint64_t s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { U128 v = acc7_value(acc[i]); s += v.lo ^ v.hi; }
    if (s == 0x1234567) sink[0] = s;
}

cudaError_t launch_imad_probe(int blocks, int threads, int iters, uint64_t *sink, cudaStream_t stream) {
    imad_probe_kernel<<<blocks, threads, 0, stream>>>(iters, sink);
    return cudaGetLastError();
}

// =====================================================================================
// IMAD.WIDE issue-rate probe: 16 independent 32x32+64 -> 64-bit multiply-add chains per thread, nothing else in the loop.
// This is the ceiling of the pipe every 64-bit modular multiplication on this path runs on (a 64x64->128-bit product is 4
// IMAD.WIDE.U32); the dependent-carry MAC probe above reaches well under half of it.  iters * 16 IMAD.WIDE per thread.
// =====================================================================================
__global__ void imad_wide_probe_kernel(int iters, uint64_t *sink) {
    uint32_t a = 0x9E3779B9u * (threadIdx.x + 1), b = 0x85EBCA6Bu + blockIdx.x;
    uint64_t acc[16];
#pragma unroll
    for (int i = 0; i < 16; i++) acc[i] = (uint64_t)i * 0x100000001ull;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 16; i++)
            asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc[i]) : "r"(a + i), "r"(b));
    }
    uint64_t s = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) s ^= acc[i];
    if (s == 0x1234567) sink[0] = s;
}

cudaError_t launch_imad_wide_probe(int blocks, int threads, int iters, uint64_t *sink, cudaStream_t stream) {
    imad_wide_probe_kernel<<<blocks, threads, 0, stream>>>(iters, sink);
    return cudaGetLastError();
}

}  // namespace crcnn
