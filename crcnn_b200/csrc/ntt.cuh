// Negacyclic NTT / inverse NTT of whole limb-polynomials resident in shared memory.
//
// One CTA transforms one limb-polynomial (n residues of one prime).  The transform is the same
// map as the reference's ntt_negacyclic_harvey / inverse_ntt_negacyclic_harvey
// (SEAL/seal/util/smallntt.cpp:195-375, smallntt.h:210-258): Cooley-Tukey forward with
// bit-reversed output, Gentleman-Sande inverse, in the reference's own table order
// (root_powers[bitrev(i)] = psi^i), so NTT-form data made by SEAL (evaluation keys, NTT plaintexts)
// is interchangeable.  Outputs are canonical [0, q); only the lazy intermediate ranges differ:
//   * forward: for q < 2^57 the Harvey correction of X is dropped altogether and the Shoup product uses an
//     approximate quotient (modarith.cuh: mulshoup_lazy4, result in [0,4q)) -- values grow by at most 4q per
//     stage (< 61q < 2^63 after 14 stages) and are reduced once at the final store.  61-bit moduli (the Bsk
//     primes of `square`) keep the exact product and the correction.
//   * inverse: the n^-1 factor is applied once at the end (one Shoup product per residue) instead of a
//     halving in every butterfly, so the tables hold the plain inverse powers; for q < 2^57 the butterflies
//     keep values in [0,4q) with the same approximate product.  Callers that multiply every output residue by a
//     constant next can leave n^-1 out altogether (NINV = false) and fold it into their constant.
// Both remove ALU-pipe work, which ncu showed to be the binding pipe (profiles/r01b_*).
//
// Schedule: log2(n) stages are grouped into passes of 3 or 4 stages done in registers
// (8 or 16 residues per thread and group); between passes the polynomial lives in shared memory
// with two pad words every 16 residues, which makes the strided passes (gaps >= 32 or 16) and the
// contiguous pass bank-conflict free and keeps every group of the contiguous pass 16-byte aligned, so it moves
// with 128-bit shared-memory accesses.  The contiguous pass gives every thread its own 15 twiddle pairs; read from
// the generic table the lanes of a warp touch 32 cache lines per load (ncu: L1 data pipe 62 % busy, two thirds of
// it these loads), so its pairs are also stored transposed (NttTable::wl / iwl: 15 rows, group index fastest).  The first forward pass reads HBM directly (coalesced),
// the last inverse pass writes HBM directly; the contiguous ends are staged through shared memory.
#pragma once
#include "modarith.cuh"
#include "params.h"

namespace crcnn {

__device__ __forceinline__ int ntt_pad(int i) { return i + ((i >> 4) << 1); }

template <int LOGN>
struct NttPlan {
    static constexpr int N = 1 << LOGN;
    static constexpr int THREADS = N / 32;  // 2 groups of 16 (4 of 8) residues per thread and pass
    static constexpr int SMEM_WORDS = N + N / 8;
    // CTAs per SM the shared-memory footprint allows (227 KB usable), capped so 85 registers per thread suffice
    static constexpr int FIT = (227 * 1024) / (SMEM_WORDS * 8);
    static constexpr int MIN_CTAS = FIT > 768 / THREADS ? 768 / THREADS : (FIT < 1 ? 1 : FIT);
    static constexpr int PASSES = (LOGN + 3) / 4;
    static constexpr int WIDE = LOGN - 3 * PASSES;  // how many passes take 4 stages (the rest take 3)
    // wide passes go last so the gaps seen by shared memory are >=32, 16 and 1 only (conflict free)
    __host__ __device__ static constexpr int bits(int pass) { return pass >= PASSES - WIDE ? 4 : 3; }
    // passes covered by sparse_skip_stages(LOGN)
    __host__ __device__ static constexpr int skip_passes() {
        int st = 0, p = 0;
        while (st < sparse_skip_stages(LOGN)) { st += bits(p); p++; }
        return p;
    }
};

// Moduli below 2^57 (every coefficient prime SEAL picks for n <= 16384) take the lazy path: the approximate Shoup
// product (mulshoup_lazy4, result in [0,4q)) and no per-stage correction in the forward transform -- values grow
// by at most 4q per stage, < 61q < 2^63 after 14 stages, and are reduced once at the final store.  Larger moduli
// (the 61-bit Bsk primes of `square`) keep the exact product and Harvey's correction.
__device__ __forceinline__ bool ntt_needs_correction(uint64_t q) { return (q >> 57) != 0; }
__device__ __forceinline__ int ntt_fwd_mode(uint64_t q) { return (q >> 57) == 0 ? 0 : ((q >> 61) == 0 ? 2 : 1); }
// inverse: the lazy butterfly keeps u, v in [0,4q) and forms T = u + 4q - v < 8q, so it serves every q < 2^61
__device__ __forceinline__ bool ntt_inv_exact(uint64_t q) { return (q >> 61) != 0; }

// Forward butterfly modes (picked per modulus by ntt_fwd_mode):
//   0  q < 2^57: approximate Shoup product, no correction of X at all (values grow by < 4q per stage)   c = nq, c2 = 4q
//   1  exact Harvey butterfly, [0,4q) -> [0,4q) (any q < 2^62)                                          c = q,  c2 = 2q
//   2  q < 2^61 (the Bsk primes): approximate product (result < 4q) with X corrected by 4q: [0,8q) -> [0,8q), 8q < 2^64
//                                                                                                       c = nq, c2 = 4q
template <int MODE>
__device__ __forceinline__ void ct_butterfly(uint64_t &x, uint64_t &y, uint64_t W, uint64_t Wp, uint64_t c, uint64_t c2) {
    if (MODE == 1) {
        uint64_t X = x >= c2 ? x - c2 : x;
        uint64_t Q = mulshoup_lazy(y, W, Wp, c);
        x = X + Q;
        y = X + c2 - Q;
    } else if (MODE == 2) {
        uint64_t X = x >= c2 ? x - c2 : x;
        uint64_t Q = mulshoup_lazy4(y, W, Wp, c);
        x = X + Q;
        y = X + c2 - Q;
    } else {
        uint64_t Q = mulshoup_lazy4(y, W, Wp, c);
        uint64_t X = x;
        x = X + Q;
        y = X + c2 - Q;
    }
}

template <bool CORR>
__device__ __forceinline__ void gs_butterfly(uint64_t &u, uint64_t &v, uint64_t W, uint64_t Wp, uint64_t c, uint64_t c2) {
    // W = psi^-k (no halving here, n^-1 is applied at the end)
    if (CORR) {
        // exact: u, v in [0,2q) -> [0,2q); c = q, c2 = 2q
        uint64_t T = u + c2 - v;
        uint64_t S = u + v;
        u = S >= c2 ? S - c2 : S;
        v = mulshoup_lazy(T, W, Wp, c);
    } else {
        // lazy: u, v in [0,4q) -> [0,4q); c = nq, c2 = 4q
        uint64_t T = u + c2 - v;
        uint64_t S = u + v;
        u = S >= c2 ? S - c2 : S;
        v = mulshoup_lazy4(T, W, Wp, c);
    }
}

// B forward stages on 2^B residues spaced g apart; m0 = number of blocks at the first stage,
// blk = this group's block index at that stage.
template <int B, int CORR>
__device__ __forceinline__ void fwd_group(uint64_t (&x)[1 << B], const ulonglong2 *__restrict__ w,
                                          uint64_t q, uint64_t twoq, int m0, int blk) {
#pragma unroll
    for (int s = 0; s < B; s++) {
        // stage s: pair distance 2^(B-1-s) (local index), 2^s local blocks each with its own twiddle
#pragma unroll
        for (int pr = 0; pr < (1 << (B - 1)); pr++) {
            const int lb = pr >> (B - 1 - s), a = pr & ((1 << (B - 1 - s)) - 1);
            const int ia = (lb << (B - s)) + a, ib = ia + (1 << (B - 1 - s));
            const int tw = ((m0 + blk) << s) + lb;
            const ulonglong2 W = __ldg(w + tw);
            ct_butterfly<CORR>(x[ia], x[ib], W.x, W.y, q, twoq);  // (q, twoq) = (c, c2) of ct_butterfly
        }
    }
}

// B inverse stages; h0 = n / (2 * distance of the first stage), blk = group index i.
template <int B, bool CORR>
__device__ __forceinline__ void inv_group(uint64_t (&x)[1 << B], const ulonglong2 *__restrict__ iw,
                                          uint64_t q, uint64_t twoq, int h0, int blk) {
#pragma unroll
    for (int s = 0; s < B; s++) {
        // stage s: pair distance 2^s, 2^(B-1-s) local blocks
#pragma unroll
        for (int pr = 0; pr < (1 << (B - 1)); pr++) {
            const int lb = pr >> s, a = pr & ((1 << s) - 1);
            const int ia = (lb << (s + 1)) + a, ib = ia + (1 << s);
            const int tw = (h0 >> s) + (blk << (B - 1 - s)) + lb;
            const ulonglong2 W = __ldg(iw + tw);
            gs_butterfly<CORR>(x[ia], x[ib], W.x, W.y, q, twoq);
        }
    }
}

// One forward pass over the whole polynomial.  SRC_GLOBAL: read `gsrc` (unpadded) instead of smem.
template <int LOGN, int B, bool SRC_GLOBAL, int CORR>
__device__ __forceinline__ void fwd_pass(uint64_t *sm, const uint64_t *__restrict__ gsrc, const NttTable &tb, int m0, int g) {
    constexpr int N = 1 << LOGN;
    const uint64_t q = CORR == 1 ? tb.mod.q : 0 - tb.mod.q, twoq = CORR == 1 ? 2 * tb.mod.q : 4 * tb.mod.q;
    for (int G = threadIdx.x; G < (N >> B); G += blockDim.x) {
        int blk = G / g, o = G - blk * g;
        int base = blk * (g << B) + o;
        uint64_t x[1 << B];
#pragma unroll
        for (int k = 0; k < (1 << B); k++) x[k] = SRC_GLOBAL ? gsrc[base + k * g] : sm[ntt_pad(base + k * g)];
        fwd_group<B, CORR>(x, reinterpret_cast<const ulonglong2 *>(tb.w), q, twoq, m0, blk);
#pragma unroll
        for (int k = 0; k < (1 << B); k++) sm[ntt_pad(base + k * g)] = x[k];
    }
}

// The contiguous 4-stage pass of the forward transform (g = 1): 16 consecutive residues per group, twiddles from the
// transposed table wl[row][G], row = 2^s - 1 + lb.
template <int LOGN, int CORR>
__device__ __forceinline__ void fwd_last_pass(uint64_t *sm, const NttTable &tb) {
    constexpr int N = 1 << LOGN, NG = N >> 4;
    const uint64_t q = CORR == 1 ? tb.mod.q : 0 - tb.mod.q, twoq = CORR == 1 ? 2 * tb.mod.q : 4 * tb.mod.q;
    const ulonglong2 *wl = reinterpret_cast<const ulonglong2 *>(tb.wl);
    for (int G = threadIdx.x; G < NG; G += blockDim.x) {
        ulonglong2 *row = reinterpret_cast<ulonglong2 *>(sm + 18 * G);
        uint64_t x[16];
#pragma unroll
        for (int m = 0; m < 8; m++) {
            const ulonglong2 v = row[m];
            x[2 * m] = v.x;
            x[2 * m + 1] = v.y;
        }
#pragma unroll
        for (int s = 0; s < 4; s++) {
#pragma unroll
            for (int lb = 0; lb < (1 << s); lb++) {
                const ulonglong2 W = __ldg(wl + ((1 << s) - 1 + lb) * NG + G);
#pragma unroll
                for (int a = 0; a < (1 << (3 - s)); a++) {
                    const int ia = (lb << (4 - s)) + a;
                    ct_butterfly<CORR>(x[ia], x[ia + (1 << (3 - s))], W.x, W.y, q, twoq);
                }
            }
        }
#pragma unroll
        for (int m = 0; m < 8; m++) row[m] = make_ulonglong2(x[2 * m], x[2 * m + 1]);
    }
}

// The contiguous 4-stage pass of the inverse transform (the first one): twiddles from iwl[row][G], row = 16 - (16 >> s) + lb.
template <int LOGN, bool CORR>
__device__ __forceinline__ void inv_first_pass(uint64_t *sm, const NttTable &tb) {
    constexpr int N = 1 << LOGN, NG = N >> 4;
    const uint64_t q = tb.mod.q;
    const uint64_t c = CORR ? q : 0 - q, c2 = CORR ? 2 * q : 4 * q;
    const ulonglong2 *iwl = reinterpret_cast<const ulonglong2 *>(tb.iwl);
    for (int G = threadIdx.x; G < NG; G += blockDim.x) {
        ulonglong2 *row = reinterpret_cast<ulonglong2 *>(sm + 18 * G);
        uint64_t x[16];
#pragma unroll
        for (int m = 0; m < 8; m++) {
            const ulonglong2 v = row[m];
            x[2 * m] = v.x;
            x[2 * m + 1] = v.y;
        }
#pragma unroll
        for (int s = 0; s < 4; s++) {
#pragma unroll
            for (int lb = 0; lb < (1 << (3 - s)); lb++) {
                const ulonglong2 W = __ldg(iwl + (16 - (16 >> s) + lb) * NG + G);
#pragma unroll
                for (int a = 0; a < (1 << s); a++) {
                    const int ia = (lb << (s + 1)) + a;
                    gs_butterfly<CORR>(x[ia], x[ia + (1 << s)], W.x, W.y, c, c2);
                }
            }
        }
#pragma unroll
        for (int m = 0; m < 8; m++) row[m] = make_ulonglong2(x[2 * m], x[2 * m + 1]);
    }
}

// DST_GLOBAL marks the last pass: the n^-1 scaling and the canonical store happen there.  NINV = false stores
// n * (the inverse transform) instead, still canonical, for a consumer whose first operation on every residue is a
// product by a constant that has absorbed n^-1 (the BEHZ lift and floor of `square`, params.h: *_n).
template <int LOGN, int B, bool DST_GLOBAL, bool CORR, bool NINV = true>
__device__ __forceinline__ void inv_pass(uint64_t *sm, uint64_t *__restrict__ gdst, const NttTable &tb, int g,
                                         const uint64_t *__restrict__ gadd = nullptr) {
    constexpr int N = 1 << LOGN;
    const uint64_t q = tb.mod.q;
    const uint64_t c = CORR ? q : 0 - q, c2 = CORR ? 2 * q : 4 * q;
    const int h0 = N / (2 * g);
    for (int G = threadIdx.x; G < (N >> B); G += blockDim.x) {
        int blk = G / g, o = G - blk * g;
        int base = blk * (g << B) + o;
        uint64_t x[1 << B];
#pragma unroll
        for (int k = 0; k < (1 << B); k++) x[k] = sm[ntt_pad(base + k * g)];
        inv_group<B, CORR>(x, reinterpret_cast<const ulonglong2 *>(tb.iw), c, c2, h0, blk);
#pragma unroll
        for (int k = 0; k < (1 << B); k++) {
            if (DST_GLOBAL) {
                uint64_t v;
                if (NINV) {
                    v = mulshoup_lazy(x[k], tb.ninv, tb.ninvp, q);  // exact product: [0,2q) for any 64-bit input
                } else {
                    v = x[k] >= 2 * q ? x[k] - 2 * q : x[k];          // [0,4q) (lazy) or [0,2q) (exact) -> [0,2q)
                }
                v = v >= q ? v - q : v;
                if (gadd) v = addmod(v, __ldg(gadd + base + k * g), q);   // fused "+ c_p" of relinearize
                gdst[base + k * g] = v;
            } else {
                sm[ntt_pad(base + k * g)] = x[k];
            }
        }
    }
}

template <int LOGN, int FIRST_PASS, int CORR>
__device__ __forceinline__ void ntt_forward_passes(uint64_t *sm, const uint64_t *__restrict__ src, const NttTable &tb) {
    using P = NttPlan<LOGN>;
    int m0 = 1, g = P::N;
#pragma unroll
    for (int p = 0; p < FIRST_PASS; p++) { g >>= P::bits(p); m0 <<= P::bits(p); }
#pragma unroll
    for (int p = FIRST_PASS; p < P::PASSES; p++) {
        g >>= P::bits(p);
        if (p == P::PASSES - 1 && P::bits(p) == 4 && !(p == 0 && src != nullptr)) {
            fwd_last_pass<LOGN, CORR>(sm, tb);
        } else if (p == 0 && src != nullptr) {
            if (P::bits(p) == 4) fwd_pass<LOGN, 4, true, CORR>(sm, src, tb, m0, g); else fwd_pass<LOGN, 3, true, CORR>(sm, src, tb, m0, g);
        } else {
            if (P::bits(p) == 4) fwd_pass<LOGN, 4, false, CORR>(sm, nullptr, tb, m0, g); else fwd_pass<LOGN, 3, false, CORR>(sm, nullptr, tb, m0, g);
        }
        m0 <<= P::bits(p);
        __syncthreads();
    }
}

// Forward transform of one polynomial: src (global, n words, canonical or < 4q) -> sm (padded, lazy).
template <int LOGN>
__device__ __forceinline__ void ntt_forward_to_smem(uint64_t *sm, const uint64_t *__restrict__ src, const NttTable &tb) {
    const int mode = ntt_fwd_mode(tb.mod.q);
    if (mode == 0) ntt_forward_passes<LOGN, 0, 0>(sm, src, tb);
    else if (mode == 2) ntt_forward_passes<LOGN, 0, 2>(sm, src, tb);
    else ntt_forward_passes<LOGN, 0, 1>(sm, src, tb);
}

// Forward transform when the polynomial is already in padded shared memory (values < 4q).
// FIRST_PASS > 0 resumes the schedule after the passes a sparse-input expansion has replaced.
template <int LOGN, int FIRST_PASS = 0>
__device__ __forceinline__ void ntt_forward_in_smem(uint64_t *sm, const NttTable &tb) {
    const int mode = ntt_fwd_mode(tb.mod.q);
    if (mode == 0) ntt_forward_passes<LOGN, FIRST_PASS, 0>(sm, nullptr, tb);
    else if (mode == 2) ntt_forward_passes<LOGN, FIRST_PASS, 2>(sm, nullptr, tb);
    else ntt_forward_passes<LOGN, FIRST_PASS, 1>(sm, nullptr, tb);
}

// Inverse transform of the polynomial in padded shared memory (values < 2q, < 4q on the lazy path) -> dst
// (global, canonical).  Pass order mirrors the forward plan (narrow passes first so the last, HBM-writing pass
// is strided).
template <int LOGN, bool CORR, bool NINV>
__device__ __forceinline__ void ntt_inverse_passes(uint64_t *sm, uint64_t *__restrict__ dst, const NttTable &tb,
                                                   const uint64_t *__restrict__ add) {
    using P = NttPlan<LOGN>;
    int g = 1;
#pragma unroll
    for (int p = P::PASSES - 1; p >= 1; p--) {
        if (p == P::PASSES - 1 && P::bits(p) == 4) inv_first_pass<LOGN, CORR>(sm, tb);
        else if (P::bits(p) == 4) inv_pass<LOGN, 4, false, CORR>(sm, nullptr, tb, g); else inv_pass<LOGN, 3, false, CORR>(sm, nullptr, tb, g);
        g <<= P::bits(p);
        __syncthreads();
    }
    if (P::bits(0) == 4) inv_pass<LOGN, 4, true, CORR, NINV>(sm, dst, tb, g, add); else inv_pass<LOGN, 3, true, CORR, NINV>(sm, dst, tb, g, add);
}

// NINV = false: the output is n times the inverse transform (see inv_pass)
template <int LOGN, bool NINV = true>
__device__ __forceinline__ void ntt_inverse_from_smem(uint64_t *sm, uint64_t *__restrict__ dst, const NttTable &tb,
                                                      const uint64_t *__restrict__ add = nullptr) {
    if (ntt_inv_exact(tb.mod.q)) ntt_inverse_passes<LOGN, true, NINV>(sm, dst, tb, add);
    else ntt_inverse_passes<LOGN, false, NINV>(sm, dst, tb, add);
}

// Coalesced copies between global (unpadded) and shared (padded).
template <int LOGN>
__device__ __forceinline__ void smem_load_poly(uint64_t *sm, const uint64_t *__restrict__ src) {
#pragma unroll 8
    for (int i = threadIdx.x; i < (1 << LOGN); i += NttPlan<LOGN>::THREADS) sm[ntt_pad(i)] = src[i];
}
// Lazy forward output (any 64-bit value) -> canonical residues in global memory.  Primes of the 2^k - delta shape take the one-fold
// reduction (1 IMAD.WIDE per residue instead of the ~9 multiplier instructions of reduce64); same residues.
template <int LOGN>
__device__ __forceinline__ void smem_store_poly_canonical(const uint64_t *sm, uint64_t *__restrict__ dst, const Mod &mod) {
    const int k = reduce64_shape_k(mod.q);
    if (k) {
#pragma unroll 8
        for (int i = threadIdx.x; i < (1 << LOGN); i += NttPlan<LOGN>::THREADS) dst[i] = reduce64_shape(sm[ntt_pad(i)], mod.q, k);
    } else {
#pragma unroll 8
        for (int i = threadIdx.x; i < (1 << LOGN); i += NttPlan<LOGN>::THREADS) dst[i] = reduce64(sm[ntt_pad(i)], mod);
    }
}

}  // namespace crcnn
