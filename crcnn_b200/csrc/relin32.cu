// Relinearisation through word-size auxiliary primes: see relin32.cuh for the algorithm and why it is bit-exact.
#include "relin32.cuh"
#include "kernels.cuh"
#include "devcfg.cuh"
#include "modarith.cuh"
#include <cmath>
#include <vector>

namespace crcnn {
namespace {

// primes k * 2^15 + 1 just below 2^30 (a primitive 2n-th root of unity exists for every n <= 16384)
const uint32_t kAuxPrimes[R32_MAXP] = {1073643521u, 1073479681u, 1073184769u, 1073053697u};

uint32_t mulm(uint32_t a, uint32_t b, uint32_t p) { return (uint32_t)((uint64_t)a * b % p); }
uint32_t powm(uint32_t a, uint64_t e, uint32_t p) {
    uint32_t r = 1;
    for (; e; e >>= 1, a = mulm(a, a, p))
        if (e & 1) r = mulm(r, a, p);
    return r;
}
uint32_t invm(uint32_t a, uint32_t p) { return powm(a % p, p - 2, p); }
uint32_t shoup_companion(uint32_t w, uint32_t p) { return (uint32_t)(((uint64_t)w << 32) / p); }
uint32_t bitrev32(uint32_t v, int bits) {
    uint32_t r = 0;
    for (int i = 0; i < bits; i++) r |= ((v >> i) & 1u) << (bits - 1 - i);
    return r;
}

// ------------------------------------------------------------------------------------------------
// 32-bit negacyclic NTT of one polynomial in shared memory.  Same map and table order as the 64-bit transform
// (ntt.cuh): Cooley-Tukey forward with bit-reversed output, Gentleman-Sande inverse; Harvey's lazy ranges
// ([0,4p) forward, [0,2p) inverse; p < 2^30).  Schedule: strided passes of 3-5 stages whose gaps are multiples of 32
// words and one contiguous pass of 5 stages (32 words per thread, moved with 128-bit shared-memory accesses).
// Four pad words after every 32 keep every access pattern bank-conflict free and every 4-word group 16-byte
// aligned.  The kernels are bound by the load/store unit, not by arithmetic (ncu: mio_throttle), hence the vector
// accesses: twiddle pairs two at a time, polynomial I/O four or eight coefficients at a time.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int pad32(int i) { return i + ((i >> 5) << 2); }
__device__ __forceinline__ uint32_t csub(uint32_t x, uint32_t m) { return min(x, x - m); }  // [0,2m) -> [0,m)
__device__ __forceinline__ uint32_t shoup32(uint32_t y, uint32_t w, uint32_t wp, uint32_t p) {
    return y * w - __umulhi(wp, y) * p;  // w*y mod p in [0,2p) for any 32-bit y
}

template <int LOGN>
struct Plan32 {
    static constexpr int N = 1 << LOGN;
    static constexpr int THREADS = N / 32 < 32 ? 32 : N / 32;
    static constexpr int SMEM_WORDS = N + N / 8;
    static constexpr int R32_TPS = 1024;  // resident threads per SM the register budget is sized for (64 registers per thread; measured 6 % faster than 768 -> 85)
    static constexpr int MIN_CTAS = R32_TPS / THREADS > 16 ? 16 : (R32_TPS / THREADS < 1 ? 1 : R32_TPS / THREADS);
    static constexpr int LAST = 5;
    static constexpr int REST = LOGN - LAST;
    static constexpr int NP = (REST + 4) / 5;  // strided passes (1 or 2 for n = 1024 ... 16384)
    __host__ __device__ static constexpr int bits(int i) { return REST / NP + (i < REST % NP ? 1 : 0); }
};

__device__ __forceinline__ void ct32(uint32_t &a, uint32_t &b, uint32_t w, uint32_t wp, uint32_t p, uint32_t twop) {
    const uint32_t X = csub(a, twop);
    const uint32_t Q = shoup32(b, w, wp, p);
    a = X + Q;
    b = X + twop - Q;
}
__device__ __forceinline__ void gs32(uint32_t &a, uint32_t &b, uint32_t w, uint32_t wp, uint32_t p, uint32_t twop) {
    const uint32_t u = a, v = b;
    a = csub(u + v, twop);
    b = shoup32(u + twop - v, w, wp, p);
}

// stage s of a forward group uses the 2^s consecutive twiddles starting at (mb << s)
template <int B>
__device__ __forceinline__ void fwd_group32(uint32_t (&x)[1 << B], const uint2 *__restrict__ w, uint32_t p, uint32_t twop, int mb) {
    {
        const uint2 W = __ldg(w + mb);
#pragma unroll
        for (int a = 0; a < (1 << (B - 1)); a++) ct32(x[a], x[a + (1 << (B - 1))], W.x, W.y, p, twop);
    }
#pragma unroll
    for (int s = 1; s < B; s++) {
        const uint4 *w4 = reinterpret_cast<const uint4 *>(w + (mb << s));
#pragma unroll
        for (int l2 = 0; l2 < (1 << (s - 1)); l2++) {
            const uint4 W = __ldg(w4 + l2);
#pragma unroll
            for (int a = 0; a < (1 << (B - 1 - s)); a++) {
                const int i0 = ((2 * l2) << (B - s)) + a, i1 = ((2 * l2 + 1) << (B - s)) + a;
                ct32(x[i0], x[i0 + (1 << (B - 1 - s))], W.x, W.y, p, twop);
                ct32(x[i1], x[i1 + (1 << (B - 1 - s))], W.z, W.w, p, twop);
            }
        }
    }
}

// stage s of an inverse group uses the 2^(B-1-s) consecutive twiddles starting at (h0 >> s) + (blk << (B-1-s))
template <int B>
__device__ __forceinline__ void inv_group32(uint32_t (&x)[1 << B], const uint2 *__restrict__ iw, uint32_t p, uint32_t twop, int h0,
                                            int blk) {
#pragma unroll
    for (int s = 0; s < B - 1; s++) {
        const uint4 *w4 = reinterpret_cast<const uint4 *>(iw + (h0 >> s) + (blk << (B - 1 - s)));
#pragma unroll
        for (int l2 = 0; l2 < (1 << (B - 2 - s)); l2++) {
            const uint4 W = __ldg(w4 + l2);
#pragma unroll
            for (int a = 0; a < (1 << s); a++) {
                const int i0 = ((2 * l2) << (s + 1)) + a, i1 = ((2 * l2 + 1) << (s + 1)) + a;
                gs32(x[i0], x[i0 + (1 << s)], W.x, W.y, p, twop);
                gs32(x[i1], x[i1 + (1 << s)], W.z, W.w, p, twop);
            }
        }
    }
    {
        const uint2 W = __ldg(iw + (h0 >> (B - 1)) + blk);
#pragma unroll
        for (int a = 0; a < (1 << (B - 1)); a++) gs32(x[a], x[a + (1 << (B - 1))], W.x, W.y, p, twop);
    }
}

// The contiguous pass gives every thread its own twiddles (31 pairs).  Read from the generic table, the lanes of a
// warp would touch 32 different cache lines per load (ncu: the L1 data pipe at 78 %, two thirds of it these loads), so
// the pairs of this pass are stored transposed: 15 rows of NG uint4 (two pairs each) + one row of NG uint2, group
// index fastest -- one fully coalesced load per row.
// (stages as template parameters: with a runtime-looking stage loop the compiler left the 32-word group in local memory)
template <int NG, int S>
__device__ __forceinline__ void fwd_last_stage(uint32_t (&x)[32], const uint4 *__restrict__ t4, uint32_t p, uint32_t twop, int G) {
    constexpr int B = 5;
#pragma unroll
    for (int l2 = 0; l2 < (1 << (S - 1)); l2++) {
        const uint4 W = __ldg(t4 + ((1 << (S - 1)) - 1 + l2) * NG + G);
#pragma unroll
        for (int a = 0; a < (1 << (B - 1 - S)); a++) {
            const int i0 = ((2 * l2) << (B - S)) + a, i1 = ((2 * l2 + 1) << (B - S)) + a;
            ct32(x[i0], x[i0 + (1 << (B - 1 - S))], W.x, W.y, p, twop);
            ct32(x[i1], x[i1 + (1 << (B - 1 - S))], W.z, W.w, p, twop);
        }
    }
}

template <int NG>
__device__ __forceinline__ void fwd_last32(uint32_t (&x)[32], const uint4 *__restrict__ t4, const uint2 *__restrict__ t1, uint32_t p,
                                           uint32_t twop, int G) {
    {
        const uint2 W = __ldg(t1 + G);
#pragma unroll
        for (int a = 0; a < 16; a++) ct32(x[a], x[a + 16], W.x, W.y, p, twop);
    }
    fwd_last_stage<NG, 1>(x, t4, p, twop, G);
    fwd_last_stage<NG, 2>(x, t4, p, twop, G);
    fwd_last_stage<NG, 3>(x, t4, p, twop, G);
    fwd_last_stage<NG, 4>(x, t4, p, twop, G);
}

template <int NG, int S>
__device__ __forceinline__ void inv_first_stage(uint32_t (&x)[32], const uint4 *__restrict__ t4, uint32_t p, uint32_t twop, int G) {
    constexpr int B = 5;
#pragma unroll
    for (int l2 = 0; l2 < (1 << (B - 2 - S)); l2++) {
        const uint4 W = __ldg(t4 + (16 - (16 >> S) + l2) * NG + G);
#pragma unroll
        for (int a = 0; a < (1 << S); a++) {
            const int i0 = ((2 * l2) << (S + 1)) + a, i1 = ((2 * l2 + 1) << (S + 1)) + a;
            gs32(x[i0], x[i0 + (1 << S)], W.x, W.y, p, twop);
            gs32(x[i1], x[i1 + (1 << S)], W.z, W.w, p, twop);
        }
    }
}

template <int NG>
__device__ __forceinline__ void inv_first32(uint32_t (&x)[32], const uint4 *__restrict__ t4, const uint2 *__restrict__ t1, uint32_t p,
                                            uint32_t twop, int G) {
    inv_first_stage<NG, 0>(x, t4, p, twop, G);
    inv_first_stage<NG, 1>(x, t4, p, twop, G);
    inv_first_stage<NG, 2>(x, t4, p, twop, G);
    inv_first_stage<NG, 3>(x, t4, p, twop, G);
    {
        const uint2 W = __ldg(t1 + G);
#pragma unroll
        for (int a = 0; a < 16; a++) gs32(x[a], x[a + 16], W.x, W.y, p, twop);
    }
}

template <int LOGN, int B, int GLOG, bool INV>
__device__ __forceinline__ void pass32(uint32_t *sm, const uint2 *__restrict__ tw, uint32_t p) {
    constexpr int N = 1 << LOGN, g = 1 << GLOG, TH = Plan32<LOGN>::THREADS;
    if constexpr (GLOG == 0) {
        // contiguous: 2^B = 32 words per group = one padded row of shared memory; `tw` is the transposed table
        static_assert(B == 5, "the contiguous pass takes 5 stages");
        constexpr int NG = N >> 5;
        const uint4 *t4 = reinterpret_cast<const uint4 *>(tw);
        const uint2 *t1 = tw + 30 * NG;
#pragma unroll 1
        for (int G = threadIdx.x; G < NG; G += TH) {
            uint4 *row = reinterpret_cast<uint4 *>(sm + G * 36);
            uint32_t x[32];
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const uint4 v = row[m];
                x[4 * m] = v.x; x[4 * m + 1] = v.y; x[4 * m + 2] = v.z; x[4 * m + 3] = v.w;
            }
            if (INV) inv_first32<NG>(x, t4, t1, p, 2 * p, G);
            else fwd_last32<NG>(x, t4, t1, p, 2 * p, G);
#pragma unroll
            for (int m = 0; m < 8; m++) row[m] = make_uint4(x[4 * m], x[4 * m + 1], x[4 * m + 2], x[4 * m + 3]);
        }
    } else {
        static_assert(GLOG >= 5, "strided passes need gaps that are multiples of 32 words");
        constexpr int PSTR = g + (g >> 5) * 4;  // pad32(base + k*g) = pad32(base) + k*PSTR
#pragma unroll 1
        for (int G = threadIdx.x; G < (N >> B); G += TH) {
            const int blk = G >> GLOG, o = G & (g - 1);
            uint32_t *col = sm + pad32((blk << (GLOG + B)) + o);
            uint32_t x[1 << B];
#pragma unroll
            for (int k = 0; k < (1 << B); k++) x[k] = col[k * PSTR];
            if (INV) inv_group32<B>(x, tw, p, 2 * p, N >> (GLOG + 1), blk);
            else fwd_group32<B>(x, tw, p, 2 * p, (N >> (GLOG + B)) + blk);
#pragma unroll
            for (int k = 0; k < (1 << B); k++) col[k * PSTR] = x[k];
        }
    }
}

// in: values < 4p in padded shared memory; out: lazy [0,4p).  Ends with a barrier.
template <int LOGN>
__device__ __forceinline__ void ntt32_forward(uint32_t *sm, const uint2 *__restrict__ w, const uint2 *__restrict__ wl, uint32_t p) {
    using P = Plan32<LOGN>;
    constexpr int b0 = P::bits(0), b1 = P::NP > 1 ? P::bits(1) : 0;
    pass32<LOGN, b0, LOGN - b0, false>(sm, w, p);
    __syncthreads();
    if constexpr (P::NP > 1) {
        pass32<LOGN, b1, LOGN - b0 - b1, false>(sm, w, p);
        __syncthreads();
    }
    pass32<LOGN, 5, 0, false>(sm, wl, p);
    __syncthreads();
}

// in: values < 2p (bit-reversed order); out: lazy [0,2p), NOT scaled by n^-1 (folded into the keys).  Ends with a barrier.
template <int LOGN>
__device__ __forceinline__ void ntt32_inverse(uint32_t *sm, const uint2 *__restrict__ iw, const uint2 *__restrict__ iwl, uint32_t p) {
    using P = Plan32<LOGN>;
    constexpr int b0 = P::bits(0), b1 = P::NP > 1 ? P::bits(1) : 0;
    pass32<LOGN, 5, 0, true>(sm, iwl, p);
    __syncthreads();
    if constexpr (P::NP > 1) {
        pass32<LOGN, b1, 5, true>(sm, iw, p);
        __syncthreads();
    }
    pass32<LOGN, b0, LOGN - b0, true>(sm, iw, p);
    __syncthreads();
}

// padded shared memory -> global, four coefficients per access; RANGE = 4 (forward output) or 2 (inverse output)
template <int LOGN, int RANGE>
__device__ __forceinline__ void store32_canonical(const uint32_t *sm, uint32_t *__restrict__ dst, uint32_t p) {
    for (int i = threadIdx.x * 4; i < (1 << LOGN); i += Plan32<LOGN>::THREADS * 4) {
        uint4 v = *reinterpret_cast<const uint4 *>(sm + pad32(i));
        if (RANGE == 4) { v.x = csub(v.x, 2 * p); v.y = csub(v.y, 2 * p); v.z = csub(v.z, 2 * p); v.w = csub(v.w, 2 * p); }
        v.x = csub(v.x, p); v.y = csub(v.y, p); v.z = csub(v.z, p); v.w = csub(v.w, p);
        *reinterpret_cast<uint4 *>(dst + i) = v;
    }
}

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
// d_i = c2_i * (q/q_i)^-1 mod q_i (evaluator.cpp:984-985), written as its dbc-bit digits (:997-1001): planes[ct][d][n] u16
__global__ void __launch_bounds__(256)
r32_scale_kernel(const DeviceParams *__restrict__ P, const Relin32Consts *__restrict__ cp, const uint64_t *__restrict__ in3,
                 uint16_t *__restrict__ planes) {
    const int n = P->n, K = P->K;
    const long pw = (long)K * n;
    const long ct = blockIdx.x;
    const long lw = ((long)blockIdx.y * 256 + threadIdx.x) * 2;  // two coefficients per thread
    const int i = (int)(lw / n), e = (int)(lw - (long)i * n);
    const ulonglong2 c2 = __ldg(reinterpret_cast<const ulonglong2 *>(in3 + (ct * 3 + 2) * pw + lw));
    const Mod mod = P->tab[i].mod;
    const uint64_t f = P->inv_qhat[i];
    const uint64_t v0 = mulmod(c2.x, f, mod), v1 = mulmod(c2.y, f, mod);
    const int dbc = cp->dbc, D = cp->D;
    const uint32_t mask = (1u << dbc) - 1;
    for (int d = cp->dfirst[i]; d < D && cp->dprime[d] == i; d++) {
        const int sh = cp->dshift[d];
        const uint32_t lo = (uint32_t)(v0 >> sh) & mask, hi = (uint32_t)(v1 >> sh) & mask;
        *reinterpret_cast<uint32_t *>(planes + (ct * D + d) * n + e) = lo | (hi << 16);
    }
}

// one CTA = (ciphertext, digit, auxiliary prime): digit polynomial -> NTT mod p_s, canonical
template <int LOGN>
__global__ void __launch_bounds__(Plan32<LOGN>::THREADS, Plan32<LOGN>::MIN_CTAS)
r32_digits_kernel(const uint16_t *__restrict__ planes, const Relin32Consts *__restrict__ cp, uint32_t *__restrict__ dig) {
    extern __shared__ uint4 sm32v[];
    uint32_t *sm32 = reinterpret_cast<uint32_t *>(sm32v);
    constexpr int N = 1 << LOGN;
    const long b = blockIdx.x;
    const int S3 = cp->S3;
    const int s = (int)(b % S3);
    const long cd = b / S3;  // ct * D + d
    const uint32_t p = cp->p[s];
    const uint2 *w = cp->w[s];
    const uint16_t *src = planes + cd * N;
    for (int i = threadIdx.x * 8; i < N; i += Plan32<LOGN>::THREADS * 8) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(src + i));
        uint4 *dst = reinterpret_cast<uint4 *>(sm32 + pad32(i));
        dst[0] = make_uint4(v.x & 0xffffu, v.x >> 16, v.y & 0xffffu, v.y >> 16);
        dst[1] = make_uint4(v.z & 0xffffu, v.z >> 16, v.w & 0xffffu, v.w >> 16);
    }
    __syncthreads();
    ntt32_forward<LOGN>(sm32, w, cp->wl[s], p);
    store32_canonical<LOGN, 4>(sm32, dig + b * N, p);
}

struct KeyMap {
    long key_off[MAXK];
    uint32_t ninv[R32_MAXP];
};

// one CTA = (digit, output o = p*K + j, auxiliary prime): key polynomial (coefficient form mod q_j) -> NTT mod p_s, times n^-1
template <int LOGN>
__global__ void __launch_bounds__(Plan32<LOGN>::THREADS, Plan32<LOGN>::MIN_CTAS)
r32_key_kernel(const uint64_t *__restrict__ coef, KeyMap km, const Relin32Consts *__restrict__ cp, int K, uint32_t *__restrict__ keys) {
    extern __shared__ uint4 sm32v[];
    uint32_t *sm32 = reinterpret_cast<uint32_t *>(sm32v);
    constexpr int N = 1 << LOGN;
    const long b = blockIdx.x;
    const int S3 = cp->S3, D = cp->D;
    const int s = (int)(b % S3);
    const int o = (int)((b / S3) % (2 * K));
    const int d = (int)(b / ((long)S3 * 2 * K));
    const int pi = o / K, j = o % K;
    const uint32_t p = cp->p[s];
    const uint64_t *src = coef + km.key_off[cp->dprime[d]] + ((long)(2 * (cp->dshift[d] / cp->dbc) + pi) * K + j) * N;
    for (int e = threadIdx.x; e < N; e += blockDim.x) sm32[pad32(e)] = (uint32_t)(__ldg(src + e) % p);
    __syncthreads();
    ntt32_forward<LOGN>(sm32, cp->w[s], cp->wl[s], p);
    uint32_t *dst = keys + (((long)s * D + d) * 2 * K + o) * N;
    const uint32_t ninv = km.ninv[s];
    for (int e = threadIdx.x; e < N; e += blockDim.x) {
        const uint32_t v = csub(csub(sm32[pad32(e)], 2 * p), p);
        dst[e] = (uint32_t)((uint64_t)v * ninv % p);
    }
}

// x mod p for any 64-bit x (p < 2^30, mu = floor(2^64/p)): the quotient estimate is at most 2 short
__device__ __forceinline__ uint32_t red64_32(uint64_t x, uint64_t mu, uint32_t p) {
    const uint32_t r = (uint32_t)x - (uint32_t)__umul64hi(x, mu) * p;
    return csub(csub(r, 2 * p), p);
}
__device__ __forceinline__ void madwide(uint64_t &acc, uint32_t a, uint32_t b) {
    asm("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc) : "r"(a), "r"(b));
}

// acc[ct][o][s][e] = sum_d dig[ct][d][s][e] * keys[s][d][o][e] mod p_s.
// One CTA = (EW coefficients, auxiliary prime s, a run of `cpb` ciphertexts): the keys of its coefficients (all digits, all
// OC = 2K outputs) are staged in shared memory once and reused for every ciphertext of the run, so the kernel streams the
// digit transforms from HBM and nothing else.  256 threads = EW coefficients x (256/EW) ciphertext lanes, T ciphertexts each.
template <int T, int OC, int EW>
__global__ void __launch_bounds__(256)
r32_mac_kernel(const uint32_t *__restrict__ dig, const uint32_t *__restrict__ keys, const Relin32Consts *__restrict__ cp, int n,
               long count, int cpb, uint32_t *__restrict__ acc) {
    extern __shared__ uint4 sm32v[];
    uint32_t *ksm = reinterpret_cast<uint32_t *>(sm32v);  // [D][OC][EW]
    constexpr int LANES = 256 / EW;
    const int el = threadIdx.x % EW, lane = threadIdx.x / EW;
    const int e = blockIdx.x * EW + el;
    const int s = blockIdx.y;
    const long ctb = (long)blockIdx.z * cpb;
    const long cte = min(ctb + cpb, count);
    const uint32_t p = cp->p[s];
    const uint64_t mu = cp->mu[s];
    const int D = cp->D, S3 = cp->S3;
    {
        // rows of EW words (16-byte vectors, several in flight per thread)
        const uint32_t *kg = keys + (long)s * D * OC * n + blockIdx.x * EW;
        constexpr int V = EW / 4;
#pragma unroll 8
        for (int i = threadIdx.x; i < D * OC * V; i += 256)
            sm32v[i] = __ldg(reinterpret_cast<const uint4 *>(kg + (long)(i / V) * n) + (i % V));
    }
    __syncthreads();
    const long dstride = (long)S3 * n;
    for (long c0 = ctb + lane * T; c0 < cte; c0 += LANES * T) {
        const uint32_t *dp[T];
#pragma unroll
        for (int t = 0; t < T; t++) dp[t] = dig + ((min(c0 + t, count - 1) * D) * S3 + s) * n + e;  // the tail repeats the last ciphertext
        uint64_t a[T][OC];
#pragma unroll
        for (int t = 0; t < T; t++)
#pragma unroll
            for (int o = 0; o < OC; o++) a[t][o] = 0;
        for (int d0 = 0; d0 < D; d0 += 16) {  // 16 products of canonical residues below 2^30 fit 64 bits
            const int dn = min(16, D - d0);
#pragma unroll 4
            for (int dd = 0; dd < dn; dd++) {
                const int d = d0 + dd;
                uint32_t dv[T];
#pragma unroll
                for (int t = 0; t < T; t++) dv[t] = __ldg(dp[t] + d * dstride);
                const uint32_t *kr = ksm + d * OC * EW + el;
#pragma unroll
                for (int o = 0; o < OC; o++) {
                    const uint32_t kv = kr[o * EW];
#pragma unroll
                    for (int t = 0; t < T; t++) madwide(a[t][o], dv[t], kv);
                }
            }
            if (d0 + 16 < D) {
#pragma unroll
                for (int t = 0; t < T; t++)
#pragma unroll
                    for (int o = 0; o < OC; o++) a[t][o] = red64_32(a[t][o], mu, p);
            }
        }
#pragma unroll
        for (int t = 0; t < T; t++)
            if (c0 + t < cte) {
                uint32_t *ap = acc + (((c0 + t) * OC) * S3 + s) * n + e;
#pragma unroll
                for (int o = 0; o < OC; o++) ap[(long)o * S3 * n] = red64_32(a[t][o], mu, p);
            }
    }
}

// The same sum for the shapes SEAL's default parameters give (D = 4K digits, OC = 2K outputs): the kernel above is bound by
// the latency of its digit loads (ncu: long_scoreboard 7.9 of 11 stall cycles per issue, 1.8 TB/s).  Here every thread keeps
// the keys of its coefficient and its two outputs in registers (2*D words, loaded once per CTA) and the digit transforms
// stream through a 6-stage cp.async ring in shared memory, two ciphertexts per stage, so dozens of KB are in flight per SM
// whatever the compute phase is doing.  32*OC threads = 64 coefficients x OC/2 output pairs.
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

template <int D, int OC>
__global__ void __launch_bounds__(32 * OC)
r32_mac_reg_kernel(const uint32_t *__restrict__ dig, const uint32_t *__restrict__ keys, const Relin32Consts *__restrict__ cp, int n,
                   long count, int cpb, uint32_t *__restrict__ acc) {
    constexpr int EW = 64, CPS = 2, NS = 6, SW = CPS * D * EW;
    extern __shared__ uint4 sm32v[];
    uint32_t *sm = reinterpret_cast<uint32_t *>(sm32v);  // [NS][CPS][D][EW]
    const int el = threadIdx.x % EW, og = threadIdx.x / EW;
    const int e0 = blockIdx.x * EW;
    const int s = blockIdx.y, S3 = cp->S3;
    const long ctb = (long)blockIdx.z * cpb;
    const long cte = min(ctb + cpb, count);
    const int nst = (int)((cte - ctb + CPS - 1) / CPS);
    const uint32_t p = cp->p[s];
    const uint64_t mu = cp->mu[s];
    uint32_t k0[D], k1[D];
    {
        const uint32_t *kg = keys + ((long)s * D * OC + og * 2) * n + e0 + el;
#pragma unroll
        for (int d = 0; d < D; d++) {
            k0[d] = __ldg(kg + (long)d * OC * n);
            k1[d] = __ldg(kg + (long)d * OC * n + n);
        }
    }
    // this thread's 16-byte chunk of every ciphertext tile: digit cd, words cpart*4 .. +3 (16*D chunks = 32*OC threads)
    const int cd = threadIdx.x / 16, cpart = threadIdx.x % 16;
    auto issue = [&](int st) {
        if (st < nst) {
            uint32_t *dst = sm + (st % NS) * SW + cd * EW + cpart * 4;
#pragma unroll
            for (int u = 0; u < CPS; u++) {
                const long ct = min(ctb + (long)st * CPS + u, count - 1);  // an odd tail repeats the last ciphertext
                cp_async16(dst + u * D * EW, dig + ((ct * D + cd) * S3 + s) * n + e0 + cpart * 4);
            }
        }
        cp_async_commit();
    };
#pragma unroll
    for (int st = 0; st < NS - 1; st++) issue(st);
    for (int st = 0; st < nst; st++) {
        cp_async_wait<NS - 2>();
        __syncthreads();
        issue(st + NS - 1);
        const uint32_t *tile = sm + (st % NS) * SW + el;
        uint64_t a[CPS][2];
#pragma unroll
        for (int u = 0; u < CPS; u++) {
            a[u][0] = 0;
            a[u][1] = 0;
        }
#pragma unroll
        for (int d = 0; d < D; d++) {
#pragma unroll
            for (int u = 0; u < CPS; u++) {
                const uint32_t x = tile[(u * D + d) * EW];
                madwide(a[u][0], x, k0[d]);
                madwide(a[u][1], x, k1[d]);
            }
            if (D > 16 && d == 15) {  // 16 products of canonical residues below 2^30 fit 64 bits
#pragma unroll
                for (int u = 0; u < CPS; u++) {
                    a[u][0] = red64_32(a[u][0], mu, p);
                    a[u][1] = red64_32(a[u][1], mu, p);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < CPS; u++) {
            const long ct = ctb + (long)st * CPS + u;
            if (ct < cte) {
                uint32_t *ap = acc + ((ct * OC + og * 2) * S3 + s) * n + e0 + el;
                ap[0] = red64_32(a[u][0], mu, p);
                ap[(long)S3 * n] = red64_32(a[u][1], mu, p);
            }
        }
    }
}

// one CTA = (ciphertext, output, auxiliary prime): inverse transform in place, canonical
template <int LOGN>
__global__ void __launch_bounds__(Plan32<LOGN>::THREADS, Plan32<LOGN>::MIN_CTAS)
r32_intt_kernel(const Relin32Consts *__restrict__ cp, uint32_t *__restrict__ acc) {
    extern __shared__ uint4 sm32v[];
    uint32_t *sm32 = reinterpret_cast<uint32_t *>(sm32v);
    constexpr int N = 1 << LOGN;
    const long b = blockIdx.x;
    const int s = (int)(b % cp->S3);
    const uint32_t p = cp->p[s];
    const uint2 *iw = cp->iw[s];
    uint32_t *poly = acc + b * N;
    for (int i = threadIdx.x * 4; i < N; i += Plan32<LOGN>::THREADS * 4)
        *reinterpret_cast<uint4 *>(sm32 + pad32(i)) = *reinterpret_cast<const uint4 *>(poly + i);
    __syncthreads();
    ntt32_inverse<LOGN>(sm32, iw, cp->iwl[s], p);
    store32_canonical<LOGN, 2>(sm32, poly, p);
}

// Garner mixed-radix digits of W mod P, sign by comparison with (P-1)/2, reduction mod q_j
struct CrtConsts {
    uint32_t p[R32_MAXP], half[R32_MAXP], ginv[R32_MAXP][R32_MAXP], ginvp[R32_MAXP][R32_MAXP];
    uint64_t c[R32_MAXP], csh[R32_MAXP], Pmodq, q;
};
template <int S3>
__device__ __forceinline__ uint64_t crt_one(const uint32_t (&r)[R32_MAXP], const CrtConsts &k) {
    uint32_t a[S3];
#pragma unroll
    for (int s = 0; s < S3; s++) {
        uint32_t t = r[s];
#pragma unroll
        for (int i = 0; i < s; i++) {
            const uint32_t ai = csub(a[i], k.p[s]);  // a_i < p_i < 2 p_s
            t = csub(shoup32(t + k.p[s] - ai, k.ginv[s][i], k.ginvp[s][i], k.p[s]), k.p[s]);
        }
        a[s] = t;
    }
    // W mod q_j = a_0 + sum_(s>0) a_s * (p_0...p_(s-1) mod q_j): Shoup products (each in [0,2q)), one lazy sum, three
    // conditional subtractions; negative W (mixed-radix digits above those of (P-1)/2) subtracts P mod q_j
    uint64_t v = a[0];
    bool neg = false, decided = false;
#pragma unroll
    for (int s = S3 - 1; s >= 0; s--) {
        if (s > 0) v += mulshoup_lazy((uint64_t)a[s], k.c[s], k.csh[s], k.q);
        if (!decided && a[s] != k.half[s]) { neg = a[s] > k.half[s]; decided = true; }
    }
    // v < 2^30 + 2(S3-1)q <= 7q
    v = v >= 4 * k.q ? v - 4 * k.q : v;
    v = v >= 2 * k.q ? v - 2 * k.q : v;
    v = v >= k.q ? v - k.q : v;
    if (neg) v = submod(v, k.Pmodq, k.q);
    return v;
}

// one CTA = (ciphertext, output o = p*K + j, 512 coefficients), two coefficients per thread: out = c_p + (W mod q_j)
template <int S3>
__global__ void __launch_bounds__(256)
r32_crt_kernel(const DeviceParams *__restrict__ P, const Relin32Consts *__restrict__ cp, const uint32_t *__restrict__ acc,
               const uint64_t *__restrict__ in3, uint64_t *__restrict__ out) {
    const int n = P->n, K = P->K;
    const int e = (blockIdx.y * 256 + threadIdx.x) * 2;
    const int o = (int)(blockIdx.x % (unsigned)(2 * K));
    const long ct = blockIdx.x / (unsigned)(2 * K);
    const int pi = o / K, j = o % K;
    CrtConsts k;
#pragma unroll
    for (int s = 0; s < S3; s++) {
        k.p[s] = cp->p[s];
        k.half[s] = cp->half[s];
        k.c[s] = cp->cmodq[j][s];
        k.csh[s] = cp->cmodq_sh[j][s];
#pragma unroll
        for (int i = 0; i < s; i++) {
            k.ginv[s][i] = cp->ginv[s][i];
            k.ginvp[s][i] = cp->ginvp[s][i];
        }
    }
    k.Pmodq = cp->Pmodq[j];
    k.q = P->tab[j].mod.q;
    const uint32_t *r = acc + ((ct * 2 * K + o) * S3) * n + e;
    uint32_t r0[R32_MAXP], r1[R32_MAXP];
#pragma unroll
    for (int s = 0; s < S3; s++) {
        const uint2 v = __ldg(reinterpret_cast<const uint2 *>(r + (long)s * n));
        r0[s] = v.x;
        r1[s] = v.y;
    }
    const long w = (long)j * n + e;
    const ulonglong2 c = __ldg(reinterpret_cast<const ulonglong2 *>(in3 + (ct * 3 + pi) * (long)K * n + w));
    ulonglong2 res;
    res.x = addmod(c.x, crt_one<S3>(r0, k), k.q);
    res.y = addmod(c.y, crt_one<S3>(r1, k), k.q);
    *reinterpret_cast<ulonglong2 *>(out + (ct * 2 + pi) * (long)K * n + w) = res;
}

// r32_intt_kernel and r32_crt_kernel in one: one CTA = (ciphertext, output o = p*K + j) transforms the S3 auxiliary-prime residues of its
// polynomial back in shared memory and reconstructs from there -- the 2 x S3 x n 32-bit words per output that the two-kernel form writes to
// and reads back from HBM (45 GB per step of the headline network) never leave the SM.  S3 * 36 KB of shared memory: two CTAs per SM at n = 8192.
template <int LOGN, int S3>
__global__ void __launch_bounds__(Plan32<LOGN>::THREADS, 2)
r32_intt_crt_kernel(const DeviceParams *__restrict__ P, const Relin32Consts *__restrict__ cp, const uint32_t *__restrict__ acc,
                    const uint64_t *__restrict__ in3, uint64_t *__restrict__ out) {
    extern __shared__ uint4 sm32v[];
    uint32_t *sm32 = reinterpret_cast<uint32_t *>(sm32v);
    constexpr int N = 1 << LOGN, SW = Plan32<LOGN>::SMEM_WORDS;
    const int K = P->K;
    const long b = blockIdx.x;                       // ct * 2K + o
    const int o = (int)(b % (2 * K));
    const long ct = b / (2 * K);
    const int pi = o / K, j = o % K;
#pragma unroll
    for (int s = 0; s < S3; s++) {
        const uint32_t *poly = acc + (b * S3 + s) * N;
        for (int i = threadIdx.x * 4; i < N; i += Plan32<LOGN>::THREADS * 4)
            *reinterpret_cast<uint4 *>(sm32 + s * SW + pad32(i)) = __ldg(reinterpret_cast<const uint4 *>(poly + i));
    }
    __syncthreads();
#pragma unroll
    for (int s = 0; s < S3; s++) ntt32_inverse<LOGN>(sm32 + s * SW, cp->iw[s], cp->iwl[s], cp->p[s]);   // ends with a barrier
    CrtConsts k;
#pragma unroll
    for (int s = 0; s < S3; s++) {
        k.p[s] = cp->p[s];
        k.half[s] = cp->half[s];
        k.c[s] = cp->cmodq[j][s];
        k.csh[s] = cp->cmodq_sh[j][s];
#pragma unroll
        for (int i = 0; i < s; i++) {
            k.ginv[s][i] = cp->ginv[s][i];
            k.ginvp[s][i] = cp->ginvp[s][i];
        }
    }
    k.Pmodq = cp->Pmodq[j];
    k.q = P->tab[j].mod.q;
    const uint64_t *cin = in3 + (ct * 3 + pi) * (long)K * N + (long)j * N;
    uint64_t *dst = out + (ct * 2 + pi) * (long)K * N + (long)j * N;
    for (int e = threadIdx.x * 2; e < N; e += Plan32<LOGN>::THREADS * 2) {
        uint32_t r0[R32_MAXP], r1[R32_MAXP];
#pragma unroll
        for (int s = 0; s < S3; s++) {
            const uint2 v = *reinterpret_cast<const uint2 *>(sm32 + s * SW + pad32(e));   // inverse output in [0, 2p): canonical first
            r0[s] = csub(v.x, k.p[s]);
            r1[s] = csub(v.y, k.p[s]);
        }
        const ulonglong2 c = __ldg(reinterpret_cast<const ulonglong2 *>(cin + e));
        ulonglong2 res;
        res.x = addmod(c.x, crt_one<S3>(r0, k), k.q);
        res.y = addmod(c.y, crt_one<S3>(r1, k), k.q);
        *reinterpret_cast<ulonglong2 *>(dst + e) = res;
    }
}

template <int LOGN>
void configure32() {
    static DeviceOnce once;
    if (!once.first()) return;
    const int smem = Plan32<LOGN>::SMEM_WORDS * 4;
    cudaFuncSetAttribute(r32_digits_kernel<LOGN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(r32_key_kernel<LOGN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(r32_intt_kernel<LOGN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(r32_digits_kernel<LOGN>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    cudaFuncSetAttribute(r32_intt_kernel<LOGN>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}

template <int T, int OC, int EW>
cudaError_t launch_mac(const uint32_t *dig, const Relin32 &r, int n, long count, int cpb, unsigned gz, size_t bytes_per_coeff, uint32_t *acc,
                       cudaStream_t stream) {
    const size_t smem = bytes_per_coeff * EW;
    // the staged size depends on the digit count of the context: set it on every launch (a cheap driver call, once per chunk)
    cudaError_t e = cudaFuncSetAttribute(r32_mac_kernel<T, OC, EW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    r32_mac_kernel<T, OC, EW><<<dim3((unsigned)(n / EW), (unsigned)r.c.S3, gz), 256, smem, stream>>>(dig, r.keys, r.dc, n, count, cpb, acc);
    return cudaGetLastError();
}

template <int D, int OC>
cudaError_t launch_mac_reg(const uint32_t *dig, const Relin32 &r, int n, long count, int cpb, unsigned gz, uint32_t *acc, cudaStream_t stream) {
    constexpr size_t smem = (size_t)6 * 2 * D * 64 * 4;
    static DeviceOnce once;
    if (once.first()) {
        cudaError_t e = cudaFuncSetAttribute(r32_mac_reg_kernel<D, OC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        cudaFuncSetAttribute(r32_mac_reg_kernel<D, OC>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    }
    r32_mac_reg_kernel<D, OC><<<dim3((unsigned)(n / 64), (unsigned)r.c.S3, gz), 32 * OC, smem, stream>>>(dig, r.keys, r.dc, n, count, cpb, acc);
    return cudaGetLastError();
}

template <int LOGN>
cudaError_t run_t(const DeviceParams *dP, int K, const Relin32 &r, const uint64_t *in3, uint64_t *out, long count, void *scratch,
                  cudaStream_t stream) {
    using Pl = Plan32<LOGN>;
    constexpr int N = 1 << LOGN;
    configure32<LOGN>();
    const Relin32Consts &c = r.c;
    const size_t smem = Pl::SMEM_WORDS * 4;
    uint32_t *dig = (uint32_t *)scratch;
    uint32_t *acc = dig + (size_t)count * c.D * c.S3 * N;
    uint16_t *planes = (uint16_t *)(acc + (size_t)count * 2 * K * c.S3 * N);
    r32_scale_kernel<<<dim3((unsigned)count, (unsigned)((long)K * N / 512)), 256, 0, stream>>>(dP, r.dc, in3, planes);
    r32_digits_kernel<LOGN><<<(unsigned)(count * c.D * c.S3), Pl::THREADS, smem, stream>>>(planes, r.dc, dig);
    {
        const int cpb = 128;
        const unsigned gz = (unsigned)((count + cpb - 1) / cpb);
        const size_t ksmem = (size_t)c.D * 2 * K * 4;  // bytes per staged coefficient
        cudaError_t e = cudaSuccess;
        if (c.D == 4 * K && K == 1) e = launch_mac_reg<4, 2>(dig, r, N, count, cpb, gz, acc, stream);
        else if (c.D == 4 * K && K == 2) e = launch_mac_reg<8, 4>(dig, r, N, count, cpb, gz, acc, stream);
        else if (c.D == 4 * K && K == 4) e = launch_mac_reg<16, 8>(dig, r, N, count, cpb, gz, acc, stream);
        else if (c.D == 4 * K && K == 8) e = launch_mac_reg<32, 16>(dig, r, N, count, cpb, gz, acc, stream);
        else
        switch (2 * K) {
            case 2: e = launch_mac<4, 2, 64>(dig, r, N, count, cpb, gz, ksmem, acc, stream); break;
            case 4: e = launch_mac<4, 4, 64>(dig, r, N, count, cpb, gz, ksmem, acc, stream); break;
            case 8: e = launch_mac<4, 8, 64>(dig, r, N, count, cpb, gz, ksmem, acc, stream); break;
            case 16: e = launch_mac<2, 16, 32>(dig, r, N, count, cpb, gz, ksmem, acc, stream); break;
            default: e = cudaErrorInvalidValue;  // relin32_applicable admits K = 1, 2, 4, 8 only
        }
        if (e != cudaSuccess) return e;
    }
    if constexpr (LOGN <= 13) {
        // fused inverse transform + reconstruction: 43.1 -> 41.4 ms per step of the headline network (two CTAs of 8 warps per SM hold it back)
        if (c.S3 == 3) {
            static DeviceOnce once3;
            const int smem3 = 3 * Pl::SMEM_WORDS * 4;
            if (once3.first()) {
                cudaFuncSetAttribute(r32_intt_crt_kernel<LOGN, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem3);
                cudaFuncSetAttribute(r32_intt_crt_kernel<LOGN, 3>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            }
            r32_intt_crt_kernel<LOGN, 3><<<(unsigned)(count * 2 * K), Pl::THREADS, smem3, stream>>>(dP, r.dc, acc, in3, out);
            return cudaGetLastError();
        }
    }
    r32_intt_kernel<LOGN><<<(unsigned)(count * 2 * K * c.S3), Pl::THREADS, smem, stream>>>(r.dc, acc);
    const dim3 gc((unsigned)(count * 2 * K), (unsigned)(N / 512));
    if (c.S3 == 2) r32_crt_kernel<2><<<gc, 256, 0, stream>>>(dP, r.dc, acc, in3, out);
    else if (c.S3 == 3) r32_crt_kernel<3><<<gc, 256, 0, stream>>>(dP, r.dc, acc, in3, out);
    else r32_crt_kernel<4><<<gc, 256, 0, stream>>>(dP, r.dc, acc, in3, out);
    return cudaGetLastError();
}

template <int LOGN>
cudaError_t build_keys_t(const uint64_t *coef, const KeyMap &km, const Relin32 &r, int K, cudaStream_t stream) {
    configure32<LOGN>();
    r32_key_kernel<LOGN><<<(unsigned)((long)r.c.D * 2 * K * r.c.S3), Plan32<LOGN>::THREADS, Plan32<LOGN>::SMEM_WORDS * 4, stream>>>(
        coef, km, r.dc, K, r.keys);
    return cudaGetLastError();
}

}  // namespace

bool relin32_applicable(int n, int K, const uint64_t *q, const int *digits, int dbc, Relin32Consts &c) {
    if (n < 1024 || n > 16384 || (n & (n - 1))) return false;
    if (dbc < 1 || dbc > 16) return false;                // digits travel as 16-bit planes
    if (K != 1 && K != 2 && K != 4 && K != 8) return false;
    c = Relin32Consts{};
    c.dbc = dbc;
    uint64_t qmax = 0;
    for (int i = 0; i < K; i++) {
        if (q[i] > qmax) qmax = q[i];
        c.dfirst[i] = c.D;
        for (int k = 0; k < digits[i]; k++) {
            if (c.D >= 32) return false;
            c.dprime[c.D] = (unsigned char)i;
            c.dshift[c.D] = (unsigned char)(k * dbc);
            c.D++;
        }
    }
    if (c.D == 0) return false;
    // |W| <= D * n * (2^dbc - 1) * (qmax - 1); need 2|W| < P.  Work in log2 with a margin far above rounding error.
    const double need = 1.0 + std::log2((double)c.D) + std::log2((double)n) + (double)dbc + std::log2((double)qmax);
    double have = 0;
    for (int s = 0; s < R32_MAXP; s++) {
        have += std::log2((double)kAuxPrimes[s]);
        if (have > need + 1e-3 && s + 1 >= 2) { c.S3 = s + 1; break; }
    }
    if (c.S3 == 0) return false;
    for (int s = 0; s < c.S3; s++) {
        c.p[s] = kAuxPrimes[s];
        c.mu[s] = (uint64_t)((((unsigned __int128)1) << 64) / kAuxPrimes[s]);
        c.half[s] = (kAuxPrimes[s] - 1) / 2;
        for (int k = 0; k < s; k++) {
            c.ginv[s][k] = invm(kAuxPrimes[k] % kAuxPrimes[s], kAuxPrimes[s]);
            c.ginvp[s][k] = shoup_companion(c.ginv[s][k], kAuxPrimes[s]);
        }
    }
    for (int j = 0; j < K; j++) {
        unsigned __int128 prod = 1;
        for (int s = 0; s < c.S3; s++) {
            c.cmodq[j][s] = (uint64_t)prod;
            c.cmodq_sh[j][s] = (uint64_t)((prod << 64) / q[j]);
            prod = prod * kAuxPrimes[s] % q[j];
        }
        c.Pmodq[j] = (uint64_t)prod;
    }
    return true;
}

cudaError_t relin32_build(const DeviceParams *dP, int logn, int K, const uint64_t *q, const uint64_t *evk_dev, const long *key_off,
                          long total_polys, Relin32 &r, cudaStream_t stream) {
    (void)q;
    const int n = 1 << logn;
    Relin32Consts &c = r.c;
    // tables: (w, w') pairs in the reference's bit-reversed order, forward and inverse, per auxiliary prime
    std::vector<uint2> host((size_t)4 * c.S3 * n);  // per prime: w, iw, transposed last-pass w, transposed first-pass iw
    const int NG = n >> 5;
    KeyMap km{};
    for (int s = 0; s < c.S3; s++) {
        const uint32_t p = c.p[s];
        uint32_t psi = 0;
        for (uint32_t z = 2; z < 1000 && !psi; z++) {
            const uint32_t cand = powm(z, (p - 1) / (2u * n), p);
            if (powm(cand, n, p) == p - 1) psi = cand;  // psi^n = -1: order exactly 2n
        }
        if (!psi) return cudaErrorInvalidValue;
        const uint32_t psi_inv = invm(psi, p);
        uint32_t pw = 1, ipw = 1;
        uint2 *w = host.data() + (size_t)(4 * s) * n, *iw = w + n, *wl = iw + n, *iwl = wl + n;
        for (int i = 0; i < n; i++) {
            const uint32_t rv = bitrev32((uint32_t)i, logn);
            w[rv] = make_uint2(pw, shoup_companion(pw, p));
            iw[rv] = make_uint2(ipw, shoup_companion(ipw, p));
            pw = mulm(pw, psi, p);
            ipw = mulm(ipw, psi_inv, p);
        }
        km.ninv[s] = invm((uint32_t)n, p);
        // transposed pairs of the contiguous pass (see fwd_last32 / inv_first32): uint4 row r, group G at uint2 index 2*(r*NG+G)
        for (int G = 0; G < NG; G++) {
            wl[30 * NG + G] = w[NG + G];
            iwl[30 * NG + G] = iw[(n >> 5) + G];
            for (int st = 1; st < 5; st++)
                for (int l2 = 0; l2 < (1 << (st - 1)); l2++) {
                    const size_t at = 2 * ((size_t)((1 << (st - 1)) - 1 + l2) * NG + G);
                    wl[at] = w[((NG + G) << st) + 2 * l2];
                    wl[at + 1] = w[((NG + G) << st) + 2 * l2 + 1];
                }
            for (int st = 0; st < 4; st++)
                for (int l2 = 0; l2 < (1 << (3 - st)); l2++) {
                    const size_t at = 2 * ((size_t)(16 - (16 >> st) + l2) * NG + G);
                    const int idx = ((n >> 1) >> st) + (G << (4 - st)) + 2 * l2;
                    iwl[at] = iw[idx];
                    iwl[at + 1] = iw[idx + 1];
                }
        }
    }
    cudaError_t e = cudaMalloc((void **)&r.tables, host.size() * sizeof(uint2));
    if (e != cudaSuccess) return e;
    e = cudaMemcpyAsync(r.tables, host.data(), host.size() * sizeof(uint2), cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) return e;
    e = cudaStreamSynchronize(stream);  // `host` goes out of scope
    if (e != cudaSuccess) return e;
    for (int s = 0; s < c.S3; s++) {
        c.w[s] = r.tables + (size_t)(4 * s) * n;
        c.iw[s] = r.tables + (size_t)(4 * s + 1) * n;
        c.wl[s] = r.tables + (size_t)(4 * s + 2) * n;
        c.iwl[s] = r.tables + (size_t)(4 * s + 3) * n;
    }
    for (int i = 0; i < MAXK; i++) km.key_off[i] = key_off[i];
    e = cudaMalloc((void **)&r.dc, sizeof(Relin32Consts));
    if (e != cudaSuccess) return e;
    e = cudaMemcpyAsync(r.dc, &c, sizeof(Relin32Consts), cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) return e;
    // keys: coefficient form (inverse 64-bit NTT of a copy), then per auxiliary prime
    const size_t words = (size_t)total_polys * K * n;
    uint64_t *coef = nullptr;
    e = cudaMalloc((void **)&coef, words * 8);
    if (e != cudaSuccess) return e;
    e = cudaMalloc((void **)&r.keys, (size_t)c.S3 * c.D * 2 * K * n * 4);
    if (e != cudaSuccess) { cudaFree(coef); return e; }
    e = cudaMemcpyAsync(coef, evk_dev, words * 8, cudaMemcpyDeviceToDevice, stream);
    if (e == cudaSuccess) e = launch_ntt(dP, logn, coef, total_polys * K, 0, K, true, stream);
    if (e == cudaSuccess) {
        switch (logn) {
            case 10: e = build_keys_t<10>(coef, km, r, K, stream); break;
            case 11: e = build_keys_t<11>(coef, km, r, K, stream); break;
            case 12: e = build_keys_t<12>(coef, km, r, K, stream); break;
            case 13: e = build_keys_t<13>(coef, km, r, K, stream); break;
            case 14: e = build_keys_t<14>(coef, km, r, K, stream); break;
            default: e = cudaErrorInvalidValue;
        }
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    cudaFree(coef);
    return e;
}

void relin32_free(Relin32 &r) {
    if (r.keys) cudaFree(r.keys);
    if (r.tables) cudaFree(r.tables);
    if (r.dc) cudaFree(r.dc);
    r.dc = nullptr;
    r.keys = nullptr;
    r.tables = nullptr;
}

size_t relin32_scratch_bytes(int n, int K, const Relin32Consts &c) {
    return (size_t)c.D * c.S3 * n * 4 + (size_t)2 * K * c.S3 * n * 4 + (size_t)c.D * n * 2;
}

cudaError_t relin32_run(const DeviceParams *dP, int logn, int K, const Relin32 &r, const uint64_t *in3, uint64_t *out, long count,
                        void *scratch, cudaStream_t stream) {
    if (count <= 0) return cudaSuccess;
    switch (logn) {
        case 10: return run_t<10>(dP, K, r, in3, out, count, scratch, stream);
        case 11: return run_t<11>(dP, K, r, in3, out, count, scratch, stream);
        case 12: return run_t<12>(dP, K, r, in3, out, count, scratch, stream);
        case 13: return run_t<13>(dP, K, r, in3, out, count, scratch, stream);
        case 14: return run_t<14>(dP, K, r, in3, out, count, scratch, stream);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace crcnn
