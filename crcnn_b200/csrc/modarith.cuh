// 64-bit modular arithmetic primitives shared by every kernel (and, compiled for the host, by
// tests/host_arith_test.cpp).  All functions are exact; results that the reference stores are
// canonical residues in [0, q), so "bit-identical to SEAL" reduces to mathematical equality
// (SURVEY.md section 0 item 5).  Moduli are <= 61 bits (coefficient primes <= 60 bits,
// SEAL/seal/util/defines.h:20; Bsk primes 61 bits, SEAL/seal/util/globals.cpp:321-340).
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define CRCNN_HD __host__ __device__ __forceinline__
#else
#define CRCNN_HD inline
#endif

namespace crcnn {

struct Mod {
    uint64_t q;   // modulus
    uint64_t r0;  // floor(2^128 / q), low word   (same constant as SmallModulus::const_ratio,
    uint64_t r1;  //                   high word   SEAL/seal/smallmodulus.cpp:62-73)
};

CRCNN_HD uint64_t mulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

struct U128 {
    uint64_t lo, hi;
};

CRCNN_HD U128 mul128(uint64_t a, uint64_t b) {
    U128 r;
    r.lo = a * b;
    r.hi = mulhi64(a, b);
    return r;
}

// a*a for a < 2^63 from three 32x32 partial products: a1^2 2^64 + 2 a0 a1 2^32 + a0^2 (2 a0 a1 < 2^64).
CRCNN_HD U128 sqr128(uint64_t a) {
    const uint64_t a0 = (uint32_t)a, a1 = a >> 32;
    const uint64_t lo = a0 * a0, mid = (a0 * a1) << 1, hi = a1 * a1;
    U128 r;
    r.lo = lo + (mid << 32);
    r.hi = hi + (mid >> 32) + (r.lo < lo);
    return r;
}

// acc += a*b (mod 2^128).  Callers bound the number of accumulated terms so this never wraps.
CRCNN_HD void mac128(U128 &acc, uint64_t a, uint64_t b) {
    uint64_t lo = a * b;
    uint64_t hi = mulhi64(a, b);
    acc.lo += lo;
    acc.hi += hi + (acc.lo < lo);
}

// Lazy multiply-accumulate with a split accumulator: `even` (128 bit) collects a0*b0 + a1*b1*2^64,
// `odd` (96 bit, weight 2^32) collects the cross products a0*b1 + a1*b0.  On the device every
// mad.lo.cc/madc.hi pair fuses into one IMAD.WIDE.U32 (carry-out) / IMAD.WIDE.U32.X (carry-in), so a
// 64x64+acc step is 4 IMAD.WIDE + 1 IADD3.X -- no explicit carry compares, no register shuffles.
// Capacity: `even` holds 2^(128 - 2*bits(q)) products like a plain 128-bit accumulator, `odd` far more.
struct Acc7 {
    uint32_t a0, a1, a2, a3;  // even accumulator, little endian
    uint32_t b0, b1, b2;      // odd accumulator (weight 2^32)
};

CRCNN_HD Acc7 acc7_zero() { return Acc7{0, 0, 0, 0, 0, 0, 0}; }

CRCNN_HD void mac7(Acc7 &c, uint64_t x, uint64_t w) {
#if defined(__CUDA_ARCH__)
    uint32_t x0 = (uint32_t)x, x1 = (uint32_t)(x >> 32), w0 = (uint32_t)w, w1 = (uint32_t)(w >> 32);
    asm("mad.lo.cc.u32 %0, %7, %9, %0;\n\t"
        "madc.hi.cc.u32 %1, %7, %9, %1;\n\t"
        "madc.lo.cc.u32 %2, %8, %10, %2;\n\t"
        "madc.hi.u32 %3, %8, %10, %3;\n\t"
        "mad.lo.cc.u32 %4, %7, %10, %4;\n\t"
        "madc.hi.cc.u32 %5, %7, %10, %5;\n\t"
        "addc.u32 %6, %6, 0;\n\t"
        "mad.lo.cc.u32 %4, %8, %9, %4;\n\t"
        "madc.hi.cc.u32 %5, %8, %9, %5;\n\t"
        "addc.u32 %6, %6, 0;\n\t"
        : "+r"(c.a0), "+r"(c.a1), "+r"(c.a2), "+r"(c.a3), "+r"(c.b0), "+r"(c.b1), "+r"(c.b2)
        : "r"(x0), "r"(x1), "r"(w0), "r"(w1));
#else
    typedef unsigned __int128 u128;
    uint64_t x0 = (uint32_t)x, x1 = x >> 32, w0 = (uint32_t)w, w1 = w >> 32;
    u128 even = ((u128)(((uint64_t)c.a3 << 32) | c.a2) << 64) | (((uint64_t)c.a1 << 32) | c.a0);
    even += (u128)(x0 * w0) + ((u128)(x1 * w1) << 64);
    u128 odd = ((u128)c.b2 << 64) | (((uint64_t)c.b1 << 32) | c.b0);
    odd += (u128)(x0 * w1) + (u128)(x1 * w0);
    c.a0 = (uint32_t)even; c.a1 = (uint32_t)(even >> 32); c.a2 = (uint32_t)(even >> 64); c.a3 = (uint32_t)(even >> 96);
    c.b0 = (uint32_t)odd; c.b1 = (uint32_t)(odd >> 32); c.b2 = (uint32_t)(odd >> 64);
#endif
}

// even + odd * 2^32 as a plain 128-bit value
CRCNN_HD U128 acc7_value(const Acc7 &c) {
    uint64_t lo = ((uint64_t)c.a1 << 32) | c.a0, hi = ((uint64_t)c.a3 << 32) | c.a2;
    uint64_t add_lo = (uint64_t)c.b0 << 32, add_hi = ((uint64_t)c.b2 << 32) | c.b1;
    U128 r;
    r.lo = lo + add_lo;
    r.hi = hi + add_hi + (r.lo < lo);
    return r;
}

CRCNN_HD Acc7 acc7_from(uint64_t v) { return Acc7{(uint32_t)v, (uint32_t)(v >> 32), 0, 0, 0, 0, 0}; }

CRCNN_HD void add128_64(U128 &acc, uint64_t v) {
    acc.lo += v;
    acc.hi += (acc.lo < v);
}

// Barrett reduction of a 128-bit value to [0, q): q_est = floor(z * floor(2^128/q) / 2^128)
// is floor(z/q) or one less, so a single conditional subtraction suffices (same bound as
// barrett_reduce_128, SEAL/seal/util/uintarithsmallmod.h:137-176).
CRCNN_HD uint64_t barrett128(U128 z, const Mod &m) {
    // word 2 of the 256-bit product z * r  (only bits [128,192) are needed)
    uint64_t carry = mulhi64(z.lo, m.r0);
    uint64_t t_lo = z.lo * m.r1;
    uint64_t t_hi = mulhi64(z.lo, m.r1);
    uint64_t s1 = t_lo + carry;
    uint64_t c1 = t_hi + (s1 < carry);
    uint64_t u_lo = z.hi * m.r0;
    uint64_t u_hi = mulhi64(z.hi, m.r0);
    uint64_t s2 = s1 + u_lo;
    uint64_t c2 = u_hi + (s2 < u_lo);
    uint64_t qest = z.hi * m.r1 + c1 + c2;
    uint64_t r = z.lo - qest * m.q;
    return r >= m.q ? r - m.q : r;
}

// x mod q for any 64-bit x: the high word of floor(2^128/q) is floor(2^64/q), so the quotient
// estimate is at most one short and one conditional subtraction finishes.
CRCNN_HD uint64_t reduce64(uint64_t x, const Mod &m) {
    uint64_t r = x - mulhi64(x, m.r1) * m.q;
    return r >= m.q ? r - m.q : r;
}

// x mod q for any 64-bit x when q = 2^k - delta with k >= 48 and delta < 2^27 (every SEAL coefficient prime and Bsk prime): one fold
// x = lo + hi 2^k = lo + hi delta (mod q), hi < 2^16 so hi delta < 2^43 is ONE 32x32 IMAD.WIDE, and lo + hi delta < 2^k + 2^43 < 2q,
// so one conditional subtraction gives the canonical residue -- the same value as reduce64.  shape_k = k, or 0 when q lacks the shape.
CRCNN_HD int reduce64_shape_k(uint64_t q) {
    int k = 0;
    for (uint64_t v = q; v; v >>= 1) k++;
    return (k >= 48 && k <= 63 && ((1ull << k) - q) < (1ull << 27)) ? k : 0;
}
CRCNN_HD uint64_t reduce64_shape(uint64_t x, uint64_t q, int k) {
    const uint32_t delta = (uint32_t)((1ull << k) - q), hi = (uint32_t)(x >> k);
    const uint64_t r = (x & ((1ull << k) - 1)) + (uint64_t)hi * delta;
    return r >= q ? r - q : r;
}

CRCNN_HD uint64_t mulmod(uint64_t a, uint64_t b, const Mod &m) { return barrett128(mul128(a, b), m); }

CRCNN_HD uint64_t addmod(uint64_t a, uint64_t b, uint64_t q) {
    uint64_t s = a + b;
    return s >= q ? s - q : s;
}
CRCNN_HD uint64_t submod(uint64_t a, uint64_t b, uint64_t q) { return a >= b ? a - b : a + q - b; }
CRCNN_HD uint64_t negmod(uint64_t a, uint64_t q) { return a ? q - a : 0; }

// Shoup / Harvey multiplication by a constant w with precomputed w' = floor(w * 2^64 / q):
// returns w*y mod q as a representative in [0, 2q) for any 64-bit y.
CRCNN_HD uint64_t mulshoup_lazy(uint64_t y, uint64_t w, uint64_t wp, uint64_t q) {
    uint64_t h = mulhi64(wp, y);
    return y * w - h * q;
}

// Cheaper Shoup product for the transforms: the quotient estimate drops the low partial products,
//   h' = wp1*y1 + hi32(wp1*y0) + hi32(wp0*y1)  in  {h-2, h-1, h},   h = floor(wp*y / 2^64),
// so the result  y*w - h'*q  (mod 2^64)  is w*y mod q as a representative in [0, 4q) for any 64-bit y
// (q < 2^62).  nq = 2^64 - q turns the subtraction into a multiply-add.  The two hi32 terms are taken as the high
// word of a mul.wide.u32 (IMAD.WIDE.U32, 2.17 clk per warp instruction on the multiplier pipe) rather than
// mul.hi.u32 (IMAD.HI, 4 clk; profiles/r01_pipe_probe.txt) -- the same value: 5 IMAD.WIDE + 4 IMAD and two carry
// adds, against 6 IMAD.WIDE + 5 IMAD and ~9 adds for the exact form.
CRCNN_HD uint64_t mulshoup_lazy4(uint64_t y, uint64_t w, uint64_t wp, uint64_t nq) {
#if defined(__CUDA_ARCH__)
    uint32_t y0 = (uint32_t)y, y1 = (uint32_t)(y >> 32), p0 = (uint32_t)wp, p1 = (uint32_t)(wp >> 32);
    uint32_t w0 = (uint32_t)w, w1 = (uint32_t)(w >> 32), n0 = (uint32_t)nq, n1 = (uint32_t)(nq >> 32);
    uint32_t a, b, h0, h1, r0, r1;
    uint64_t wa, wb;
    asm("mul.wide.u32 %0, %2, %3;\n\t"
        "mul.wide.u32 %1, %4, %5;\n\t"
        : "=l"(wa), "=l"(wb) : "r"(p1), "r"(y0), "r"(p0), "r"(y1));
    a = (uint32_t)(wa >> 32);
    b = (uint32_t)(wb >> 32);
    asm("mad.lo.cc.u32 %0, %2, %3, %4;\n\t"
        "madc.hi.u32 %1, %2, %3, 0;\n\t"
        "add.cc.u32 %0, %0, %5;\n\t"
        "addc.u32 %1, %1, 0;\n\t"
        : "=r"(h0), "=r"(h1) : "r"(p1), "r"(y1), "r"(a), "r"(b));
    asm("mul.lo.u32 %0, %2, %3;\n\t"
        "mul.hi.u32 %1, %2, %3;\n\t"
        "mad.lo.cc.u32 %0, %4, %5, %0;\n\t"
        "madc.hi.u32 %1, %4, %5, %1;\n\t"
        "mad.lo.u32 %1, %2, %6, %1;\n\t"
        "mad.lo.u32 %1, %7, %3, %1;\n\t"
        "mad.lo.u32 %1, %4, %8, %1;\n\t"
        "mad.lo.u32 %1, %9, %5, %1;\n\t"
        : "=&r"(r0), "=&r"(r1) : "r"(y0), "r"(w0), "r"(h0), "r"(n0), "r"(w1), "r"(y1), "r"(n1), "r"(h1));
    return ((uint64_t)r1 << 32) | r0;
#else
    uint64_t y0 = (uint32_t)y, y1 = y >> 32, p0 = (uint32_t)wp, p1 = wp >> 32;
    uint64_t h = p1 * y1 + ((p1 * y0) >> 32) + ((p0 * y1) >> 32);
    return y * w + h * nq;
#endif
}

// ------------------------------------------------------------------------------------------------------------
// Reduction of the 13 weight-class sums of the limb-split GEMM (tcn_mac.cuh) for primes of SEAL's shape
// q = 2^k - delta (SEAL/seal/util/globals.cpp:50-74: the 54/55-bit primes have delta < 2^25), without forming the
// 128-bit integer and without a generic Barrett step:  z = sum_w S_w 2^(8w) (+ bias)  ->  z mod q in [0, q).
//   La, Lb, Ha, Hb = the classes 0-3, 4-6, 7-10, 11-12 as four sums of weight 2^0, 2^32, 2^56, 2^88 (the
//   multiply-adds by 2^8, 2^16, 2^24 take their factor from a run-time operand, so each is ONE IMAD.WIDE instead
//   of shifts and carry chains);  2^56 = T (mod q) with T = 2^(56-k) delta < 2^28 folds the upper two into the
//   lower two:   z = [La + Ha0 T] + 2^32 [Lb + Ha1 T + Hb0 T] + 2^64 [Hb1 T]   (< 2^100);
//   the bits above k fold through delta twice (67 bits, then < 2q; the bias joins in between), one conditional
//   subtraction.  Every step is an identity mod q and the result is canonical, so it equals
//   barrett128(tcn_combine(S)) (+ bias mod q) bit for bit; host_selftest.cpp checks it against unsigned __int128.
struct TcnFold {
    uint32_t T;           // 2^56 mod q
    uint32_t delta;       // 2^k - q
    uint32_t sh, mask;    // k - 32, 2^(k-32) - 1
    uint32_t c8, c16, c24;
    uint32_t ok;          // 0: this prime does not have the shape (the kernels then take the generic path)
    uint32_t ok7;         // tcn7_fold_reduce is exact for this prime (seven-class sums of the pre-shifted GEMM)
};

// worst case of tcn7_fold_reduce (below) for q = 2^k - delta: every class sum 2^31 - 1, bias q - 1
inline bool tcn7_fold_bound(uint64_t q, int k, uint64_t delta) {
    typedef unsigned __int128 u128;
    const u128 one = 1, cmax = 0x7fffffffu;
    u128 z = 0;
    for (int a = 6; a >= 0; a--) z = (z << 8) + cmax;
    const u128 h = z >> k;
    const u128 v = h * delta + ((one << k) - 1) + (q - 1);
    if (h >> 32 || v >> 64) return false;
    return (v >> k) * delta + ((one << k) - 1) < 2 * (u128)q;
}

// Worst-case magnitudes of every intermediate for S_w <= 2^31 - 1 and bias <= q - 1, checked numerically.
inline TcnFold tcn_fold_make(uint64_t q) {
    typedef unsigned __int128 u128;
    TcnFold f{};
    int k = 0;
    for (uint64_t v = q; v; v >>= 1) k++;
    if (k < 48 || k > 56) return f;
    const uint64_t delta = (1ull << k) - q;
    if (delta == 0 || delta >> 28) return f;
    const u128 T = (u128)delta << (56 - k);
    if (T >> 32 || T >= q) return f;
    const u128 one = 1, smax = 0x7fffffffu, w32 = 0xffffffffu;
    const u128 La = smax * (1 + (one << 8) + (one << 16) + (one << 24)), Lb = smax * (1 + (one << 8) + (one << 16));
    const u128 Ha = La, Hb = smax * (1 + (one << 8));
    const u128 a = w32 * T + La, b = (Ha >> 32) * T + Lb + w32 * T, e = (Hb >> 32) * T;
    if (a >> 64 || b >> 64 || e >> 60) return f;
    const u128 y = a + (b << 32) + (e << 64);                   // < 2^101
    const u128 h1 = (y >> k) >> 32;
    const u128 v = w32 * delta + ((one << k) - 1) + (q - 1), w = h1 * delta;
    if (h1 >> 32 || v >> 64 || w >> 62) return f;
    const u128 V = v + (w << 32);
    const u128 g = V >> k;
    if (V >> 96 || g >> 32) return f;
    if (g * delta + ((one << k) - 1) >= 2 * (u128)q) return f;
    f.T = (uint32_t)T; f.delta = (uint32_t)delta; f.sh = (uint32_t)(k - 32); f.mask = (1u << (k - 32)) - 1;
    f.c8 = 1u << 8; f.c16 = 1u << 16; f.c24 = 1u << 24; f.ok = 1;
    f.ok7 = tcn7_fold_bound(q, k, delta) ? 1 : 0;
    return f;
}

CRCNN_HD uint32_t tcn_shr64(uint32_t lo, uint32_t hi, uint32_t sh) {   // low word of (hi:lo) >> sh, 0 < sh < 32
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, sh);
#else
    return (lo >> sh) | (hi << (32 - sh));
#endif
}

// s[w] = class sum S_w (< 2^31), bias < q (0 when there is none)
CRCNN_HD uint64_t tcn_fold_reduce(const uint32_t (&s)[13], uint64_t bias, const TcnFold &f, uint64_t q) {
    const uint64_t La = (uint64_t)s[3] * f.c24 + ((uint64_t)s[2] * f.c16 + ((uint64_t)s[1] * f.c8 + s[0]));
    const uint64_t Lb = (uint64_t)s[6] * f.c16 + ((uint64_t)s[5] * f.c8 + s[4]);
    const uint64_t Ha = (uint64_t)s[10] * f.c24 + ((uint64_t)s[9] * f.c16 + ((uint64_t)s[8] * f.c8 + s[7]));
    const uint64_t Hb = (uint64_t)s[12] * f.c8 + s[11];
    const uint64_t a = (uint64_t)(uint32_t)Ha * f.T + La;
    const uint64_t b = (uint64_t)(uint32_t)Hb * f.T + ((Ha >> 32) * f.T + Lb);
    const uint64_t e = (Hb >> 32) * f.T;
    // y = a + 2^32 b + 2^64 e  as words y0..y3
    const uint32_t y0 = (uint32_t)a;
    const uint64_t m1 = (a >> 32) + (uint32_t)b;
    const uint32_t y1 = (uint32_t)m1;
    const uint64_t m2 = (b >> 32) + (uint64_t)(uint32_t)e + (m1 >> 32);
    const uint32_t y2 = (uint32_t)m2;
    const uint32_t y3 = (uint32_t)(e >> 32) + (uint32_t)(m2 >> 32);
    // first fold of the bits above k, bias added: V = v + 2^32 w
    const uint32_t h0 = tcn_shr64(y1, y2, f.sh), h1 = tcn_shr64(y2, y3, f.sh);
    const uint64_t l = ((uint64_t)(y1 & f.mask) << 32) | y0;
    const uint64_t v = (uint64_t)h0 * f.delta + l + bias;
    const uint64_t w = (uint64_t)h1 * f.delta;
    const uint64_t m3 = (v >> 32) + (uint32_t)w;
    const uint32_t V1 = (uint32_t)m3, V2 = (uint32_t)(w >> 32) + (uint32_t)(m3 >> 32);
    // second fold
    const uint32_t g = tcn_shr64(V1, V2, f.sh);
    const uint64_t lo = ((uint64_t)(V1 & f.mask) << 32) | (uint32_t)v;
    const uint64_t r = (uint64_t)g * f.delta + lo;
    return r >= q ? r - q : r;
}

// ------------------------------------------------------------------------------------------------------------
// Reduction of the SEVEN accumulator classes of the pre-shifted limb-split GEMM (tcn_mac.cuh: the weights are staged as
// W'_b = W 2^(8b) mod q, so every product lands in class a = weight byte and z = sum_a C_a 2^(8a)).  C_a < 2^31 gives
// z < 2^80 = 2^(48+32): for 48 <= k <= 56 the bits above k are ONE word h, and two folds through delta (the bias joins the
// first) leave r < 2q.  tcn_fold_make checks the worst case per prime (TcnFold::ok7); the result is canonical, so it equals
// (z + bias) mod q bit for bit (host_selftest.cpp checks it against unsigned __int128).
// C[a] = class sum of weight byte a (< 2^31), bias < q (0 when there is none)
CRCNN_HD uint64_t tcn7_fold_reduce(const uint32_t (&C)[7], uint64_t bias, const TcnFold &f, uint64_t q) {
    const uint64_t La = (uint64_t)C[3] * f.c24 + ((uint64_t)C[2] * f.c16 + ((uint64_t)C[1] * f.c8 + C[0]));   // weight 2^0, < 2^56
    const uint64_t Lb = (uint64_t)C[6] * f.c16 + ((uint64_t)C[5] * f.c8 + C[4]);                             // weight 2^32, < 2^48
    const uint64_t m1 = (La >> 32) + (uint32_t)Lb;
    const uint32_t y0 = (uint32_t)La, y1 = (uint32_t)m1, y2 = (uint32_t)(Lb >> 32) + (uint32_t)(m1 >> 32);
    const uint32_t h = tcn_shr64(y1, y2, f.sh);                                   // z >> k: one word since z < 2^(k+32)
    const uint64_t v = (uint64_t)h * f.delta + ((((uint64_t)(y1 & f.mask)) << 32) | y0) + bias;
    const uint32_t vh = (uint32_t)(v >> 32);
    const uint64_t r = (uint64_t)(vh >> f.sh) * f.delta + ((((uint64_t)(vh & f.mask)) << 32) | (uint32_t)v);
    return r >= q ? r - q : r;
}

// The same 80-bit value as a U128, for the generic (Barrett) reduction
CRCNN_HD U128 tcn7_combine(const uint32_t (&C)[7]) {
    const uint64_t La = ((uint64_t)C[3] << 24) + (((uint64_t)C[2] << 16) + (((uint64_t)C[1] << 8) + C[0]));
    const uint64_t Lb = ((uint64_t)C[6] << 16) + (((uint64_t)C[5] << 8) + C[4]);
    const uint64_t m1 = (La >> 32) + (uint32_t)Lb;
    U128 z;
    z.lo = (m1 << 32) | (uint32_t)La;
    z.hi = (Lb >> 32) + (m1 >> 32);
    return z;
}

// ------------------------------------------------------------------------------------------------------------
// The same idea for ANY 128-bit value (the lazy sums of the BEHZ and relinearize kernels): z mod q for q = 2^k - delta, 54 <= k <= 61,
// delta < 2^27 -- every coefficient prime and every Bsk prime of SEAL 2.3.1 (SEAL/seal/util/globals.cpp:50-74, 321-340).  Three folds of
// the bits above k through delta (6 IMAD.WIDE in all, against 18 multiply-pipe instructions of barrett128) and one conditional
// subtraction; canonical result, so it equals barrett128(z, mod) bit for bit.  Used by the BEHZ kernels and the tensor products of
// `square` (kernels.cu: behz_reduce); host_selftest.cpp checks it against unsigned __int128 for every modulus of the context.
struct Fold128 {
    uint64_t q;
    uint32_t delta, sh, mask, ok;   // 2^k - q, k - 32, 2^(k-32) - 1
};

inline Fold128 fold128_make(uint64_t q) {
    typedef unsigned __int128 u128;
    Fold128 f{};
    f.q = q;
    int k = 0;
    for (uint64_t v = q; v; v >>= 1) k++;
    if (k < 54 || k > 61) return f;
    const uint64_t delta = (1ull << k) - q;
    if (delta == 0 || delta >> 27) return f;
    // worst cases: z = 2^128 - 1;  y = l + h delta  < 2^k + 2^(128-k) delta;  V = l' + h' delta;  r = l'' + g delta < 2q
    const u128 one = 1, zmax = ~(u128)0;
    const u128 y = ((one << k) - 1) + (zmax >> k) * delta;
    const u128 V = ((one << k) - 1) + (y >> k) * delta;
    const u128 g = V >> k;
    if (y >> 112 || (y >> k) >> 64 || V >> 96 || g >> 32) return f;
    if (g * delta + ((one << k) - 1) >= 2 * (u128)q) return f;
    f.delta = (uint32_t)delta; f.sh = (uint32_t)(k - 32); f.mask = (1u << (k - 32)) - 1; f.ok = 1;
    return f;
}

CRCNN_HD uint64_t reduce128_fold(U128 z, const Fold128 &f) {
    const uint32_t z0 = (uint32_t)z.lo, z1 = (uint32_t)(z.lo >> 32), z2 = (uint32_t)z.hi, z3 = (uint32_t)(z.hi >> 32);
    // fold 1: h = z >> k (three words), l = z mod 2^k;  y = l + h delta as words y0..y3
    const uint32_t h0 = tcn_shr64(z1, z2, f.sh), h1 = tcn_shr64(z2, z3, f.sh), h2 = z3 >> f.sh;
    const uint64_t l = ((uint64_t)(z1 & f.mask) << 32) | z0;
    const uint64_t t0 = (uint64_t)h0 * f.delta + l;
    const uint64_t u = (uint64_t)h1 * f.delta + (t0 >> 32);                 // weight 2^32
    const uint64_t u2 = (uint64_t)h2 * f.delta + (u >> 32);                 // weight 2^64
    const uint32_t y0 = (uint32_t)t0, y1 = (uint32_t)u, y2 = (uint32_t)u2, y3 = (uint32_t)(u2 >> 32);
    // fold 2: h' = y >> k (two words);  V = l' + h' delta as words V0..V2
    const uint32_t g0 = tcn_shr64(y1, y2, f.sh), g1 = tcn_shr64(y2, y3, f.sh);
    const uint64_t l2 = ((uint64_t)(y1 & f.mask) << 32) | y0;
    const uint64_t v = (uint64_t)g0 * f.delta + l2;
    const uint64_t w = (uint64_t)g1 * f.delta + (v >> 32);                  // weight 2^32
    const uint32_t V0 = (uint32_t)v, V1 = (uint32_t)w, V2 = (uint32_t)(w >> 32);
    // fold 3
    const uint32_t g = tcn_shr64(V1, V2, f.sh);
    const uint64_t l3 = ((uint64_t)(V1 & f.mask) << 32) | V0;
    const uint64_t r = (uint64_t)g * f.delta + l3;
    return r >= f.q ? r - f.q : r;
}

}  // namespace crcnn
