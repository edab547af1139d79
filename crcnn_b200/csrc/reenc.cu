// See reenc.cuh.
#include "reenc.cuh"
#include "modarith.cuh"

namespace crcnn {

typedef unsigned __int128 u128h;

ReencConsts make_reenc_consts(const DeviceParams &d) {
    ReencConsts c{};
    c.n = d.n; c.K = d.K; c.t = d.t; c.half = d.half; c.gamma = REENC_GAMMA;
    c.tm = make_mod(d.t);
    c.gm = make_mod(REENC_GAMMA);
    auto prod_except = [&](int skip, const Mod &m) {
        uint64_t r = 1 % m.q;
        for (int i = 0; i < d.K; i++)
            if (i != skip) r = mulmod(r, d.tab[i].mod.q % m.q, m);
        return r;
    };
    for (int i = 0; i < d.K; i++) {
        const Mod &m = d.tab[i].mod;
        c.q[i] = m;
        const uint64_t tg = mulmod(d.t % m.q, REENC_GAMMA % m.q, m);          // plain_gamma_product_mod_coeff_array_, baseconverter.cpp:345-349
        c.dec_c[i] = mulmod(tg, d.inv_qhat[i], m);
        c.qhat_t[i] = prod_except(i, c.tm);                                  // baseconverter.cpp:315-323
        c.qhat_g[i] = prod_except(i, c.gm);
        c.delta[i] = d.delta[i];
        c.rho[i] = d.rho[i];
    }
    c.neg_inv_q_t = inv_mod(negmod(prod_except(-1, c.tm), c.tm.q), c.tm.q);    // baseconverter.cpp:325-335
    c.neg_inv_q_g = inv_mod(negmod(prod_except(-1, c.gm), c.gm.q), c.gm.q);
    c.inv_gamma_t = inv_mod(REENC_GAMMA % d.t, d.t);                          // baseconverter.cpp:337-343
    return c;
}

CrtConsts make_crt_consts(const uint64_t *moduli, int M, int own) {
    CrtConsts c{};
    c.M = M;
    uint64_t p = 1;
    for (int k = 0; k < M; k++) {
        c.tm[k] = make_mod(moduli[k]);
        c.prefix[k] = p;
        c.inv[k] = k ? inv_mod(p % moduli[k], moduli[k]) : 0;
        p *= moduli[k];
    }
    c.T = p; c.half = (p + 1) >> 1;
    c.t_own = moduli[own];
    return c;
}

// w[NB_WORDS] *= v
static void words_mul(uint64_t *w, uint64_t v) {
    u128h carry = 0;
    for (int j = 0; j < NB_WORDS; j++) {
        const u128h p = (u128h)w[j] * v + carry;
        w[j] = (uint64_t)p;
        carry = p >> 64;
    }
}

BudgetConsts make_budget_consts(const DeviceParams &d) {
    BudgetConsts c{};
    c.n = d.n; c.K = d.K;
    c.qw[0] = 1;
    for (int i = 0; i < d.K; i++) {
        const Mod &m = d.tab[i].mod;
        c.q[i] = m;
        c.c[i] = mulmod(d.t % m.q, d.inv_qhat[i], m);
        c.qhat[i][0] = 1;
        for (int j = 0; j < d.K; j++)
            if (j != i) words_mul(c.qhat[i], d.tab[j].mod.q);
        words_mul(c.qw, m.q);
    }
    // (q + 1) / 2: q is odd, so this is q / 2 rounded up = (q >> 1) + 1
    for (int j = 0; j < NB_WORDS; j++) c.half[j] = (c.qw[j] >> 1) | (j + 1 < NB_WORDS ? c.qw[j + 1] << 63 : 0);
    for (int j = 0; j < NB_WORDS && ++c.half[j] == 0; j++) {}
    for (int j = 0; j < NB_WORDS; j++)
        if (c.qw[j]) c.q_bits = 64 * j + 64 - __builtin_clzll(c.qw[j]);
    return c;
}

// ---------------------------------------------------------------------------------------------- decrypt
__global__ void __launch_bounds__(256)
dec_dot_kernel(const __grid_constant__ ReencConsts c, const uint64_t *__restrict__ ct, int ct_is_ntt, const uint64_t *__restrict__ sk,
               uint64_t *__restrict__ tmp, long total) {
    const long w = (long)blockIdx.x * 256 + threadIdx.x;
    if (w >= total) return;
    const int n = c.n, K = c.K;
    const int k = (int)(w % n), i = (int)((w / n) % K);
    const long cti = w / ((long)n * K);
    const Mod m = c.q[i];
    const uint64_t s = __ldg(sk + (long)i * n + k);
    if (ct_is_ntt) {
        const uint64_t *c0 = ct + (cti * 2 * K + i) * (long)n + k;
        tmp[w] = addmod(mulmod(__ldg(c0 + (long)K * n), s, m), __ldg(c0), m.q);
    } else {
        tmp[w] = mulmod(tmp[w], s, m);        // dyadic_product_coeffmod, decryptor.cpp:160
    }
}

// The K residues of c0 + c1 s at coefficient k of ciphertext cti -> the plaintext coefficient (decryptor.cpp:172-234)
__device__ __forceinline__ uint64_t dec_scale_coeff(const ReencConsts &c, const uint64_t *__restrict__ ct, const uint64_t *__restrict__ tmp,
                                                    long cti, int k) {
    const int n = c.n, K = c.K;
    Acc7 at = acc7_zero(), ag = acc7_zero();
    for (int i = 0; i < K; i++) {
        uint64_t d = __ldg(tmp + (cti * K + i) * (long)n + k);
        if (ct) d += __ldg(ct + (cti * 2 * K + i) * (long)n + k);      // lazy "+ c0" (decryptor.cpp:181-183): < 2q, the product below reduces it
        const uint64_t v = mulmod(d, c.dec_c[i], c.q[i]);              // x |gamma t|_qi (:186) and x (q/q_i)^-1 (baseconverter.cpp:767), both canonical
        mac7(at, v, c.qhat_t[i]);                                      // baseconverter.cpp:781-792
        mac7(ag, v, c.qhat_g[i]);
    }
    const uint64_t a_t = mulmod(barrett128(acc7_value(at), c.tm), c.neg_inv_q_t, c.tm);   // decryptor.cpp:196-201
    const uint64_t a_g = mulmod(barrett128(acc7_value(ag), c.gm), c.neg_inv_q_g, c.gm);
    uint64_t r;
    if (a_g > (c.gamma >> 1)) r = addmod(a_t, reduce64(c.gamma - a_g, c.tm), c.t);          // :207-217
    else r = submod(a_t, reduce64(a_g, c.tm), c.t);                                         // :219-224
    return mulmod(r, c.inv_gamma_t, c.tm);                                                  // :233-234
}

// One thread per coefficient: plain[count][n]
__global__ void __launch_bounds__(128)
dec_scale_kernel(const __grid_constant__ ReencConsts c, const uint64_t *__restrict__ ct, const uint64_t *__restrict__ tmp,
                 uint64_t *__restrict__ plain, long total) {
    const long w = (long)blockIdx.x * 128 + threadIdx.x;
    if (w >= total) return;
    plain[w] = dec_scale_coeff(c, ct, tmp, w / c.n, (int)(w % c.n));
}

// One thread per slot: slots[count][96], slot j < 64 is coefficient j, slot j >= 64 coefficient n - 96 + j
__global__ void __launch_bounds__(128)
dec_scale_slots_kernel(const __grid_constant__ ReencConsts c, const uint64_t *__restrict__ ct, const uint64_t *__restrict__ tmp,
                       uint64_t *__restrict__ slots, long total) {
    const long w = (long)blockIdx.x * 128 + threadIdx.x;
    if (w >= total) return;
    const int j = (int)(w % REENC_SLOTS);
    slots[w] = dec_scale_coeff(c, ct, tmp, w / REENC_SLOTS, j < 64 ? j : c.n - REENC_SLOTS + j);
}

// x -= y when x >= y (NB_WORDS words each); returns whether it subtracted
__device__ __forceinline__ bool words_sub_if_ge(uint64_t (&x)[NB_WORDS], const uint64_t (&y)[NB_WORDS]) {
    uint64_t d[NB_WORDS], borrow = 0;
#pragma unroll
    for (int j = 0; j < NB_WORDS; j++) {
        const uint64_t yj = y[j] + borrow;
        const uint64_t nb = (uint64_t)(yj < borrow) | (uint64_t)(x[j] < yj);
        d[j] = x[j] - yj;
        borrow = nb;
    }
    if (borrow) return false;
#pragma unroll
    for (int j = 0; j < NB_WORDS; j++) x[j] = d[j];
    return true;
}

// One thread per coefficient: the K residues of c0 + c1 s -> bit length of the centred t (c0 + c1 s) mod q (decryptor.cpp:
// invariant_noise_budget), maximised over the ciphertext's n coefficients into bits[cti].  Every thread reaches the warp reduction
// (no early return); n is a multiple of 32 and blocks are 128 threads, so a warp never straddles two ciphertexts or the end.
__global__ void __launch_bounds__(128)
noise_bits_kernel(const __grid_constant__ BudgetConsts c, const uint64_t *__restrict__ ct, const uint64_t *__restrict__ tmp,
                  int *__restrict__ bits, long total) {
    const long w = (long)blockIdx.x * 128 + threadIdx.x;
    const int n = c.n, K = c.K;
    const long cti = w / n;
    int b = 0;
    if (w < total) {
        const int k = (int)(w % n);
        uint64_t x[NB_WORDS];
#pragma unroll
        for (int j = 0; j < NB_WORDS; j++) x[j] = 0;
#pragma unroll
        for (int i = 0; i < MAXK; i++) {
            if (i >= K) break;
            uint64_t d = __ldg(tmp + (cti * K + i) * (long)n + k);
            if (ct) d += __ldg(ct + (cti * 2 * K + i) * (long)n + k);   // lazy "+ c0": < 2 q_i, the product below reduces it
            const uint64_t a = mulmod(d, c.c[i], c.q[i]);              // [t y_i (q/q_i)^-1]_{q_i}  (baseconverter.cpp: compose)
            // x += a (q/q_i): q/q_i has at most K-1 nonzero words; the partial sum stays below K q < 2^(64 K + 3), so the carry out of
            // word K-1 lands in word K without overflowing it
            uint64_t carry = 0;
#pragma unroll
            for (int j = 0; j < MAXK; j++) {
                if (j >= K) break;
                const uint64_t lo = a * c.qhat[i][j], hi = __umul64hi(a, c.qhat[i][j]);
                uint64_t s = x[j] + lo;
                uint64_t cy = s < lo;
                s += carry;
                cy += s < carry;
                x[j] = s;
                carry = hi + cy;              // a * qhat + x + carry < 2^128: no overflow
            }
#pragma unroll
            for (int j = 1; j < NB_WORDS; j++)
                if (j == K) x[j] += carry;
        }
        // x < K q: at most K - 1 subtractions of q bring it into [0, q)  (compose's final modulo_uint_inplace)
#pragma unroll 1
        for (int r = 1; r < K; r++)
            if (!words_sub_if_ge(x, c.qw)) break;
        // |x| = q - x for x >= (q + 1) / 2 (poly_infty_norm_coeffmod)
        uint64_t h[NB_WORDS];
#pragma unroll
        for (int j = 0; j < NB_WORDS; j++) h[j] = x[j];
        if (words_sub_if_ge(h, c.half)) {
            uint64_t borrow = 0;
#pragma unroll
            for (int j = 0; j < NB_WORDS; j++) {
                const uint64_t xj = x[j] + borrow;
                const uint64_t nb = (uint64_t)(xj < borrow) | (uint64_t)(c.qw[j] < xj);
                x[j] = c.qw[j] - xj;
                borrow = nb;
            }
        }
#pragma unroll
        for (int j = 0; j < NB_WORDS; j++)
            if (x[j]) b = 64 * j + 64 - __clzll((long long)x[j]);     // get_significant_bit_count_uint
    }
    // the bit length of the maximum is the maximum of the bit lengths: no multi-word maximum is needed
    b = __reduce_max_sync(0xffffffffu, b);
    if ((threadIdx.x & 31) == 0 && w < total) atomicMax(bits + cti, b);
}

// ---------------------------------------------------------------------------------------------- decode -> float -> encode
// IEEE double arithmetic with explicit round-to-nearest intrinsics: no fused multiply-add may change a digit.

// BalancedFractionalEncoder::decode / BalancedEncoder::decode_int64 (SEAL/seal/encoder.cpp) under plain modulus t with
// coeff_neg_threshold_ half = (t + 1) >> 1; coef(j) is slot j of the plaintext: coefficient j for j < 64, coefficient n - 96 + j above.
// The single-modulus path reads a decrypted plaintext, the CRT ensembles compose each coefficient from the instances' residues.
template <class Coef>
__device__ __forceinline__ double decode_fractional(uint64_t t, uint64_t half, const Coef &coef) {
    long long ip = 0;
    for (int i = 63; i >= 0; i--) {
        const uint64_t cf = coef(i);
        const long long v = cf >= half ? -(long long)(t - cf) : (long long)cf;
        ip = (long long)((unsigned long long)ip * 3ull) + v;
    }
    double frac = 0;
    for (int i = 0; i < 32; i++) {
        const uint64_t cf = coef(64 + i);
        const long long v = cf >= half ? -(long long)(t - cf) : (long long)cf;
        frac = __ddiv_rn(__dadd_rn(frac, (double)v), 3.0);
    }
    return __dadd_rn((double)ip, -frac);
}

__device__ __forceinline__ double decode_plain(const ReencConsts &c, const uint64_t *p) {
    const int tail = c.n - REENC_SLOTS;
    return decode_fractional(c.t, c.half, [p, tail](int j) { return p[j < 64 ? j : tail + j]; });
}

// BalancedFractionalEncoder::encode of value (the restatement of params.cpp: encode_fractional_sparse, checked against the oracle):
// s[96] = coefficients 0..63 and n-32..n-1
__device__ __forceinline__ void encode_fractional(uint64_t t, double value, uint64_t *s) {
    for (int i = 0; i < REENC_SLOTS; i++) s[i] = 0;
    const long long ipart = (long long)round(value);
    {
        const bool ng = ipart < 0;
        unsigned long long mag = ng ? (unsigned long long)(-ipart) : (unsigned long long)ipart;
        for (int pos = 0; mag && pos < 64; pos++) {
            const unsigned long long rem = mag % 3;
            int digit = rem == 0 ? 0 : (rem == 1 ? 1 : -1);
            mag = (mag + 1) / 3;
            if (ng) digit = -digit;
            if (digit) s[pos] = digit > 0 ? 1 : t - 1;
        }
    }
    double fr = __dadd_rn(value, -(double)ipart);
    if (fr != 0) {
        for (int i = 0; i < 32; i++) {
            fr = __dmul_rn(fr, 3.0);
            const int sign = fr >= 0 ? 1 : -1;
            const long long digit = (long long)(sign * ceil(__dadd_rn(fabs(fr), -0.5)));
            fr = __dadd_rn(fr, -(double)digit);
            if (digit) s[64 + 31 - i] = digit > 0 ? t - (uint64_t)digit : (uint64_t)(-digit);     // coefficient n-1-i
        }
    }
}

__global__ void __launch_bounds__(128)
reencode_kernel(const __grid_constant__ ReencConsts c, const uint64_t *__restrict__ plain, uint64_t *__restrict__ slots,
                float *__restrict__ values, long count) {
    const long cti = (long)blockIdx.x * 128 + threadIdx.x;
    if (cti >= count) return;
    const float f = (float)decode_plain(c, plain + cti * (long)c.n);          // floatCube (CrCNN/src/globals.h:16): the value passes through a float
    if (values) values[cti] = f;
    encode_fractional(c.t, (double)f, slots + cti * REENC_SLOTS);
}

// encryptImage's encoding: fraencoder->encode(image[z][x][y]), the float promoted to double (CrCNN/src/globals.cpp:207-226)
__global__ void __launch_bounds__(128)
encode_values_kernel(const __grid_constant__ ReencConsts c, const float *__restrict__ values, uint64_t *__restrict__ slots, long count) {
    const long cti = (long)blockIdx.x * 128 + threadIdx.x;
    if (cti >= count) return;
    encode_fractional(c.t, (double)values[cti], slots + cti * REENC_SLOTS);
}

// decryptImage's decoding: (float) fraencoder->decode(plain) (CrCNN/src/globals.cpp:127-142)
__global__ void __launch_bounds__(128)
decode_values_kernel(const __grid_constant__ ReencConsts c, const uint64_t *__restrict__ plain, float *__restrict__ values, long count) {
    const long cti = (long)blockIdx.x * 128 + threadIdx.x;
    if (cti >= count) return;
    values[cti] = (float)decode_plain(c, plain + cti * (long)c.n);
}

// ---------------------------------------------------------------------------------------------- CRT ensembles
// Garner's recombination of slot j of ciphertext cti from slots[M][total][96]
__device__ __forceinline__ uint64_t crt_compose(const CrtConsts &c, const uint64_t *__restrict__ slots, long total, long cti, int j) {
    const long stride = total * REENC_SLOTS, at = cti * REENC_SLOTS + j;
    uint64_t x = __ldg(slots + at);
    for (int k = 1; k < c.M; k++) {
        const Mod &m = c.tm[k];
        const uint64_t v = mulmod(submod(__ldg(slots + k * stride + at), reduce64(x, m), m.q), c.inv[k], m);
        x += v * c.prefix[k];                 // x < t_1 ... t_k <= T
    }
    return x;
}

__device__ __forceinline__ double crt_decode(const CrtConsts &c, const uint64_t *slots, long total, long cti) {
    return decode_fractional(c.T, c.half, [&](int j) { return crt_compose(c, slots, total, cti, j); });
}

// decryptImage's decoding under T: (float) FractionalEncoder::decode of the composed plaintext
__global__ void __launch_bounds__(128)
crt_decode_values_kernel(const __grid_constant__ CrtConsts c, const uint64_t *__restrict__ slots, float *__restrict__ values, long count) {
    const long cti = (long)blockIdx.x * 128 + threadIdx.x;
    if (cti >= count) return;
    values[cti] = (float)crt_decode(c, slots, count, cti);
}

// reencode_kernel's step for an ensemble: decode under T, through a float (floatCube), encode under this instance's t
__global__ void __launch_bounds__(128)
crt_reencode_kernel(const __grid_constant__ CrtConsts c, const uint64_t *__restrict__ slots, long total, long first,
                    uint64_t *__restrict__ out, long count) {
    const long r = (long)blockIdx.x * 128 + threadIdx.x;
    if (r >= count) return;
    const float f = (float)crt_decode(c, slots, total, first + r);
    encode_fractional(c.t_own, (double)f, out + r * REENC_SLOTS);
}

// ---------------------------------------------------------------------------------------------- encrypt
// Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3"): counter = (ciphertext, coefficient), key = seed
__device__ __forceinline__ void philox4x32(uint32_t (&ctr)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * ctr[0], p1 = (uint64_t)0xCD9E8D57u * ctr[2];
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ ctr[1] ^ k0, n2 = (uint32_t)(p0 >> 32) ^ ctr[3] ^ k1;
        ctr[1] = (uint32_t)p1; ctr[3] = (uint32_t)p0; ctr[0] = n0; ctr[2] = n2;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

__global__ void __launch_bounds__(256)
enc_sample_kernel(const __grid_constant__ ReencConsts c, uint64_t seed, long first_ct, double sigma, double max_dev,
                  const int8_t *__restrict__ given, uint64_t *__restrict__ U, int8_t *__restrict__ e, long total) {
    const long w = (long)blockIdx.x * 256 + threadIdx.x;
    if (w >= total) return;
    const int n = c.n, K = c.K;
    const int k = (int)(w % n);
    const long cti = w / n;
    int u, e0, e1;
    if (given) {
        u = given[(cti * 3 + 0) * (long)n + k]; e0 = given[(cti * 3 + 1) * (long)n + k]; e1 = given[(cti * 3 + 2) * (long)n + k];
    } else {
        // u uniform in {-1, 0, 1} (Encryptor::set_poly_coeffs_zero_one_negone, encryptor.cpp:202-239); e0, e1 a normal sample of
        // standard deviation sigma, redrawn while beyond max_dev, truncated toward zero (set_poly_coeffs_normal :241-287,
        // util/clipnormal.cpp)
        const uint64_t gct = (uint64_t)(first_ct + cti);
        bool ok = false;
        u = e0 = e1 = 0;
        for (uint32_t attempt = 0; attempt < 16 && !ok; attempt++) {
            uint32_t ctr[4] = {(uint32_t)gct, (uint32_t)(gct >> 32), (uint32_t)k, attempt};
            philox4x32(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
            u = (int)(((uint64_t)ctr[0] * 3u) >> 32) - 1;       // multiply-shift map of 32 uniform bits onto {-1, 0, 1}: bias below 2^-32
            const double u1 = ((double)ctr[1] + 0.5) * (1.0 / 4294967296.0), u2 = ((double)ctr[2] + 0.5) * (1.0 / 4294967296.0);
            const double rad = sqrt(-2.0 * log(u1)) * sigma;
            double sn, cs;
            sincospi(2.0 * u2, &sn, &cs);
            const double z0 = rad * cs, z1 = rad * sn;
            ok = fabs(z0) <= max_dev && fabs(z1) <= max_dev;
            e0 = (int)z0; e1 = (int)z1;
        }
    }
    for (int i = 0; i < K; i++) U[(cti * K + i) * (long)n + k] = u > 0 ? 1 : (u < 0 ? c.q[i].q - 1 : 0);
    e[(cti * 2 + 0) * (long)n + k] = (int8_t)e0;
    e[(cti * 2 + 1) * (long)n + k] = (int8_t)e1;
}

__global__ void __launch_bounds__(256)
enc_mul_kernel(const __grid_constant__ ReencConsts c, const uint64_t *__restrict__ U, const uint64_t *__restrict__ pk,
               uint64_t *__restrict__ out, long total) {
    const long w = (long)blockIdx.x * 256 + threadIdx.x;    // over count * K * n
    if (w >= total) return;
    const int n = c.n, K = c.K;
    const int k = (int)(w % n), i = (int)((w / n) % K);
    const long cti = w / ((long)n * K);
    const Mod m = c.q[i];
    const uint64_t un = __ldg(U + w);
    out[((cti * 2 + 0) * K + i) * (long)n + k] = mulmod(un, __ldg(pk + ((long)0 * K + i) * n + k), m);    // ntt_double_multiply_poly_nttpoly
    out[((cti * 2 + 1) * K + i) * (long)n + k] = mulmod(un, __ldg(pk + ((long)1 * K + i) * n + k), m);
}

__global__ void __launch_bounds__(256)
enc_finish_kernel(const __grid_constant__ ReencConsts c, const uint64_t *__restrict__ slots, const int8_t *__restrict__ e,
                  uint64_t *__restrict__ out, long total) {
    const long w = (long)blockIdx.x * 256 + threadIdx.x;    // over count * n
    if (w >= total) return;
    const int n = c.n, K = c.K;
    const int k = (int)(w % n);
    const long cti = w / n;
    uint64_t pm = 0;                                         // plaintext coefficient k of this ciphertext
    if (k < 64) pm = __ldg(slots + cti * REENC_SLOTS + k);
    else if (k >= n - 32) pm = __ldg(slots + cti * REENC_SLOTS + 64 + (k - (n - 32)));
    const int e0 = e[(cti * 2 + 0) * (long)n + k], e1 = e[(cti * 2 + 1) * (long)n + k];
    for (int i = 0; i < K; i++) {
        const Mod m = c.q[i];
        uint64_t *p0 = out + ((cti * 2 + 0) * K + i) * (long)n + k, *p1 = p0 + (long)K * n;
        uint64_t v0 = *p0;
        if (pm) {                                            // Encryptor::preencrypt, encryptor.cpp:168-200
            U128 z = mul128(c.delta[i], pm);
            if (pm >= c.half) add128_64(z, c.rho[i]);
            v0 = addmod(v0, barrett128(z, m), m.q);
        }
        const uint64_t n0 = e0 > 0 ? (uint64_t)e0 : (e0 < 0 ? m.q - (uint64_t)(-e0) : 0);
        const uint64_t n1 = e1 > 0 ? (uint64_t)e1 : (e1 < 0 ? m.q - (uint64_t)(-e1) : 0);
        *p0 = addmod(n0, v0, m.q);
        *p1 = addmod(n1, *p1, m.q);
    }
}

static unsigned blocks(long total, int per) { return (unsigned)((total + per - 1) / per); }

cudaError_t launch_dec_dot(const ReencConsts &c, const uint64_t *ct, int ct_is_ntt, const uint64_t *sk, uint64_t *tmp, long count, cudaStream_t s) {
    const long total = count * c.K * (long)c.n;
    if (total <= 0) return cudaSuccess;
    dec_dot_kernel<<<blocks(total, 256), 256, 0, s>>>(c, ct, ct_is_ntt, sk, tmp, total);
    return cudaGetLastError();
}
cudaError_t launch_dec_scale(const ReencConsts &c, const uint64_t *ct, const uint64_t *tmp, uint64_t *plain, long count, cudaStream_t s) {
    const long total = count * (long)c.n;
    if (total <= 0) return cudaSuccess;
    dec_scale_kernel<<<blocks(total, 128), 128, 0, s>>>(c, ct, tmp, plain, total);
    return cudaGetLastError();
}
cudaError_t launch_dec_scale_slots(const ReencConsts &c, const uint64_t *ct, const uint64_t *tmp, uint64_t *slots, long count, cudaStream_t s) {
    const long total = count * REENC_SLOTS;
    if (total <= 0) return cudaSuccess;
    dec_scale_slots_kernel<<<blocks(total, 128), 128, 0, s>>>(c, ct, tmp, slots, total);
    return cudaGetLastError();
}
cudaError_t launch_noise_bits(const BudgetConsts &c, const uint64_t *ct, const uint64_t *tmp, int *bits, long count, cudaStream_t s) {
    const long total = count * (long)c.n;
    if (total <= 0) return cudaSuccess;
    if (c.n % 32) return cudaErrorInvalidValue;      // the warp reduction needs whole warps per ciphertext
    noise_bits_kernel<<<blocks(total, 128), 128, 0, s>>>(c, ct, tmp, bits, total);
    return cudaGetLastError();
}
cudaError_t launch_reencode(const ReencConsts &c, const uint64_t *plain, uint64_t *slots, float *values, long count, cudaStream_t s) {
    if (count <= 0) return cudaSuccess;
    reencode_kernel<<<blocks(count, 128), 128, 0, s>>>(c, plain, slots, values, count);
    return cudaGetLastError();
}
cudaError_t launch_encode_values(const ReencConsts &c, const float *values, uint64_t *slots, long count, cudaStream_t s) {
    if (count <= 0) return cudaSuccess;
    encode_values_kernel<<<blocks(count, 128), 128, 0, s>>>(c, values, slots, count);
    return cudaGetLastError();
}
cudaError_t launch_decode_values(const ReencConsts &c, const uint64_t *plain, float *values, long count, cudaStream_t s) {
    if (count <= 0) return cudaSuccess;
    decode_values_kernel<<<blocks(count, 128), 128, 0, s>>>(c, plain, values, count);
    return cudaGetLastError();
}
cudaError_t launch_crt_decode_values(const CrtConsts &c, const uint64_t *slots, float *values, long count, cudaStream_t s) {
    if (count <= 0) return cudaSuccess;
    crt_decode_values_kernel<<<blocks(count, 128), 128, 0, s>>>(c, slots, values, count);
    return cudaGetLastError();
}
cudaError_t launch_crt_reencode(const CrtConsts &c, const uint64_t *slots, long total, long first, uint64_t *out, long count, cudaStream_t s) {
    if (count <= 0) return cudaSuccess;
    crt_reencode_kernel<<<blocks(count, 128), 128, 0, s>>>(c, slots, total, first, out, count);
    return cudaGetLastError();
}
cudaError_t launch_enc_sample(const ReencConsts &c, uint64_t seed, long first_ct, double sigma, double max_dev, const int8_t *given,
                              uint64_t *U, int8_t *e, long count, cudaStream_t s) {
    const long total = count * (long)c.n;
    if (total <= 0) return cudaSuccess;
    enc_sample_kernel<<<blocks(total, 256), 256, 0, s>>>(c, seed, first_ct, sigma, max_dev, given, U, e, total);
    return cudaGetLastError();
}
cudaError_t launch_enc_mul(const ReencConsts &c, const uint64_t *U, const uint64_t *pk, uint64_t *out, long count, cudaStream_t s) {
    const long total = count * c.K * (long)c.n;
    if (total <= 0) return cudaSuccess;
    enc_mul_kernel<<<blocks(total, 256), 256, 0, s>>>(c, U, pk, out, total);
    return cudaGetLastError();
}
cudaError_t launch_enc_finish(const ReencConsts &c, const uint64_t *slots, const int8_t *e, uint64_t *out, long count, cudaStream_t s) {
    const long total = count * (long)c.n;
    if (total <= 0) return cudaSuccess;
    enc_finish_kernel<<<blocks(total, 256), 256, 0, s>>>(c, slots, e, out, total);
    return cudaGetLastError();
}

}  // namespace crcnn
