/* TEST INFRASTRUCTURE ONLY.  CPU restatement of Decryptor::invariant_noise_budget (SEAL 2.3.1, seal/decryptor.cpp) after the dot
 * product: given d = c0 + c1 s mod q_i in coefficient form (the dot product of Decryptor::decrypt, formed by tests/fv_keygen.py
 * with the oracle's transforms), it computes y = d t mod q_i (multiply_poly_scalar_coeffmod), x = BaseConverter::compose(y) in
 * [0, q) (util/baseconverter.cpp: sum_i [y_i (q/q_i)^-1]_{q_i} (q/q_i), reduced mod q after every term by add_uint_uint_mod), the
 * centred absolute value at (q + 1) / 2 (poly_infty_norm_coeffmod, util/polyarithmod.cpp), the maximum over the coefficients and
 * budget = max(0, bits(q) - bits(norm) - 1).  Multi-word integers in unsigned __int128 arithmetic, K <= 15. */
#include <stdint.h>
#include <string.h>

typedef unsigned __int128 u128;
#define MAXK 15
#define NBW (MAXK + 1)

static uint64_t mulmod(uint64_t a, uint64_t b, uint64_t q) { return (uint64_t)((u128)a * b % q); }

static uint64_t invmod(uint64_t a, uint64_t q) {   /* extended Euclid, gcd(a, q) = 1 */
    __int128 r0 = q, r1 = a % q, s0 = 0, s1 = 1;
    while (r1) {
        __int128 k = r0 / r1, r = r0 - k * r1, s = s0 - k * s1;
        r0 = r1; r1 = r; s0 = s1; s1 = s;
    }
    return (uint64_t)(s0 < 0 ? s0 + q : s0);
}

static int bit_count(uint64_t v) { int b = 0; while (v) { b++; v >>= 1; } return b; }
static int words_bits(const uint64_t *a, int w) {
    for (int j = w - 1; j >= 0; j--) if (a[j]) return 64 * j + bit_count(a[j]);
    return 0;
}
static int words_ge(const uint64_t *a, const uint64_t *b, int w) {
    for (int j = w - 1; j >= 0; j--) if (a[j] != b[j]) return a[j] > b[j];
    return 1;
}
static void words_sub(uint64_t *a, const uint64_t *b, int w) {   /* a -= b, a >= b */
    unsigned borrow = 0;
    for (int j = 0; j < w; j++) {
        u128 d = (u128)a[j] - b[j] - borrow;
        a[j] = (uint64_t)d;
        borrow = (unsigned)((d >> 64) & 1);
    }
}

/* d: [count][K][n+1] canonical residues of c0 + c1 s; out: count budgets.  Returns 0, or -1 for K out of range. */
int fvb_noise_budget(int n, int K, const uint64_t *primes, uint64_t t, const uint64_t *d, int count, int *out) {
    if (K < 1 || K > MAXK) return -1;
    const int W = K + 1;
    const size_t st = (size_t)n + 1;
    uint64_t q[NBW] = {1}, half[NBW], qhat[MAXK][NBW], inv_qhat[MAXK];
    for (int i = 0; i < K; i++) { memset(qhat[i], 0, sizeof qhat[i]); qhat[i][0] = 1; }
    for (int p = 0; p < K; p++)                            /* q = prod q_p, qhat[i] = prod_{p != i} q_p (coeff_products_array_) */
        for (int i = -1; i < K; i++) {
            if (i == p) continue;
            uint64_t *w = i < 0 ? q : qhat[i];
            u128 carry = 0;
            for (int j = 0; j < W; j++) { u128 v = (u128)w[j] * primes[p] + carry; w[j] = (uint64_t)v; carry = v >> 64; }
        }
    for (int i = 0; i < K; i++) {                          /* inv_coeff_products_mod_coeff_array_ */
        uint64_t r = 1;
        for (int p = 0; p < K; p++) if (p != i) r = mulmod(r, primes[p] % primes[i], primes[i]);
        inv_qhat[i] = invmod(r, primes[i]);
    }
    for (int j = 0; j < W; j++) half[j] = (q[j] >> 1) | (j + 1 < W ? q[j + 1] << 63 : 0);   /* (q + 1) / 2, q odd */
    for (int j = 0; j < W && ++half[j] == 0; j++) {}
    const int q_bits = words_bits(q, W);                   /* total_coeff_modulus_bit_count */
    for (int c = 0; c < count; c++) {
        int norm_bits = 0;
        for (int k = 0; k < n; k++) {
            uint64_t x[NBW] = {0};
            for (int i = 0; i < K; i++) {
                const uint64_t y = mulmod(d[((size_t)c * K + i) * st + k], t % primes[i], primes[i]);
                const uint64_t a = mulmod(y, inv_qhat[i], primes[i]);
                u128 carry = 0;
                for (int j = 0; j < W; j++) {                 /* x += a qhat_i (multiply_uint_uint64, add_uint_uint) */
                    u128 v = (u128)a * qhat[i][j] + x[j] + carry;
                    x[j] = (uint64_t)v; carry = v >> 64;
                }
                if (words_ge(x, q, W)) words_sub(x, q, W);    /* add_uint_uint_mod: both terms below q */
            }
            if (words_ge(x, half, W)) {                       /* |x| = q - x */
                uint64_t r[NBW];
                memcpy(r, q, sizeof r);
                words_sub(r, x, W);
                memcpy(x, r, sizeof r);
            }
            const int b = words_bits(x, W);
            if (b > norm_bits) norm_bits = b;
        }
        const int budget = q_bits - norm_bits - 1;
        out[c] = budget < 0 ? 0 : budget;
    }
    return 0;
}
