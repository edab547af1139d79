// See params.h.  Host-only code (compiled by nvcc's host pass or g++).
#include "params.h"
#include <cmath>
#include <stdexcept>

namespace crcnn {

typedef unsigned __int128 u128;

static const uint64_t kAuxPrimes[] = {
    // 61-bit primes = 1 mod 2^18, in the order the reference's BaseConverter consumes them
    // (SEAL/seal/util/globals.cpp:330-333)
    0x1fffffffffb40001ULL, 0x1fffffffff500001ULL, 0x1fffffffff380001ULL, 0x1fffffffff000001ULL,
    0x1ffffffffef00001ULL, 0x1ffffffffee80001ULL, 0x1ffffffffeb40001ULL, 0x1ffffffffe780001ULL,
    0x1ffffffffe600001ULL, 0x1ffffffffe4c0001ULL};
static const uint64_t kMsk = 0x1fffffffffe00001ULL;  // SEAL/seal/util/globals.cpp:324
static const uint64_t kMtilde = 1ULL << 32;          // SEAL/seal/util/globals.cpp:327

static int bits_of(uint64_t v) {
    int b = 0;
    for (; v; v >>= 1) b++;
    return b;
}

Mod make_mod(uint64_t q) {
    // floor(2^128 / q) without a 192-bit divide: (2^128-1)/q, corrected when q divides 2^128.
    u128 ones = ~(u128)0;
    u128 quo = ones / q;
    if (ones % q == (u128)(q - 1)) quo++;
    Mod m;
    m.q = q;
    m.r0 = (uint64_t)quo;
    m.r1 = (uint64_t)(quo >> 64);
    return m;
}

uint64_t pow_mod(uint64_t a, uint64_t e, const Mod &m) {
    uint64_t r = 1 % m.q;
    a %= m.q;
    for (; e; e >>= 1) {
        if (e & 1) r = mulmod(r, a, m);
        a = mulmod(a, a, m);
    }
    return r;
}

uint64_t inv_mod(uint64_t a, uint64_t q) {
    // extended Euclid on signed 128-bit; q may be composite (m_tilde = 2^32)
    __int128 r0 = q, r1 = a % q, s0 = 0, s1 = 1;
    while (r1 != 0) {
        __int128 k = r0 / r1;
        __int128 r2 = r0 - k * r1, s2 = s0 - k * s1;
        r0 = r1; r1 = r2; s0 = s1; s1 = s2;
    }
    if (r0 != 1) throw std::invalid_argument("inv_mod: operand not invertible");
    if (s0 < 0) s0 += q;
    return (uint64_t)s0;
}

bool minimal_primitive_root(uint64_t degree, const Mod &m, uint64_t &root) {
    // The reference picks a random primitive degree-th root, then scans all its odd powers for
    // the smallest (SEAL/seal/util/uintarithsmallmod.cpp:83-108) -- the minimum over the whole set
    // of primitive roots, hence independent of the starting point.  We start from g^((q-1)/degree)
    // for the first small g that yields a primitive root.
    if ((m.q - 1) % degree) return false;
    uint64_t cof = (m.q - 1) / degree, start = 0;
    for (uint64_t g = 2; g < 1u << 16 && !start; g++) {
        uint64_t c = pow_mod(g, cof, m);
        if (pow_mod(c, degree / 2, m) == m.q - 1) start = c;
    }
    if (!start) return false;
    uint64_t step = mulmod(start, start, m), cur = start, best = start;
    for (uint64_t i = 0; i < degree / 2; i++) {  // the degree/2 odd powers
        if (cur < best) best = cur;
        cur = mulmod(cur, step, m);
    }
    root = best;
    return true;
}

static uint32_t bit_reverse(uint32_t x, int bits) {
    uint32_t r = 0;
    for (int i = 0; i < bits; i++, x >>= 1) r = (r << 1) | (x & 1);
    return r;
}

static uint64_t product_mod(const uint64_t *v, int count, int skip, const Mod &m) {
    uint64_t r = 1 % m.q;
    for (int i = 0; i < count; i++)
        if (i != skip) r = mulmod(r, v[i] % m.q, m);
    return r;
}

static void build_tables(HostParams &hp, int slot, int logn, const Mod &m) {
    int n = 1 << logn;
    uint64_t psi;
    if (!minimal_primitive_root(2ull * n, m, psi))
        throw std::invalid_argument("modulus " + std::to_string(m.q) + " has no primitive 2n-th root of unity");
    uint64_t psi_inv = inv_mod(psi, m.q);
    auto &w = hp.w[slot], &wp = hp.wp[slot], &iw = hp.iw[slot], &iwp = hp.iwp[slot];
    auto &iwf = hp.iwf[slot], &iwfp = hp.iwfp[slot];
    w.assign(n, 0); wp.assign(n, 0); iw.assign(n, 0); iwp.assign(n, 0); iwf.assign(n, 0); iwfp.assign(n, 0);
    uint64_t pw = 1, ipw = 1;
    for (int i = 0; i < n; i++) {
        uint32_t r = bit_reverse((uint32_t)i, logn);
        w[r] = pw;
        // inverse power halved mod q (q odd): x/2 = (x + (x odd ? q : 0)) >> 1
        iw[r] = (ipw & 1) ? (uint64_t)(((u128)ipw + m.q) >> 1) : (ipw >> 1);
        iwf[r] = ipw;
        pw = mulmod(pw, psi, m);
        ipw = mulmod(ipw, psi_inv, m);
    }
    for (int i = 0; i < n; i++) {
        wp[i] = (uint64_t)((((u128)w[i]) << 64) / m.q);
        iwp[i] = (uint64_t)((((u128)iw[i]) << 64) / m.q);
        iwfp[i] = (uint64_t)((((u128)iwf[i]) << 64) / m.q);
    }
    hp.d.tab[slot].ninv = inv_mod((uint64_t)n % m.q, m.q);
    hp.d.tab[slot].ninvp = (uint64_t)((((u128)hp.d.tab[slot].ninv) << 64) / m.q);
    hp.roots[slot] = psi;
}

HostParams derive_params(int n, int K, const uint64_t *q, uint64_t t) {
    int logn = 0;
    while ((1 << logn) < n) logn++;
    if (n < 1024 || n > 16384 || (1 << logn) != n) throw std::invalid_argument("n must be a power of two in [1024, 16384]");
    if (K < 1 || K > MAXK) throw std::invalid_argument("coefficient modulus count must be in [1, 8]");
    if (t < 2) throw std::invalid_argument("plain modulus must be at least 2");
    int total_bits = 0;
    for (int i = 0; i < K; i++) {
        if (bits_of(q[i]) > 60 || q[i] < 2) throw std::invalid_argument("coefficient primes must be at most 60 bits");
        if (q[i] <= t) throw std::invalid_argument("plain modulus must be smaller than every coefficient prime (fast plain lift)");
        for (int j = 0; j < i; j++)
            if (q[i] == q[j]) throw std::invalid_argument("coefficient primes must be distinct");
        total_bits += bits_of(q[i]);
    }
    HostParams hp;
    DeviceParams &d = hp.d;
    d.n = n; d.logn = logn; d.K = K; d.t = t; d.half = (t + 1) >> 1;
    // aux base: K primes, one more if K*n*t*q^2 might not fit under q*M*m_sk
    // (SEAL/seal/util/baseconverter.cpp:47-58)
    d.L = K + ((32 + bits_of(t) + total_bits >= 61 * K + 61) ? 1 : 0);
    d.S = d.L + 1;
    int slots = K + d.S;
    hp.w.resize(slots); hp.wp.resize(slots); hp.iw.resize(slots); hp.iwp.resize(slots); hp.iwf.resize(slots); hp.iwfp.resize(slots); hp.roots.resize(slots);

    std::vector<uint64_t> bsk(d.S);
    for (int i = 0; i < d.L; i++) bsk[i] = kAuxPrimes[i];
    bsk[d.L] = kMsk;
    for (int i = 0; i < K; i++) { d.tab[i].mod = make_mod(q[i]); build_tables(hp, i, logn, d.tab[i].mod); }
    for (int k = 0; k < d.S; k++) { d.tab[K + k].mod = make_mod(bsk[k]); build_tables(hp, K + k, logn, d.tab[K + k].mod); }
    for (int s = 0; s < slots; s++) d.t_mod[s] = t % d.tab[s].mod.q;
    // Sparse-input forward NTT: after `skip` Cooley-Tukey stages a coefficient sitting in the top 32
    // positions of the polynomial has only been multiplied, stage by stage, by +W (lower child block) or
    // -W (upper child block); block b therefore holds it times  prod_s (+-) w[2^s + (b >> (skip - s))].
    hp.tf.resize(K);
    const int skip = sparse_skip_stages(logn);
    for (int j = 0; j < K; j++) {
        const Mod &m = d.tab[j].mod;
        hp.tf[j].assign((size_t)1 << skip, 0);
        for (int b = 0; b < (1 << skip); b++) {
            uint64_t c = 1;
            for (int s = 0; s < skip; s++) {
                uint64_t w = hp.w[j][((size_t)1 << s) + (b >> (skip - s))];
                if ((b >> (skip - 1 - s)) & 1) w = negmod(w, m.q);
                c = mulmod(c, w, m);
            }
            hp.tf[j][b] = c;
        }
    }

    Mod mt = make_mod(kMtilde), msk = make_mod(kMsk), tm = make_mod(t);
    // Delta = floor(Q/t), rho = Q - t*Delta = Q mod t.  t*Delta = Q - rho, so modulo q_j
    // (where Q = 0): Delta = -rho * t^-1.
    uint64_t rho = product_mod(q, K, -1, tm);
    for (int j = 0; j < K; j++) {
        const Mod &m = d.tab[j].mod;
        d.rho[j] = rho % m.q;
        d.delta[j] = mulmod(negmod(d.rho[j], m.q), inv_mod(t % m.q, m.q), m);
        d.lift_inc[j] = m.q - t;
        d.inv_qhat[j] = inv_mod(product_mod(q, K, j, m), m.q);
        d.mt_inv_qhat[j] = mulmod(d.inv_qhat[j], kMtilde % m.q, m);
        d.qhat_mod_mt[j] = product_mod(q, K, j, mt);
        d.M_mod_q[j] = product_mod(bsk.data(), d.L, -1, m);
        d.neg_M_mod_q[j] = m.q - d.M_mod_q[j];
        for (int i = 0; i < d.L; i++) d.Mhat_mod_q[j][i] = product_mod(bsk.data(), d.L, i, m);
    }
    d.neg_inv_q_mod_mt = (kMtilde - inv_mod(product_mod(q, K, -1, mt), kMtilde)) % kMtilde;
    for (int k = 0; k < d.S; k++) {
        const Mod &m = d.tab[K + k].mod;
        for (int i = 0; i < K; i++) d.qhat_mod_bsk[k][i] = product_mod(q, K, i, m);
        d.q_mod_bsk[k] = product_mod(q, K, -1, m);
        d.inv_q_mod_bsk[k] = inv_mod(d.q_mod_bsk[k], m.q);
        d.inv_mt_mod_bsk[k] = inv_mod(kMtilde % m.q, m.q);
    }
    for (int i = 0; i < d.L; i++) {
        const Mod &m = d.tab[K + i].mod;
        d.inv_Mhat[i] = inv_mod(product_mod(bsk.data(), d.L, i, m), m.q);
        d.Mhat_mod_msk[i] = product_mod(bsk.data(), d.L, i, msk);
    }
    d.inv_M_mod_msk = inv_mod(product_mod(bsk.data(), d.L, -1, msk), kMsk);
    // folded constants (see params.h)
    for (int j = 0; j < K; j++) {
        const Mod &m = d.tab[j].mod;
        d.fl_c[j] = mulmod(mulmod(t % m.q, d.inv_qhat[j], m), d.tab[j].ninv, m);
        d.mt_inv_qhat_n[j] = mulmod(d.mt_inv_qhat[j], d.tab[j].ninv, m);
    }
    for (int k = 0; k < d.S; k++) {
        const Mod &m = d.tab[K + k].mod;
        const uint64_t fold = k < d.L ? mulmod(d.inv_q_mod_bsk[k], d.inv_Mhat[k], m) : d.inv_q_mod_bsk[k];
        d.lift_b[k] = mulmod(d.q_mod_bsk[k], d.inv_mt_mod_bsk[k], m);
        d.fl_T[k] = mulmod(mulmod(t % m.q, fold, m), d.tab[K + k].ninv, m);
        for (int i = 0; i < K; i++) {
            d.lift_a[k][i] = mulmod(d.qhat_mod_bsk[k][i], d.inv_mt_mod_bsk[k], m);
            d.fl_N[k][i] = negmod(mulmod(d.qhat_mod_bsk[k][i], fold, m), m.q);
        }
    }
    for (int i = 0; i < d.L; i++) d.fl_P[i] = mulmod(d.Mhat_mod_msk[i], d.inv_M_mod_msk, msk);
    return hp;
}

// ---- balanced base-3 fractional encoder (weights loader; SURVEY.md section 8(f) row N1) ----
static void encode_integer_b3(int64_t v, uint64_t t, std::vector<uint32_t> &idx, std::vector<uint64_t> &val) {
    // balanced ternary digits of v, least significant first (SEAL/seal/encoder.cpp:408-481)
    bool neg = v < 0;
    uint64_t mag = neg ? (uint64_t)(-v) : (uint64_t)v;
    for (uint32_t pos = 0; mag; pos++) {
        uint64_t rem = mag % 3;
        int digit = rem == 0 ? 0 : (rem == 1 ? 1 : -1);  // 2 == -1 with carry
        mag = (mag + 1) / 3;                              // (mag + base/2)/base, identical for both signs at base 3
        if (neg) digit = -digit;
        if (digit) { idx.push_back(pos); val.push_back(digit > 0 ? 1 : t - 1); }
    }
}

void encode_fractional_sparse(double value, int n, uint64_t t, std::vector<uint32_t> &idx,
                              std::vector<uint64_t> &val) {
    int64_t ip = (int64_t)std::round(value);
    encode_integer_b3(ip, t, idx, val);
    double frac = value - (double)ip;
    if (frac == 0) return;
    // 32 fractional trits, most significant first at x^(n-1) with flipped sign
    // (x^n = -1 makes -x^(n-k) play the role of 3^-k)
    for (int i = 0; i < 32; i++) {
        frac *= 3.0;
        int sign = frac >= 0 ? 1 : -1;
        int64_t digit = (int64_t)(sign * std::ceil(std::fabs(frac) - 0.5));
        frac -= (double)digit;
        if (digit) { idx.push_back((uint32_t)(n - 1 - i)); val.push_back(digit > 0 ? t - (uint64_t)digit : (uint64_t)(-digit)); }
    }
}

}  // namespace crcnn
