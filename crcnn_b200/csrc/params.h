// Host-side derivation of every constant the kernels need, from (n, q_1..q_K, t) alone.
//
// Mirrors what the reference derives in SEALContext / Evaluator / BaseConverter /
// SmallNTTTables so that NTT-form data produced by SEAL (evaluation keys, NTT-form plaintexts)
// is directly consumable:
//   - Barrett ratios                      SEAL/seal/smallmodulus.cpp:62-73
//   - minimal primitive 2n-th roots, bit-reversed power tables, Shoup companions,
//     inverse powers pre-divided by two   SEAL/seal/util/smallntt.cpp:37-92, 162-184
//   - Delta = floor(q/t) and q mod t per prime, plain-lift increments
//                                         SEAL/seal/evaluator.cpp:66-105
//   - BEHZ base-conversion constants, aux/Bsk primes, m_sk, m_tilde
//                                         SEAL/seal/util/baseconverter.cpp:20-349,
//                                         SEAL/seal/util/globals.cpp:321-340
#pragma once
#include <cstdint>
#include <string>
#include <vector>
#include "modarith.cuh"

namespace crcnn {

constexpr int MAXK = 8;    // coefficient primes (n <= 16384 at 128-bit security)
constexpr int MAXS = 10;   // Bsk primes = aux (K or K+1) + m_sk
constexpr int MAXDIG = 4;  // 16-bit relinearisation digits per prime (<= 60-bit primes)

// One NTT modulus with device pointers to its four n-entry tables.
struct NttTable {
    Mod mod;
    const uint64_t *w;    // interleaved (root_power, scaled_root_power) pairs: w[2i] = psi^bitrev(i), w[2i+1] = floor(w[2i] * 2^64 / q)
    const uint64_t *iw;   // interleaved inverse pairs psi^-bitrev(i) (NOT pre-halved: the kernels scale by n^-1 once at the end)
    uint64_t ninv, ninvp; // n^-1 mod q and floor(n^-1 * 2^64 / q)
    const uint64_t *tf;   // top-block factors for the sparse-input forward transform (see ntt.cuh), 2^skip entries
    const uint64_t *wl;   // pairs of the contiguous 4-stage forward pass, transposed: [15 rows][n/16 groups] (ntt.cuh: fwd_last_pass)
    const uint64_t *iwl;  // same for the first (contiguous) inverse pass
};

// Forward-NTT stages that can be skipped for FractionalEncoder-shaped plaintexts (support in
// [0,64) U [n-32,n)): whole passes of the NttPlan schedule while the block length stays >= 128.
#if defined(__CUDACC__)
__host__ __device__
#endif
constexpr int sparse_skip_stages(int logn) { return logn == 13 ? 6 : logn == 12 ? 4 : logn == 14 ? 6 : 3; }

// Everything the kernels read; lives in device global memory, one per context.
struct DeviceParams {
    int n, logn, K, L, S;
    uint64_t t, half;               // plain modulus, (t+1)>>1
    NttTable tab[MAXK + MAXS];      // [0,K): coefficient primes, [K,K+S): Bsk primes (aux..., m_sk)
    uint64_t delta[MAXK];           // floor(q/t) mod q_j
    uint64_t rho[MAXK];             // (q mod t) mod q_j          (upper_half_increment)
    uint64_t lift_inc[MAXK];        // q_j - t                     (fast plain lift)
    // BEHZ (names follow BaseConverter's members)
    uint64_t inv_qhat[MAXK];            // (q/q_i)^-1 mod q_i
    uint64_t mt_inv_qhat[MAXK];         // m_tilde * (q/q_i)^-1 mod q_i
    uint64_t qhat_mod_bsk[MAXS][MAXK];  // (q/q_i) mod p_k
    uint64_t qhat_mod_mt[MAXK];         // (q/q_i) mod m_tilde
    uint64_t neg_inv_q_mod_mt;          // -(q^-1) mod m_tilde  (32-bit)
    uint64_t q_mod_bsk[MAXS];           // q mod p_k
    uint64_t inv_mt_mod_bsk[MAXS];      // m_tilde^-1 mod p_k
    uint64_t inv_q_mod_bsk[MAXS];       // q^-1 mod p_k
    uint64_t inv_Mhat[MAXS];            // (M/m_i)^-1 mod m_i
    uint64_t Mhat_mod_q[MAXK][MAXS];    // (M/m_i) mod q_j
    uint64_t Mhat_mod_msk[MAXS];        // (M/m_i) mod m_sk
    uint64_t inv_M_mod_msk;             // M^-1 mod m_sk
    uint64_t M_mod_q[MAXK];             // M mod q_j
    uint64_t neg_M_mod_q[MAXK];         // q_j - (M mod q_j)
    uint64_t t_mod[MAXK + MAXS];        // t mod each modulus (the scalar multiply inside square)
    // Folded constants: products of the above that let each base-conversion output be ONE lazy
    // 128-bit sum followed by ONE Barrett reduction (same residues, fewer reductions).
    uint64_t lift_a[MAXS][MAXK];        // (q/q_i mod p_k) * m_tilde^-1 mod p_k
    uint64_t lift_b[MAXS];              // (q mod p_k) * m_tilde^-1 mod p_k
    uint64_t fl_c[MAXK];                // t * (q/q_i)^-1 mod q_i
    uint64_t fl_T[MAXS];                // t * q^-1 [* (M/m_k)^-1 for k < L] mod p_k
    uint64_t fl_N[MAXS][MAXK];          // -(q/q_i mod p_k) * q^-1 [* (M/m_k)^-1 for k < L] mod p_k
    uint64_t fl_P[MAXS];                // (M/m_i mod m_sk) * M^-1 mod m_sk
    // The same first-step constants times n^-1 (mod q_i resp. p_k): for lift / floor inputs that an inverse transform left
    // multiplied by n (kernels.cuh: ninv_in = false), so the transform saves its n^-1 product per residue.
    uint64_t mt_inv_qhat_n[MAXK];       // mt_inv_qhat * n^-1 mod q_i
    uint64_t fl_c_n[MAXK];              // fl_c * n^-1 mod q_i
    uint64_t fl_T_n[MAXS];              // fl_T * n^-1 mod p_k
};

// Host copy: the scalar part of DeviceParams plus the tables as vectors.
struct HostParams {
    DeviceParams d{};                               // table pointers left null
    std::vector<std::vector<uint64_t>> w, wp, iw, iwp;  // per modulus, n entries (iw/iwp = SEAL's pre-halved inverse tables, for cross-checks)
    std::vector<std::vector<uint64_t>> iwf, iwfp;       // un-halved inverse powers: what the device uses
    std::vector<uint64_t> roots;                    // minimal primitive 2n-th root per modulus
    std::vector<std::vector<uint64_t>> tf;          // per coefficient prime: top-block factors
};

// Throws std::invalid_argument on parameters the reference's SEALContext would reject
// (non power-of-two n, q_i != 1 mod 2n, duplicate primes, t >= q_i i.e. no fast plain lift).
HostParams derive_params(int n, int K, const uint64_t *q, uint64_t t);

Mod make_mod(uint64_t q);
uint64_t inv_mod(uint64_t a, uint64_t q);
uint64_t pow_mod(uint64_t a, uint64_t e, const Mod &m);
bool minimal_primitive_root(uint64_t degree, const Mod &m, uint64_t &root);

// Balanced base-3 fractional encoding used for every CrCNN weight:
// FractionalEncoder(t, x^n+1, 64 integer coeffs, 32 fraction coeffs, base 3)
// (CrCNN/src/globals.cpp:52, SEAL/seal/encoder.cpp:1013-1076).  Appends (index, value<t) pairs.
void encode_fractional_sparse(double value, int n, uint64_t t, std::vector<uint32_t> &idx,
                              std::vector<uint64_t> &val);

}  // namespace crcnn
