// Re-encryption on the device (SURVEY 8(f) row N4): the reference's Network::forward decrypts and re-encrypts the whole activation
// tensor before layer 6 to reset the noise (CrCNN/src/network.cpp:30-33 -> decryptImage / encryptImage, CrCNN/src/globals.cpp:127-142,
// 207-226).  Done by the reference on the host with the SECRET key (3.2 s per image at n = 4096, Doc/Tesi.lyx:13020-13700); here the
// same three client-side steps run on the GPU next to the activations:
//   Decryptor::decrypt          (SEAL/seal/decryptor.cpp:107-234; BEHZ scaling through {t, gamma}: util/baseconverter.cpp:744-795)
//   decode -> float -> encode   (FractionalEncoder(64, 32, base 3), SEAL/seal/encoder.cpp; floatCube holds floats, CrCNN/src/globals.h:16)
//   Encryptor::encrypt          (SEAL/seal/encryptor.cpp:95-200), noise from a counter-based generator (Philox4x32-10) on the device
// Decryption and the re-encoding are deterministic and bit-identical to SEAL's; encryption is randomised by definition, so it is
// byte-checked against the oracle with the sampled polynomials supplied, and against the reference's own Decryptor (same plaintext,
// fresh noise budget).  Moving the secret key next to the evaluator changes the trust model -- exactly as the reference's own
// in-process re-encryption does; it is opt-in (crcnn_keys_upload) and nothing else in the library ever sees a key.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "params.h"

namespace crcnn {

constexpr uint64_t REENC_GAMMA = 0x1fffffffffc80001ULL;   // SEAL/seal/util/globals.cpp:330 (internal_mods::gamma)
constexpr int REENC_SLOTS = 96;                            // 64 integer + 32 fraction coefficients of the encoder

struct ReencConsts {
    int n, K;
    uint64_t t, half, gamma;
    Mod q[MAXK], tm, gm;
    uint64_t dec_c[MAXK];                 // (t * gamma mod q_i) * (q/q_i)^-1 mod q_i: decryptor.cpp:186 and baseconverter.cpp:767 folded
    uint64_t qhat_t[MAXK], qhat_g[MAXK];  // (q/q_i) mod t, mod gamma (coeff_products_mod_plain_gamma_array_)
    uint64_t neg_inv_q_t, neg_inv_q_g;    // (-q)^-1 mod t, mod gamma (neg_inv_coeff_products_all_mod_plain_gamma_array_)
    uint64_t inv_gamma_t;                 // gamma^-1 mod t
    uint64_t delta[MAXK], rho[MAXK];      // floor(q/t) mod q_i, (q mod t) mod q_i: Encryptor::preencrypt
};

ReencConsts make_reenc_consts(const DeviceParams &d);

// Decryptor::invariant_noise_budget (SEAL/seal/decryptor.cpp): t (c0 + c1 s) mod q composed by CRT (BaseConverter::compose) as
// sum_i [y_i (q/q_i)^-1]_{q_i} (q/q_i), reduced below q, centred (poly_infty_norm_coeffmod).  Multi-word integers are MAXK + 1
// little-endian 64-bit words: primes are <= 60 bits, so q < 2^480 and a sum of K terms below q stays below 2^(64 K + 3).
constexpr int NB_WORDS = MAXK + 1;
struct BudgetConsts {
    int n, K, q_bits;                     // q_bits: total_coeff_modulus_bit_count
    Mod q[MAXK];
    uint64_t c[MAXK];                     // t (q/q_i)^-1 mod q_i: multiply_poly_scalar_coeffmod by t and compose's first step folded
    uint64_t qhat[MAXK][NB_WORDS];        // q/q_i
    uint64_t qw[NB_WORDS], half[NB_WORDS];   // q and (q + 1) / 2 (modulus_neg_threshold)
};

BudgetConsts make_budget_consts(const DeviceParams &d);

// tmp[count][K][n] = NTT(c1) on entry (coefficient-form input) -> tmp (.) sk;  NTT-form input: tmp = c1 (.) sk + c0
cudaError_t launch_dec_dot(const ReencConsts &c, const uint64_t *ct, int ct_is_ntt, const uint64_t *sk, uint64_t *tmp, long count, cudaStream_t s);
// tmp = INTT(...) on entry; plain[count][n] = Decryptor::decrypt's result
cudaError_t launch_dec_scale(const ReencConsts &c, const uint64_t *ct /* null when c0 is already in tmp */, const uint64_t *tmp,
                             uint64_t *plain, long count, cudaStream_t s);
// tmp as for launch_dec_scale; bits[count] (zeroed by the caller) = max over coefficients of the bit length of |t (c0 + c1 s) mod q|
cudaError_t launch_noise_bits(const BudgetConsts &c, const uint64_t *ct /* null when c0 is already in tmp */, const uint64_t *tmp,
                              int *bits, long count, cudaStream_t s);
// decode -> (float) -> encode: slots[count][96] = coefficients 0..63 and n-32..n-1 of the re-encoded plaintext; values[count] (may be null)
cudaError_t launch_reencode(const ReencConsts &c, const uint64_t *plain, uint64_t *slots, float *values, long count, cudaStream_t s);
// slots[count][96] = FractionalEncoder::encode((double) values[i]), laid out as launch_reencode's
cudaError_t launch_encode_values(const ReencConsts &c, const float *values, uint64_t *slots, long count, cudaStream_t s);
// values[count] = (float) FractionalEncoder::decode(plain[i]), plain[count][n] as launch_dec_scale leaves it
cudaError_t launch_decode_values(const ReencConsts &c, const uint64_t *plain, float *values, long count, cudaStream_t s);
// Decryptor::decrypt restricted to the coefficients the fractional decoder reads: slots[count][96] = coefficients 0..63 and
// n-32..n-1 of launch_dec_scale's plaintexts (tmp and ct as for launch_dec_scale)
cudaError_t launch_dec_scale_slots(const ReencConsts &c, const uint64_t *ct, const uint64_t *tmp, uint64_t *slots, long count, cudaStream_t s);
// u (as residues, U[count][K][n]) and e[count][2][n] (int8): sampled from (seed, ciphertext index, coefficient) or copied from `given`
// ([count][3][n] int8: u, e0, e1)
cudaError_t launch_enc_sample(const ReencConsts &c, uint64_t seed, long first_ct, double sigma, double max_dev, const int8_t *given,
                              uint64_t *U, int8_t *e, long count, cudaStream_t s);
// out[count][2][K][n] = U (.) pk[p]   (U in NTT form)
cudaError_t launch_enc_mul(const ReencConsts &c, const uint64_t *U, const uint64_t *pk, uint64_t *out, long count, cudaStream_t s);
// out (coefficient form after the inverse transform) += e_p (+ Delta * m on polynomial 0)
cudaError_t launch_enc_finish(const ReencConsts &c, const uint64_t *slots, const int8_t *e, uint64_t *out, long count, cudaStream_t s);

// CRT plaintext-modulus ensembles: M instances under pairwise coprime t_1 .. t_M stand for one under T = t_1 ... t_M.  A coefficient
// is rebuilt modulo T from its M residues by Garner's mixed-radix recombination, x = r_1 + v_2 t_1 + v_3 t_1 t_2 + ..., with
// v_k = (r_k - x_{k-1}) (t_1 ... t_{k-1})^-1 mod t_k; T is below every coefficient prime (< 2^61), so every partial sum fits a word.
constexpr int CRT_MAX_MODULI = 16;
struct CrtConsts {
    int M;
    uint64_t T, half;                     // the product and BalancedEncoder's negative threshold (T + 1) >> 1 under it
    Mod tm[CRT_MAX_MODULI];               // t_k
    uint64_t prefix[CRT_MAX_MODULI];      // t_1 ... t_{k-1} (prefix[0] = 1)
    uint64_t inv[CRT_MAX_MODULI];         // (t_1 ... t_{k-1})^-1 mod t_k (inv[0] unused)
    uint64_t t_own;                       // this instance's modulus, the one re-encoded plaintexts are written under
};

// moduli[M] pairwise coprime with a product below 2^62 (the caller checks); own: index of this instance's modulus
CrtConsts make_crt_consts(const uint64_t *moduli, int M, int own);
// values[count] = (float) BalancedFractionalEncoder::decode under T of the coefficients composed from slots[M][count][96]
// (instance k's block of launch_dec_scale_slots output at slots + k count 96)
cudaError_t launch_crt_decode_values(const CrtConsts &c, const uint64_t *slots, float *values, long count, cudaStream_t s);
// ciphertexts [first, first + count) of slots[M][total][96]: compose, decode under T, round to float, encode under t_own into
// out[count][96] (launch_reencode's layout, ready for launch_enc_finish)
cudaError_t launch_crt_reencode(const CrtConsts &c, const uint64_t *slots, long total, long first, uint64_t *out, long count, cudaStream_t s);

}  // namespace crcnn
