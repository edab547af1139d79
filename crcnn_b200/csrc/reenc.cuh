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
// u (as residues, U[count][K][n]) and e[count][2][n] (int8): sampled from (seed, ciphertext index, coefficient) or copied from `given`
// ([count][3][n] int8: u, e0, e1)
cudaError_t launch_enc_sample(const ReencConsts &c, uint64_t seed, long first_ct, double sigma, double max_dev, const int8_t *given,
                              uint64_t *U, int8_t *e, long count, cudaStream_t s);
// out[count][2][K][n] = U (.) pk[p]   (U in NTT form)
cudaError_t launch_enc_mul(const ReencConsts &c, const uint64_t *U, const uint64_t *pk, uint64_t *out, long count, cudaStream_t s);
// out (coefficient form after the inverse transform) += e_p (+ Delta * m on polynomial 0)
cudaError_t launch_enc_finish(const ReencConsts &c, const uint64_t *slots, const int8_t *e, uint64_t *out, long count, cudaStream_t s);

}  // namespace crcnn
