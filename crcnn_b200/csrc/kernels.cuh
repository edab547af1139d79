// Launch wrappers for every device kernel of the encrypted-forward hot path.  All pointers are
// device pointers; limb-polynomials are dense (stride n, no SEAL pad word).  Ciphertext tensors are
// uint64[count][size][K][n].  Every wrapper enqueues on `stream` and returns the launch error.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "params.h"

namespace crcnn {

// ---- NTT over `npolys` limb-polynomials; polynomial p uses modulus slot slot_base + p % slot_count.
cudaError_t launch_ntt(const DeviceParams *P, int logn, uint64_t *data, long npolys, int slot_base, int slot_count,
                       bool inverse, cudaStream_t stream);

// Same for polynomials that sit `slot_count` in a row at offset group_off inside records of group_polys polynomials
// (e.g. only the Bsk limbs of [count][2][K+S][n]).
// src (inverse transform only): read the polynomials from src instead of data (out of place, same indexing).
// addend (inverse only): output polynomial p = transform + polynomial (p / add_group) * add_stride + p % add_group of addend.
// ninv = false (inverse only): the output is n times the inverse transform, canonical -- for a consumer that multiplies
// every residue by a constant carrying n^-1 next (launch_behz_lift with ninv_in = false).
cudaError_t launch_ntt_grouped(const DeviceParams *P, int logn, uint64_t *data, long npolys, int slot_base, int slot_count,
                               bool inverse, int group_polys, int group_off, cudaStream_t stream, const uint64_t *src = nullptr,
                               const uint64_t *addend = nullptr, int add_group = 1, int add_stride = 1, bool ninv = true);

// ---- plaintext packs: sparse coefficient form -> dense NTT form, one CTA per (plaintext, limb).
// mode 0: lifted residues (multiplicative use: weights, scale factors)  [evaluator.cpp:1465-1486]
// mode 1: Delta-scaled residues (additive use: biases, means)           [evaluator.cpp:1169-1191]
cudaError_t launch_plain_expand(const DeviceParams *P, int logn, int K, const uint32_t *offsets, const uint32_t *idx,
                                const uint64_t *val, long first, long count, int mode, bool to_ntt, uint64_t *out,
                                cudaStream_t stream);

// ---- fused weighted sum (conv / fully connected), NTT domain.
struct MacArgs {
    const uint64_t *x;       // inputs  [num_in][2][K][n] (NTT form)
    const uint64_t *w;       // weights [M][R][K][n]      (NTT form, lifted)
    const uint64_t *bias;    // [M][K][n] NTT of Delta-scaled bias, added to poly 0 (may be null)
    const int *in_index;     // [Npos][R] input ciphertext index for output position p, term r
    uint64_t *out;           // output ct index = (p / Pimg) * (Mtotal * Pimg) + (m0 + m) * Pimg + p % Pimg
    int R, M, Npos, Pimg, Mtotal, m0;
    int K, n;
    int chunk_terms;         // terms that may be accumulated in 128 bits before a reduction
};
cudaError_t launch_mac(const DeviceParams *P, const MacArgs &a, cudaStream_t stream);

// ---- window sum (sum-pool / avg-pool): out[o] = (sum_r in[in_index[o][r]]) (* scale[K][n] if given)
// scale_shoup = Shoup companions of scale_ntt (launch_shoup_companion); sum_fits_64: R * max(q) < 2^64
cudaError_t launch_pool(const DeviceParams *P, int n, int K, const uint64_t *in, const int *in_index, int Nout, int R,
                        const uint64_t *scale_ntt, const uint64_t *scale_shoup, bool sum_fits_64, uint64_t *out,
                        cudaStream_t stream, int per_channel = 1, int channels = 0, const uint64_t *sub = nullptr);
cudaError_t launch_pool_bn_consts(const DeviceParams *P, const uint64_t *S, const uint64_t *V, const uint64_t *M, long words,
                                  uint64_t *C, uint64_t *D, cudaStream_t stream);

// ---- batch-norm, NTT domain: c0' = (c0 - mean_ntt[z]) * invstd_ntt[z], c1' = c1 * invstd_ntt[z]
// ciphertext i belongs to channel (i / per_channel) % channels.
cudaError_t launch_bn(const DeviceParams *P, int n, int K, const uint64_t *in, long count, int per_channel, int channels,
                      const uint64_t *mean_ntt, const uint64_t *invstd_ntt, const uint64_t *invstd_shoup, uint64_t *out,
                      cudaStream_t stream);

// ---- coefficient-domain multiply_plain by a +-1-digit plaintext, fused with a window sum and a plaintext subtraction
struct TapMulArgs {
    const uint64_t *in;       // ciphertexts [..][2][K][n], COEFFICIENT form
    const int *in_index;      // [nout][R] inputs summed for output o (pooling); null: input o itself, R ignored
    int R;
    const uint64_t *sub;      // [channels][K][n] Delta-scaled plaintext subtracted from polynomial 0 first (batch-norm mean); may be null
    const uint32_t *t_off;    // sparse form of the multiplier pack: plaintext z has terms [t_off[z], t_off[z+1])
    const uint32_t *t_idx;    //   exponents, in [0,64) U [n-32,n)
    const uint64_t *t_val;    //   values, 1 or t-1
    int per_channel, channels;  // output o uses plaintext z = (o / per_channel) % channels (channels == 1: always plaintext 0)
    uint64_t *out;            // [nout][2][K][n] coefficient form
    long nout;
};
cudaError_t launch_tapmul(const DeviceParams *P, int n, int K, const TapMulArgs &a, cudaStream_t stream);

// ---- Shoup companions floor(v * 2^64 / q_j) of `words` canonical residues laid out [..][K][n]
// data[row] = data[row] (.) C[row / group] - D[row / group] over rows of poly_words residues (D may be null)
cudaError_t launch_fold_affine(const DeviceParams *P, uint64_t *data, long rows, long poly_words, int group, const uint64_t *C,
                               const uint64_t *D, cudaStream_t stream);
// Bias[k] -= sum_r W[k][r] (.) D[r / per_channel]; W[k][r] (.)= C[r / per_channel]   (W: [out_dim][in_dim][poly_words], NTT form)
cudaError_t launch_fold_fc_input_affine(const DeviceParams *P, uint64_t *W, int out_dim, int in_dim, long poly_words, int per_channel,
                                        const uint64_t *C, const uint64_t *D, uint64_t *Bias, cudaStream_t stream);
cudaError_t launch_scale_small(const DeviceParams *P, uint64_t *data, long words, int times, cudaStream_t stream);   // data *= times (mod q), times small
cudaError_t launch_shoup_companion(const DeviceParams *P, const uint64_t *data, long words, uint64_t *out, cudaStream_t stream);

// ---- generic plaintext ops on `count` ciphertexts of `size` polys (evaluator-level API)
// op 0: every poly *= pl (pl in NTT lifted form, data in NTT form); op 1/2: poly0 +=/-= pl (scaled form,
// same domain as data)
cudaError_t launch_plain_op(const DeviceParams *P, int n, int K, uint64_t *data, long count, int size, const uint64_t *pl, const uint64_t *pl_sh, int op,
                            cudaStream_t stream);

// ---- FV square (BEHZ), staged exactly as evaluator.cpp:742-883
// lift:   in [count][2][K][n] (coefficient form) -> ext [count][2][K+S][n] (q limbs copied, Bsk limbs computed)
// (lift and floor take the HOST copy of the parameter block: it travels as a by-value kernel argument, so every
// base-conversion constant is a constant-bank operand)
// in_ntt (optional): the same ciphertexts in NTT form; the q limbs of ext are then left unwritten (launch_ntt_inv_tensor reads them from in_ntt) and only the Bsk
// limbs still need the forward transform
// ninv_in = false: `in` holds n times the coefficients (an inverse transform without its n^-1, launch_ntt_grouped ninv = false);
// the lift then multiplies by mt_inv_qhat_n.  Only together with in_ntt: the q limbs of `in` are not copied to ext then.
cudaError_t launch_behz_lift(const DeviceParams &hp, int n, const uint64_t *in, const uint64_t *in_ntt, long count, uint64_t *ext,
                             cudaStream_t stream, bool ninv_in = true);
// floor:  prod (coefficient form) -> out [count][3][K][n]: multiply by t, fast_floor, fastbconv_sk
// ninv_in = false: prod holds n times the products (launch_ntt_inv_tensor with ninv = false); fl_c_n / fl_T_n absorb the factor.
cudaError_t launch_behz_floor(const DeviceParams &hp, int n, const uint64_t *prod, long count, uint64_t *out, cudaStream_t stream,
                              bool ninv_in = true);
// true when every modulus of the context (q and Bsk) has the 2^k - delta shape of reduce128_fold (modarith.cuh)
bool behz_fold_ok(const DeviceParams &hp);

// ---- relinearize 3 -> 2 with 16-bit digits (evaluator.cpp:934-1069)
// in3 [count][3][K][n] (coefficient), keys: for prime i, digit k: polys (2k, 2k+1) at
// evk + key_off[i] + (2k)*K*n, each [K][n] NTT form;  out [count][2][K][n] coefficient form.
struct RelinArgs {
    const uint64_t *in3;
    const uint64_t *evk;
    long key_off[MAXK];
    int digits[MAXK];
    int dbc;
    uint64_t *out;
    long count;
    // scratch (per call): dsc [count][K][n], dig [count][sum digits][K][n], acc [count][2][K][n]
    uint64_t *dsc, *dig, *acc;
};
// ---- tensor square (c0*c0, 2*c0*c1, c1*c1 in q U Bsk) fused into the inverse transform of each product polynomial:
// ext = [count][2][KS][n] NTT form (qntt != null: its q limbs are taken from qntt = [count][2][K][n] instead),
// prod = [count][3][KS][n] coefficient form
// fold: reduce the products with reduce128_fold (requires behz_fold_ok; only with ninv = false).  ninv = false: prod holds n times
// the products, for launch_behz_floor with ninv_in = false.
cudaError_t launch_ntt_inv_tensor(const DeviceParams *P, int logn, const uint64_t *ext, const uint64_t *qntt, long count, int KS, uint64_t *prod,
                                  bool fold, bool ninv, cudaStream_t stream);

// stages 1-3 (scale, digit NTTs, key MAC); then the caller inverse-NTTs `acc` and calls launch_relin_finish
cudaError_t launch_relin(const DeviceParams *P, int logn, int K, const RelinArgs &a, cudaStream_t stream);
cudaError_t launch_relin_finish(const DeviceParams *P, int n, int K, const RelinArgs &a, cudaStream_t stream);

// ---- residues stored lazily in [0,4q) (evaluation keys) -> canonical, in place; data = [..][K][n]
cudaError_t launch_canonicalize(const DeviceParams *P, uint64_t *data, long words, cudaStream_t stream);

// ---- host layout (limb stride n+1) -> device layout (stride n) for `rows` limb-polynomials already on the device
cudaError_t launch_strip_pad(const uint64_t *src_padded, uint64_t *dst, long rows, int n, cudaStream_t stream);

// ---- integer-pipe roofline probe: register-only 64x64->128 multiply-accumulate loop.
// Returns nothing; caller times it.  total MACs = blocks * threads * iters * 8.
cudaError_t launch_imad_probe(int blocks, int threads, int iters, uint64_t *sink, cudaStream_t stream);
cudaError_t launch_imad_wide_probe(int blocks, int threads, int iters, uint64_t *sink, cudaStream_t stream);

}  // namespace crcnn
