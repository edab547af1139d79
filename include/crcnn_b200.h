/* crcnn_b200 -- C ABI of the B200-native engine for CrCNN's encrypted-inference forward pass.
 *
 * The reference (barlettacarmen/CrCNN) has no FFI: its hot path sits behind the virtual
 * Layer::forward(ciphertext3D) (CrCNN/src/layer.h:20) and a process-global seal::Evaluator
 * (CrCNN/src/globals.h:23).  This header is the boundary a drop-in replacement binds instead of
 * that Evaluator; each entry point names the reference interface it replaces.  INTEGRATION.md
 * shows the reference-side binding (the C++17 layer classes in crcnn_b200/cpp/ are that binding).
 *
 * Conventions
 *  - extern "C", opaque handles, plain pointers and sizes; every call returns 0 on success or a
 *    negative crcnn_status; crcnn_last_error() gives the message.  No exceptions cross the ABI.
 *  - Host buffers use SEAL 2.3.1's in-memory layout (SEAL/seal/ciphertext.h:448-452, :647-660):
 *      ciphertext = uint64[size][K][n+1]  (limb stride n+1, trailing pad word 0)
 *      plaintext  = uint64[coeff_count], values < t
 *      NTT-form plaintext / evaluation-key polys = uint64[K][n+1]
 *    Device buffers are re-strided to n on upload and re-padded (pad = 0) on download.
 *  - A context is bound to one GPU and one CUDA stream; calls on one context must be serialised by
 *    the caller, different contexts are independent.  Forward calls never change the value of their
 *    inputs (the reference transforms the caller's copy and the layer's weights in place,
 *    CrCNN/src/convolutionalLayer.cpp:113,155).
 *  - All results are canonical residues and bit-identical to SEAL 2.3.1's Evaluator for the same
 *    inputs.  There is no CPU fallback: without a CUDA device crcnn_ctx_create fails.
 */
#ifndef CRCNN_B200_H
#define CRCNN_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct crcnn_ctx crcnn_ctx;
typedef struct crcnn_tensor crcnn_tensor; /* device tensor of ciphertexts */
typedef struct crcnn_plain crcnn_plain;   /* device pack of plaintexts (weights, biases, scale factors) */
typedef struct crcnn_evk crcnn_evk;       /* device copy of evaluation (relinearisation) keys */
typedef struct crcnn_keys crcnn_keys;     /* device copy of the key holder's secret and public key (opt-in: GPU re-encryption) */
typedef struct crcnn_comm crcnn_comm;     /* NCCL communicator of a group of contexts, one per GPU (output-neuron sharding) */

typedef enum {
    CRCNN_OK = 0,
    CRCNN_ERR_INVALID_ARGUMENT = -1, /* what SEAL reports as std::invalid_argument */
    CRCNN_ERR_CUDA = -2,
    CRCNN_ERR_NO_DEVICE = -3,
    CRCNN_ERR_OUT_OF_MEMORY = -4,
    CRCNN_ERR_UNSUPPORTED = -5,
    CRCNN_ERR_OUT_OF_BUDGET = -6     /* the host library's OutOfBudgetException (crcnn_b200.hpp): a ciphertext ran out of noise budget */
} crcnn_status;

/* Message for the most recent failing call on `ctx` (or, with ctx == NULL, for the most recent
 * failing crcnn_ctx_create on this thread). */
const char *crcnn_last_error(const crcnn_ctx *ctx);

/* ---- context ---------------------------------------------------------------------------
 * Replaces: setParameters (CrCNN/src/globals.cpp:25-56) as far as the Evaluator is concerned:
 * SEALContext + Evaluator + BaseConverter + SmallNTTTables constant derivation
 * (SEAL/seal/context.cpp:23-165, evaluator.cpp:19-121, util/baseconverter.cpp:20-349).
 * n: power of two in [1024,16384]; q[K]: distinct NTT primes (= 1 mod 2n), <= 60 bits, K <= 8;
 * t: plain modulus, t < every q_i.  device: CUDA ordinal. */
int crcnn_ctx_create(int n, int K, const uint64_t *q, uint64_t t, int device, crcnn_ctx **out);
int crcnn_ctx_destroy(crcnn_ctx *ctx);
/* Run on a caller-owned cudaStream_t (e.g. torch's current stream); NULL selects the legacy default stream. */
int crcnn_ctx_set_stream(crcnn_ctx *ctx, void *cuda_stream);
int crcnn_ctx_sync(crcnn_ctx *ctx);
/* Device-memory allocator counters since the context was created (DESIGN.md section 3): out[0] blocks >= 32 MB taken from the
 * CUDA pool, out[1] taken from the context's exact-size cache, out[2] returned to the CUDA pool because the cache was full,
 * out[3] cache flushes after an out-of-memory answer, out[4] small allocations, out[5] bytes the cache holds now.  A steady-state
 * step should only move out[1] and out[4]. */
int crcnn_ctx_alloc_stats(crcnn_ctx *ctx, long long out[6]);
/* Upper bound (bytes) for NTT-form weights kept resident per plaintext pack; larger packs are
 * expanded chunk by chunk into a scratch buffer during forward.  Default 24 GiB. */
int crcnn_ctx_set_weight_cache_bytes(crcnn_ctx *ctx, size_t bytes);
/* Weighted sums (conv / fc) whose weights are FractionalEncoder base-3 plaintexts with |w| < 1/2 (every
 * weight of the reference's models) and whose fan-in is >= min_fanin run as a u8 x s8 -> s32 GEMM on the
 * tcgen05 tensor cores in the coefficient domain (crcnn_b200/csrc/tc_mac.cuh); results are the same canonical
 * residues.  mode 0 forces the CUDA-core NTT-domain kernel (also the fallback for any other weights); mode 2 takes the
 * tensor-core kernel for every eligible layer with fan-in >= min_fanin, however few outputs it has.
 * min_fanin <= 0 / scratch_bytes == 0 keep the current values (defaults 256, 12 GiB; layers with fewer than 32 outputs also
 * stay on the CUDA cores: measured on B200 the NTT-domain kernel wins for conv2 (fan-in 180) and fc4 (10 outputs)).  Env CRCNN_TC=0|1 sets the
 * initial mode. */
int crcnn_ctx_set_tensor_core_mode(crcnn_ctx *ctx, int mode, int min_fanin, size_t scratch_bytes);
/* Every other weighted sum (any plaintext weights: convolutions, small fully connected layers) runs in the NTT domain
 * as a limb-split GEMM on the same tensor cores: residues of weights and inputs are split into 7 byte planes, the 49
 * plane products accumulate per weight class in TMEM and are recombined and reduced once
 * (crcnn_b200/csrc/tcn_mac.cuh).  It needs primes of at most 56 bits and its staged weights (7 bytes per residue)
 * within the weight cache; otherwise, or with mode 0, the CUDA-core kernel runs.  Modes 2 and 3 force one of its two
 * kernel shapes (outputs / columns on the UMMA rows) instead of choosing by layer shape.  Env CRCNN_TCN sets the
 * initial mode (default 1).  The scratch budget is the one of crcnn_ctx_set_tensor_core_mode. */
int crcnn_ctx_set_limb_split_mode(crcnn_ctx *ctx, int mode);
/* How the limb-split GEMM turns its 13 class sums into a residue: mode 1 (default) uses the shape of SEAL's coefficient primes,
 * q = 2^k - delta with delta < 2^25 (SEAL/seal/util/globals.cpp:50-74): the classes are gathered into four sums, 2^56 and the bits
 * above k are folded through 2^56 mod q and delta, one conditional subtraction (crcnn_b200/csrc/modarith.cuh: tcn_fold_reduce); it
 * applies when every prime of the context has that shape (the engine checks: tcn_fold_make(q).ok), otherwise, or with mode 0, the classes are recombined into a 128-bit
 * integer and reduced by the generic Barrett step (barrett_reduce_128, SEAL/seal/util/uintarithsmallmod.h:137-176).  Both produce
 * the canonical residue, i.e. the same bytes.  Env CRCNN_TCN_FOLD sets the initial mode. */
int crcnn_ctx_set_limb_split_reduction(crcnn_ctx *ctx, int mode);
/* relinearize (Evaluator::relinearize, SEAL/seal/evaluator.cpp:886-1069): mode 1 (default) evaluates the digit (x) key
 * product sums over three or four NTT-friendly primes below 2^30 and reconstructs each coefficient exactly before reducing it
 * mod q_j (crcnn_b200/csrc/relin32.cuh) -- the same canonical residues from 32-bit transforms; it applies when
 * 2 * D * n * (2^dbc - 1) * max q_j is below the product of those primes (every SEAL default with dbc <= 16), otherwise, or
 * with mode 0, the 64-bit transforms of the reference's own procedure run. */
int crcnn_ctx_set_relin_mode(crcnn_ctx *ctx, int mode);
/* Derived constants, for cross-checking against SEAL: which = 0 root_powers, 1 scaled_root_powers,
 * 2 inv_root_powers_div_two, 3 scaled_inv_root_powers_div_two (SEAL/seal/util/smallntt.cpp:37-92);
 * slot in [0,K) = coefficient primes, [K,K+S) = Bsk primes.  out has n words. */
int crcnn_ctx_ntt_table(const crcnn_ctx *ctx, int slot, int which, uint64_t *out);
int crcnn_ctx_bsk_count(const crcnn_ctx *ctx);

/* ---- ciphertext tensors ------------------------------------------------------------------
 * Replaces: the ciphertext3D by-value hand-off between layers (CrCNN/src/globals.h:10). */
int crcnn_tensor_upload(crcnn_ctx *ctx, const uint64_t *host_words, long count, int ct_size, crcnn_tensor **out);
/* ntt_form != 0: the host data is already in NTT form (as after Evaluator::transform_to_ntt). */
int crcnn_tensor_upload_ex(crcnn_ctx *ctx, const uint64_t *host_words, long count, int ct_size, int ntt_form,
                           crcnn_tensor **out);
/* Double buffering: enqueue the host->device copy on a caller-owned copy stream so it overlaps the
 * forward pass running on the context's stream; call crcnn_ctx_wait_stream(ctx, copy_stream) before the
 * first use of the tensor.  host_words should be pinned and must stay valid until the copy has run. */
int crcnn_tensor_upload_on(crcnn_ctx *ctx, const uint64_t *host_words, long count, int ct_size, int ntt_form,
                           void *copy_stream, crcnn_tensor **out);
/* Steady-state form of the above: overwrite an EXISTING tensor (same count and ct_size) with new host data, through a
 * staging buffer the context keeps, so a serving loop that alternates between two input tensors allocates nothing per
 * request.  Enqueued on copy_stream (NULL: the context's stream); uploads sharing the staging buffer must use one
 * copy stream.  The tensor must not be in use by work still running on the context's stream. */
int crcnn_tensor_upload_into(crcnn_ctx *ctx, const uint64_t *host_words, crcnn_tensor *t, int ntt_form, void *copy_stream);
/* Make the context's stream wait for everything enqueued so far on other_stream (event, no host sync). */
int crcnn_ctx_wait_stream(crcnn_ctx *ctx, void *other_stream);
/* Always delivers coefficient form unless want_ntt_form != 0. Blocks until the copy has finished. */
int crcnn_tensor_download(crcnn_ctx *ctx, crcnn_tensor *t, uint64_t *host_words);
int crcnn_tensor_download_ex(crcnn_ctx *ctx, crcnn_tensor *t, int want_ntt_form, uint64_t *host_words);
int crcnn_tensor_free(crcnn_ctx *ctx, crcnn_tensor *t);
long crcnn_tensor_count(const crcnn_tensor *t);
int crcnn_tensor_ct_size(const crcnn_tensor *t);
/* New tensor holding ciphertexts [first, first+count) of t (device copy). */
int crcnn_tensor_slice(crcnn_ctx *ctx, crcnn_tensor *t, long first, long count, crcnn_tensor **out);
/* Raw device pointer (uint64[count][size][K][n]) and domain flag (0 coefficient, 1 NTT), for
 * collectives over NVLink done by the caller (NCCL all-gather of activations). */
int crcnn_tensor_device_ptr(crcnn_tensor *t, void **dev_ptr, int *ntt_form);
int crcnn_tensor_wrap_alloc(crcnn_ctx *ctx, long count, int ct_size, int ntt_form, crcnn_tensor **out);

/* ---- plaintext packs ----------------------------------------------------------------------
 * Replaces: plaintext2D/plaintext4D weights + vector<Plaintext> biases held by the layers
 * (CrCNN/src/convolutionalLayer.h:30-31, fullyConnectedLayer.h:19-20) and their lazy
 * Evaluator::transform_to_ntt(Plaintext&) (SEAL/seal/evaluator.cpp:1418-1493). */
/* `count` plaintexts, each `stride` words apart, of which the first coeff_count are significant. */
int crcnn_plain_upload(crcnn_ctx *ctx, const uint64_t *host_words, long count, int coeff_count, long stride,
                       crcnn_plain **out);
/* Sparse form: plaintext i has coefficients (idx[e], val[e]) for e in [offsets[i], offsets[i+1]). */
int crcnn_plain_upload_sparse(crcnn_ctx *ctx, const uint32_t *idx, const uint64_t *val, const uint32_t *offsets,
                              long count, crcnn_plain **out);
/* Encode floats exactly as CnnBuilder does: FractionalEncoder(t, x^n+1, 64, 32, base 3).encode(v)
 * (CrCNN/src/cnnBuilder.cpp:25-105, CrCNN/src/globals.cpp:52) -- SURVEY 8(f) row N1. */
int crcnn_plain_encode(crcnn_ctx *ctx, const float *values, long count, crcnn_plain **out);
/* The same encoder on doubles: FractionalEncoder::encode takes a double, and the reference hands it one where it does not come
 * from a float tensor -- AvgPoolingLayer's div_factor = encode(1./(xf*yf)) (CrCNN/src/avgPoolingLayer.cpp:10-13): for a window
 * area that is not a power of two the base-3 digits of the float and the double differ from about the 15th on. */
int crcnn_plain_encode_f64(crcnn_ctx *ctx, const double *values, long count, crcnn_plain **out);
/* Coefficient-form words of plaintext `index` (n+1 words, zero padded) -- for parity checks. */
int crcnn_plain_get(crcnn_ctx *ctx, const crcnn_plain *p, long index, uint64_t *out_words);
int crcnn_plain_free(crcnn_ctx *ctx, crcnn_plain *p);
long crcnn_plain_count(const crcnn_plain *p);

/* ---- evaluation keys -----------------------------------------------------------------------
 * Replaces: EvaluationKeys *ev_keys16 (CrCNN/src/globals.h:27).  host_words = keys_[0][i] back to
 * back for i in [0,K), each a ciphertext of sizes[i] polys in SEAL layout [sizes[i]][K][n+1]
 * (SEAL/seal/keygenerator.cpp:198-215, 652-702); dbc = decomposition bit count. */
int crcnn_evk_upload(crcnn_ctx *ctx, const uint64_t *host_words, int dbc, const int *sizes, crcnn_evk **out);
int crcnn_evk_free(crcnn_ctx *ctx, crcnn_evk *k);

/* ---- layers --------------------------------------------------------------------------------
 * Tensors are [batch][z][x][y] ciphertexts of size 2 (batch independent images; the reference
 * processes one image per forward call, i.e. batch = 1).  Each call returns a new tensor. */

/* Replaces ConvolutionalLayer::forward (CrCNN/src/convolutionalLayer.cpp:159-197, :56-93).
 * weights: nf*zd*xf*yf plaintexts in [nf][zd][xf][yf] order; biases: nf plaintexts. */
int crcnn_conv_forward(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *weights, crcnn_plain *biases, int batch,
                       int xd, int yd, int zd, int xs, int ys, int xf, int yf, int nf, crcnn_tensor **out);
/* As above for output channels [k0, k0+kc) only (output-neuron sharding across GPUs, SURVEY 8(e)). */
int crcnn_conv_forward_shard(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *weights, crcnn_plain *biases, int batch,
                             int xd, int yd, int zd, int xs, int ys, int xf, int yf, int nf, int k0, int kc,
                             crcnn_tensor **out);
/* Replaces FullyConnectedLayer::forward (CrCNN/src/fullyConnectedLayer.cpp:113-168); the input is
 * the row-major flattening reshapeInput produces (:38-56).  weights [out_dim][in_dim]. */
int crcnn_fc_forward(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *weights, crcnn_plain *biases, int batch,
                     int in_dim, int out_dim, crcnn_tensor **out);
int crcnn_fc_forward_shard(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *weights, crcnn_plain *biases, int batch,
                           int in_dim, int out_dim, int o0, int oc, crcnn_tensor **out);
/* Replaces PoolingLayer::forward (scale == NULL, CrCNN/src/poolingLayer.cpp:22-44) and
 * AvgPoolingLayer::forward (scale = pack holding encode(1/(xf*yf)), CrCNN/src/avgPoolingLayer.cpp:16-45). */
int crcnn_pool_forward(crcnn_ctx *ctx, crcnn_tensor *in, int batch, int xd, int yd, int zd, int xs, int ys, int xf,
                       int yf, crcnn_plain *scale, crcnn_tensor **out);
/* Replaces BatchNormLayer::forward (CrCNN/src/batchNormLayer.cpp:29-40): sub_plain(mean[z]) then
 * multiply_plain(invstd[z]). */
int crcnn_bn_forward(crcnn_ctx *ctx, crcnn_tensor *in, int batch, int zd, int xd, int yd, crcnn_plain *mean,
                     crcnn_plain *invstd, crcnn_tensor **out);
/* AvgPoolingLayer::forward immediately followed by BatchNormLayer::forward (CrCNN/src/avgPoolingLayer.cpp:16-45,
 * batchNormLayer.cpp:29-40 -- layers 1+2 and 5+6 of the reference's nine-layer networks, cnnBuilder.cpp:115-134) in one pass over
 * NTT-form activations: out = (window sum) * (scale (.) invstd_z) - mean_z (.) invstd_z, the same canonical residues as the two
 * calls.  Coefficient-form activations run the two layers one after the other.  The result has the batch-norm layer's shape.
 * scale = NULL: PoolingLayer (window sum without a factor, poolingLayer.cpp:23-47 -- the WoPad topology) in place of AvgPoolingLayer;
 * the same holds for crcnn_conv_pool_bn_forward and crcnn_pool_bn_fc_fc_forward. */
int crcnn_pool_bn_forward(crcnn_ctx *ctx, crcnn_tensor *in, int batch, int xd, int yd, int zd, int xs, int ys, int xf, int yf,
                          crcnn_plain *scale, crcnn_plain *mean, crcnn_plain *invstd, crcnn_tensor **out);
/* ConvolutionalLayer::forward, AvgPoolingLayer::forward and BatchNormLayer::forward in a row (layers 0-2 of the reference's
 * nine-layer networks, CrCNN/src/cnnBuilder.cpp:109-134; convolutionalLayer.cpp:136-196, avgPoolingLayer.cpp:16-45,
 * batchNormLayer.cpp:29-40), producing the batch-norm layer's output ciphertexts -- the same bytes as the three calls.  The work
 * is done on the pooled grid: the pooling windows are summed over the layer's INPUT (dilated by the convolution stride), the
 * convolution runs at stride (pool stride x conv stride) over those sums, and the pooling scale and the batch-norm are folded into
 * the convolution's weights and bias once (W' = W (.) scale (.) invstd_k, B' = |window| B (.) scale (.) invstd_k - mean_k (.) invstd_k,
 * NTT domain).  All three layers are affine over Z_q[x]/(x^n+1), so the canonical residues are identical while one weighted sum over
 * the pooled positions replaces three layers and two full-size intermediates.  Geometries where the combined stride exceeds the
 * filter, or contexts without the limb-split tensor-core GEMM, run crcnn_conv_forward + crcnn_pool_bn_forward.  conv: (xd,yd,zd)
 * input, stride (xs,ys), filter (xf,yf), nf kernels; pool: stride (pxs,pys), window (pxf,pyf).  Environment CRCNN_NO_POOLED_CONV=1
 * forces the layer-by-layer path (A/B timing, tests). */
int crcnn_conv_pool_bn_forward(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w, crcnn_plain *b, int batch, int xd, int yd, int zd,
                               int xs, int ys, int xf, int yf, int nf, int pxs, int pys, int pxf, int pyf, crcnn_plain *scale,
                               crcnn_plain *mean, crcnn_plain *invstd, crcnn_tensor **out);
/* Output channels [k0, k0+kc) of the same (one GPU's share of the reference's filter split, convolutionalLayer.cpp:177-187; pooling and
 * batch-norm are per channel).  Only on the pooled grid: CRCNN_ERR_UNSUPPORTED where the whole-layer call would fall back. */
int crcnn_conv_pool_bn_forward_shard(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w, crcnn_plain *b, int batch, int xd, int yd, int zd,
                                     int xs, int ys, int xf, int yf, int nf, int pxs, int pys, int pxf, int pyf, crcnn_plain *scale,
                                     crcnn_plain *mean, crcnn_plain *invstd, int k0, int kc, crcnn_tensor **out);
/* Two FullyConnectedLayer::forward calls in a row with no layer between them (fc3 -> fc4, the tail of every reference topology:
 * CrCNN/src/cnnBuilder.cpp:121-122, 132-133, 153-154; fullyConnectedLayer.cpp:96-166), producing the second layer's output
 * ciphertexts -- the same bytes as the two calls.  fc2(fc1(x)) = (W2 W1) x + (W2 Delta b1 + Delta b2) over Z_q[x]/(x^n+1): the composed
 * weights (out_dim x in_dim ring elements, NTT form, staged as byte planes for the limb-split GEMM) and bias are computed on the device
 * at the first call and kept in w1; every later call is ONE weighted sum with out_dim x in_dim terms instead of
 * mid_dim x (in_dim + out_dim).  Falls back to the two calls when that is not smaller, when the composed planes do not fit the weight
 * cache, or without the limb-split GEMM.  Environment CRCNN_NO_FC_COMPOSE=1 forces the two-call path (A/B timing, tests). */
int crcnn_fc_fc_forward(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_plain *w1, crcnn_plain *b1, crcnn_plain *w2, crcnn_plain *b2, int batch,
                        int in_dim, int mid_dim, int out_dim, crcnn_tensor **out);
/* AvgPoolingLayer, BatchNormLayer, FullyConnectedLayer, FullyConnectedLayer::forward in a row (layers 5-8 of the reference's
 * nine-layer networks, CrCNN/src/cnnBuilder.cpp:118-122), producing the last layer's output ciphertexts -- the same bytes as the four
 * calls: the pooling windows are summed, then ONE composed fully connected layer carries the pooling scale, the batch-norm and both
 * weight matrices (crcnn_fc_fc_forward's composition with W[k,r] (.)= scale (.) invstd_c(r) and B_k -= sum_r W[k,r] (.) mean_c(r) (.) invstd_c(r)).
 * (xd,yd,zd): input of the pooling layer; the first fully connected layer has zd * pooled positions inputs.  Falls back to
 * crcnn_pool_bn_forward + crcnn_fc_fc_forward under the conditions stated there. */
int crcnn_pool_bn_fc_fc_forward(crcnn_ctx *ctx, crcnn_tensor *in, int batch, int xd, int yd, int zd, int pxs, int pys, int pxf, int pyf,
                                crcnn_plain *scale, crcnn_plain *mean, crcnn_plain *invstd, crcnn_plain *w1, crcnn_plain *b1,
                                crcnn_plain *w2, crcnn_plain *b2, int mid_dim, int out_dim, crcnn_tensor **out);
/* Replaces SquareLayer::forward (CrCNN/src/squareLayer.cpp:22-71): Evaluator::square + relinearize. */
int crcnn_square_forward(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_evk *evk, crcnn_tensor **out);

/* ---- Evaluator-level operations (parity tests and the kernel sweep) --------------------------- */
/* Evaluator::transform_to_ntt / transform_from_ntt (SEAL/seal/evaluator.cpp:1495-1539); in place. */
int crcnn_transform_to_ntt(crcnn_ctx *ctx, crcnn_tensor *t);
int crcnn_transform_from_ntt(crcnn_ctx *ctx, crcnn_tensor *t);
/* Evaluator::transform_to_ntt(Plaintext&): K*(n+1) words of plaintext `index` in SEAL NTT form. */
int crcnn_plain_get_ntt(crcnn_ctx *ctx, crcnn_plain *p, long index, uint64_t *out_words);
/* op 0: Evaluator::multiply_plain (SEAL/seal/evaluator.cpp:1243-1416; also multiply_plain_ntt :1541-1585),
 * op 1: add_plain (:1145-1192), op 2: sub_plain (:1194-1241); plaintext `index` of the pack is applied
 * to every ciphertext of t, in place. */
int crcnn_plain_op(crcnn_ctx *ctx, crcnn_tensor *t, crcnn_plain *p, long index, int op);
/* Evaluator::add_many over all ciphertexts of t (SEAL/seal/evaluator.cpp:296-308) -> 1 ciphertext. */
int crcnn_add_many(crcnn_ctx *ctx, crcnn_tensor *t, crcnn_tensor **out);
/* Evaluator::square, size 2 -> 3 (SEAL/seal/evaluator.cpp:702-884). */
int crcnn_square(crcnn_ctx *ctx, crcnn_tensor *in, crcnn_tensor **out3);
/* Evaluator::relinearize, size 3 -> 2 (SEAL/seal/evaluator.cpp:886-1069). */
int crcnn_relinearize(crcnn_ctx *ctx, crcnn_tensor *in3, crcnn_evk *evk, crcnn_tensor **out2);

/* ---- host support for a serving loop ------------------------------------------------------------
 * Replaces: nothing in the reference (its inference loop, CrCNN/src/mainparams.cpp:64-116, is synchronous host code);
 * these are what a C++17 caller needs to drive the double-buffered loop of crcnn_tensor_upload_into without linking the
 * CUDA runtime itself: page-locked staging memory, a copy stream, events to order the streams and to time on the device. */
int crcnn_pinned_alloc(size_t bytes, void **out);
int crcnn_pinned_free(void *p);
int crcnn_stream_create(crcnn_ctx *ctx, void **stream);
int crcnn_stream_destroy(crcnn_ctx *ctx, void *stream);
int crcnn_event_create(crcnn_ctx *ctx, void **event);
int crcnn_event_record(crcnn_ctx *ctx, void *event, void *stream);      /* stream NULL: the context's stream */
int crcnn_stream_wait_event(crcnn_ctx *ctx, void *stream, void *event); /* stream NULL: the context's stream */
int crcnn_event_elapsed_ms(crcnn_ctx *ctx, void *first, void *second, double *ms); /* waits for `second` */
int crcnn_event_destroy(crcnn_ctx *ctx, void *event);
/* Enqueue the download of t (coefficient form, pad words written) into PINNED host memory on the context's stream and return;
 * the data is complete when an event recorded afterwards has fired.  Lets the score download of request i overlap request i+1. */
int crcnn_tensor_download_async(crcnn_ctx *ctx, crcnn_tensor *t, uint64_t *host_words);

/* ---- output-neuron sharding across GPUs ------------------------------------------------------------
 * Replaces: the reference's split of a layer's output filters / rows over std::threads
 * (CrCNN/src/convolutionalLayer.cpp:177-187, fullyConnectedLayer.cpp:148-158); across GPUs the same split is
 * crcnn_conv_forward_shard / crcnn_fc_forward_shard on every rank followed by this all-gather of the layer's output
 * ciphertexts over NVLink before the next layer that consumes every channel (SURVEY 8(e) item 3).
 * One process per GPU: rank 0 calls crcnn_comm_unique_id and hands the 128 bytes to the other ranks by any means (file, socket,
 * torch.distributed), every rank then calls crcnn_comm_create with its context.  NCCL is loaded at run time (libnccl.so.2;
 * env CRCNN_NCCL_LIB overrides), CRCNN_ERR_UNSUPPORTED if it is absent. */
int crcnn_comm_unique_id(void *id128);
int crcnn_comm_create(crcnn_ctx *ctx, const void *id128, int world, int rank, crcnn_comm **out);
int crcnn_comm_destroy(crcnn_ctx *ctx, crcnn_comm *comm);
/* local holds batch x counts[rank] ciphertexts ([batch][own channels][positions]); *out gets batch x sum(counts), image b being
 * rank 0's ciphertexts of b, then rank 1's, ... .  Enqueued on the context's stream as ONE NCCL group of sends / receives, no
 * host synchronisation.  want_ntt_form 0 / 1: every rank first brings its block into that domain; -1: the blocks are exchanged as
 * they are (all ranks of a sharded layer produce one domain: kernels are chosen from the layer's total output count). */
int crcnn_comm_all_gather(crcnn_ctx *ctx, crcnn_comm *comm, crcnn_tensor *local, int batch, const long *counts,
                          int want_ntt_form, crcnn_tensor **out);

/* ---- re-encryption on the device (opt-in) -----------------------------------------------------------
 * Replaces: the noise reset inside Network::forward (CrCNN/src/network.cpp:30-33): decryptImage -> encryptImage
 * (CrCNN/src/globals.cpp:127-142, 207-226), i.e. Decryptor::decrypt (SEAL/seal/decryptor.cpp:107-234), FractionalEncoder::decode,
 * the float the reference stores in its floatCube, FractionalEncoder::encode and Encryptor::encrypt
 * (SEAL/seal/encryptor.cpp:95-200) for every ciphertext of the tensor.  The reference runs it in-process with the SECRET key;
 * so does this, on the GPU -- uploading keys is the caller's decision and nothing else in the library touches key material.
 * secret_key_ntt: SecretKey::data() as SEAL keeps it, NTT form, uint64[K][n+1];  public_key_ntt: PublicKey::data(),
 * uint64[2][K][n+1], NTT form. */
int crcnn_keys_upload(crcnn_ctx *ctx, const uint64_t *secret_key_ntt, const uint64_t *public_key_ntt, crcnn_keys **out);
int crcnn_keys_free(crcnn_ctx *ctx, crcnn_keys *keys);   /* the device copy of the secret key is zeroed first */
/* Decryptor::decrypt of every (size-2) ciphertext of t: host_plain gets count plaintexts of n+1 words (values < t, pad word 0),
 * bit-identical to SEAL's. */
int crcnn_decrypt(crcnn_ctx *ctx, crcnn_keys *keys, crcnn_tensor *t, uint64_t *host_plain);
/* Decryptor::invariant_noise_budget (SEAL/seal/decryptor.cpp) of every size-2 ciphertext of t, either domain.
 * host_budgets: count ints (may be NULL); min_budget: the minimum over t (may be NULL). Needs the secret key. */
int crcnn_noise_budget(crcnn_ctx *ctx, crcnn_keys *keys, crcnn_tensor *t, int *host_budgets, int *min_budget);
/* decrypt -> decode -> (float) -> encode -> encrypt of every ciphertext of `in`, activations never leaving the device.  The three
 * sampled polynomials of an encryption (u uniform in {-1,0,1}; e0, e1 clipped normal, standard deviation
 * noise_standard_deviation (<= 0: SEAL's default 3.19), redrawn beyond 6 sigma, truncated toward zero) come from a counter-based
 * generator keyed by `seed` -- or, for byte-exact checks, from host_noise: int8[count][3][n] = u, e0, e1.  Optional outputs:
 * host_reencoded (count x (n+1) words: the plaintexts that were encrypted), host_values (count floats: the decoded values). */
int crcnn_reencrypt(crcnn_ctx *ctx, crcnn_keys *keys, crcnn_tensor *in, uint64_t seed, double noise_standard_deviation,
                    const int8_t *host_noise, crcnn_tensor **out, uint64_t *host_reencoded, float *host_values);

/* ---- the client's two ends on the device (opt-in, the same keys) ----------------------------------------
 * Replaces: encryptImage / decryptImage (CrCNN/src/globals.cpp:127-142, 207-233) for a key holder who runs the evaluator.
 * encryptImage's inner loop: FractionalEncoder(64, 32, base 3).encode((double) v) + Encryptor::encrypt for every value; *out is a
 * new coefficient-form tensor of `count` size-2 ciphertexts, ciphertext i encrypting host_values[i].  Noise as crcnn_reencrypt:
 * (seed, ciphertext index, coefficient) -> Philox, or host_noise int8[count][3][n] = u, e0, e1.  The values are encoded exactly as
 * crcnn_plain_encode encodes them, which accepts every float; SEAL leaves the integer part of a value outside the int64 range (and
 * NaN) undefined, and so does this call.
 * Seeds: the same (seed, ciphertext index) always draws the same u, e0, e1 -- in this call and in crcnn_reencrypt alike -- so a seed
 * must never serve two calls: two encryptions under one u reveal the difference of their plaintexts. */
int crcnn_encrypt_values(crcnn_ctx *ctx, crcnn_keys *keys, const float *host_values, long count, uint64_t seed,
                         double noise_standard_deviation, const int8_t *host_noise, crcnn_tensor **out);
/* decryptImage's inner loop: host_values[i] = (float) FractionalEncoder::decode(Decryptor::decrypt(ciphertext i of t)), size-2
 * ciphertexts in either domain; only the count floats leave the device. */
int crcnn_decrypt_values(crcnn_ctx *ctx, crcnn_keys *keys, crcnn_tensor *t, float *host_values);

/* ---- measurement ------------------------------------------------------------------------------
 * Kernel classes are timed with CUDA events on the context's stream while profiling is on. */
int crcnn_prof_enable(crcnn_ctx *ctx, int on);
int crcnn_prof_reset(crcnn_ctx *ctx);
int crcnn_prof_count(crcnn_ctx *ctx); /* number of kernel classes */
/* name: >= 32 bytes.  launches counts since the last reset (always maintained); ms only while enabled. */
int crcnn_prof_get(crcnn_ctx *ctx, int cls, char *name, long *launches, double *ms);
/* Algorithmic work enqueued for class `cls` since the last reset (SURVEY 8(d) figures, counted at launch time):
 * bytes = compulsory HBM bytes (every distinct input and output once); ops = butterflies for the NTT classes
 * (ntt_forward, ntt_inverse, plain_expand_ntt, relinearize), 64x64->128-bit multiply-accumulates or modular
 * multiplies for the CUDA-core classes, int8 multiply-accumulates for weighted_sum_tc_i8. */
int crcnn_prof_get_work(crcnn_ctx *ctx, int cls, double *bytes, double *ops);
/* Register-only 64x64->128-bit multiply-accumulate probe (integer-pipe roofline): runs
 * blocks*threads*iters*8 MACs and returns the elapsed device time in ms. */
int crcnn_probe_imad(crcnn_ctx *ctx, int blocks, int threads, int iters, double *ms);
/* Roofline denominators measured on the device the context is bound to, at the clocks of the run (SURVEY 8(d): "integer-pipe
 * peak must be measured on the box"); *ops = operations issued, *ms = elapsed device time.
 *   which 0: the dependent 64x64->128-bit multiply-accumulate chain above          (ops = multiply-accumulates)
 *   which 1: independent IMAD.WIDE.U32 chains, nothing else in the loop: the issue-rate ceiling of the pipe every 64-bit
 *            modular product runs on (4 IMAD.WIDE per 64x64 product)                (ops = IMAD.WIDE thread-instructions)
 *   which 2: tcgen05.mma kind::i8, M128 x N256 x K32, operands resident in shared memory, no epilogue, one CTA per SM
 *            (blocks = SM count, threads ignored)                                   (ops = int8 multiply-accumulates) */
int crcnn_probe_pipe(crcnn_ctx *ctx, int which, int blocks, int threads, int iters, double *ms, double *ops);

#ifdef __cplusplus
}
#endif
#endif
