// Limb-split tensor-core realisation of the plaintext-weight weighted sum in the NTT domain -- the "int8
// limb-split tcgen05 kind::i8 path" of BASELINE.json's north_star, for ANY plaintext weights (tc_mac.cuh covers
// ternary-tap weights in the coefficient domain; this one is what convolutional layers use).
//
// In NTT form a layer is, independently for every slot s = (limb j, position c) of the transform,
//       Y[m][col] = sum_r W[m][r][s] * X[col][r][s]   mod q_j,        col = (output position p, polynomial 0/1),
// a small dense GEMM of 55-bit residues (conv2 of PlainModel.h5: 50 x 576 x 180 for each of 32768 slots).  Both
// operands are split into 7 (8) unsigned byte planes, W = sum_a Wa 2^(8a), X = sum_b Xb 2^(8b), so that
//       Y = sum_{w=0..12} 2^(8w) * S_w,      S_w = sum_{a+b=w} sum_r Wa[m][r] * Xb[col][r]
// and every S_w is a u8 x u8 -> s32 GEMM accumulated in ONE TMEM accumulator (at most 7 plane pairs share a
// weight class; 7 * R * 255^2 < 2^31 for R <= 4096).  The epilogue recombines the 13 classes into a 128-bit
// integer and reduces it mod q_j once: the same canonical residue multiply_plain_ntt + add_many produce.
//
// Kernel shapes: one persistent CTA per SM, warp 0 = TMA producer, warp 1 = tcgen05.mma.cta_group::1.kind::i8 issuer,
// warps 2-9 = epilogue (tcgen05.ld of the 13 classes -> 128-bit recombination -> Barrett -> bias -> store).  The 7 planes
// of one operand are stacked along N, so ONE MMA of N = 7 x 32 multiplies a plane of the other operand with all of
// them and its 7 products land in 7 consecutive weight classes (TMEM columns [32 (a+b), +32)); 7 MMAs per K step.
//   tcn_mac_kernel   (fully connected shapes: few columns): outputs on the UMMA rows, M = 64, work item = slot x 64 outputs,
//                    columns in chunks of 32, weight and input planes streamed per K block
//   tcn2_mac_kernel  (convolutions: many columns, few outputs): columns on the UMMA rows, M = 128, work item = slot x 32
//                    outputs whose weight planes stay resident in shared memory, input planes streamed one per stage
// Operand staging (tcn_split_kernel) gathers the layer's inputs per output position and writes byte planes with
// the fan-in index contiguous (K-major); weights are staged once per layer the same way.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "params.h"

namespace crcnn {

constexpr int TCN_BM = 64;     // outputs per tile (UMMA M)
constexpr int TCN_NB = 32;     // columns per chunk (UMMA N)
constexpr int TCN_MAX_R = 4096;

// byte planes of a residue of this context (7 for <= 56-bit primes, else 8)
inline int tcn_planes_for(const DeviceParams &d) {
    int maxbits = 0;
    for (int j = 0; j < d.K; j++) {
        int b = 0;
        for (uint64_t v = d.tab[j].mod.q; v; v >>= 1) b++;
        maxbits = b > maxbits ? b : maxbits;
    }
    return maxbits <= 56 ? 7 : 8;
}

// Row pitch (bytes) of the staged operands for fan-in R, and the K block the kernel streams:
// R <= 32: 32-byte rows, one K step (32B swizzle); otherwise rows padded to a multiple of 32 (at least 128) and
// K blocks of 128 bytes (128B swizzle; the tail of the last block is filled with zeros by TMA).
inline int tcn_kpad(int R) { return R <= 32 ? 32 : ((R + 31) / 32 * 32 < 128 ? 128 : (R + 31) / 32 * 32); }
inline int tcn_bk(int R) { return R <= 32 ? 32 : 128; }

struct TcnSplitArgs {
    const uint64_t *src;   // items of `item_polys` limb-polynomial groups: [item][item_polys][K][n], NTT form
    const int *index;      // [ncols / item_polys][R] item of (column group, term r); null: item = group * R + r
    uint8_t *dst;          // [slot - slot0][planes][ncols][Kpad]
    int item_polys;        // 2 for ciphertexts (column = position * 2 + poly), 1 for plaintext weights (column = output)
    int R, Kpad, planes, ncols;
    int slot0, nslots;     // slots (j * n + c) of this launch; slot0 and nslots are multiples of 32
    int n, K;
};

struct TcnMacArgs {
    const uint8_t *W;      // staged weights [K*n][planes][Mall][Kpad]
    const uint8_t *X;      // staged inputs  [nslots][planes][ncols][Kpad]
    const uint64_t *bias;  // [Mall][K][n] NTT of the Delta-scaled bias (may be null), added to polynomial 0
    uint64_t *out;         // output ciphertext of (position p, output m): (p / Pimg) * (Mtotal * Pimg) + (m0 + m) * Pimg + p % Pimg
    int Mall, m_first, M;  // outputs [m_first, m_first + M) of the layer's Mall
    int R, Kpad, planes, ncols;
    int slot0, nslots;
    int Pimg, Mtotal, m0;
    int n, K;
    int use_fold;          // 1: reduce the class sums with tcn_fold_reduce when fold[j].ok for every prime (0: 128-bit recombination + Barrett)
    TcnFold fold[MAXK];    // per coefficient prime (modarith.cuh: tcn_fold_make)
    int variant;           // 0: pick by shape; 1: outputs on the UMMA rows (64 x 32 tiles); 2: columns on the UMMA rows (128 x 32 tiles, fan-in <= 256)
    int preshift;          // 1: W holds the pre-shifted planes [7 (b)][K*n][planes][Mall][Kpad] (W 2^(8b) mod q_j; block b = 0 is the
                           //    plain staging) and the shape is tcn_preshift_shape: seven-class kernel.  0: 13-class kernels on block 0
};

size_t tcn_x_bytes_per_slot(int planes, int ncols, int Kpad);
size_t tcn_w_bytes(int planes, int Mall, int Kpad, int K, int n);
cudaError_t launch_tcn_split(const TcnSplitArgs &a, cudaStream_t stream);
// shapes that run on pre-shifted weights: fan-in <= 32 on the column-major kernel (variant as in TcnMacArgs)
bool tcn_preshift_shape(int R, int ncols, int M, int variant);
// dst = src 2^(8b) mod q_j for every residue of `words` limb-major words ([..][K][n]); q = the K primes (host array), 1 <= b <= 6
cudaError_t launch_tcn_preshift(const uint64_t *q, const uint64_t *src, uint64_t *dst, long words, int b, int n, int K, cudaStream_t stream);
cudaError_t launch_tcn_mac(const DeviceParams *P, const TcnMacArgs &a, int sm_count, cudaStream_t stream);

}  // namespace crcnn
