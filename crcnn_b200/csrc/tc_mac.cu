// tcgen05 kind::i8 weighted-sum path (see tc_mac.cuh for the algorithm and the exactness argument).
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdio>
#include "devcfg.cuh"
#include "modarith.cuh"
#include "tc_mac.cuh"
#include "tc_ptx.cuh"

namespace crcnn {

namespace {

constexpr int TC_A_STAGE = TC_BM * TC_BK;  // 16 KB
constexpr int TC_THREADS = 192;            // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr int TC_ACC_STRIDE = 256;         // TMEM columns between the two accumulator buffers
constexpr int TC_SCRATCH_WARP = 64 * 32 * 4;

using namespace tcptx;

// ------------------------------------------------------------------------------------ the GEMM kernel
template <int PLANES>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_mac_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
              const DeviceParams *__restrict__ P, TcMacArgs a) {
    constexpr int N = PLANES * TC_CB;               // UMMA N: 224 or 256
    constexpr int B_BLK = N * TC_BK;                // 28 / 32 KB
    // two 128-byte K blocks per ring stage (2 stages of 88 KB, half as many barrier flips and tcgen05.commits as four stages of
    // 44 KB): fc3 of the bench 64.8 -> 62.1 ms on B200
    constexpr int SUB = 2;
    constexpr int TC_STAGES = 4 / SUB;
    constexpr int NACC = 2;                                 // accumulators in tensor memory
    constexpr uint32_t TMEM_COLS = 512;
    constexpr int SCRATCH = 4 * TC_SCRATCH_WARP;
    constexpr int A_STAGE = SUB * TC_A_STAGE, B_STAGE = SUB * B_BLK;
    constexpr uint32_t IDESC = (2u << 4)            // accumulator format S32
                               | (1u << 7)          // A = signed 8 bit
                               | (0u << 10)         // B = unsigned 8 bit
                               | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);  // K-major A and B

    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t sA = base, sB = base + TC_STAGES * A_STAGE;
    const uint32_t off_scratch = TC_STAGES * (A_STAGE + B_STAGE);
    const uint32_t off_bar = off_scratch + SCRATCH;
    const uint32_t bar_full = base + off_bar, bar_empty = bar_full + 8 * TC_STAGES;
    const uint32_t bar_tfull = bar_empty + 8 * TC_STAGES, bar_tempty = bar_tfull + 16;
    const uint32_t tmem_slot = bar_tempty + 16;
    volatile uint32_t *tmem_slot_ptr = reinterpret_cast<volatile uint32_t *>(base_ptr + off_bar + 16 * TC_STAGES + 32);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = a.n, K = a.K;
    const int m_tiles = a.Mpad / TC_BM;
    const long items = (long)a.npos * 2 * K * m_tiles;
    const int NU = n / TC_CB + 1;                   // coefficient blocks incl. the negated wrap-around block
    const int ksteps = (a.R + 31) / 32;
    const int KBLK = (ksteps + 3) / 4;                // 128-byte K blocks
    const int KB = (KBLK + SUB - 1) / SUB;            // ring stages per coefficient block

    if (threadIdx.x == 0) {
        for (int s = 0; s < TC_STAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int s = 0; s < 2; s++) { mbar_init(bar_tfull + 8 * s, 1); mbar_init(bar_tempty + 8 * s, 4); }
        fence_barrier_init();
        prefetch_tmap(&tmA);
        prefetch_tmap(&tmB);
    }
    if (warp == 0) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp == 0) {
        // ===================================================================== TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (long item = blockIdx.x; item < items; item += gridDim.x) {
                const int g = (int)(item / m_tiles), mt = (int)(item % m_tiles);
                for (int u = 0; u < NU; u++)
                    for (int kb = 0; kb < KB; kb++) {
                        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                        const int nsub = min(SUB, KBLK - kb * SUB);
                        mbar_expect_tx(bar_full + 8 * stage, nsub * (TC_A_STAGE + B_BLK));
                        for (int sb = 0; sb < nsub; sb++) {
                            tma_load_2d(sA + stage * A_STAGE + sb * TC_A_STAGE, &tmA, bar_full + 8 * stage, (kb * SUB + sb) * TC_BK, mt * TC_BM);
                            tma_load_4d(sB + stage * B_STAGE + sb * B_BLK, &tmB, bar_full + 8 * stage, (kb * SUB + sb) * TC_BK, u * TC_CB, 0, g);
                        }
                        if (++stage == TC_STAGES) { stage = 0; phase ^= 1; }
                    }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================================================================== MMA issuer
        if (lane == 0) {
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (long item = blockIdx.x; item < items; item += gridDim.x)
                for (int u = 0; u < NU; u++) {
                    mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + acc * TC_ACC_STRIDE;
                    for (int kb = 0; kb < KB; kb++) {
                        mbar_wait(bar_full + 8 * stage, phase);
                        tc_fence_after();
                        for (int sb = 0; sb < SUB && kb * SUB + sb < KBLK; sb++) {
                            const uint64_t da = umma_desc_sw128(sA + stage * A_STAGE + sb * TC_A_STAGE), db = umma_desc_sw128(sB + stage * B_STAGE + sb * B_BLK);
                            const int nks = min(4, ksteps - (kb * SUB + sb) * 4);
                            for (int ks = 0; ks < nks; ks++)
                                umma_i8(d_tmem, da + 2 * ks, db + 2 * ks, IDESC, (kb | sb | ks) != 0);  // +32 B per K-step
                        }
                        umma_commit(bar_empty + 8 * stage);
                        if (++stage == TC_STAGES) { stage = 0; phase ^= 1; }
                    }
                    umma_commit(bar_tfull + 8 * acc);
                    if (++acc == NACC) { acc = 0; acc_phase ^= 1; }
                }
        }
        __syncwarp();
    } else {
        // ===================================================================== epilogue
        const int lg = warp & 3;  // TMEM lane group this warp may read = output (mt*4 + lg), lane = tap-1
        int *S = reinterpret_cast<int *>(base_ptr + off_scratch + (warp - 2) * TC_SCRATCH_WARP);
        int acc = 0;
        uint32_t acc_phase = 0;
        for (long item = blockIdx.x; item < items; item += gridDim.x) {
            const int g = (int)(item / m_tiles), mt = (int)(item % m_tiles);
            const int j = g % K, poly = (g / K) & 1, p = g / (2 * K);
            const int m = mt * 4 + lg;
            const bool valid = m < a.M;
            const Mod mod = P->tab[j].mod;
            // offset q * 2^s >= 2^84 that makes the signed plane sum non-negative before the reduction
            const int s = 85 - (64 - __clzll(mod.q));
            const uint64_t off_lo = mod.q << s, off_hi = mod.q >> (64 - s);
            const int pg = a.p0 + p;  // position index within the whole layer
            const long oct = (long)(pg / a.Pimg) * ((long)a.Mtotal * a.Pimg) + (long)(a.m0 + m) * a.Pimg + pg % a.Pimg;
            uint64_t *optr = a.out + ((oct * 2 + poly) * K + j) * (long)n;
            const uint64_t *bptr = (a.bias && poly == 0 && valid) ? a.bias + ((long)m * K + j) * n : nullptr;
            int carry[PLANES];
#pragma unroll
            for (int l = 0; l < PLANES; l++) carry[l] = 0;
            for (int u = 0; u < NU; u++) {
                mbar_wait(bar_tfull + 8 * acc, acc_phase);
                tc_fence_after();
                int lo[PLANES], hi[PLANES];
#pragma unroll
                for (int l = 0; l < PLANES; l++) {
                    int v[32];
                    tmem_ld32(tmem_base + ((uint32_t)(lg * 32) << 16) + acc * TC_ACC_STRIDE + l * TC_CB, v);
                    // D[(m,tap), cc] belongs to output coefficient cc - tap of this block (tap = lane+1):
                    // skew into S[cc - tap + 32][lane]; rows < 32 finish the previous block, rows >= 32 start this one
                    // D[(m,tap), cc] belongs to output coefficient cc - tap of this block (tap = lane+1):
                    // skew into S[cc - tap + 32][lane]; rows < 32 finish the previous block, rows >= 32 start this one
#pragma unroll
                    for (int cc = 0; cc < 32; cc++) S[(cc - lane + 31) * 32 + lane] = v[cc];
                    __syncwarp();
                    int slo = 0, shi = 0;
#pragma unroll
                    for (int st = 0; st < 32; st++) {
                        const int i = (st + lane) & 31;
                        const bool is_lo = i >= 31 - lane;
                        const int val = S[(lane + (is_lo ? 0 : 32)) * 32 + i];
                        slo += is_lo ? val : 0;
                        shi += is_lo ? 0 : val;
                    }
                    __syncwarp();
                    lo[l] = slo;
                    hi[l] = shi;
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
                if (++acc == NACC) { acc = 0; acc_phase ^= 1; }
                if (u >= 1 && valid) {
                    long long v0 = 0, v1 = 0;
#pragma unroll
                    for (int l = 0; l < PLANES; l++) {
                        const long long pl = (long long)(carry[l] + lo[l]);
                        if (l < 4) v0 += pl << (8 * l); else v1 += pl << (8 * (l - 4));
                    }
                    // total = v0 + v1 * 2^32 as a 128-bit two's complement number, plus the offset
                    U128 z;
                    const uint64_t t_lo = (uint64_t)v1 << 32;
                    z.lo = (uint64_t)v0 + t_lo;
                    z.hi = (uint64_t)(v0 >> 63) + (uint64_t)(v1 >> 32) + (z.lo < t_lo);
                    const uint64_t l2 = z.lo + off_lo;
                    z.hi += off_hi + (l2 < off_lo);
                    z.lo = l2;
                    uint64_t r = barrett128(z, mod);
                    const int c = (u - 1) * TC_CB + lane;
                    if (bptr) r = addmod(r, __ldg(bptr + c), mod.q);
                    optr[c] = r;
                }
#pragma unroll
                for (int l = 0; l < PLANES; l++) carry[l] = hi[l];
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------ tensor-pipe roofline probe
// kind::i8 UMMA peak of this GPU: one CTA per SM issues M = 128, N = 256, K = 32 tcgen05.mma instructions back to back on operand
// tiles that stay in shared memory (no TMA, no epilogue), alternating between two TMEM accumulators.  What it measures is the
// denominator of the tensor-bound kernels' roofline fraction (int8 multiply-accumulates per second), on the box and at the clocks
// of the run -- not a figure derived from the bf16 GEMM of MEASURED_PEAKS.json.
// VAR 0: N = 256, one operand tile reused by every MMA (the peak).  VAR 1: N = 224 (the ternary GEMM's tile), same.  VAR 2: N = 224,
// operands taken in turn from four 44 KB stages, tcgen05.commit after every fourth MMA (the ternary GEMM's issue pattern without
// its TMA traffic and epilogue).
template <int VAR>
__global__ void __launch_bounds__(128, 1)
umma_i8_probe_kernel(int iters) {
    constexpr int N = VAR == 0 ? 256 : 224;
    constexpr int NST = VAR == 2 ? 4 : 1;
    constexpr int STAGE = (TC_BM + N) * TC_BK;
    constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (0u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *bp = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t bar = base + NST * STAGE, tmem_slot = bar + 64;
    for (int i = threadIdx.x; i < NST * STAGE / 4; i += blockDim.x)
        reinterpret_cast<uint32_t *>(bp)[i] = 0x01010101u * (uint32_t)((i * 2654435761u) >> 28);   // small bytes: products stay far from overflow
    if (threadIdx.x == 0) { for (int b = 0; b < 5; b++) mbar_init(bar + 8 * b, 1); fence_barrier_init(); }
    fence_proxy_async();
    if (threadIdx.x < 32) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(bp + (tmem_slot - base));
    if (threadIdx.x == 0) {
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int half = 0; half < 2; half++) {
                const uint32_t st = VAR == 2 ? (uint32_t)((2 * it + half) & 3) : 0u;
                const uint64_t da = umma_desc_sw128(base + st * STAGE), db = umma_desc_sw128(base + st * STAGE + TC_BM * TC_BK);
#pragma unroll
                for (int ks = 0; ks < 4; ks++) umma_i8(tmem_base + half * 256, da + 2 * ks, db + 2 * ks, IDESC, (it | ks) != 0);
                if (VAR == 2) umma_commit(bar + 8 * (1 + st));     // nobody waits on these: the cost of the commit itself
            }
        }
        umma_commit(bar);
        mbar_wait(bar, 0);
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------ operand staging
// Gathers the layer's input ciphertexts per output position, splits every residue into byte planes and
// writes them transposed (fan-in index contiguous) with the 32 negated wrap-around coefficients appended:
//   B[g][l][c][r] = byte l of X~_(in_index[p][r])[poly][j][c],   g = (p*2 + poly)*K + j,  c in [0, n+32)
__global__ void __launch_bounds__(256)
tc_split_kernel(const DeviceParams *__restrict__ P, TcMacArgs a) {
    __shared__ uint64_t tile[32][133];    // [c][(r & 3) * 33 + (r >> 2)]; row stride 133 = 5 mod 16: conflict free both ways
    const int n = a.n, K = a.K;
    const int ct = blockIdx.x;            // coefficient block, n/32 = the wrap-around block
    const int g = blockIdx.y;
    const int r0 = blockIdx.z * 128;
    const int j = g % K, poly = (g / K) & 1, p = g / (2 * K);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t q = P->tab[j].mod.q;
    const bool wrap = ct == n / 32;
    for (int rr = warp; rr < 128; rr += 8) {
        const int r = r0 + rr;
        uint64_t v = 0;
        const long ctx = r < a.R ? __ldg(a.in_index + (long)p * a.R + r) : -1;
        if (ctx >= 0) {             // index -1: a padded border's zero ciphertext, zero wrap coefficients included
            const uint64_t *src = a.x + ((ctx * 2 + poly) * K + j) * (long)n;
            if (!wrap) v = __ldg(src + ct * 32 + lane);
            else { v = __ldg(src + lane); v = v ? q - v : 0; }
        }
        tile[lane][(rr & 3) * 33 + (rr >> 2)] = v;
    }
    __syncthreads();
    const long plane_stride = (long)(n + 32) * a.Kpad;
    uint8_t *dst = a.B + (long)g * a.planes * plane_stride + (long)(ct * 32) * a.Kpad + r0;
    for (int w = threadIdx.x; w < a.planes * 1024; w += 256) {
        const int l = w >> 10, c = (w >> 5) & 31, rw = w & 31;
        const int sh = 8 * l;
        const uint32_t word = (uint32_t)((tile[c][rw] >> sh) & 0xff) | (uint32_t)((tile[c][33 + rw] >> sh) & 0xff) << 8 |
                              (uint32_t)((tile[c][66 + rw] >> sh) & 0xff) << 16 | (uint32_t)((tile[c][99 + rw] >> sh) & 0xff) << 24;
        *reinterpret_cast<uint32_t *>(dst + l * plane_stride + (long)c * a.Kpad + 4 * rw) = word;
    }
}

// ------------------------------------------------------------------------------------ host side
template <int PLANES>
size_t tc_smem_bytes() {
    return 1024 + (size_t)4 * (TC_A_STAGE + PLANES * TC_CB * TC_BK) + 4 * TC_SCRATCH_WARP + 16 * 4 + 32 + 16;
}

template <int PLANES>
cudaError_t launch_tc_mac_t(const DeviceParams *P, const TcMacArgs &a, int sm_count, cudaStream_t stream) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return cudaErrorNotSupported;
    CUtensorMap tmA, tmB;
    {
        cuuint64_t dims[2] = {(cuuint64_t)a.Kpad, (cuuint64_t)a.Mpad};
        cuuint64_t strides[1] = {(cuuint64_t)a.Kpad};
        cuuint32_t box[2] = {TC_BK, TC_BM}, es[2] = {1, 1};
        if (enc(&tmA, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, (void *)a.A, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    {
        const cuuint64_t rows = (cuuint64_t)a.n + 32, groups = (cuuint64_t)a.npos * 2 * a.K;
        cuuint64_t dims[4] = {(cuuint64_t)a.Kpad, rows, (cuuint64_t)PLANES, groups};
        cuuint64_t strides[3] = {(cuuint64_t)a.Kpad, rows * a.Kpad, rows * a.Kpad * PLANES};
        cuuint32_t box[4] = {TC_BK, TC_CB, PLANES, 1}, es[4] = {1, 1, 1, 1};
        if (enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, (void *)a.B, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    const size_t smem = tc_smem_bytes<PLANES>();
    static DeviceOnce once;
    if (once.first()) {
        cudaError_t e = cudaFuncSetAttribute(tc_mac_kernel<PLANES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const long items = (long)a.npos * 2 * a.K * (a.Mpad / TC_BM);
    const unsigned grid = (unsigned)(items < sm_count ? items : sm_count);
    tc_mac_kernel<PLANES><<<grid, TC_THREADS, smem, stream>>>(tmA, tmB, P, a);
    return cudaGetLastError();
}

}  // namespace

size_t tc_b_bytes(const TcMacArgs &a) { return (size_t)a.npos * 2 * a.K * a.planes * (size_t)(a.n + 32) * a.Kpad; }

cudaError_t tc_mac_available() { return encode_tiled() ? cudaSuccess : cudaErrorNotSupported; }

// blocks CTAs (one per SM), iters * 8 UMMAs of 128 x N x 32 each; *macs = int8 multiply-accumulates issued in total
template <int VAR>
static cudaError_t launch_umma_probe_t(int blocks, int iters, double *macs, cudaStream_t stream) {
    constexpr int N = VAR == 0 ? 256 : 224;
    const size_t smem = 1024 + (size_t)(VAR == 2 ? 4 : 1) * (TC_BM + N) * TC_BK + 128;
    static DeviceOnce once;
    if (once.first()) {
        cudaError_t e = cudaFuncSetAttribute(umma_i8_probe_kernel<VAR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    umma_i8_probe_kernel<VAR><<<blocks, 128, smem, stream>>>(iters);
    if (macs) *macs = (double)blocks * iters * 8.0 * TC_BM * N * 32;
    return cudaGetLastError();
}
cudaError_t launch_umma_i8_probe(int blocks, int iters, int variant, double *macs, cudaStream_t stream) {
    if (variant == 1) return launch_umma_probe_t<1>(blocks, iters, macs, stream);
    if (variant == 2) return launch_umma_probe_t<2>(blocks, iters, macs, stream);
    return launch_umma_probe_t<0>(blocks, iters, macs, stream);
}

cudaError_t launch_tc_split(const DeviceParams *P, const TcMacArgs &a, cudaStream_t stream) {
    if (a.npos <= 0) return cudaSuccess;
    dim3 grid((unsigned)(a.n / 32 + 1), (unsigned)(a.npos * 2 * a.K), (unsigned)(a.Kpad / 128));
    tc_split_kernel<<<grid, 256, 0, stream>>>(P, a);
    return cudaGetLastError();
}

cudaError_t launch_tc_mac(const DeviceParams *P, const TcMacArgs &a, int sm_count, cudaStream_t stream) {
    if (a.npos <= 0 || a.M <= 0) return cudaSuccess;
    if (a.Kpad % TC_BK || a.Mpad % TC_BM || a.n % TC_CB || (long)a.npos * 2 * a.K > 65535) return cudaErrorInvalidValue;
    if (a.planes == 7) return launch_tc_mac_t<7>(P, a, sm_count, stream);
    if (a.planes == 8) return launch_tc_mac_t<8>(P, a, sm_count, stream);
    return cudaErrorInvalidValue;
}

}  // namespace crcnn
