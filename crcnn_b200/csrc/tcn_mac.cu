// NTT-domain limb-split weighted sum on tcgen05 kind::i8 (see tcn_mac.cuh for the algorithm and the exactness argument).
#include <cuda.h>
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdio>
#include "devcfg.cuh"
#include "modarith.cuh"
#include "tc_ptx.cuh"
#include "tcn_mac.cuh"

namespace crcnn {

namespace {

using namespace tcptx;

constexpr int TCN_PLANES = 7;
constexpr int TCN_CLASSES = 2 * TCN_PLANES - 1;       // weight classes a + b
constexpr int TCN_EPI_WARPS = 8;
constexpr int TCN_THREADS = 32 * (2 + TCN_EPI_WARPS);  // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue
constexpr int TCN_TMEM_COLS = 512;                     // 13 classes x 32 columns = 416 used

// sum_w S_w 2^(8w) of the 13 weight classes of one output as a 128-bit integer.  Classes 0,4,8,12 are whole words;
// 1,5,9 / 2,6,10 / 3,7,11 are three more word-aligned numbers shifted by 8 / 16 / 24 bits: 9 funnel shifts and three
// 4-word carry chains.
__device__ __forceinline__ U128 tcn_combine(const uint32_t (&S)[TCN_CLASSES][4], int i) {
    uint32_t z0 = S[0][i], z1 = S[4][i], z2 = S[8][i], z3 = S[12][i];
#define CRCNN_ADD4(a0, a1, a2, a3)                                                                                     \
    asm("add.cc.u32 %0, %0, %4;\n\taddc.cc.u32 %1, %1, %5;\n\taddc.cc.u32 %2, %2, %6;\n\taddc.u32 %3, %3, %7;"          \
        : "+r"(z0), "+r"(z1), "+r"(z2), "+r"(z3)                                                                       \
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3))
    CRCNN_ADD4(S[1][i] << 8, __funnelshift_l(S[1][i], S[5][i], 8), __funnelshift_l(S[5][i], S[9][i], 8), S[9][i] >> 24);
    CRCNN_ADD4(S[2][i] << 16, __funnelshift_l(S[2][i], S[6][i], 16), __funnelshift_l(S[6][i], S[10][i], 16), S[10][i] >> 16);
    CRCNN_ADD4(S[3][i] << 24, __funnelshift_l(S[3][i], S[7][i], 24), __funnelshift_l(S[7][i], S[11][i], 24), S[11][i] >> 8);
#undef CRCNN_ADD4
    U128 z;
    z.lo = ((uint64_t)z1 << 32) | z0;
    z.hi = ((uint64_t)z3 << 32) | z2;
    return z;
}

// output i of a group of four through the folded reduction (modarith.cuh: tcn_fold_reduce); bias = 0 when there is none
__device__ __forceinline__ uint64_t tcn_fold_out(const uint32_t (&S)[TCN_CLASSES][4], int i, uint64_t bias, const TcnFold &f, uint64_t q) {
    uint32_t s[TCN_CLASSES];
#pragma unroll
    for (int w = 0; w < TCN_CLASSES; w++) s[w] = S[w][i];
    return tcn_fold_reduce(s, bias, f, q);
}

template <int BK> struct TcnCfg {
    static constexpr int A_STAGE = TCN_PLANES * TCN_BM * BK;   // weight planes of one K block
    static constexpr int B_STAGE = TCN_PLANES * TCN_NB * BK;   // input planes of one K block
    static constexpr int STAGES = BK == 128 ? 2 : 4;
    static constexpr size_t SMEM = 1024 + (size_t)STAGES * (A_STAGE + B_STAGE) + 8 * (2 * STAGES + 2) + 16;
};

// ------------------------------------------------------------------------------------ the GEMM kernel
template <int BK, bool FOLD>
__global__ void __launch_bounds__(TCN_THREADS, 1)
tcn_mac_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmX,
               const DeviceParams *__restrict__ P, TcnMacArgs a) {
    using Cfg = TcnCfg<BK>;
    constexpr int STAGES = Cfg::STAGES, A_STAGE = Cfg::A_STAGE, B_STAGE = Cfg::B_STAGE;
    constexpr uint32_t IDESC_BASE = (2u << 4)   // accumulator format S32; A and B formats 0 = unsigned 8 bit, both K-major; N is added per MMA
                                    | ((uint32_t)(TCN_BM >> 4) << 24);

    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t sA = base, sB = base + STAGES * A_STAGE;
    const uint32_t off_bar = STAGES * (A_STAGE + B_STAGE);
    const uint32_t bar_full = base + off_bar, bar_empty = bar_full + 8 * STAGES;
    const uint32_t bar_tfull = bar_empty + 8 * STAGES, bar_tempty = bar_tfull + 8;
    const uint32_t tmem_slot = bar_tempty + 8;
    volatile uint32_t *tmem_slot_ptr = reinterpret_cast<volatile uint32_t *>(base_ptr + off_bar + 8 * (2 * STAGES + 2));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = a.n;
    const int m_tiles = (a.M + TCN_BM - 1) / TCN_BM;
    const long items = (long)a.nslots * m_tiles;
    const int chunks = (a.ncols + TCN_NB - 1) / TCN_NB;
    const int ksteps = (a.R + 31) / 32;
    const int KB = (ksteps * 32 + BK - 1) / BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        mbar_init(bar_tfull, 1);
        mbar_init(bar_tempty, TCN_EPI_WARPS);
        fence_barrier_init();
        prefetch_tmap(&tmW);
        prefetch_tmap(&tmX);
    }
    if (warp == 0) tmem_alloc(tmem_slot, TCN_TMEM_COLS);
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
                const int sl = (int)(item / m_tiles), mt = (int)(item % m_tiles);
                for (int ch = 0; ch < chunks; ch++)
                    for (int kb = 0; kb < KB; kb++) {
                        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                        mbar_expect_tx(bar_full + 8 * stage, A_STAGE + B_STAGE);
                        tma_load_4d(sA + stage * A_STAGE, &tmW, bar_full + 8 * stage, kb * BK, mt * TCN_BM, 0, a.slot0 + sl);
                        tma_load_4d(sB + stage * B_STAGE, &tmX, bar_full + 8 * stage, kb * BK, ch * TCN_NB, 0, sl);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================================================================== MMA issuer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (long item = blockIdx.x; item < items; item += gridDim.x)
                for (int ch = 0; ch < chunks; ch++) {
                    mbar_wait(bar_tempty, acc_phase ^ 1);
                    tc_fence_after();
                    for (int kb = 0; kb < KB; kb++) {
                        mbar_wait(bar_full + 8 * stage, phase);
                        tc_fence_after();
                        const uint32_t aS = sA + stage * A_STAGE, bS = sB + stage * B_STAGE;
                        const int nks = BK == 128 ? min(4, ksteps - kb * 4) : 1;
                        // One MMA per weight plane pa: its B operand is ALL input planes stacked (N = 7 x 32), so the product with
                        // input plane pb lands in columns [32 (pa + pb), +32) = weight class pa + pb.  The first K step of a chunk
                        // must overwrite: plane 0 initialises classes 0-6, plane 6 against input planes 1-6 initialises 7-12.
                        for (int ks = 0; ks < nks; ks++) {
                            const bool fresh = (kb | ks) == 0;
                            auto descA = [&](int pa) { return (BK == 128 ? umma_desc_sw128(aS + pa * (TCN_BM * BK)) : umma_desc_sw32(aS + pa * (TCN_BM * BK))) + 2 * ks; };
                            auto descB = [&](int pb) { return (BK == 128 ? umma_desc_sw128(bS + pb * (TCN_NB * BK)) : umma_desc_sw32(bS + pb * (TCN_NB * BK))) + 2 * ks; };
                            constexpr uint32_t ID_ALL = IDESC_BASE | ((uint32_t)((TCN_PLANES * TCN_NB) >> 3) << 17);
                            constexpr uint32_t ID_HI = IDESC_BASE | ((uint32_t)(((TCN_PLANES - 1) * TCN_NB) >> 3) << 17);
                            constexpr uint32_t ID_ONE = IDESC_BASE | ((uint32_t)(TCN_NB >> 3) << 17);
                            if (fresh) {
                                umma_i8(tmem_base, descA(0), descB(0), ID_ALL, 0u);
                                umma_i8(tmem_base + TCN_PLANES * TCN_NB, descA(TCN_PLANES - 1), descB(1), ID_HI, 0u);
                                umma_i8(tmem_base + (TCN_PLANES - 1) * TCN_NB, descA(TCN_PLANES - 1), descB(0), ID_ONE, 1u);
#pragma unroll
                                for (int pa = 1; pa < TCN_PLANES - 1; pa++) umma_i8(tmem_base + pa * TCN_NB, descA(pa), descB(0), ID_ALL, 1u);
                            } else {
#pragma unroll
                                for (int pa = 0; pa < TCN_PLANES; pa++) umma_i8(tmem_base + pa * TCN_NB, descA(pa), descB(0), ID_ALL, 1u);
                            }
                        }
                        umma_commit(bar_empty + 8 * stage);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                    umma_commit(bar_tfull);
                    acc_phase ^= 1;
                }
        }
        __syncwarp();
    } else {
        // ===================================================================== epilogue
        // UMMA M = 64 keeps output row m in TMEM lane (m % 16) + 32 * (m / 16): a warp owns lane quadrant warp % 4,
        // lanes 0-15 of it hold rows; the two warps of a quadrant split the chunk's 8 groups of 4 columns
        const int qd = warp & 3, half = (warp - 2) >> 2;
        const long pw = (long)a.K * n;
        uint32_t acc_phase = 0;
        for (long item = blockIdx.x; item < items; item += gridDim.x) {
            const int sl = (int)(item / m_tiles), mt = (int)(item % m_tiles);
            const int slot = a.slot0 + sl, j = slot / n, c = slot - j * n;
            const Mod mod = P->tab[j].mod;
            const TcnFold fold = a.fold[FOLD ? j : 0];
            const int m = mt * TCN_BM + qd * 16 + lane;     // output row of this thread (lanes >= 16 hold nothing)
            const bool valid = lane < 16 && m < a.M;
            const uint64_t bias = (a.bias && valid) ? __ldg(a.bias + (long)m * pw + (long)j * n + c) : 0;
            const long row_off = (long)(a.m0 + m) * a.Pimg;
            for (int ch = 0; ch < chunks; ch++) {
                mbar_wait(bar_tfull, acc_phase);
                tc_fence_after();
#pragma unroll 1
                for (int g = 0; g < 4; g++) {
                    const int col0 = ch * TCN_NB + (half * 4 + g) * 4;
                    uint32_t S[TCN_CLASSES][4];
#pragma unroll
                    for (int w = 0; w < TCN_CLASSES; w++)
                        tmem_ld4(tmem_base + ((uint32_t)(qd * 32) << 16) + w * TCN_NB + (half * 4 + g) * 4, S[w]);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const int col = col0 + i;
                        if (!valid || col >= a.ncols) continue;
                        const int p = col >> 1, poly = col & 1;
                        uint64_t r;
                        if constexpr (FOLD) {
                            r = tcn_fold_out(S, i, poly == 0 ? bias : 0, fold, mod.q);   // bias is 0 without a bias pack
                        } else {
                            r = barrett128(tcn_combine(S, i), mod);
                            if (poly == 0 && a.bias) r = addmod(r, bias, mod.q);
                        }
                        const long oct = (long)(p / a.Pimg) * ((long)a.Mtotal * a.Pimg) + row_off + p % a.Pimg;
                        a.out[((oct * 2 + poly) * a.K + j) * (long)n + c] = r;
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_tempty);
                acc_phase ^= 1;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, TCN_TMEM_COLS);
}

// ------------------------------------------------------------------------------------ the GEMM kernel, column-major variant
// For layers with many columns and few outputs (convolutions: 576 / 3136 columns, 50 / 20 outputs) the roles swap:
// the COLUMNS fill the 128 UMMA rows (A operand = one input plane, [128 columns][BK]) and the outputs sit on the N
// side (B operand = all 7 weight planes of a tile of 32 outputs stacked, N = 224), so one MMA per input plane and K
// step covers 128 columns -- 4x the work per tensor-pipe cycle of the 64-row form for these shapes -- and every
// epilogue lane holds a column.  The weights of a work item (slot, 32 outputs) stay resident in shared memory
// (fan-in of at most 2 K blocks); input planes stream through a ring, one plane tile per stage.
constexpr int TCN2_CB = 128;   // columns per chunk (UMMA M)
constexpr int TCN2_MT = 32;    // outputs per tile (N per weight class)
constexpr int TCN2_KBMAX = 2;
constexpr int TCN2_EPI_WARPS = 12;                      // three per TMEM lane quadrant
constexpr int TCN2_THREADS = 32 * (2 + TCN2_EPI_WARPS);

// -DCRCNN_TCN2_TRACE: CTA 0 records clock64() at the hand-over points of its three roles (tools/tcn2_trace.py reads them
// back).  Every record costs a global-memory round trip (~340 cycles): compare intervals that contain the same number of records.
#ifdef CRCNN_TCN2_TRACE
constexpr int TCN2_TRACE_N = 8192;
__device__ unsigned long long g_tcn2_trace[3][TCN2_TRACE_N];
__device__ int g_tcn2_trace_n[3];
#define TCN2_TR(role, tag)                                                                                    \
    do {                                                                                                      \
        if (blockIdx.x == 0) {                                                                                \
            const int i_ = g_tcn2_trace_n[role];                                                              \
            if (i_ < TCN2_TRACE_N) { g_tcn2_trace[role][i_] = ((unsigned long long)(tag) << 56) | (clock64() & 0xffffffffffffffull); g_tcn2_trace_n[role] = i_ + 1; } \
        }                                                                                                     \
    } while (0)
#else
#define TCN2_TR(role, tag) do { } while (0)
#endif

template <int BK> struct Tcn2Cfg {
    static constexpr int W_BLOCK = TCN_PLANES * TCN2_MT * BK;   // weight planes of one K block: [7][32][BK]
    static constexpr int X_STAGE = TCN2_CB * BK;                // one input plane of one K block: [128][BK]
    static constexpr int NS = BK == 32 ? 4 : 1;                 // consecutive slots per work item (see tcn2_mac_kernel)
    // ring depth: measured on B200, 40 / 9 stages instead of 8 / 6 made conv1 slower (42.6 -> 62.8 ms) and left conv2 unchanged,
    // although 39 % of the samples of the 8-stage kernel wait on the accumulator-full barrier (profiles/r01f_ncu_source_top.txt)
    static constexpr int STAGES = BK == 128 ? 6 : 8;
    static constexpr size_t BARS = (8 * (2 * STAGES + 4) + 16 + 127) / 128 * 128;   // barriers + TMEM slot, padded so that the output staging is 128-byte aligned
    // staged: results of the first NS - 1 slots of an item wait in shared memory, [slot][output][column] words, for the whole-sector store
    static constexpr size_t smem(bool staged) {
        const size_t ops = 1024 + (size_t)NS * TCN2_KBMAX * W_BLOCK + (size_t)STAGES * X_STAGE;
        return staged ? ops + BARS + (size_t)(NS - 1) * TCN2_MT * TCN2_CB * 8 : ops + 8 * (2 * STAGES + 4) + 16;
    }
};

// one 256-bit store: a whole 32-byte sector from one thread (STG.E.256, sm_100)
__device__ __forceinline__ void tcn_store_sector(uint64_t *p, uint64_t a, uint64_t b, uint64_t c, uint64_t d) {
    asm volatile("st.global.v4.u64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}

// NS = Tcn2Cfg<BK>::NS consecutive slots per work item.  BK 128 (fan-in > 32): one slot per item.  BK 32 (fan-in <= 32: conv1):
// the four slots of one 32-byte output sector belong to ONE item, loop order chunk-outer / slot-inner with the four slots' weight
// planes resident, so a sector's four 8-byte writes come from the same thread a few microseconds apart instead of from four CTAs
// that have to stay in step (DESIGN.md section 6, "Correction").
// STAGED (BK 32 only): the results of slots 0-2 wait in shared memory (each thread reads back only what it wrote, no
// synchronisation) and slot 3 writes all four as ONE 32-byte sector per (column, output): a quarter of the sector writes.
template <int BK, bool FOLD, bool STAGED = false>
__global__ void __launch_bounds__(TCN2_THREADS, 1)
tcn2_mac_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmX,
                const DeviceParams *__restrict__ P, TcnMacArgs a) {
    using Cfg = Tcn2Cfg<BK>;
    constexpr int NS = Cfg::NS, STAGES = Cfg::STAGES, W_BLOCK = Cfg::W_BLOCK, X_STAGE = Cfg::X_STAGE;
    static_assert(!STAGED || NS == 4, "the staged whole-sector store needs four slots per item");
    constexpr uint32_t IDESC_BASE = (2u << 4) | ((uint32_t)(TCN2_CB >> 4) << 24);  // S32 accumulators, u8 x u8, K-major, M = 128
    constexpr uint32_t ID_ALL = IDESC_BASE | ((uint32_t)((TCN_PLANES * TCN2_MT) >> 3) << 17);
    constexpr uint32_t ID_HI = IDESC_BASE | ((uint32_t)(((TCN_PLANES - 1) * TCN2_MT) >> 3) << 17);
    constexpr uint32_t ID_ONE = IDESC_BASE | ((uint32_t)(TCN2_MT >> 3) << 17);

    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t sW = base, sX = base + NS * TCN2_KBMAX * W_BLOCK;
    const uint32_t off_bar = NS * TCN2_KBMAX * W_BLOCK + STAGES * X_STAGE;
    const uint32_t bar_full = base + off_bar, bar_empty = bar_full + 8 * STAGES;
    const uint32_t bar_wfull = bar_empty + 8 * STAGES, bar_wempty = bar_wfull + 8;
    const uint32_t bar_tfull = bar_wempty + 8, bar_tempty = bar_tfull + 8;
    const uint32_t tmem_slot = bar_tempty + 8;
    volatile uint32_t *tmem_slot_ptr = reinterpret_cast<volatile uint32_t *>(base_ptr + off_bar + 8 * (2 * STAGES + 4));
    uint64_t *out_stage = reinterpret_cast<uint64_t *>(base_ptr + off_bar + Cfg::BARS);   // [NS - 1][TCN2_MT][TCN2_CB], STAGED only

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = a.n;
    const int m_tiles = (a.M + TCN2_MT - 1) / TCN2_MT;
    // item = (group of NS consecutive slots, output tile).  A CTA takes slot groups round robin and runs ALL output tiles of a group back to
    // back: the second tile streams the group's input planes again, now from L2 (conv2: 4.3 MB per slot) instead of from DRAM -- with the
    // tiles of a group on neighbouring CTAs the kernel read 26.8 GB for 12.5 GB of staged planes (ncu r01g).
    const long groups = a.nslots / NS;
    const long items = (groups > blockIdx.x ? (groups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0) * m_tiles;   // items of THIS CTA
    auto item_group = [&](long it) { return (long)blockIdx.x + (it / m_tiles) * gridDim.x; };
    const int chunks = (a.ncols + TCN2_CB - 1) / TCN2_CB;
    const int ksteps = (a.R + 31) / 32;
    const int KB = (ksteps * 32 + BK - 1) / BK;   // <= TCN2_KBMAX (checked by the launcher)

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        mbar_init(bar_wfull, 1);
        mbar_init(bar_wempty, 1);
        mbar_init(bar_tfull, 1);
        mbar_init(bar_tempty, TCN2_EPI_WARPS);
        fence_barrier_init();
        prefetch_tmap(&tmW);
        prefetch_tmap(&tmX);
    }
    if (warp == 0) tmem_alloc(tmem_slot, TCN_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    // input planes are streamed in the order 0, 6, 1, 2, 3, 4, 5: planes 0 and 6 initialise the 13 weight classes
    auto plane_of = [](int bi) { return bi == 0 ? 0 : (bi == 1 ? TCN_PLANES - 1 : bi - 1); };

    if (warp == 0) {
        // ===================================================================== TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0, wphase = 0;
            for (long item = 0; item < items; item++) {
                const int sl = (int)item_group(item) * NS, mt = (int)(item % m_tiles);
                mbar_wait(bar_wempty, wphase ^ 1);
                mbar_expect_tx(bar_wfull, NS * KB * W_BLOCK);
                for (int s = 0; s < NS; s++)
                    for (int kb = 0; kb < KB; kb++)
                        tma_load_4d(sW + (s * TCN2_KBMAX + kb) * W_BLOCK, &tmW, bar_wfull, kb * BK, mt * TCN2_MT, 0, a.slot0 + sl + s);
                wphase ^= 1;
                for (int ch = 0; ch < chunks; ch++)
                    for (int s = 0; s < NS; s++)
                        for (int kb = 0; kb < KB; kb++)
                            for (int bi = 0; bi < TCN_PLANES; bi++) {
                                mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                                TCN2_TR(0, bi);                         // stage free: load of plane bi issued now
                                mbar_expect_tx(bar_full + 8 * stage, X_STAGE);
                                tma_load_4d(sX + stage * X_STAGE, &tmX, bar_full + 8 * stage, kb * BK, ch * TCN2_CB, plane_of(bi), sl + s);
                                if (++stage == STAGES) { stage = 0; phase ^= 1; }
                            }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================================================================== MMA issuer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0, acc_phase = 0, wphase = 0;
            for (long item = 0; item < items; item++) {
                mbar_wait(bar_wfull, wphase);
                wphase ^= 1;
                tc_fence_after();
                for (int chs = 0; chs < chunks * NS; chs++) {       // (chunk, slot of the item), slot fastest
                    const int s = NS == 1 ? 0 : chs % NS;
                    TCN2_TR(1, 100);                                // waiting for the accumulator
                    mbar_wait(bar_tempty, acc_phase ^ 1);
                    TCN2_TR(1, 101);                                // accumulator free
                    tc_fence_after();
                    for (int kb = 0; kb < KB; kb++) {
                        const uint32_t wS = sW + (s * TCN2_KBMAX + kb) * W_BLOCK;
                        const int nks = BK == 128 ? min(4, ksteps - kb * 4) : 1;
                        for (int bi = 0; bi < TCN_PLANES; bi++) {
                            const int pb = plane_of(bi);
                            mbar_wait(bar_full + 8 * stage, phase);
                            TCN2_TR(1, kb * 8 + bi);                    // plane tile arrived
                            tc_fence_after();
                            const uint32_t xS = sX + stage * X_STAGE;
                            for (int ks = 0; ks < nks; ks++) {
                                const uint64_t dx = (BK == 128 ? umma_desc_sw128(xS) : umma_desc_sw32(xS)) + 2 * ks;
                                auto descW = [&](int pa) { return (BK == 128 ? umma_desc_sw128(wS + pa * (TCN2_MT * BK)) : umma_desc_sw32(wS + pa * (TCN2_MT * BK))) + 2 * ks; };
                                // D[column, (class, output)]: input plane pb against all weight planes lands in classes pb .. pb+6
                                if ((kb | ks) == 0 && pb == 0) {
                                    umma_i8(tmem_base, dx, descW(0), ID_ALL, 0u);
                                } else if ((kb | ks) == 0 && pb == TCN_PLANES - 1) {
                                    umma_i8(tmem_base + TCN_PLANES * TCN2_MT, dx, descW(1), ID_HI, 0u);         // classes 7-12: overwrite
                                    umma_i8(tmem_base + (TCN_PLANES - 1) * TCN2_MT, dx, descW(0), ID_ONE, 1u);  // class 6: accumulate
                                } else {
                                    umma_i8(tmem_base + pb * TCN2_MT, dx, descW(0), ID_ALL, 1u);
                                }
                            }
                            umma_commit(bar_empty + 8 * stage);
                            if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        }
                    }
                    umma_commit(bar_tfull);
                    TCN2_TR(1, 102);                                // all MMAs of the chunk issued
                    acc_phase ^= 1;
                }
                umma_commit(bar_wempty);   // every MMA that reads this item's weights has been issued before this commit
            }
        }
        __syncwarp();
    } else {
        // ===================================================================== epilogue
        // UMMA M = 128: TMEM lane = column of the chunk; a warp owns lane quadrant warp % 4, the three warps of a
        // quadrant take the tile's groups of 4 outputs round robin
        const int qd = warp & 3, sub = (warp - 2) >> 2;
        const long pw = (long)a.K * n;
        const long m_stride = 2L * a.Pimg * pw;      // words between consecutive outputs of one column
        uint32_t acc_phase = 0;
        for (long item = 0; item < items; item++) {
            const int sl = (int)item_group(item) * NS, mt = (int)(item % m_tiles);
            const int slot = a.slot0 + sl, j = slot / n, c = slot - j * n;   // first slot of the item; its NS slots share the limb j (n and slot0 are multiples of NS)
            const Mod mod = P->tab[j].mod;
            const TcnFold fold = a.fold[FOLD ? j : 0];
            const long slot_off = (long)j * n + c;
            const int m_valid = min(TCN2_MT, a.M - mt * TCN2_MT);
            const int groups = (m_valid + 3) >> 2;
            // the bias residue of output m of this item does not depend on the column: lane m fetches it once per item and the
            // loop below broadcasts it by shuffle (a load per output inside the loop put an L2 round trip into every output's chain)
            uint64_t bias_lane[NS];
#pragma unroll
            for (int s = 0; s < NS; s++)
                bias_lane[s] = (a.bias && lane < m_valid) ? __ldg(a.bias + (long)(mt * TCN2_MT + lane) * pw + slot_off + s) : 0;
            for (int ch = 0; ch < chunks; ch++) {
                const int col = ch * TCN2_CB + qd * 32 + lane;
                const bool valid = col < a.ncols;
                const int p = col >> 1, poly = col & 1;
                const long colbase = (long)(p / a.Pimg) * ((long)a.Mtotal * a.Pimg) + p % a.Pimg;
                uint64_t *out_col = a.out + (colbase * 2 + poly) * pw + slot_off + (long)(a.m0 + mt * TCN2_MT) * m_stride;
                const bool add_bias = poly == 0;
#pragma unroll
              for (int s = 0; s < NS; s++) {                    // slot sl + s of the item: residue position c + s
                if (warp == 2 && lane == 0) TCN2_TR(2, 200);    // waiting for the accumulator
                mbar_wait(bar_tfull, acc_phase);
                if (warp == 2 && lane == 0) TCN2_TR(2, 201);    // accumulator complete
                tc_fence_after();
#pragma unroll 1
                for (int g = sub; g < groups; g += TCN2_EPI_WARPS / 4) {
                    const int mloc = g * 4;
                    uint32_t S[TCN_CLASSES][4];
#pragma unroll
                    for (int w = 0; w < TCN_CLASSES; w++)
                        tmem_ld4(tmem_base + ((uint32_t)(qd * 32) << 16) + w * TCN2_MT + mloc, S[w]);
                    tmem_ld_wait();
                    uint64_t *op = out_col + (long)mloc * m_stride + s;
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        if (mloc + i < m_valid) {                // warp uniform
                            const uint64_t bias_m = __shfl_sync(0xffffffffu, bias_lane[s], mloc + i);
                            uint64_t r;
                            if constexpr (FOLD) {
                                r = tcn_fold_out(S, i, add_bias ? bias_m : 0, fold, mod.q);
                            } else {
                                r = barrett128(tcn_combine(S, i), mod);
                                if (add_bias) r = addmod(r, bias_m, mod.q);
                            }
                            if constexpr (STAGED) {
                                uint64_t *st = out_stage + (mloc + i) * TCN2_CB + qd * 32 + lane;
                                if (s < NS - 1) st[s * (TCN2_MT * TCN2_CB)] = r;
                                else if (valid) tcn_store_sector(op - (NS - 1), st[0], st[TCN2_MT * TCN2_CB], st[2 * TCN2_MT * TCN2_CB], r);
                            } else if (valid) *op = r;
                        }
                        op += m_stride;
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_tempty);
                if (warp == 2 && lane == 0) TCN2_TR(2, 202);    // this warp's share of the chunk recombined and stored
                acc_phase ^= 1;
              }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, TCN_TMEM_COLS);
}

// ------------------------------------------------------------------------------------ the column-major GEMM on pre-shifted weights
// The weights are staged as W'_b = W 2^(8b) mod q_j for b = 0..6, each split into its 7 byte planes W'_(b,a).  Then
//       W X = sum_b X_b W'_b = sum_a 2^(8a) C_a  (mod q_j),      C_a = sum_b sum_r Xb[col][r] W'_(b,a)[m][r],
// SEVEN classes instead of 13 (C_a <= 7 R 255^2 < 2^31 as before; the recombined value is < 2^80).  Input plane b is
// multiplied against the 7 stacked planes of W'_b (N = 224) into the SAME 224 accumulator columns for every b: no
// column shift, no special first step, and two accumulators fit TMEM (2 x 224 of 512 columns), so the epilogue of one
// (chunk, slot) runs while the MMAs of the next one are issued.  Fan-in <= 32 (one 32-byte K block: conv1) and four
// consecutive slots per item, as tcn2_mac_kernel<32, .>: the pre-shifted planes of the four slots stay resident
// (4 x 49 KB), which leaves no shared memory for output staging -- instead each epilogue thread keeps the results of
// slots 0-2 in registers and slot 3 writes all four as one 32-byte sector (STAGED, layers of at most 24 outputs).
constexpr int TCN2P_NS = 4;
constexpr int TCN2P_WB = TCN_PLANES * TCN2_MT * 32;           // one b block [a][32 outputs][32 bytes]
constexpr int TCN2P_WSLOT = TCN_PLANES * TCN2P_WB;            // [b][a][32][32] of one slot
constexpr int TCN2P_X = TCN2_CB * 32;                         // one input plane tile [128][32]
constexpr int TCN2P_STAGES = 7;
constexpr int TCN2P_ACC = TCN_PLANES * TCN2_MT;               // 224 columns per accumulator
// groups of 4 outputs per epilogue warp: 3 cover a 32-output tile; the STAGED kernel keeps 2 x 4 x 3 results in registers and
// takes tiles of at most 24 outputs (3 groups would need more registers than 448 threads can have)
template <bool STAGED> __host__ __device__ constexpr int tcn2p_gpw() { return STAGED ? 2 : (TCN2_MT / 4 + TCN2_EPI_WARPS / 4 - 1) / (TCN2_EPI_WARPS / 4); }
constexpr int TCN2P_STAGED_MAX_M = 4 * 2 * (TCN2_EPI_WARPS / 4);
constexpr size_t TCN2P_SMEM = 1024 + (size_t)TCN2P_NS * TCN2P_WSLOT + (size_t)TCN2P_STAGES * TCN2P_X + 8 * (2 * TCN2P_STAGES + 6) + 16;

template <bool FOLD, bool STAGED>
__global__ void __launch_bounds__(TCN2_THREADS, 1)
tcn2p_mac_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmX,
                 const DeviceParams *__restrict__ P, TcnMacArgs a) {
    constexpr int NS = TCN2P_NS, STAGES = TCN2P_STAGES, GPW = tcn2p_gpw<STAGED>();
    constexpr uint32_t ID = (2u << 4) | ((uint32_t)(TCN2_CB >> 4) << 24) | ((uint32_t)(TCN2P_ACC >> 3) << 17);   // S32, u8 x u8, M 128, N 224

    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t sW = base, sX = base + NS * TCN2P_WSLOT;
    const uint32_t off_bar = NS * TCN2P_WSLOT + STAGES * TCN2P_X;
    const uint32_t bar_full = base + off_bar, bar_empty = bar_full + 8 * STAGES;
    const uint32_t bar_wfull = bar_empty + 8 * STAGES, bar_wempty = bar_wfull + 8;
    const uint32_t bar_tfull = bar_wempty + 8, bar_tempty = bar_tfull + 16;   // one pair per accumulator
    const uint32_t tmem_slot = bar_tempty + 16;
    volatile uint32_t *tmem_slot_ptr = reinterpret_cast<volatile uint32_t *>(base_ptr + off_bar + 8 * (2 * STAGES + 6));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = a.n;
    const int m_tiles = (a.M + TCN2_MT - 1) / TCN2_MT;
    const long groups = a.nslots / NS;
    const long items = (groups > blockIdx.x ? (groups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0) * m_tiles;   // items of THIS CTA
    auto item_group = [&](long it) { return (long)blockIdx.x + (it / m_tiles) * gridDim.x; };
    const int chunks = (a.ncols + TCN2_CB - 1) / TCN2_CB;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        mbar_init(bar_wfull, 1);
        mbar_init(bar_wempty, 1);
        for (int b = 0; b < 2; b++) { mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, TCN2_EPI_WARPS); }
        fence_barrier_init();
        prefetch_tmap(&tmW);
        prefetch_tmap(&tmX);
    }
    if (warp == 0) tmem_alloc(tmem_slot, TCN_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp == 0) {
        // ===================================================================== TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0, wphase = 0;
            for (long item = 0; item < items; item++) {
                const int sl = (int)item_group(item) * NS, mt = (int)(item % m_tiles);
                mbar_wait(bar_wempty, wphase ^ 1);
                mbar_expect_tx(bar_wfull, NS * TCN2P_WSLOT);
                for (int s = 0; s < NS; s++) tma_load_5d(sW + s * TCN2P_WSLOT, &tmW, bar_wfull, 0, mt * TCN2_MT, 0, a.slot0 + sl + s, 0);
                wphase ^= 1;
                for (int ch = 0; ch < chunks; ch++)
                    for (int s = 0; s < NS; s++)
                        for (int b = 0; b < TCN_PLANES; b++) {
                            mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                            TCN2_TR(0, b);                          // stage free: load of plane b issued now
                            mbar_expect_tx(bar_full + 8 * stage, TCN2P_X);
                            tma_load_4d(sX + stage * TCN2P_X, &tmX, bar_full + 8 * stage, 0, ch * TCN2_CB, b, sl + s);
                            if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================================================================== MMA issuer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0, wphase = 0, use = 0;   // use: accumulator fills so far; buffer use & 1, its phase (use >> 1) & 1
            for (long item = 0; item < items; item++) {
                mbar_wait(bar_wfull, wphase);
                wphase ^= 1;
                tc_fence_after();
                for (int chs = 0; chs < chunks * NS; chs++, use++) {   // (chunk, slot of the item), slot fastest
                    const int s = chs % NS;
                    const uint32_t buf = use & 1;
                    TCN2_TR(1, 100);                                // waiting for the accumulator
                    mbar_wait(bar_tempty + 8 * buf, ((use >> 1) & 1) ^ 1);
                    TCN2_TR(1, 101);                                // accumulator free
                    tc_fence_after();
                    const uint32_t acc = tmem_base + buf * TCN2P_ACC;
                    for (int b = 0; b < TCN_PLANES; b++) {
                        mbar_wait(bar_full + 8 * stage, phase);
                        TCN2_TR(1, b);                              // plane tile arrived
                        tc_fence_after();
                        // D[column, (a, output)] += X_b[column] . W'_(b,a)[output]
                        umma_i8(acc, umma_desc_sw32(sX + stage * TCN2P_X), umma_desc_sw32(sW + s * TCN2P_WSLOT + b * TCN2P_WB), ID, b ? 1u : 0u);
                        umma_commit(bar_empty + 8 * stage);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                    umma_commit(bar_tfull + 8 * buf);
                    TCN2_TR(1, 102);                                // all MMAs of the chunk issued
                }
                umma_commit(bar_wempty);   // every MMA that reads this item's weights has been issued before this commit
            }
        }
        __syncwarp();
    } else {
        // ===================================================================== epilogue
        // TMEM lane = column of the chunk; a warp owns lane quadrant warp % 4, the three warps of a quadrant take the tile's
        // groups of 4 outputs round robin (at most GPW each)
        const int qd = warp & 3, sub = (warp - 2) >> 2;
        const long pw = (long)a.K * n;
        const long m_stride = 2L * a.Pimg * pw;      // words between consecutive outputs of one column
        uint32_t use = 0;
        for (long item = 0; item < items; item++) {
            const int sl = (int)item_group(item) * NS, mt = (int)(item % m_tiles);
            const int slot = a.slot0 + sl, j = slot / n, c = slot - j * n;   // first slot of the item; its NS slots share the limb j
            const Mod mod = P->tab[j].mod;
            const TcnFold fold = a.fold[FOLD ? j : 0];
            const long slot_off = (long)j * n + c;
            const int m_valid = min(TCN2_MT, a.M - mt * TCN2_MT);
            const int groups = (m_valid + 3) >> 2;
            // lane m holds the bias residues of output m of this item; the loop broadcasts them by shuffle
            uint64_t bias_lane[NS];
#pragma unroll
            for (int s = 0; s < NS; s++)
                bias_lane[s] = (a.bias && lane < m_valid) ? __ldg(a.bias + (long)(mt * TCN2_MT + lane) * pw + slot_off + s) : 0;
            for (int ch = 0; ch < chunks; ch++) {
                const int col = ch * TCN2_CB + qd * 32 + lane;
                const bool valid = col < a.ncols;
                const int p = col >> 1, poly = col & 1;
                const long colbase = (long)(p / a.Pimg) * ((long)a.Mtotal * a.Pimg) + p % a.Pimg;
                uint64_t *out_col = a.out + (colbase * 2 + poly) * pw + slot_off + (long)(a.m0 + mt * TCN2_MT) * m_stride;
                const bool add_bias = poly == 0 && a.bias != nullptr;
                uint64_t keep[GPW][4][NS - 1];    // STAGED: results of slots 0 .. NS-2 until slot NS-1 completes the sector
#pragma unroll
                for (int s = 0; s < NS; s++, use++) {   // slot sl + s of the item: residue position c + s
                    const uint32_t buf = use & 1;
                    if (warp == 2 && lane == 0) TCN2_TR(2, 200);    // waiting for the accumulator
                    mbar_wait(bar_tfull + 8 * buf, (use >> 1) & 1);
                    if (warp == 2 && lane == 0) TCN2_TR(2, 201);    // accumulator complete
                    tc_fence_after();
#pragma unroll
                    for (int gi = 0; gi < GPW; gi++) {
                        const int g = sub + gi * (TCN2_EPI_WARPS / 4);
                        if (g >= groups) break;                   // warp uniform
                        const int mloc = g * 4;
                        uint32_t C[TCN_PLANES][4];
#pragma unroll
                        for (int w = 0; w < TCN_PLANES; w++)
                            tmem_ld4(tmem_base + ((uint32_t)(qd * 32) << 16) + buf * TCN2P_ACC + w * TCN2_MT + mloc, C[w]);
                        tmem_ld_wait();
                        uint64_t *op = out_col + (long)mloc * m_stride + s;
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            if (mloc + i < m_valid) {                // warp uniform
                                const uint64_t bias_m = __shfl_sync(0xffffffffu, bias_lane[s], mloc + i);
                                uint32_t Ci[TCN_PLANES];
#pragma unroll
                                for (int w = 0; w < TCN_PLANES; w++) Ci[w] = C[w][i];
                                uint64_t r;
                                if constexpr (FOLD) {
                                    r = tcn7_fold_reduce(Ci, add_bias ? bias_m : 0, fold, mod.q);
                                } else {
                                    r = barrett128(tcn7_combine(Ci), mod);
                                    if (add_bias) r = addmod(r, bias_m, mod.q);
                                }
                                if constexpr (STAGED) {
                                    if (s < NS - 1) keep[gi][i][s < NS - 1 ? s : 0] = r;
                                    else if (valid) tcn_store_sector(op - (NS - 1), keep[gi][i][0], keep[gi][i][1], keep[gi][i][2], r);
                                } else if (valid) {
                                    *op = r;
                                }
                            }
                            op += m_stride;
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_tempty + 8 * buf);
                    if (warp == 2 && lane == 0) TCN2_TR(2, 202);    // this warp's share of the chunk recombined and stored
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, TCN_TMEM_COLS);
}

// W'_b = W 2^(8b) mod q_j (Shoup product by a per-limb constant), b = 1..6, for the pre-shifted staging
struct TcnShift { uint64_t q[MAXK], w[MAXK], wp[MAXK]; };   // per limb: q_j, 2^(8b) mod q_j, floor(w 2^64 / q_j)
__global__ void tcn_preshift_kernel(const uint64_t *__restrict__ src, uint64_t *__restrict__ dst, long words, int n, int K, TcnShift c) {
    const long pw = (long)K * n;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (long)gridDim.x * blockDim.x) {
        const int j = (int)((i % pw) / n);
        const uint64_t q = c.q[j];
        const uint64_t r = mulshoup_lazy(__ldg(src + i), c.w[j], c.wp[j], q);
        dst[i] = r >= q ? r - q : r;
    }
}

// ------------------------------------------------------------------------------------ operand staging
// dst[slot - slot0][l][col][r] = byte l of src item (col group, r), polynomial col % item_polys, residue of `slot`.
// One CTA: 32 consecutive slots x 128 consecutive (column, term) bytes of a plane row -- one column x 128 terms, or
// four columns x 32 terms when rows are 32 bytes -- transposed through shared memory, so every store is 128 B wide.
__global__ void __launch_bounds__(256)
tcn_split_kernel(TcnSplitArgs a) {
    __shared__ uint64_t tile[32][133];    // [slot][(e & 3) * 33 + (e >> 2)], e = byte within the 128; row stride 133 = 5 mod 16: conflict free both ways
    __shared__ long src_off[128];         // word offset of source row e (-1: tile padding or a zero ciphertext)
    const int n = a.n, K = a.K;
    const int rows_per = a.Kpad < 128 ? 128 / a.Kpad : 1;   // columns per CTA
    const int col0 = blockIdx.x * rows_per;
    const int st = blockIdx.y;            // tile of 32 slots
    const int r0 = blockIdx.z * 128;      // only rows of >= 128 bytes have more than one z block
    const int slot = a.slot0 + st * 32;
    const int j = slot / n, c0 = slot - j * n;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < 128) {
        const int e = threadIdx.x;
        const int col = col0 + (rows_per > 1 ? e / a.Kpad : 0);
        const int r = rows_per > 1 ? e % a.Kpad : r0 + e;
        long off = -1;
        if (r < a.R && col < a.ncols) {
            const int group = col / a.item_polys, poly = col - group * a.item_polys;
            const long item = a.index ? (long)__ldg(a.index + (long)group * a.R + r) : (long)group * a.R + r;
            if (item >= 0) off = ((item * a.item_polys + poly) * K + j) * (long)n + c0;   // index -1: a padded border's zero ciphertext
        }
        src_off[e] = off;
    }
    __syncthreads();
#pragma unroll 4
    for (int e = warp; e < 128; e += 8) {
        const long off = src_off[e];
        tile[lane][(e & 3) * 33 + (e >> 2)] = off >= 0 ? __ldg(a.src + off + lane) : 0;
    }
    __syncthreads();
    const long plane_stride = (long)a.ncols * a.Kpad;
    const long row_bytes = plane_stride - (long)col0 * a.Kpad - r0;   // bytes left in the plane row from this CTA's start
    uint8_t *dst = a.dst + ((long)st * 32 * a.planes) * plane_stride + (long)col0 * a.Kpad + r0;
    // one thread: 4 consecutive source rows of one slot -> one 32-bit word of each of the 7 planes (3 byte permutes per word)
#pragma unroll
    for (int it = 0; it < 4; it++) {
        const int w = threadIdx.x + 256 * it;
        const int c = w >> 5, rw = w & 31;
        if (rows_per > 1 ? 4 * rw >= row_bytes : r0 + 4 * rw >= a.Kpad) continue;
        const uint64_t x0 = tile[c][rw], x1 = tile[c][33 + rw], x2 = tile[c][66 + rw], x3 = tile[c][99 + rw];
        uint8_t *d = dst + (long)c * a.planes * plane_stride + 4 * rw;
#pragma unroll
        for (int l = 0; l < 7; l++) {
            const uint32_t a0 = l < 4 ? (uint32_t)x0 : (uint32_t)(x0 >> 32), a1 = l < 4 ? (uint32_t)x1 : (uint32_t)(x1 >> 32);
            const uint32_t a2 = l < 4 ? (uint32_t)x2 : (uint32_t)(x2 >> 32), a3 = l < 4 ? (uint32_t)x3 : (uint32_t)(x3 >> 32);
            const uint32_t sel = (uint32_t)(l & 3) | ((uint32_t)(4 + (l & 3)) << 4);
            const uint32_t w01 = __byte_perm(a0, a1, sel), w23 = __byte_perm(a2, a3, sel);
            *reinterpret_cast<uint32_t *>(d + (long)l * plane_stride) = __byte_perm(w01, w23, 0x5410);
        }
    }
}

// ------------------------------------------------------------------------------------ host side
template <int BK, bool FOLD>
cudaError_t launch_tcn_mac_t(const DeviceParams *P, const TcnMacArgs &a, int sm_count, cudaStream_t stream) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return cudaErrorNotSupported;
    const CUtensorMapSwizzle sw = BK == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_32B;
    CUtensorMap tmW, tmX;
    {
        // rows m of the shard only: tiles that reach past M are zero filled by TMA, no padding rows in memory
        const cuuint64_t rowsW = (cuuint64_t)a.Mall * a.Kpad;
        cuuint64_t dims[4] = {(cuuint64_t)a.Kpad, (cuuint64_t)a.M, (cuuint64_t)TCN_PLANES, (cuuint64_t)a.K * a.n};
        cuuint64_t strides[3] = {(cuuint64_t)a.Kpad, rowsW, rowsW * TCN_PLANES};
        cuuint32_t box[4] = {BK, TCN_BM, TCN_PLANES, 1}, es[4] = {1, 1, 1, 1};
        if (enc(&tmW, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, (void *)(a.W + (size_t)a.m_first * a.Kpad), dims, strides, box, es,
                CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    {
        const cuuint64_t rowsX = (cuuint64_t)a.ncols * a.Kpad;
        cuuint64_t dims[4] = {(cuuint64_t)a.Kpad, (cuuint64_t)a.ncols, (cuuint64_t)TCN_PLANES, (cuuint64_t)a.nslots};
        cuuint64_t strides[3] = {(cuuint64_t)a.Kpad, rowsX, rowsX * TCN_PLANES};
        cuuint32_t box[4] = {BK, TCN_NB, TCN_PLANES, 1}, es[4] = {1, 1, 1, 1};
        if (enc(&tmX, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, (void *)a.X, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    auto k = tcn_mac_kernel<BK, FOLD>;
    const size_t smem = TcnCfg<BK>::SMEM;
    static DeviceOnce once;
    if (once.first()) {
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const long items = (long)a.nslots * ((a.M + TCN_BM - 1) / TCN_BM);
    const unsigned grid = (unsigned)(items < sm_count ? items : sm_count);
    k<<<grid, TCN_THREADS, smem, stream>>>(tmW, tmX, P, a);
    return cudaGetLastError();
}

template <int BK, bool FOLD, bool STAGED = false>
cudaError_t launch_tcn2_mac_t(const DeviceParams *P, const TcnMacArgs &a, int sm_count, cudaStream_t stream) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return cudaErrorNotSupported;
    const CUtensorMapSwizzle sw = BK == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_32B;
    CUtensorMap tmW, tmX;
    {
        const cuuint64_t rowsW = (cuuint64_t)a.Mall * a.Kpad;
        cuuint64_t dims[4] = {(cuuint64_t)a.Kpad, (cuuint64_t)a.M, (cuuint64_t)TCN_PLANES, (cuuint64_t)a.K * a.n};
        cuuint64_t strides[3] = {(cuuint64_t)a.Kpad, rowsW, rowsW * TCN_PLANES};
        cuuint32_t box[4] = {BK, TCN2_MT, TCN_PLANES, 1}, es[4] = {1, 1, 1, 1};
        if (enc(&tmW, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, (void *)(a.W + (size_t)a.m_first * a.Kpad), dims, strides, box, es,
                CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    {
        const cuuint64_t rowsX = (cuuint64_t)a.ncols * a.Kpad;
        cuuint64_t dims[4] = {(cuuint64_t)a.Kpad, (cuuint64_t)a.ncols, (cuuint64_t)TCN_PLANES, (cuuint64_t)a.nslots};
        cuuint64_t strides[3] = {(cuuint64_t)a.Kpad, rowsX, rowsX * TCN_PLANES};
        cuuint32_t box[4] = {BK, TCN2_CB, 1, 1}, es[4] = {1, 1, 1, 1};
        if (enc(&tmX, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, (void *)a.X, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    auto k = tcn2_mac_kernel<BK, FOLD, STAGED>;
    const size_t smem = Tcn2Cfg<BK>::smem(STAGED);
    static DeviceOnce once;
    if (once.first()) {
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const long groups = a.nslots / Tcn2Cfg<BK>::NS;      // a CTA runs every output tile of its slot groups
    const unsigned grid = (unsigned)(groups < sm_count ? groups : sm_count);
    k<<<grid, TCN2_THREADS, smem, stream>>>(tmW, tmX, P, a);
    return cudaGetLastError();
}

template <bool FOLD, bool STAGED>
cudaError_t launch_tcn2p_mac_t(const DeviceParams *P, const TcnMacArgs &a, int sm_count, cudaStream_t stream) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return cudaErrorNotSupported;
    CUtensorMap tmW, tmX;
    {
        // pre-shifted planes [b][K*n][a][Mall][Kpad]; one box = the 49 planes of 32 outputs of one slot, landing as [b][a][m][32]
        const cuuint64_t rowsW = (cuuint64_t)a.Mall * a.Kpad, slotW = rowsW * TCN_PLANES;
        cuuint64_t dims[5] = {(cuuint64_t)a.Kpad, (cuuint64_t)a.M, (cuuint64_t)TCN_PLANES, (cuuint64_t)a.K * a.n, (cuuint64_t)TCN_PLANES};
        cuuint64_t strides[4] = {(cuuint64_t)a.Kpad, rowsW, slotW, slotW * a.K * a.n};
        cuuint32_t box[5] = {32, TCN2_MT, TCN_PLANES, 1, TCN_PLANES}, es[5] = {1, 1, 1, 1, 1};
        if (enc(&tmW, CU_TENSOR_MAP_DATA_TYPE_UINT8, 5, (void *)(a.W + (size_t)a.m_first * a.Kpad), dims, strides, box, es,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    {
        const cuuint64_t rowsX = (cuuint64_t)a.ncols * a.Kpad;
        cuuint64_t dims[4] = {(cuuint64_t)a.Kpad, (cuuint64_t)a.ncols, (cuuint64_t)TCN_PLANES, (cuuint64_t)a.nslots};
        cuuint64_t strides[3] = {(cuuint64_t)a.Kpad, rowsX, rowsX * TCN_PLANES};
        cuuint32_t box[4] = {32, TCN2_CB, 1, 1}, es[4] = {1, 1, 1, 1};
        if (enc(&tmX, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, (void *)a.X, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B,
                CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    auto k = tcn2p_mac_kernel<FOLD, STAGED>;
    static DeviceOnce once;
    if (once.first()) {
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TCN2P_SMEM);
        if (e != cudaSuccess) return e;
    }
    const long groups = a.nslots / TCN2P_NS;
    const unsigned grid = (unsigned)(groups < sm_count ? groups : sm_count);
    k<<<grid, TCN2_THREADS, TCN2P_SMEM, stream>>>(tmW, tmX, P, a);
    return cudaGetLastError();
}

}  // namespace

bool tcn_preshift_shape(int R, int ncols, int M, int variant) {
    return R >= 1 && R <= 32 && variant != 1 && (variant == 2 || ncols >= 4 * M);
}

cudaError_t launch_tcn_preshift(const uint64_t *q, const uint64_t *src, uint64_t *dst, long words, int b, int n, int K, cudaStream_t stream) {
    if (words <= 0) return cudaSuccess;
    if (b < 1 || b >= TCN_PLANES || K > MAXK) return cudaErrorInvalidValue;
    TcnShift c{};
    for (int j = 0; j < K; j++) {
        c.q[j] = q[j];
        c.w[j] = (uint64_t)(((unsigned __int128)1 << (8 * b)) % q[j]);
        c.wp[j] = (uint64_t)(((unsigned __int128)c.w[j] << 64) / q[j]);
    }
    const long blocks = std::min<long>((words + 255) / 256, 148L * 16);
    tcn_preshift_kernel<<<(unsigned)blocks, 256, 0, stream>>>(src, dst, words, n, K, c);
    return cudaGetLastError();
}

size_t tcn_x_bytes_per_slot(int planes, int ncols, int Kpad) { return (size_t)planes * ncols * Kpad; }
size_t tcn_w_bytes(int planes, int Mall, int Kpad, int K, int n) { return (size_t)K * n * planes * Mall * Kpad; }

cudaError_t launch_tcn_split(const TcnSplitArgs &a, cudaStream_t stream) {
    if (a.ncols <= 0 || a.nslots <= 0) return cudaSuccess;
    if (a.nslots % 32 || a.slot0 % 32 || a.Kpad % 32 || a.planes != TCN_PLANES || a.nslots / 32 > 65535) return cudaErrorInvalidValue;
    const int rows_per = a.Kpad < 128 ? 128 / a.Kpad : 1;
    dim3 grid((unsigned)((a.ncols + rows_per - 1) / rows_per), (unsigned)(a.nslots / 32), (unsigned)((a.Kpad + 127) / 128));
    tcn_split_kernel<<<grid, 256, 0, stream>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_tcn_mac(const DeviceParams *P, const TcnMacArgs &a, int sm_count, cudaStream_t stream) {
    if (a.nslots <= 0 || a.M <= 0 || a.ncols <= 0) return cudaSuccess;
    if (a.planes != TCN_PLANES || a.R > TCN_MAX_R || a.Kpad != tcn_kpad(a.R)) return cudaErrorInvalidValue;
    const int forced = a.variant;   // 1 / 2 force the row-major / column-major kernel (tests, sweeps)
    const int bk = tcn_bk(a.R);
    const bool fits2 = ((a.R + 31) / 32 * 32 + bk - 1) / bk <= TCN2_KBMAX;
    const bool use2 = fits2 && (forced == 2 || (forced != 1 && a.ncols >= 4 * a.M));
    // folded reduction of the class sums (modarith.cuh: tcn_fold_reduce) when every prime of the context has SEAL's shape
    bool fold = a.use_fold != 0;
    for (int j = 0; j < a.K && fold; j++) fold = a.fold[j].ok != 0;
    // staged whole-sector stores (STG.E.256) need a 32-byte aligned output, and the pre-shift kernel's register budget at most
    // TCN2P_STAGED_MAX_M outputs
    const bool staged = a.M <= TCN2P_STAGED_MAX_M && (reinterpret_cast<uintptr_t>(a.out) & 31) == 0;
    // Pre-shifted weights (a.preshift, staged by the caller for tcn_preshift_shape): seven accumulator classes, double-buffered
    // accumulator, four slots per item
    if (a.preshift) {
        if (!tcn_preshift_shape(a.R, a.ncols, a.M, forced) || a.nslots % TCN2P_NS || a.slot0 % TCN2P_NS || a.n % TCN2P_NS) return cudaErrorInvalidValue;
        bool fold7 = a.use_fold != 0;
        for (int j = 0; j < a.K && fold7; j++) fold7 = a.fold[j].ok7 != 0;
        if (staged) return fold7 ? launch_tcn2p_mac_t<true, true>(P, a, sm_count, stream) : launch_tcn2p_mac_t<false, true>(P, a, sm_count, stream);
        return fold7 ? launch_tcn2p_mac_t<true, false>(P, a, sm_count, stream) : launch_tcn2p_mac_t<false, false>(P, a, sm_count, stream);
    }
    // The 32-byte-row kernel (fan-in <= 32: conv1) takes items of FOUR consecutive slots, stages slots 0-2 of an item in shared
    // memory and writes whole 32-byte sectors (one STG.E.256 per (column, output)): a sector is then completed by ONE thread
    // instead of four CTAs that have to stay in step (DESIGN.md section 6).  Measured on B200 (profiles/r02a_first.txt): conv1's
    // GEMM 23.6 -> 21.3 ms per step (20.1 with the folded reduction).
    if (use2 && bk == 32) {
        if (a.nslots % 4 || a.slot0 % 4 || a.n % 4) return cudaErrorInvalidValue;
        if (staged) return fold ? launch_tcn2_mac_t<32, true, true>(P, a, sm_count, stream) : launch_tcn2_mac_t<32, false, true>(P, a, sm_count, stream);
        return fold ? launch_tcn2_mac_t<32, true>(P, a, sm_count, stream) : launch_tcn2_mac_t<32, false>(P, a, sm_count, stream);
    }
    if (use2) return fold ? launch_tcn2_mac_t<128, true>(P, a, sm_count, stream) : launch_tcn2_mac_t<128, false>(P, a, sm_count, stream);
    if (fold) return bk == 128 ? launch_tcn_mac_t<128, true>(P, a, sm_count, stream) : launch_tcn_mac_t<32, true>(P, a, sm_count, stream);
    return bk == 128 ? launch_tcn_mac_t<128, false>(P, a, sm_count, stream) : launch_tcn_mac_t<32, false>(P, a, sm_count, stream);
}

}  // namespace crcnn

#ifdef CRCNN_TCN2_TRACE
// debug builds only: reset / read back the trace of CTA 0 (role 0 producer, 1 MMA issuer, 2 first epilogue warp)
extern "C" int crcnn_debug_tcn2_trace_reset() {
    int z[3] = {0, 0, 0};
    return (int)cudaMemcpyToSymbol(crcnn::g_tcn2_trace_n, z, sizeof(z));
}
extern "C" int crcnn_debug_tcn2_trace_read(int role, unsigned long long *out, int cap) {
    int n[3];
    if (cudaMemcpyFromSymbol(n, crcnn::g_tcn2_trace_n, sizeof(n)) != cudaSuccess) return -1;
    const int cnt = n[role] < cap ? n[role] : cap;
    if (cudaMemcpyFromSymbol(out, crcnn::g_tcn2_trace, (size_t)cnt * 8, (size_t)role * crcnn::TCN2_TRACE_N * 8) != cudaSuccess) return -1;
    return cnt;
}
#endif
