// Host-only dump of everything derive_params() computes, for the CPU test-suite to compare with the
// oracle (tests/test_host_params.py).  No CUDA involved: modarith.cuh compiles as plain C++.
//   host_selftest <n> <t> <q_1> ... <q_K>   -> text on stdout
#include <cinttypes>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "params.h"

using namespace crcnn;

static uint64_t fnv(const std::vector<uint64_t> &v) {
    uint64_t h = 1469598103934665603ULL;
    for (uint64_t x : v) { h ^= x; h *= 1099511628211ULL; }
    return h;
}

int main(int argc, char **argv) {
    if (argc < 4) { fprintf(stderr, "usage: host_selftest n t q...\n"); return 2; }
    int n = atoi(argv[1]);
    uint64_t t = strtoull(argv[2], nullptr, 0);
    std::vector<uint64_t> q;
    for (int i = 3; i < argc; i++) q.push_back(strtoull(argv[i], nullptr, 0));
    try {
        HostParams hp = derive_params(n, (int)q.size(), q.data(), t);
        const DeviceParams &d = hp.d;
        printf("K %d L %d S %d half %" PRIu64 "\n", d.K, d.L, d.S, d.half);
        for (int s = 0; s < d.K + d.S; s++) {
            printf("slot %d q %" PRIu64 " r0 %" PRIu64 " r1 %" PRIu64 " root %" PRIu64 " w %" PRIu64 " wp %" PRIu64 " iw %" PRIu64 " iwp %" PRIu64 "\n",
                   s, d.tab[s].mod.q, d.tab[s].mod.r0, d.tab[s].mod.r1, hp.roots[s], fnv(hp.w[s]), fnv(hp.wp[s]), fnv(hp.iw[s]), fnv(hp.iwp[s]));
        }
        for (int j = 0; j < d.K; j++)
            printf("prime %d delta %" PRIu64 " rho %" PRIu64 " lift %" PRIu64 "\n", j, d.delta[j], d.rho[j], d.lift_inc[j]);
        // modular arithmetic spot checks against unsigned __int128
        uint64_t x = 0x123456789abcdef1ULL, y = 0xfedcba9876543211ULL;
        for (int s = 0; s < d.K + d.S; s++) {
            const Mod &m = d.tab[s].mod;
            for (int it = 0; it < 1000; it++) {
                x = x * 6364136223846793005ULL + 1442695040888963407ULL;
                y = y * 2862933555777941757ULL + 3037000493ULL;
                uint64_t a = x % (4 * m.q), b = y % m.q;
                uint64_t want = (uint64_t)(((unsigned __int128)a * b) % m.q);
                if (mulmod(a, b, m) != want) { printf("MULMOD MISMATCH\n"); return 1; }
                uint64_t wp = (uint64_t)((((unsigned __int128)b) << 64) / m.q);
                uint64_t lazy = mulshoup_lazy(a, b, wp, m.q);
                if (lazy >= 2 * m.q || lazy % m.q != want) { printf("SHOUP MISMATCH\n"); return 1; }
            }
        }
        // folded reduction of the limb-split GEMM's class sums (modarith.cuh: tcn_fold_reduce) against unsigned __int128
        for (int j = 0; j < d.K; j++) {
            const Mod &m = d.tab[j].mod;
            const TcnFold f = tcn_fold_make(m.q);
            printf("fold %d ok %u T %u delta %u\n", j, f.ok, f.T, f.delta);
            if (!f.ok) continue;
            for (int it = 0; it < 200000; it++) {
                uint32_t s[13];
                const int mode = it % 8;
                for (int w = 0; w < 13; w++) {
                    x = x * 6364136223846793005ULL + 1442695040888963407ULL;
                    const uint32_t r = (uint32_t)(x >> 33);                 // < 2^31
                    s[w] = mode == 0 ? 0x7fffffffu : mode == 1 ? 0u : mode == 2 ? ((x >> 20) & 1 ? 0x7fffffffu : 0u)
                         : mode == 3 ? 7u * 4096u * 255u * 255u - (r & 3) : mode == 4 ? (r >> (x & 31)) : r;
                }
                y = y * 2862933555777941757ULL + 3037000493ULL;
                const uint64_t bias = mode == 0 ? m.q - 1 : (it & 1) ? y % m.q : 0;
                unsigned __int128 z = 0;
                for (int w = 12; w >= 0; w--) z = (z << 8) + s[w];
                const uint64_t want = (uint64_t)((z + bias) % m.q);
                if (tcn_fold_reduce(s, bias, f, m.q) != want) { printf("FOLD MISMATCH\n"); return 1; }
            }
        }
        // pre-shifted limb-split GEMM (tcn_mac.cu: tcn2p_mac_kernel): the byte planes of W' = W 2^(8b) mod q recombine to W' and give
        // W X mod q through the seven classes; tcn7_fold_reduce and tcn7_combine against unsigned __int128, all-(q-1) operands at R = 4096.
        // Seven byte planes hold residues of primes up to 56 bits only; above that the engine does not take the limb-split GEMM.
        bool seven_planes = true;
        for (int j = 0; j < d.K; j++) seven_planes = seven_planes && (d.tab[j].mod.q >> 56) == 0;
        for (int j = 0; j < d.K && seven_planes; j++) {
            const Mod &m = d.tab[j].mod;
            const TcnFold f = tcn_fold_make(m.q);
            long checked = 0;
            for (int it = 0; it < 20000; it++) {
                x = x * 6364136223846793005ULL + 1442695040888963407ULL;
                y = y * 2862933555777941757ULL + 3037000493ULL;
                const uint64_t W = it < 2 ? m.q - 1 : x % m.q, X = it < 2 ? m.q - 1 : y % m.q;
                uint32_t C[7] = {0, 0, 0, 0, 0, 0, 0};
                for (int b = 0; b < 7; b++) {
                    const uint64_t wb = (uint64_t)(((unsigned __int128)1 << (8 * b)) % m.q);
                    const uint64_t wbp = (uint64_t)(((unsigned __int128)wb << 64) / m.q);
                    uint64_t Wb = mulshoup_lazy(W, wb, wbp, m.q);
                    Wb = Wb >= m.q ? Wb - m.q : Wb;
                    if (Wb != (uint64_t)(((unsigned __int128)W << (8 * b)) % m.q)) { printf("PRESHIFT MISMATCH\n"); return 1; }
                    uint64_t back = 0;
                    for (int a = 6; a >= 0; a--) back = (back << 8) | ((Wb >> (8 * a)) & 0xff);
                    if (back != Wb) { printf("PLANE MISMATCH\n"); return 1; }
                    for (int a = 0; a < 7; a++) C[a] += (uint32_t)(((X >> (8 * b)) & 0xff) * ((Wb >> (8 * a)) & 0xff));
                }
                const uint64_t bias = (it & 1) ? y % m.q : 0;
                const uint64_t want = (uint64_t)(((unsigned __int128)W * X + bias) % m.q);
                const U128 z = tcn7_combine(C);
                if (addmod(barrett128(z, m), bias, m.q) != want) { printf("SEVEN-CLASS MISMATCH\n"); return 1; }
                if (f.ok7 && tcn7_fold_reduce(C, bias, f, m.q) != want) { printf("FOLD7 MISMATCH\n"); return 1; }
                checked++;
            }
            // largest class sums the kernel admits: every byte 0xff in all 7 x 4096 plane pairs of a class
            const uint32_t cmax = 7u * 4096u * 255u * 255u;
            for (int it = 0; it < 2000 && f.ok7; it++) {
                uint32_t C[7];
                x = x * 6364136223846793005ULL + 1442695040888963407ULL;
                for (int a = 0; a < 7; a++) C[a] = it == 0 ? cmax : cmax - (uint32_t)((x >> (4 * a)) % 4096);
                const uint64_t bias = it == 0 ? m.q - 1 : x % m.q;
                unsigned __int128 z = 0;
                for (int a = 6; a >= 0; a--) z = (z << 8) + C[a];
                if (z >> 80) { printf("FOLD7 BOUND\n"); return 1; }
                if (tcn7_fold_reduce(C, bias, f, m.q) != (uint64_t)((z + bias) % m.q)) { printf("FOLD7 MISMATCH\n"); return 1; }
                checked++;
            }
            printf("fold7 %d ok7 %u checked %ld\n", j, f.ok7, checked);
        }
        // three-fold reduction of arbitrary 128-bit values (modarith.cuh: reduce128_fold) for every modulus, against barrett128 and __int128
        for (int sidx = 0; sidx < d.K + d.S; sidx++) {
            const Mod &m = d.tab[sidx].mod;
            const Fold128 f = fold128_make(m.q);
            printf("fold128 %d ok %u delta %u\n", sidx, f.ok, f.delta);
            if (!f.ok) continue;
            for (int it = 0; it < 200000; it++) {
                x = x * 6364136223846793005ULL + 1442695040888963407ULL;
                y = y * 2862933555777941757ULL + 3037000493ULL;
                U128 z;
                const int mode = it % 8;
                z.lo = mode == 0 ? ~0ull : mode == 1 ? 0 : mode == 2 ? m.q - 1 : mode == 3 ? m.q : x;
                z.hi = mode == 0 ? ~0ull : mode == 1 ? 0 : mode == 2 ? 0 : mode == 3 ? (y >> (y & 63)) : mode == 4 ? (y >> 40) : y;
                const uint64_t want = (uint64_t)(((((unsigned __int128)z.hi) << 64) | z.lo) % m.q);
                if (reduce128_fold(z, f) != want || barrett128(z, m) != want) { printf("FOLD128 MISMATCH\n"); return 1; }
            }
        }
        // square without n^-1 in its inverse transforms: the lift / floor constants that absorb it (params.h: *_n)
        typedef unsigned __int128 u128;
        for (int s = 0; s < d.K + d.S; s++) {
            const uint64_t q = d.tab[s].mod.q;
            const bool ok_ninv = (u128)d.tab[s].ninv * (uint64_t)n % q == 1;
            bool ok = ok_ninv;
            if (s < d.K) {
                ok = ok && d.mt_inv_qhat_n[s] < q && (u128)d.mt_inv_qhat_n[s] * (uint64_t)n % q == d.mt_inv_qhat[s];
                ok = ok && d.fl_c_n[s] < q && (u128)d.fl_c_n[s] * (uint64_t)n % q == d.fl_c[s];
            } else {
                ok = ok && d.fl_T_n[s - d.K] < q && (u128)d.fl_T_n[s - d.K] * (uint64_t)n % q == d.fl_T[s - d.K];
            }
            printf("ninv %d ok %d\n", s, ok ? 1 : 0);
            if (!ok) { printf("NINV CONSTANT MISMATCH\n"); return 1; }
        }
        // the transforms' approximate Shoup product (modarith.cuh: mulshoup_lazy4, host form of the same quotient estimate) on edge
        // operands: result in [0,4q) and = w*y mod q; and the three-partial-product square of the tensor stage
        for (int s = 0; s < d.K + d.S; s++) {
            const uint64_t q = d.tab[s].mod.q, nq = 0 - q;
            const uint64_t ws[] = {0, 1, q - 1, q / 2, 0x5555555555555555ULL % q, 0};
            long checked = 0;
            for (int wi = 0; wi < 6; wi++) {
                uint64_t w = ws[wi];
                for (int it = 0; it < 20000; it++) {
                    x = x * 6364136223846793005ULL + 1442695040888963407ULL;
                    y = y * 2862933555777941757ULL + 3037000493ULL;
                    if (wi == 5) w = y % q;
                    const uint64_t wp = (uint64_t)(((u128)w << 64) / q);
                    const int mode = it % 8;
                    const uint64_t yv = mode == 0 ? 0 : mode == 1 ? ~0ull : mode == 2 ? (x % (~0ull / q + 1)) * q
                                      : mode == 3 ? (~0ull / q) * q : mode == 4 ? q - 1 : mode == 5 ? 8 * q - 1 - (x & 7) : x;
                    const uint64_t r = mulshoup_lazy4(yv, w, wp, nq);
                    if (r >= 4 * q || r % q != (uint64_t)((u128)w * yv % q)) { printf("SHOUP4 MISMATCH\n"); return 1; }
                    const uint64_t a = x % q;
                    const U128 z = sqr128(a);
                    if (((u128)z.hi << 64 | z.lo) != (u128)a * a) { printf("SQR128 MISMATCH\n"); return 1; }
                    checked++;
                }
            }
            printf("shoup4 %d checked %ld\n", s, checked);
            // one-fold reduction of the forward transforms' final store (modarith.cuh: reduce64_shape), any 64-bit input
            const int k = reduce64_shape_k(q);
            if (k) {
                for (int it = 0; it < 200000; it++) {
                    x = x * 6364136223846793005ULL + 1442695040888963407ULL;
                    const int mode = it % 6;
                    const uint64_t v = mode == 0 ? ~0ull : mode == 1 ? 0 : mode == 2 ? q : mode == 3 ? q - 1 : mode == 4 ? (x % 16) * q + (x >> 60) : x;
                    if (reduce64_shape(v, q, k) != v % q || reduce64(v, d.tab[s].mod) != v % q) { printf("REDUCE64 MISMATCH\n"); return 1; }
                }
            }
            printf("reduce64_shape %d k %d\n", s, k);
        }
        // fractional encoder
        for (int i = 4; i >= 0; i--) {
            double vals[] = {0.0867, -3.25, 0.0, 1.0, 2.8215};
            std::vector<uint32_t> idx; std::vector<uint64_t> val;
            encode_fractional_sparse(vals[i], n, t, idx, val);
            printf("enc %.4f nnz %zu", vals[i], idx.size());
            for (size_t e = 0; e < idx.size(); e++) printf(" %u:%" PRIu64, idx[e], val[e]);
            printf("\n");
        }
        printf("OK\n");
    } catch (const std::exception &e) {
        printf("ERROR %s\n", e.what());
        return 1;
    }
    return 0;
}
