// ldscore.cu -- LD Scores of a reference panel (ldsc.py --l2): a banded, exact integer Gram of the kept SNPs, reduced to one
// number per SNP on the device.  No correlation matrix is ever stored.
//
// For kept SNPs i, k of one chromosome (int8 allele-count rows g, call-mask rows M, n_i calls, allele sum S_i,
// d_i = n_i sum g_i^2 - S_i^2):
//     r_ik = num_ik / sqrt(n_i n_k d_i d_k),   num_ik = n_i n_k Q_ik - n_i S_k A_ik - n_k S_i A_ki + S_i S_k N_ik
// (Q = g.g, A_ik = g_i.M_k, N = M.M; gram.cu's integer planes), which is ldsc's r = Y_i^T Y_k / n of the mean-imputed,
// standardised (ddof 0) genotypes.  Without missing calls it is (n Q_ik - S_i S_k) / sqrt(d_i d_k).  The LD Score is
//     l_i = sum_{k in W(i)} r2adj(i, k),   r2adj = r^2 - (1 - r^2) / (n - 2)   (denominator n when n <= 2)
// computed as (1 + a) sum r^2 - a |W(i)|, a = 1 / denominator.  W(i) is a symmetric window over the kept SNPs of i's
// chromosome, given per row as an inclusive range [lo_i, hi_i] of padded row indices (the host applies ldsc's rule).
//
// The rows of a chromosome are laid out from a 128-row boundary (padding rows up to the next one), and the host lists,
// per row tile t, the 128 x 128 tiles (t, c), c >= t, that meet a window of one of t's rows.  ld_band_kernel<kMiss> is
// gram.cu's persistent, warp-specialised shape:
//   warp 0   TMA producer: int8 code tiles [128 rows x 128 B], SWIZZLE_128B, multi-stage ring
//   warp 1   TMEM allocator + tcgen05.mma.kind::i8 issuer (whole-warp loop, one elected lane issues; s32 accumulators)
//   warps 2-9 epilogue: tcgen05.ld -> r^2 in FP64 -> window select -> row and column partial sums
// A TMEM lane is a row j of tile c (the A operand), a TMEM column a row i of tile t (the B operand).  The epilogue writes
// no matrix: for every row i of t the sum over the tile's columns (row partial) and, off the diagonal, for every row j of c
// the sum over the tile's rows (column partial: the windows are symmetric).  Each goes to its own slot -- one per (SNP,
// tile column of its window) -- and ld_reduce_kernel adds a SNP's slots in ascending tile-column order.  Every sum has a
// fixed order, there are no floating-point atomics, and a tile's partials do not depend on which CTA ran it, on the
// segment it was streamed in, or on the other chromosomes of the call: the result is deterministic.
//   kMiss = false  one plane (Q), 128 TMEM columns per accumulator, four accumulators: the epilogue of a tile overlaps
//                  the main loop of the next ones;
//   kMiss = true   four planes: g_j . [g_i | M_i] and M_j . [g_i | M_i] as two MMAs of N = 256, all 512 TMEM columns.
// Which kernel owns a tile is decided on the device: ld_group_flags_kernel marks the 128-row groups with a missing call
// from the decoder's counts, and a tile is four-plane if either of its groups is marked.
// Partitioned LD Scores (ld_band_kernel<kMiss, true>, ld_annot_reduce_kernel): L_c(i) = sum_{k in W(i)} r2adj(i, k) a_kc
// over the FULL band (tiles (t, c) for every c that t's windows reach, both sides): no column partials and no transpose,
// each epilogue lane contracts its SNP's r2adj with the partners' annotation rows, register group by register group.
#include <algorithm>
#include "common.cuh"
#include "kernels.h"

namespace dbslmm {

static constexpr int kLdTile = 128;
static constexpr int kLdTileBytes = kLdTile * 128;     // one operand: 128 rows x 128 B (K chunk = 128 samples)
static constexpr int kLdThreads = 320;

static constexpr int kLdGroup = 16;                     // annotations per register group of the annotated epilogue

// kAnnot: the annotated band (ld_band_kernel<kMiss, true>).  It is FP64-bound, so its TMA ring is shallower, and the
// space freed holds one group of annotation values per epilogue warp: its 64 partner rows x kLdGroup doubles.
template <bool kMiss, bool kAnnot = false>
struct LdCfg {
    static constexpr int kStages = kAnnot ? (kMiss ? 2 : 3) : (kMiss ? 3 : 6);
    static constexpr int kStageBytes = (kMiss ? 4 : 2) * kLdTileBytes;
    static constexpr int kAcc = kMiss ? 1 : 4;           // accumulator buffers
    static constexpr int kAccCols = kMiss ? 512 : 128;   // TMEM columns of one
    static constexpr int kAnnotBytes = kAnnot ? 8 * 64 * kLdGroup * (int)sizeof(double) : 0;
    static constexpr int kSmem = kStages * kStageBytes + kAnnotBytes + 1024;
};

__device__ __forceinline__ void ld_tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}

__device__ __forceinline__ LdTile ld_tile_rec(const LdTile* p) {
    const int4* q = reinterpret_cast<const int4*>(p);
    const int4 x = __ldg(q), y = __ldg(q + 1);
    LdTile t;
    t.ti = x.x; t.tj = x.y; t.sr_stride = x.z; t.sc_stride = x.w;
    t.sr = (int64_t)(((uint64_t)(uint32_t)y.y << 32) | (uint64_t)(uint32_t)y.x);
    t.sc = (int64_t)(((uint64_t)(uint32_t)y.w << 32) | (uint64_t)(uint32_t)y.z);
    return t;
}

__device__ __forceinline__ bool ld_tile_missing(const LdArgs& a, const LdTile& t) {
    return (__ldg(a.gflags + t.ti) | __ldg(a.gflags + t.tj)) != 0;
}

// x[k] of every lane -> lane l holds the sum of x[l] over the 32 lanes (31 shuffles instead of 5 x 32; fixed order)
__device__ __forceinline__ double lane_transpose_sum(double (&x)[32], int lane) {
#pragma unroll
    for (int w = 16; w >= 1; w >>= 1) {
        const bool upper = (lane & w) != 0;
#pragma unroll
        for (int k = 0; k < w; ++k) {
            const double send = upper ? x[k] : x[k + w];
            const double keep = upper ? x[k + w] : x[k];
            x[k] = keep + __shfl_xor_sync(0xffffffffu, send, w);
        }
    }
    return x[0];
}

// The annotated epilogue, annotations [c0, c0 + W) of one tile (t, c) of the full band: this lane's row j of c (a scored
// SNP) against this warp's 64 partner rows i of t.  For every annotation the sum runs over the partners in ascending
// order, one r2adj = fma(1 + alpha, r^2, -alpha) per pair and acc = fma(r2adj, a_ic, acc): it depends neither on W nor on
// the number of annotations.  The sums go to slots[slot + c0 .. c0 + W).
template <bool kMiss, int W>
__device__ __forceinline__ void ld_annot_group(const LdArgs& a, const LdTile& tl, const LdRow* rs, const LdRow& rj, bool diag,
                                               int half, int jl, int lane, uint32_t tlane, double* stage, int c0, double* slot) {
    const int64_t i0 = (int64_t)tl.ti * kLdTile + half * 64;
    __syncwarp();                                                    // every lane is done with the previous group's values
    for (int e = lane; e < 64 * W; e += 32) stage[e] = a.annot[(i0 + e / W) * a.n_annot + c0 + e % W];
    __syncwarp();
    double acc[W];
#pragma unroll
    for (int g = 0; g < W; ++g) acc[g] = 0.0;
    const double alpha = a.alpha, ap1 = 1.0 + alpha;
    auto term = [&](int r, double rr) {
        double r2 = rr * rr;
        if (diag && half * 64 + r == jl) r2 = 1.0;
        const int ig = (int)i0 + r;
        const double v = (ig >= rj.lo && ig <= rj.hi) ? fma(ap1, r2, -alpha) : 0.0;   // a select: padding rows carry NaN
        const double* av = stage + r * W;                                           // warp-uniform: a broadcast
#pragma unroll
        for (int g = 0; g < W; ++g) acc[g] = fma(v, av[g], acc[g]);
    };
    if (!kMiss) {
        const double dn = (double)a.n_ref, Sj = rj.S, wj = rj.w * dn;
#pragma unroll 1
        for (int c8 = 0; c8 < 8; ++c8) {
            uint32_t v[8];
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                         : "r"(tlane + (uint32_t)(c8 * 8))
                         : "memory");
            tmem_ld_wait();
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const LdRow& ri = rs[c8 * 8 + k];
                term(c8 * 8 + k, fma(-ri.S, Sj, u32_to_f64(v[k]) * dn) * ri.w * wj);
            }
        }
    } else {
        const int64_t Nj = rj.N, Sj = (int64_t)rj.S;
#pragma unroll 1
        for (int c16 = 0; c16 < 4; ++c16) {
            const uint32_t col0 = (uint32_t)(c16 * 16);
            uint32_t v0[16], v1[16], v2[16], v3[16];
            ld_tmem_ld16(tlane + col0, v0);
            ld_tmem_ld16(tlane + kLdTile + col0, v1);
            ld_tmem_ld16(tlane + 2 * kLdTile + col0, v2);
            ld_tmem_ld16(tlane + 3 * kLdTile + col0, v3);
            tmem_ld_wait();
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const LdRow& ri = rs[c16 * 16 + k];
                const int64_t Ni = ri.N, Si = (int64_t)ri.S;
                const int64_t num = Ni * Nj * (int64_t)v0[k] - Ni * Sj * (int64_t)v2[k] - Nj * Si * (int64_t)v1[k] +
                                    Si * Sj * (int64_t)v3[k];
                term(c16 * 16 + k, (double)num * ri.w * rj.w);
            }
        }
    }
#pragma unroll
    for (int g = 0; g < W; ++g) slot[c0 + g] = acc[g];
}

template <bool kMiss, bool kAnnot = false>
__global__ void __launch_bounds__(kLdThreads, 1)
ld_band_kernel(const __grid_constant__ CUtensorMap tmap, const LdArgs a) {
    using Cfg = LdCfg<kMiss, kAnnot>;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[Cfg::kStages], empty_bar[Cfg::kStages], acc_full[Cfg::kAcc], acc_empty[Cfg::kAcc];
    __shared__ __align__(16) LdRow rows_s[8][64];        // per epilogue warp: the constants of its 64 rows of tile t
    __shared__ double red_r[2][2][4][64];                // [tile parity][row half][lane quarter][row]: row partials
    __shared__ double red_c[2][2][kLdTile];              // [tile parity][row half][column]: column partials
    __shared__ uint32_t tmem_slot;
    if (kMiss && *a.any == 0) return;                    // no row of this segment has a missing call
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int nk = a.nk;
    const int t0 = (int)blockIdx.x, tstride = (int)gridDim.x, n_tiles = a.n_tiles;

    if (threadIdx.x == 0) {
        for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int b = 0; b < Cfg::kAcc; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 8); }
        mbar_fence_init();
        tma_prefetch_desc(&tmap);
    }
    if (warp == 1) tmem_alloc<512>(&tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        uint32_t it = 0;
        for (int t = t0; t < n_tiles; t += tstride) {
            const LdTile tl = ld_tile_rec(a.tiles + t);
            if (ld_tile_missing(a, tl) != kMiss) continue;
            const bool diag = (tl.ti == tl.tj);
            const int32_t rowJ = tl.tj * kLdTile, rowI = tl.ti * kLdTile;
            const uint32_t bytes = kMiss ? 4u * kLdTileBytes : (uint32_t)((diag ? 1 : 2) * kLdTileBytes);
            for (int ks = 0; ks < nk; ++ks, ++it) {
                const int s = it % Cfg::kStages;
                mbar_wait(&empty_bar[s], ((it / Cfg::kStages) & 1u) ^ 1u);
                uint8_t* st = smem + (size_t)s * Cfg::kStageBytes;
                if (elect_one()) {
                    mbar_expect_tx(&full_bar[s], bytes);
                    tma_load_2d(st, &tmap, ks * 128, rowJ, &full_bar[s]);
                    if (kMiss) {
                        // [g_j | M_j | g_i | M_i]: the I-side rows and masks are adjacent, one B operand of 256 rows
                        tma_load_2d(st + kLdTileBytes, &tmap, ks * 128, rowJ + a.mask_off, &full_bar[s]);
                        tma_load_2d(st + 2 * kLdTileBytes, &tmap, ks * 128, rowI, &full_bar[s]);
                        tma_load_2d(st + 3 * kLdTileBytes, &tmap, ks * 128, rowI + a.mask_off, &full_bar[s]);
                    } else if (!diag) {
                        tma_load_2d(st + kLdTileBytes, &tmap, ks * 128, rowI, &full_bar[s]);
                    }
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = make_i8_idesc(kLdTile, kMiss ? 2 * kLdTile : kLdTile);
        uint32_t it = 0, lt = 0;
        for (int t = t0; t < n_tiles; t += tstride) {
            const LdTile tl = ld_tile_rec(a.tiles + t);
            if (ld_tile_missing(a, tl) != kMiss) continue;
            const bool diag = (tl.ti == tl.tj);
            const uint32_t as = lt % Cfg::kAcc;
            mbar_wait(&acc_empty[as], ((lt / Cfg::kAcc) & 1u) ^ 1u);      // the epilogue has drained this accumulator
            tc_fence_after();
            const uint32_t tm = tmem_base + as * Cfg::kAccCols;
            for (int ks = 0; ks < nk; ++ks, ++it) {
                const int s = it % Cfg::kStages;
                mbar_wait(&full_bar[s], (it / Cfg::kStages) & 1u);
                tc_fence_after();
                const uint32_t st = smem_u32(smem + (size_t)s * Cfg::kStageBytes);
                if (elect_one()) {
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const uint32_t acc = (ks > 0 || kk > 0) ? 1u : 0u;
                        const uint64_t adv = (uint64_t)(kk * 2);         // +32 bytes inside the 128 B swizzle atom
                        if (kMiss) {
                            const uint64_t dI = make_sw128_kmajor_desc(st + 2 * kLdTileBytes);
                            umma_i8(tm, make_sw128_kmajor_desc(st) + adv, dI + adv, idesc, acc);                       // Q | P1
                            umma_i8(tm + 2 * kLdTile, make_sw128_kmajor_desc(st + kLdTileBytes) + adv, dI + adv, idesc, acc);   // P2 | N
                        } else {
                            const uint64_t dJ = make_sw128_kmajor_desc(st), dI = make_sw128_kmajor_desc(diag ? st : st + kLdTileBytes);
                            umma_i8(tm, dJ + adv, dI + adv, idesc, acc);
                        }
                    }
                    umma_commit(&empty_bar[s]);
                    if (ks == nk - 1) umma_commit(&acc_full[as]);
                }
                __syncwarp();
            }
            ++lt;
        }
    } else if (kAnnot) {
        // full band: a tile (t, c) scores the rows of c (TMEM lanes) against the partners of t; one slot per (row, tile,
        // half, annotation), added in order by ld_annot_reduce_kernel
        const int e = warp - 2, q = warp & 3, half = e >> 2;
        LdRow* rs = rows_s[e];
        double* stage = reinterpret_cast<double*>(smem + (size_t)Cfg::kStages * Cfg::kStageBytes) + e * 64 * kLdGroup;
        const int jl = q * 32 + lane, C = a.n_annot;
        uint32_t lt = 0;
        for (int t = t0; t < n_tiles; t += tstride) {
            const LdTile tl = ld_tile_rec(a.tiles + t);
            if (ld_tile_missing(a, tl) != kMiss) continue;
            const bool diag = (tl.ti == tl.tj);
            const LdRow rj = a.rows[tl.tj * kLdTile + jl];
            __syncwarp();
            rs[lane] = a.rows[tl.ti * kLdTile + half * 64 + lane];
            rs[32 + lane] = a.rows[tl.ti * kLdTile + half * 64 + 32 + lane];
            __syncwarp();
            const uint32_t as = lt % Cfg::kAcc;
            mbar_wait(&acc_full[as], (lt / Cfg::kAcc) & 1u);
            tc_fence_after();
            const uint32_t tlane = tmem_base + as * Cfg::kAccCols + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * 64);
            double* slot = a.slots + tl.sr + (int64_t)jl * tl.sr_stride + half * C;
            // groups of kLdGroup, then 8, 4, 2, 1: the accumulator stays in TMEM until the last one is done
            int c0 = 0;
            for (; c0 + kLdGroup <= C; c0 += kLdGroup) ld_annot_group<kMiss, kLdGroup>(a, tl, rs, rj, diag, half, jl, lane, tlane, stage, c0, slot);
            if (C - c0 >= 8) { ld_annot_group<kMiss, 8>(a, tl, rs, rj, diag, half, jl, lane, tlane, stage, c0, slot); c0 += 8; }
            if (C - c0 >= 4) { ld_annot_group<kMiss, 4>(a, tl, rs, rj, diag, half, jl, lane, tlane, stage, c0, slot); c0 += 4; }
            if (C - c0 >= 2) { ld_annot_group<kMiss, 2>(a, tl, rs, rj, diag, half, jl, lane, tlane, stage, c0, slot); c0 += 2; }
            if (C - c0 >= 1) ld_annot_group<kMiss, 1>(a, tl, rs, rj, diag, half, jl, lane, tlane, stage, c0, slot);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[as]);
            ++lt;
        }
    } else {
        const int e = warp - 2, q = warp & 3, half = e >> 2;         // TMEM lane quarter (rows of c), half of t's rows
        LdRow* rs = rows_s[e];
        const double dn = (double)a.n_ref;
        const int jl = q * 32 + lane;                                 // this lane's row of tile c
        uint32_t lt = 0;
        for (int t = t0; t < n_tiles; t += tstride) {
            const LdTile tl = ld_tile_rec(a.tiles + t);
            if (ld_tile_missing(a, tl) != kMiss) continue;
            const bool diag = (tl.ti == tl.tj);
            const int jg = tl.tj * kLdTile + jl;                       // padded row index of j in the segment
            const LdRow rj = a.rows[jg];
            __syncwarp();                                             // every lane is done with the previous tile's table
            rs[lane] = a.rows[tl.ti * kLdTile + half * 64 + lane];
            rs[32 + lane] = a.rows[tl.ti * kLdTile + half * 64 + 32 + lane];
            __syncwarp();
            const uint32_t as = lt % Cfg::kAcc, par = lt & 1u;
            mbar_wait(&acc_full[as], (lt / Cfg::kAcc) & 1u);
            tc_fence_after();
            const uint32_t tlane = tmem_base + as * Cfg::kAccCols + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * 64);
            double col = 0.0;
            // r^2 of row i (this warp's row `r`) and this lane's column j, the window select, the column partial; x[] keeps
            // the values for the row partials
            auto finish = [&](int r, double rr, double (&x)[32], int k) {
                const LdRow& ri = rs[r];
                double r2 = rr * rr;
                if (diag && half * 64 + r == jl) r2 = 1.0;
                const double val = (jg >= ri.lo && jg <= ri.hi) ? r2 : 0.0;     // a select: padding rows carry NaN
                col += val;
                x[k] = val;
            };
            if (!kMiss) {
                uint32_t v[2][32];
                tmem_ld32(tlane, v[0]);
                tmem_ld32(tlane + 32, v[1]);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[as]);           // accumulator copied out: MMA may reuse it
                const double Sj = rj.S, wj = rj.w * dn;
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    double x[32];
#pragma unroll
                    for (int k = 0; k < 32; ++k) {
                        const LdRow& ri = rs[c * 32 + k];
                        // n Q - S_i S_j is an exact integer below 2^53: one FMA, no rounding
                        const double num = fma(-ri.S, Sj, u32_to_f64(v[c][k]) * dn);
                        finish(c * 32 + k, num * ri.w * wj, x, k);
                    }
                    const double s = lane_transpose_sum(x, lane);
                    red_r[par][half][q][c * 32 + lane] = s;
                }
            } else {
                const int64_t Nj = rj.N, Sj = (int64_t)rj.S;
#pragma unroll 1
                for (int c = 0; c < 2; ++c) {
                    double x[32];
#pragma unroll
                    for (int c16 = 0; c16 < 2; ++c16) {
                        const uint32_t col0 = (uint32_t)(c * 32 + c16 * 16);
                        uint32_t v0[16], v1[16], v2[16], v3[16];
                        ld_tmem_ld16(tlane + col0, v0);                       // Q    = g_j . g_i
                        ld_tmem_ld16(tlane + kLdTile + col0, v1);             // P1   = g_j . M_i
                        ld_tmem_ld16(tlane + 2 * kLdTile + col0, v2);         // P2   = M_j . g_i
                        ld_tmem_ld16(tlane + 3 * kLdTile + col0, v3);         // N    = M_j . M_i
                        tmem_ld_wait();
#pragma unroll
                        for (int k = 0; k < 16; ++k) {
                            const int r = c * 32 + c16 * 16 + k;
                            const LdRow& ri = rs[r];
                            const int64_t Ni = ri.N, Si = (int64_t)ri.S;
                            // the exact numerator in int64: every term is below 4 n^3 <= 2.8e17 for n <= 409,344
                            const int64_t num = Ni * Nj * (int64_t)v0[k] - Ni * Sj * (int64_t)v2[k] - Nj * Si * (int64_t)v1[k] +
                                                Si * Sj * (int64_t)v3[k];
                            finish(r, (double)num * ri.w * rj.w, x, c16 * 16 + k);
                        }
                    }
                    const double s = lane_transpose_sum(x, lane);
                    red_r[par][half][q][c * 32 + lane] = s;
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[as]);
            }
            red_c[par][half][jl] = col;
            asm volatile("bar.sync 1, 256;" ::: "memory");            // the eight epilogue warps: partials of tile t are in
            // one thread per row of t (row partial: lane quarters in order) and, off the diagonal, per row of c (column
            // partial: row halves in order).  The tables are double-buffered by tile parity: the barrier of the next tile
            // orders these reads before the tile after it overwrites them.
            const int u = e * 32 + lane;
            if (u < kLdTile) {
                const int h = u >> 6, rr = u & 63;
                const double s = ((red_r[par][h][0][rr] + red_r[par][h][1][rr]) + red_r[par][h][2][rr]) + red_r[par][h][3][rr];
                a.slots[tl.sr + (int64_t)u * tl.sr_stride] = s;
            } else if (!diag) {
                const int j = u - kLdTile;
                a.slots[tl.sc + (int64_t)j * tl.sc_stride] = red_c[par][0][j] + red_c[par][1][j];
            }
            ++lt;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// Warps 0 and 1 of ld_pairs_kernel: the TMA producer and the MMA issuer of ld_band_kernel, for the tiles of this CTA that
// belong to the kMiss kernel.  (ld_band_kernel keeps its own copy of these loops: factored through these functions its
// register allocation, and so its code, would change.)
template <bool kMiss, class Cfg>
__device__ __forceinline__ void ld_band_produce(const CUtensorMap& tmap, const LdArgs& a, uint8_t* smem, uint64_t* full_bar,
                                                uint64_t* empty_bar, int t0, int tstride, int n_tiles, int nk) {
    uint32_t it = 0;
    for (int t = t0; t < n_tiles; t += tstride) {
        const LdTile tl = ld_tile_rec(a.tiles + t);
        if (ld_tile_missing(a, tl) != kMiss) continue;
        const bool diag = (tl.ti == tl.tj);
        const int32_t rowJ = tl.tj * kLdTile, rowI = tl.ti * kLdTile;
        const uint32_t bytes = kMiss ? 4u * kLdTileBytes : (uint32_t)((diag ? 1 : 2) * kLdTileBytes);
        for (int ks = 0; ks < nk; ++ks, ++it) {
            const int s = it % Cfg::kStages;
            mbar_wait(&empty_bar[s], ((it / Cfg::kStages) & 1u) ^ 1u);
            uint8_t* st = smem + (size_t)s * Cfg::kStageBytes;
            if (elect_one()) {
                mbar_expect_tx(&full_bar[s], bytes);
                tma_load_2d(st, &tmap, ks * 128, rowJ, &full_bar[s]);
                if (kMiss) {
                    // [g_j | M_j | g_i | M_i]: the I-side rows and masks are adjacent, one B operand of 256 rows
                    tma_load_2d(st + kLdTileBytes, &tmap, ks * 128, rowJ + a.mask_off, &full_bar[s]);
                    tma_load_2d(st + 2 * kLdTileBytes, &tmap, ks * 128, rowI, &full_bar[s]);
                    tma_load_2d(st + 3 * kLdTileBytes, &tmap, ks * 128, rowI + a.mask_off, &full_bar[s]);
                } else if (!diag) {
                    tma_load_2d(st + kLdTileBytes, &tmap, ks * 128, rowI, &full_bar[s]);
                }
            }
            __syncwarp();
        }
    }
}

template <bool kMiss, class Cfg>
__device__ __forceinline__ void ld_band_mma(const LdArgs& a, uint8_t* smem, uint64_t* full_bar, uint64_t* empty_bar, uint64_t* acc_full,
                                            uint64_t* acc_empty, uint32_t tmem_base, int t0, int tstride, int n_tiles, int nk) {
    constexpr uint32_t idesc = make_i8_idesc(kLdTile, kMiss ? 2 * kLdTile : kLdTile);
    uint32_t it = 0, lt = 0;
    for (int t = t0; t < n_tiles; t += tstride) {
        const LdTile tl = ld_tile_rec(a.tiles + t);
        if (ld_tile_missing(a, tl) != kMiss) continue;
        const bool diag = (tl.ti == tl.tj);
        const uint32_t as = lt % Cfg::kAcc;
        mbar_wait(&acc_empty[as], ((lt / Cfg::kAcc) & 1u) ^ 1u);      // the epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tm = tmem_base + as * Cfg::kAccCols;
        for (int ks = 0; ks < nk; ++ks, ++it) {
            const int s = it % Cfg::kStages;
            mbar_wait(&full_bar[s], (it / Cfg::kStages) & 1u);
            tc_fence_after();
            const uint32_t st = smem_u32(smem + (size_t)s * Cfg::kStageBytes);
            if (elect_one()) {
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const uint32_t acc = (ks > 0 || kk > 0) ? 1u : 0u;
                    const uint64_t adv = (uint64_t)(kk * 2);         // +32 bytes inside the 128 B swizzle atom
                    if (kMiss) {
                        const uint64_t dI = make_sw128_kmajor_desc(st + 2 * kLdTileBytes);
                        umma_i8(tm, make_sw128_kmajor_desc(st) + adv, dI + adv, idesc, acc);                       // Q | P1
                        umma_i8(tm + 2 * kLdTile, make_sw128_kmajor_desc(st + kLdTileBytes) + adv, dI + adv, idesc, acc);   // P2 | N
                    } else {
                        const uint64_t dJ = make_sw128_kmajor_desc(st), dI = make_sw128_kmajor_desc(diag ? st : st + kLdTileBytes);
                        umma_i8(tm, dJ + adv, dI + adv, idesc, acc);
                    }
                }
                umma_commit(&empty_bar[s]);
                if (ks == nk - 1) umma_commit(&acc_full[as]);
            }
            __syncwarp();
        }
        ++lt;
    }
}

// SNP pairs (ld_pairs_kernel<kMiss, kEmit>, dbslmm_b200_ld_pairs): tiles (T, P), P >= T, of
// the upper band, T on the TMEM lanes (tj) and P the partner tile (ti).  A pair (a, b) of padded rows passes when b > a,
// b <= hi_a (a's window; -1 for a row that never forms a pair), b is a row with called genotypes and nonzero variance
// (g >= 0) and ld_pair_pass(r).  Both passes decide every pair through this one function on the same bits of r.
__device__ __forceinline__ bool ld_pair_pass(double r, double r2_min) { return __dmul_rn(r, r) >= r2_min; }

// The epilogue of both pair passes: this lane owns row a = jl of T, this warp the 64 partners of one half of P, walked in
// ascending order.  The count pass writes the number of passing partners to the slot of (a, P, half),
// cnt[sr + jl sr_stride + half]; the emit pass writes b (the caller's row index) and r of each at
// rowoff[a] + off[slot] - base, counts again, and raises *err where the counts differ (never writing past its slot).
template <bool kMiss, bool kEmit>
__device__ __forceinline__ void ld_pairs_epilogue(const LdArgs& a, const LdPairArgs& p, LdRow* rs, uint64_t* acc_full, uint64_t* acc_empty,
                                                  uint32_t tmem_base, int warp, int lane, int t0, int tstride, int n_tiles) {
    using Cfg = LdCfg<kMiss>;
    const int e = warp - 2, q = warp & 3, half = e >> 2;
    const int jl = q * 32 + lane;
    const double dn = (double)a.n_ref, r2_min = p.r2_min;
    uint32_t lt = 0;
    for (int t = t0; t < n_tiles; t += tstride) {
        const LdTile tl = ld_tile_rec(a.tiles + t);
        if (ld_tile_missing(a, tl) != kMiss) continue;
        const int ag = tl.tj * kLdTile + jl, i0 = tl.ti * kLdTile + half * 64;
        const LdRow rj = a.rows[ag];
        __syncwarp();
        rs[lane] = a.rows[i0 + lane];
        rs[32 + lane] = a.rows[i0 + 32 + lane];
        __syncwarp();
        const int64_t slot = tl.sr + (int64_t)jl * tl.sr_stride + half;
        int64_t o = 0;
        int32_t n = 0, cap = 0, ra = 0;
        uint32_t nmiss = 0;
        if (kEmit) {
            cap = p.cnt[slot];
            o = p.rowoff[ag] + p.off[slot] - p.base;
            ra = p.rid[ag];
        }
        const bool amiss = rj.N != a.n_ref;
        const uint32_t as = lt % Cfg::kAcc;
        mbar_wait(&acc_full[as], (lt / Cfg::kAcc) & 1u);
        tc_fence_after();
        const uint32_t tlane = tmem_base + as * Cfg::kAccCols + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * 64);
        auto visit = [&](int r, double rr) {
            const LdRow& ri = rs[r];
            const int ig = i0 + r;
            if (ri.g >= 0 && ig > ag && ig <= rj.hi && ld_pair_pass(rr, r2_min)) {
                if (kEmit && n < cap) {
                    p.b[o] = ra + (ig - ag);          // the rows of a chromosome are consecutive padded rows
                    p.r[o] = rr;
                    ++o;
                    nmiss += (amiss || ri.N != a.n_ref) ? 1u : 0u;
                }
                ++n;
            }
        };
        if (!kMiss) {
            uint32_t v[2][32];
            tmem_ld32(tlane, v[0]);
            tmem_ld32(tlane + 32, v[1]);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[as]);
            const double Sj = rj.S, wj = rj.w * dn;
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    const LdRow& ri = rs[c * 32 + k];
                    visit(c * 32 + k, fma(-ri.S, Sj, u32_to_f64(v[c][k]) * dn) * ri.w * wj);
                }
        } else {
            const int64_t Nj = rj.N, Sj = (int64_t)rj.S;
#pragma unroll 1
            for (int c16 = 0; c16 < 4; ++c16) {
                const uint32_t col0 = (uint32_t)(c16 * 16);
                uint32_t v0[16], v1[16], v2[16], v3[16];
                ld_tmem_ld16(tlane + col0, v0);
                ld_tmem_ld16(tlane + kLdTile + col0, v1);
                ld_tmem_ld16(tlane + 2 * kLdTile + col0, v2);
                ld_tmem_ld16(tlane + 3 * kLdTile + col0, v3);
                tmem_ld_wait();
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const LdRow& ri = rs[c16 * 16 + k];
                    const int64_t Ni = ri.N, Si = (int64_t)ri.S;
                    const int64_t num = Ni * Nj * (int64_t)v0[k] - Ni * Sj * (int64_t)v2[k] - Nj * Si * (int64_t)v1[k] +
                                        Si * Sj * (int64_t)v3[k];
                    visit(c16 * 16 + k, (double)num * ri.w * rj.w);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[as]);
        }
        if (!kEmit) {
            p.cnt[slot] = n;
        } else {
            if (n != cap) atomicOr(p.err, 1);
            for (int w = 16; w >= 1; w >>= 1) nmiss += __shfl_xor_sync(0xffffffffu, nmiss, w);
            if (lane == 0 && nmiss) atomicAdd(p.nmiss, (unsigned long long)nmiss);
        }
        ++lt;
    }
}

// The pair passes over the upper band (see ld_pairs_epilogue): ld_band_kernel's warp roles, with LdCfg<kMiss>'s ring.
template <bool kMiss, bool kEmit>
__global__ void __launch_bounds__(kLdThreads, 1)
ld_pairs_kernel(const __grid_constant__ CUtensorMap tmap, const LdArgs a, const LdPairArgs p) {
    using Cfg = LdCfg<kMiss>;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[Cfg::kStages], empty_bar[Cfg::kStages], acc_full[Cfg::kAcc], acc_empty[Cfg::kAcc];
    __shared__ __align__(16) LdRow rows_s[8][64];        // per epilogue warp: the constants of its 64 partner rows
    __shared__ uint32_t tmem_slot;
    if (kMiss && *a.any == 0) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int t0 = (int)blockIdx.x, tstride = (int)gridDim.x, n_tiles = a.n_tiles;
    if (threadIdx.x == 0) {
        for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int b = 0; b < Cfg::kAcc; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 8); }
        mbar_fence_init();
        tma_prefetch_desc(&tmap);
    }
    if (warp == 1) tmem_alloc<512>(&tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;
    if (warp == 0) ld_band_produce<kMiss, Cfg>(tmap, a, smem, full_bar, empty_bar, t0, tstride, n_tiles, a.nk);
    else if (warp == 1) ld_band_mma<kMiss, Cfg>(a, smem, full_bar, empty_bar, acc_full, acc_empty, tmem_base, t0, tstride, n_tiles, a.nk);
    else ld_pairs_epilogue<kMiss, kEmit>(a, p, rows_s[warp - 2], acc_full, acc_empty, tmem_base, warp, lane, t0, tstride, n_tiles);
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// gflags[grp] = some row of 128-row group grp has a missing call (from the decoder's counts rowN); *any |= gflags.  One warp
// per group.
__global__ void ld_group_flags_kernel(const LdRow* __restrict__ rows, int32_t n_groups, const int32_t* __restrict__ rowN,
                                      int32_t n_ref, int32_t* __restrict__ gflags, int32_t* __restrict__ any) {
    const int grp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (grp >= n_groups) return;
    const int lane = threadIdx.x & 31;
    int miss = 0;
    for (int r = lane; r < kLdTile; r += 32) {
        const int32_t g = rows[(int64_t)grp * kLdTile + r].g;
        miss |= (g >= 0 && rowN[g] != n_ref);
    }
    miss = __any_sync(0xffffffffu, miss);
    if (lane == 0) {
        gflags[grp] = miss ? 1 : 0;
        if (miss) atomicOr(any, 1);
    }
}

// l2[p] = (1 + a) sum_u slots[base(p) + u] - a wcount[p] over the slots of padded row p in ascending tile-column order;
// NaN for padding rows (wcount 0).  base(p) = tbase[p / 128] + (p % 128) * tnslot[p / 128].
__global__ void ld_reduce_kernel(const double* __restrict__ slots, const int64_t* __restrict__ tbase, const int32_t* __restrict__ tnslot,
                                 const int32_t* __restrict__ wcount, int64_t n_prows, double a, double* __restrict__ l2) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_prows) return;
    const int32_t w = wcount[p];
    if (w == 0) { l2[p] = __longlong_as_double(0x7FF8000000000000ll); return; }
    const int64_t T = p / kLdTile;
    const int32_t ns = tnslot[T];
    const double* s = slots + tbase[T] + (p % kLdTile) * ns;
    double sum = 0.0;
    for (int32_t u = 0; u < ns; ++u) sum += s[u];
    l2[p] = fma(sum, 1.0 + a, -(a * (double)w));
}

// The annotated sums of one segment: l2[p][c] = sum_u slots[base(p) + u C + c] over the 2 x (tile columns) slots of
// scored row p in ascending (tile column, half) order, base(p) = sbase[p / 128] + (p % 128) * 2 nslot[p / 128] * C; NaN for
// padding rows.  rows[row0 + p] is the LdRow of scored row p.
__global__ void ld_annot_reduce_kernel(const double* __restrict__ slots, const int64_t* __restrict__ sbase,
                                       const int32_t* __restrict__ nslot, const LdRow* __restrict__ rows, int64_t row0,
                                       int64_t n_rows, int32_t C, double* __restrict__ l2) {
    const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= n_rows * C) return;
    const int64_t p = x / C, T = p / kLdTile;
    const int c = (int)(x - p * C);
    if (rows[row0 + p].g < 0) { l2[x] = __longlong_as_double(0x7FF8000000000000ll); return; }
    const int32_t ns = 2 * nslot[T];
    const double* s = slots + sbase[T] + (p % kLdTile) * ns * (int64_t)C + c;
    double sum = 0.0;
    for (int32_t u = 0; u < ns; ++u) sum += s[(int64_t)u * C];
    l2[x] = sum;
}

cudaError_t launch_ld_group_flags(const LdRow* rows, int32_t n_groups, const int32_t* rowN, int32_t n_ref, int32_t* gflags,
                                  int32_t* any, cudaStream_t st) {
    if (n_groups == 0) return cudaSuccess;
    ld_group_flags_kernel<<<(n_groups + 7) / 8, 256, 0, st>>>(rows, n_groups, rowN, n_ref, gflags, any);
    return cudaGetLastError();
}

// Both band kernels over the same tile list: the one-plane kernel takes the tiles without a missing call, the four-plane
// kernel the others (and returns at once when *a.any == 0).
cudaError_t launch_ld_band(const CUtensorMap& tmap, const LdArgs& a, int n_sm, cudaStream_t st) {
    if (a.n_tiles == 0) return cudaSuccess;
    const int grid = std::min(a.n_tiles, n_sm);
    cudaError_t e = cudaFuncSetAttribute(ld_band_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, LdCfg<false>::kSmem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ld_band_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LdCfg<true>::kSmem);
    if (e != cudaSuccess) return e;
    ld_band_kernel<false><<<grid, kLdThreads, LdCfg<false>::kSmem, st>>>(tmap, a);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ld_band_kernel<true><<<grid, kLdThreads, LdCfg<true>::kSmem, st>>>(tmap, a);
    return cudaGetLastError();
}

// The annotated band: both kernels over the same full-band tile list, as launch_ld_band.
cudaError_t launch_ld_band_annot(const CUtensorMap& tmap, const LdArgs& a, int n_sm, cudaStream_t st) {
    if (a.n_tiles == 0) return cudaSuccess;
    const int grid = std::min(a.n_tiles, n_sm);
    cudaError_t e = cudaFuncSetAttribute(ld_band_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LdCfg<false, true>::kSmem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ld_band_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LdCfg<true, true>::kSmem);
    if (e != cudaSuccess) return e;
    ld_band_kernel<false, true><<<grid, kLdThreads, LdCfg<false, true>::kSmem, st>>>(tmap, a);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ld_band_kernel<true, true><<<grid, kLdThreads, LdCfg<true, true>::kSmem, st>>>(tmap, a);
    return cudaGetLastError();
}

cudaError_t launch_ld_annot_reduce(const double* slots, const int64_t* sbase, const int32_t* nslot, const LdRow* rows, int64_t row0,
                                   int64_t n_rows, int32_t n_annot, double* l2, cudaStream_t st) {
    const int64_t n = n_rows * n_annot;
    if (n == 0) return cudaSuccess;
    ld_annot_reduce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(slots, sbase, nslot, rows, row0, n_rows, n_annot, l2);
    return cudaGetLastError();
}

cudaError_t launch_ld_reduce(const double* slots, const int64_t* tbase, const int32_t* tnslot, const int32_t* wcount,
                             int64_t n_prows, double a, double* l2, cudaStream_t st) {
    if (n_prows == 0) return cudaSuccess;
    ld_reduce_kernel<<<(unsigned)((n_prows + 255) / 256), 256, 0, st>>>(slots, tbase, tnslot, wcount, n_prows, a, l2);
    return cudaGetLastError();
}

// The pair offsets of one segment, after its count pass.  Row p of the segment's scored tiles (T = p / 128) has the
// 2 nslot[T] slots sbase[T] + (p % 128) 2 nslot[T] + u, u in (tile, half) order: off[slot] = the pairs of p's earlier
// slots, rowcnt[p] = all of p's pairs.
__global__ void ld_pair_rowscan_kernel(const int32_t* __restrict__ cnt, const int64_t* __restrict__ sbase,
                                       const int32_t* __restrict__ nslot, int64_t n_rows, int64_t* __restrict__ off,
                                       int64_t* __restrict__ rowcnt) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_rows) return;
    const int64_t T = p / kLdTile;
    const int32_t ns = 2 * nslot[T];
    const int64_t b = sbase[T] + (p % kLdTile) * ns;
    int64_t s = 0;
    for (int32_t u = 0; u < ns; ++u) {
        off[b + u] = s;
        s += cnt[b + u];
    }
    rowcnt[p] = s;
}

// rowoff[p] = sum of rowcnt[0..p) for p <= n_rows, in place over rowcnt[0..n_rows] (one CTA: each thread scans a contiguous
// run of rows, then the runs' totals are scanned in shared memory)
__global__ void __launch_bounds__(1024) ld_pair_offsets_kernel(int64_t* __restrict__ row, int64_t n_rows) {
    __shared__ int64_t part[1024];
    const int64_t per = (n_rows + 1023) / 1024, r0 = min(n_rows, (int64_t)threadIdx.x * per), r1 = min(n_rows, r0 + per);
    int64_t s = 0;
    for (int64_t p = r0; p < r1; ++p) s += row[p];
    part[threadIdx.x] = s;
    __syncthreads();
    for (int w = 1; w < 1024; w <<= 1) {
        const int64_t x = threadIdx.x >= (unsigned)w ? part[threadIdx.x - w] : 0;
        __syncthreads();
        part[threadIdx.x] += x;
        __syncthreads();
    }
    int64_t acc = part[threadIdx.x] - s;
    for (int64_t p = r0; p < r1; ++p) {
        const int64_t c = row[p];
        row[p] = acc;
        acc += c;
    }
    if (threadIdx.x == 1023) row[n_rows] = part[1023];
}

// The pair passes: one-plane and four-plane kernels over the same tile list, as launch_ld_band.
cudaError_t launch_ld_pairs(const CUtensorMap& tmap, const LdArgs& a, const LdPairArgs& p, bool emit, int n_sm, cudaStream_t st) {
    if (a.n_tiles == 0) return cudaSuccess;
    const int grid = std::min(a.n_tiles, n_sm);
    auto go = [&](auto k0, auto k1) {
        cudaError_t e = cudaFuncSetAttribute(k0, cudaFuncAttributeMaxDynamicSharedMemorySize, LdCfg<false>::kSmem);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, LdCfg<true>::kSmem);
        if (e != cudaSuccess) return e;
        k0<<<grid, kLdThreads, LdCfg<false>::kSmem, st>>>(tmap, a, p);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        k1<<<grid, kLdThreads, LdCfg<true>::kSmem, st>>>(tmap, a, p);
        return cudaGetLastError();
    };
    return emit ? go(ld_pairs_kernel<false, true>, ld_pairs_kernel<true, true>)
                : go(ld_pairs_kernel<false, false>, ld_pairs_kernel<true, false>);
}

cudaError_t launch_ld_pair_scan(const int32_t* cnt, const int64_t* sbase, const int32_t* nslot, int64_t n_rows, int64_t* off,
                                int64_t* rowoff, cudaStream_t st) {
    if (n_rows > 0) {
        ld_pair_rowscan_kernel<<<(unsigned)((n_rows + 255) / 256), 256, 0, st>>>(cnt, sbase, nslot, n_rows, off, rowoff);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    ld_pair_offsets_kernel<<<1, 1024, 0, st>>>(rowoff, n_rows);
    return cudaGetLastError();
}

}  // namespace dbslmm
