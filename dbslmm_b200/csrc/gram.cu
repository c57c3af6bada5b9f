// gram.cu -- correlation builder (K3): exact int8 tensor-core Gram + FP64 centre/scale epilogue.
//
// Replaces the FP64 dsyrk/dgemm call sites of DBSLMMFIT::estBlock (reference
// scr/dbslmmfit.cpp:698-709, 752-756) and the per-column z-scoring of nomalizeVec
// (scr/dtpr.cpp:375-380).  For one LD block with SNP rows i, j (small SNPs first, then
// large ones), raw allele counts g in {0,1,2} (missing -> 0) and call mask M:
//     Q_ij = sum g_i g_j,  A_ij = sum g_i M_j,  N_ij = sum M_i M_j          (exact, s32)
//     num_ij = n_i n_j Q_ij - n_i S_j A_ij - n_j S_i A_ji + S_i S_j N_ij      (an integer; see gram_missing_kernel)
//     Sigma_ij = num_ij * r_i * r_j + (1 - tau) [i == j],   r_i = sqrt(tau (n-1) / (n n_i d_i)),
//     d_i = n_i Q_ii - S_i^2
// which equals tau * X^T X / n + (1 - tau) I for the mean-imputed, (N-1)-standardised X of
// the reference (SURVEY.md 8a).  Blocks without missing calls need only Q
// (A_ij = S_i, N_ij = n): one accumulator plane; blocks with missing calls use four.
//
// Kernel shape (all kernels are persistent, walking a tile list, warp-specialised; details at each kernel):
//   warp 0   TMA producer: int8 code tiles [rows x 128 B], SWIZZLE_128B, multi-stage ring
//   warp 1   TMEM allocator + tcgen05.mma.kind::i8 issuer (whole-warp loop, one elected lane issues; s32 accumulators in
//            TMEM: four of 128 columns in the one-plane kernels, two sets of four planes in the four-plane kernel)
//   warps 2-9 epilogue: tcgen05.ld -> FP64 transform -> coalesced stores of the LOWER tile, overlapping the next tiles'
//            main loops.
//   gram_persistent_kernel  one plane, 128 x 128 tiles, one CTA per SM (default)
//   gram_pair_kernel        one plane, 256 x 256 super tiles by CTA pairs (tcgen05 cta_group::2; DBSLMM_B200_GRAM=pair)
//   gram_packed_kernel      one plane from packed 2-bit rows, unpacked in shared memory (DBSLMM_B200_GRAM=packed)
//   gram_missing_kernel     four planes (blocks with missing calls)
// The A operand is the J (column) side and the B operand the I (row) side, so a TMEM lane
// holds one Sigma column and consecutive lanes store consecutive addresses of one Sigma row.
// Which kernel owns a block is decided ON THE DEVICE: block_flags_kernel (decode.cu) sets flags[b] from the counts the
// decoder just produced; the one-plane kernel skips flagged blocks, the four-plane kernel the others.
#include <algorithm>
#include "common.cuh"
#include "kernels.h"

namespace dbslmm {

static constexpr int kTile = 128;            // output tile edge and UMMA M = N
static constexpr int kTileBytes = kTile * 128;   // one operand stage: 128 rows x 128 B (K chunk = 128 samples)

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}

// FP64 transform + stores of NV * 32 rows (i0 ...) x this warp's 32 Sigma columns (jl = this lane's column) from the raw
// s32 accumulators v (one TMEM column per row): n Q - S_i S_j (exact) -> scale -> coalesced row stores of the lower
// triangle.  rc[r] = {S_i, r_i} of row i0 + r; `below` = every entry of the chunk lies strictly below the diagonal.
template <class Desc, int NV>      // Desc = BlockDesc or TileRec: m, mp, ld, moff
__device__ __forceinline__ void store_half_tile(const GramArgs& a, const Desc& bd, const uint32_t (&v)[NV][32], const double2* rc,
                                                bool below, int i0, int jl, double Sj, double rj) {
    constexpr int NR = 32 * NV;
    if (i0 >= bd.mp) return;                                  // warp-uniform: nothing of this half is inside the block
    const double dn = (double)a.n_ref;
    double* sig = a.sigma + bd.moff;
    const size_t ld = (size_t)bd.ld;
    if (below && i0 + NR <= bd.m && !a.full && a.intQ == nullptr) {
        // interior half tile (every entry below the diagonal, every row a real SNP): straight-line code
        double* p = sig + (size_t)i0 * ld + jl;
        // kB rows at a time, stage by stage: the five FP64 operations of a row form one dependent chain (~10 cycles each),
        // and left to itself ptxas walks the rows one after the other in the same registers (~100 cycles per row and warp,
        // ncu round 2); written this way the chains of kB rows overlap
        constexpr int kB = 8;
#pragma unroll
        for (int r0 = 0; r0 < NR; r0 += kB) {
            double2 c[kB];
            double t[kB];
#pragma unroll
            for (int i = 0; i < kB; ++i) c[i] = rc[r0 + i];
#pragma unroll
            for (int i = 0; i < kB; ++i) t[i] = u32_to_f64(v[(r0 + i) >> 5][(r0 + i) & 31]);
#pragma unroll
            for (int i = 0; i < kB; ++i) t[i] *= dn;
            // n Q - S_i S_j is an exact integer below 2^53: one FMA, no rounding
#pragma unroll
            for (int i = 0; i < kB; ++i) t[i] = fma(-c[i].x, Sj, t[i]);
#pragma unroll
            for (int i = 0; i < kB; ++i) t[i] *= c[i].y;
#pragma unroll
            for (int i = 0; i < kB; ++i) t[i] *= rj;
#pragma unroll
            for (int i = 0; i < kB; ++i) {
                if (a.hint & 2) __stcs(p + (size_t)(r0 + i) * ld, t[i]);
                else p[(size_t)(r0 + i) * ld] = t[i];
            }
        }
        return;
    }
    const int nreal = bd.m - i0;                           // rows r < nreal are real SNPs
    double* p = sig + (size_t)i0 * ld + jl;
    if (!a.full && a.intQ == nullptr) {
        // half tile on the diagonal or in the last tile row: the same staged arithmetic for every row (the table is zero
        // beyond the block), then PREDICATED stores -- no branch per row
        constexpr int kB = 8;
#pragma unroll
        for (int r0 = 0; r0 < NR; r0 += kB) {
            double2 c[kB];
            double t[kB];
#pragma unroll
            for (int i = 0; i < kB; ++i) c[i] = rc[r0 + i];
#pragma unroll
            for (int i = 0; i < kB; ++i) t[i] = u32_to_f64(v[(r0 + i) >> 5][(r0 + i) & 31]);
#pragma unroll
            for (int i = 0; i < kB; ++i) t[i] *= dn;
#pragma unroll
            for (int i = 0; i < kB; ++i) t[i] = fma(-c[i].x, Sj, t[i]);
#pragma unroll
            for (int i = 0; i < kB; ++i) t[i] *= c[i].y;
#pragma unroll
            for (int i = 0; i < kB; ++i) t[i] *= rj;
#pragma unroll
            for (int i = 0; i < kB; ++i) {
                const int il = i0 + r0 + i;
                const double val = (il == jl) ? t[i] + a.one_minus_tau : t[i];
                if (r0 + i < nreal && jl <= il) p[(size_t)(r0 + i) * ld] = val;
            }
        }
        for (int il = max(bd.m, i0); il < min(bd.mp, i0 + NR); ++il)      // identity padding rows m .. mp-1 (at most 7 per block)
            if (jl <= il) sig[(size_t)il * ld + jl] = (il == jl) ? 1.0 : 0.0;
        return;
    }
    // debug planes / upper triangle on request: same arithmetic, row by row
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const int il = i0 + r;
        const double2 c = rc[r];
        const double t = fma(-c.x, Sj, dn * u32_to_f64(v[r >> 5][r & 31]));
        double val = t * c.y * rj;
        if (il == jl) val += a.one_minus_tau;
        if (r < nreal && jl <= il) {
            p[(size_t)r * ld] = val;
            if (a.full && jl < il) sig[(size_t)jl * ld + il] = val;
            if (a.intQ != nullptr) {
                a.intQ[(size_t)bd.moff + (size_t)il * ld + jl] = (int32_t)v[r >> 5][r & 31];
                a.intQ[(size_t)bd.moff + (size_t)jl * ld + il] = (int32_t)v[r >> 5][r & 31];
            }
        }
    }
    // identity padding rows m .. mp-1 (at most 7 per block)
    for (int il = max(bd.m, i0); il < min(bd.mp, i0 + NR); ++il)
        if (jl <= il) sig[(size_t)il * ld + jl] = (il == jl) ? 1.0 : 0.0;
}

// FP64 epilogue of one 128 x 128 one-plane tile for one epilogue warp (TMEM lane quarter q = Sigma columns, row half):
// tcgen05.ld -> n Q - S_i S_j (exact) -> scale -> coalesced row stores of the lower triangle.  Shared by the int8-row and the
// packed-row kernels.  rc: this warp's 64 x {S_i, r_i} staging in shared memory.
__device__ __forceinline__ void plain_epilogue_tile(const GramArgs& a, const GramTile& tile, const BlockDesc& bd, uint32_t tmem_acc,
                                                    int q, int half, int lane, double2* rc, uint64_t* acc_full_bar,
                                                    uint32_t full_parity, uint64_t* acc_empty_bar) {
    const double dn = (double)a.n_ref;
    const int jl = tile.tj * kTile + q * 32 + lane;
    const int i0 = tile.ti * kTile + half * 64;          // first row of this warp's half
    double Sj = 0.0, rj = 0.0;
    if (jl < bd.m) { Sj = (double)a.rowS[bd.goff + jl]; rj = a.rowR[bd.goff + jl] * dn; }
    // per-row constants go through shared memory (one broadcast LDS.128 per row instead of four shuffles);
    // their global loads overlap the wait for the accumulator
    __syncwarp();
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
        const int il = i0 + 32 * hh + lane;
        double2 c = make_double2(0.0, 0.0);
        if (il < bd.m) c = make_double2((double)a.rowS[bd.goff + il], a.rowR[bd.goff + il]);
        rc[32 * hh + lane] = c;
    }
    __syncwarp();
    mbar_wait(acc_full_bar, full_parity);
    tc_fence_after();
    const uint32_t tlane = tmem_acc + ((uint32_t)(q * 32) << 16);
    uint32_t v[2][32];
    tmem_ld32(tlane + half * 64, v[0]);
    tmem_ld32(tlane + half * 64 + 32, v[1]);
    tmem_ld_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(acc_empty_bar);                // accumulator copied out: MMA may reuse it
    store_half_tile(a, bd, v, rc, tile.ti > tile.tj, i0, jl, Sj, rj);
}

// ------------------------------------------------------------------------------------------
// Blocks WITHOUT missing calls (one accumulator plane), two kernels of the same shape: persistent, warp-specialised,
//   warp 0: TMA producer   warp 1: TMEM alloc + MMA issuer   warps 2-9: FP64 epilogue
// the s32 accumulator double-buffered in TMEM so the epilogue of tile n overlaps the TMA/MMA main loop of tile n+1.
//
// What bounds them (ncu, round 2): not the tensor pipe, L2 or DRAM, but LATENCY between tiles.  Until session 3 every role
// began a tile with a chain of dependent global loads (tile -> block descriptor -> per-row constants, 0.7-2 us each under
// load) and the producer / MMA issuer ran inside `if (lane == 0)`, where each UTMALDG / UTCIMMA / UTCBAR is wrapped in a
// vote-elect-broadcast loop (~18 SASS instructions).  Now:
//   * the tile list holds self-contained RECORDS (TileRec, 48 B, built by the host); every role fetches the record of
//     the NEXT tile before it starts on the current one;
//   * the epilogue warps stage {S_i, r_i} of their rows and columns (rowC, written by the decoder) with cp.async into a
//     double-buffered shared-memory table one tile ahead -- no register ever waits for them;
//   * warps 0 and 1 run their loops with all 32 lanes and elect one lane per issue (elect_one in common.cuh).
// Tiles are assigned round-robin (tile t0 + n * stride); blocks whose device-side flag says "missing calls" are skipped.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ TileRec ld_rec(const TileRec* p) {
    const int4* q = reinterpret_cast<const int4*>(p);
    const int4 x = __ldg(q), y = __ldg(q + 1), z = __ldg(q + 2);
    TileRec r;
    r.blk = x.x; r.ti = x.y; r.tj = x.z; r.croff = x.w;
    r.goff = y.x; r.m = y.y; r.mp = y.z; r.ld = y.w;
    r.moff = (int64_t)(((uint64_t)(uint32_t)z.y << 32) | (uint64_t)(uint32_t)z.x);
    r.pad = 0;
    return r;
}

static constexpr int kPThreads = 320;
template <int kPStages>
struct PCfg { static constexpr int kSmem = kPStages * 2 * kTileBytes + 1024; };

// 128 x 128 tiles, one CTA per SM (DBSLMM_B200_GRAM=single).
// (min-blocks 2 only caps the registers at 102 per thread: with the 3-stage ring a Gram CTA then fits next to a
//  Cholesky panel CTA during a streaming fit)
// kAcc accumulator buffers of 128 TMEM columns (4 = all 512 columns: the MMA issuer runs up to three tiles ahead of the
// epilogue and practically never waits for an accumulator to be handed back)
template <int kPStages, int kMinB, int kAcc>
__global__ void __launch_bounds__(kPThreads, kMinB)
gram_persistent_kernel(const __grid_constant__ CUtensorMap tmap, const GramArgs a) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[kPStages], empty_bar[kPStages], acc_full[kAcc], acc_empty[kAcc];
    __shared__ __align__(16) double2 row_consts[8][2][64 + 32];  // per epilogue warp, two tiles: {S, r} of its 64 rows, then of its 32 columns
    __shared__ uint32_t tmem_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int nk = a.nk;
    const uint64_t l2hint = (a.hint & 1) ? 0x14F0000000000000ull : 0x1000000000000000ull;      // evict last / normal
    const int t0 = (int)blockIdx.x, tstride = (int)gridDim.x, n_tiles = a.n_tiles;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kPStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int b = 0; b < kAcc; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 8); }
        mbar_fence_init();
        tma_prefetch_desc(&tmap);
    }
    if (warp == 1) tmem_alloc<128 * kAcc>(&tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        uint32_t it = 0;
        int t = t0;
        TileRec cur = ld_rec(a.recs + min(t, n_tiles - 1)), nxt = cur;
        while (t < n_tiles) {
            const int tn = t + tstride;
            if (tn < n_tiles) nxt = ld_rec(a.recs + tn);
            if (__ldg(a.flags + cur.blk) == 0) {                  // (else: missing calls, the four-plane kernel's block)
                const bool diag = (cur.ti == cur.tj);
                const int32_t rowJ = cur.croff + cur.tj * kTile, rowI = cur.croff + cur.ti * kTile;
                const uint32_t bytes = (uint32_t)((diag ? 1 : 2) * kTileBytes);
                for (int ks = 0; ks < nk; ++ks, ++it) {
                    const int s = it % kPStages;
                    const uint32_t ph = (it / kPStages) & 1u;
                    mbar_wait(&empty_bar[s], ph ^ 1u);
                    uint8_t* st = smem + (size_t)s * 2 * kTileBytes;
                    if (elect_one()) {
                        mbar_expect_tx(&full_bar[s], bytes);
                        tma_load_2d_hint(st, &tmap, ks * 128, rowJ, &full_bar[s], l2hint);
                        if (!diag) tma_load_2d_hint(st + kTileBytes, &tmap, ks * 128, rowI, &full_bar[s], l2hint);
                    }
                    __syncwarp();
                }
            }
            cur = nxt;
            t = tn;
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = make_i8_idesc(kTile, kTile);
        uint32_t it = 0, lt = 0;
        int t = t0;
        TileRec cur = ld_rec(a.recs + min(t, n_tiles - 1)), nxt = cur;
        while (t < n_tiles) {
            const int tn = t + tstride;
            if (tn < n_tiles) nxt = ld_rec(a.recs + tn);
            if (__ldg(a.flags + cur.blk) == 0) {
                const bool diag = (cur.ti == cur.tj);
                const uint32_t as = lt % kAcc;
                mbar_wait(&acc_empty[as], ((lt / kAcc) & 1u) ^ 1u);    // epilogue has drained this accumulator
                tc_fence_after();
                for (int ks = 0; ks < nk; ++ks, ++it) {
                    const int s = it % kPStages;
                    const uint32_t ph = (it / kPStages) & 1u;
                    mbar_wait(&full_bar[s], ph);
                    tc_fence_after();
                    const uint32_t st = smem_u32(smem + (size_t)s * 2 * kTileBytes);
                    const uint64_t dJ = make_sw128_kmajor_desc(st), dI = make_sw128_kmajor_desc(diag ? st : st + kTileBytes);
                    if (elect_one()) {
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)
                            umma_i8(tmem_base + as * kTile, dJ + (uint64_t)(kk * 2), dI + (uint64_t)(kk * 2), idesc,
                                    (ks > 0 || kk > 0) ? 1u : 0u);
                        umma_commit(&empty_bar[s]);
                        if (ks == nk - 1) umma_commit(&acc_full[as]);
                    }
                    __syncwarp();
                }
                ++lt;
            }
            cur = nxt;
            t = tn;
        }
    } else {
        const int q = warp & 3, half = (warp - 2) >> 2;              // TMEM lane quarter (Sigma columns), row half
        double2 (*rcb)[64 + 32] = row_consts[warp - 2];
        const double dn = (double)a.n_ref;
        // {S, r} of tile r's rows and columns -> table `buf` (zero beyond the block), asynchronously
        auto stage = [&](int buf, const TileRec& r) {
            const double2* src = a.rowC + r.goff;
            const int i0 = r.ti * kTile + half * 64;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                const int il = i0 + 32 * hh + lane;
                cp_async16(&rcb[buf][32 * hh + lane], src + (il < r.m ? il : 0), il < r.m);
            }
            const int jl = r.tj * kTile + q * 32 + lane;
            cp_async16(&rcb[buf][64 + lane], src + (jl < r.m ? jl : 0), jl < r.m);
        };
        uint32_t lt = 0, n = 0;
        int t = t0;
        TileRec cur = ld_rec(a.recs + min(t, n_tiles - 1)), nxt = cur;
        if (t < n_tiles) stage(0, cur);
        cp_async_commit();
        if (t + tstride < n_tiles) nxt = ld_rec(a.recs + t + tstride);
        while (t < n_tiles) {
            const int tn = t + tstride, tnn = tn + tstride;
            TileRec nn = nxt;
            if (tnn < n_tiles) nn = ld_rec(a.recs + tnn);
            __syncwarp();                                        // every lane is done with the table of tile n - 1
            if (tn < n_tiles) stage((int)((n + 1) & 1u), nxt);
            cp_async_commit();
            if (__ldg(a.flags + cur.blk) == 0) {
                const uint32_t as = lt % kAcc;
                const int jl = cur.tj * kTile + q * 32 + lane;
                const int i0 = cur.ti * kTile + half * 64;
                cp_async_wait<1>();                              // this tile's table has landed (only the group just committed may be pending)
                __syncwarp();
                const double2* rc = rcb[n & 1u];
                const double2 cj = rc[64 + lane];
                const double Sj = cj.x, rj = cj.y * dn;
                mbar_wait(&acc_full[as], (lt / kAcc) & 1u);
                tc_fence_after();
                const uint32_t tlane = tmem_base + as * kTile + ((uint32_t)(q * 32) << 16);
                uint32_t v[2][32];
                tmem_ld32(tlane + half * 64, v[0]);
                tmem_ld32(tlane + half * 64 + 32, v[1]);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[as]);      // accumulator copied out: MMA may reuse it
                store_half_tile(a, cur, v, rc, cur.ti > cur.tj, i0, jl, Sj, rj);
                ++lt;
            }
            cur = nxt;
            nxt = nn;
            t = tn;
            ++n;
        }
        cp_async_wait<0>();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<128 * kAcc>(tmem_base);
}

// ------------------------------------------------------------------------------------------
// CTA-pair version (DBSLMM_B200_GRAM=pair).  The 128 x 128-tile kernel above moves 32 KB of operands from L2 per
// 128-sample K step and tile -- 17 GB per genome-wide fit, 11.5 TB/s: once its epilogue was out of the way (session 3) it
// ran at the L2 -> SM limit of the chip (~12 TB/s).  Here the two CTAs of a 2-CTA cluster (one TPC) work on a 256 x 256
// SUPER tile of the block's lower triangle with tcgen05.mma.cta_group::2: CTA r loads 128 J rows (its half of A = its 128
// Sigma columns, the TMEM lanes) and 2 x 64 I rows (its halves of the two B operands), 32 KB per K step for FOUR 128 x 128
// units instead of one -- half the operand traffic per unit.  The super tile is computed as TWO MMAs of M = 256, N = 128
// (I rows 0..127 and 128..255) into separate 128-column accumulators, four of which fill TMEM: every epilogue warp then
// owns 64 rows x 32 columns of a unit, copies them out with two tcgen05.ld and hands the accumulator back BEFORE its FP64
// work, exactly like the one-CTA kernel (a 256-column accumulator forced each warp through 64 rows of arithmetic before
// the hand-over, and the MMA issuer waited for it half of the time).  The upper-right unit of a diagonal super tile is
// computed and dropped; a last I half beyond the block is not computed at all.
//   warp 0 (both CTAs)  TMA producer; completion bytes of both CTAs are counted on the LEADER's full barrier
//   warp 1              TMEM allocator (both CTAs); the leader's warp issues the MMAs and commits to both CTAs
//   warps 2-9 (both)    epilogue: lane quarter = warp % 4, 64-row half of the unit = (warp - 2) / 4
// ------------------------------------------------------------------------------------------
static constexpr int kSuper = 256;
static constexpr int kPairAcc = 4;                               // accumulator buffers (128 TMEM columns each)
template <int kStages>
struct PairCfg { static constexpr int kSmem = kStages * 2 * kTileBytes + 1024; };

// (kMinB = 2 only caps the registers at 102 per thread: the 3-stage version then fits next to a Cholesky panel CTA
//  during a streaming fit, like the one-CTA kernel's)
template <int kStages, int kMinB>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPThreads, kMinB)
gram_pair_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap64, const GramArgs a) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[kStages], empty_bar[kStages], acc_full[kPairAcc], acc_empty[kPairAcc];
    __shared__ __align__(16) double2 row_consts[8][2][128 + 32]; // per epilogue warp, two super tiles: {S, r} of its 2 x 64 rows, then of its 32 columns
    __shared__ uint32_t tmem_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int t0 = (int)(blockIdx.x >> 1), tstride = (int)(gridDim.x >> 1), n_tiles = a.n_tiles;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int nk = a.nk;
    const uint64_t l2hint = (a.hint & 1) ? 0x14F0000000000000ull : 0x1000000000000000ull;      // evict last / normal

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int b = 0; b < kPairAcc; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 16); }      // 8 epilogue warps x 2 CTAs
        mbar_fence_init();
        tma_prefetch_desc(&tmap);
        tma_prefetch_desc(&tmap64);
    }
    cluster_sync_all();                                          // both CTAs are running, all barriers exist
    if (warp == 1) tmem_alloc_pair<128 * kPairAcc>(&tmem_slot);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;
    // units of a super tile: the I rows 256 ti .. +127 always, 256 ti + 128 .. +255 if they reach into the block
    auto two_units = [](const TileRec& r) { return r.ti * kSuper + kTile < r.mp; };

    if (warp == 0) {
        uint32_t it = 0;
        int t = t0;
        TileRec cur = ld_rec(a.recs + min(t, n_tiles - 1)), nxt = cur;
        while (t < n_tiles) {
            const int tn = t + tstride;
            if (tn < n_tiles) nxt = ld_rec(a.recs + tn);
            if (__ldg(a.flags + cur.blk) == 0) {                  // (else: missing calls, the four-plane kernel's block)
                const bool two = two_units(cur);
                const int32_t rowJ = cur.croff + cur.tj * kSuper + (int32_t)rank * kTile;      // this CTA's Sigma columns (A)
                const int32_t rowI = cur.croff + cur.ti * kSuper + (int32_t)rank * 64;         // its half of the first 128 Sigma rows (B0); B1 = + 128
                const uint32_t bytes = (uint32_t)((two ? 4 : 3) * kTileBytes);                 // of BOTH CTAs
                for (int ks = 0; ks < nk; ++ks, ++it) {
                    const int s = it % kStages;
                    const uint32_t ph = (it / kStages) & 1u;
                    mbar_wait(&empty_bar[s], ph ^ 1u);
                    uint8_t* st = smem + (size_t)s * 2 * kTileBytes;
                    if (elect_one()) {
                        if (rank == 0) mbar_expect_tx(&full_bar[s], bytes);
                        tma_load_2d_pair(st, &tmap, ks * 128, rowJ, &full_bar[s], l2hint);
                        tma_load_2d_pair(st + kTileBytes, &tmap64, ks * 128, rowI, &full_bar[s], l2hint);
                        if (two) tma_load_2d_pair(st + kTileBytes + kTileBytes / 2, &tmap64, ks * 128, rowI + kTile, &full_bar[s], l2hint);
                    }
                    __syncwarp();
                }
            }
            cur = nxt;
            t = tn;
        }
    } else if (warp == 1) {
        if (rank == 0) {
            constexpr uint32_t idesc = make_i8_idesc(kSuper, kTile);
            uint32_t it = 0, ut = 0;                              // ring uses, units issued so far
            int t = t0;
            TileRec cur = ld_rec(a.recs + min(t, n_tiles - 1)), nxt = cur;
            while (t < n_tiles) {
                const int tn = t + tstride;
                if (tn < n_tiles) nxt = ld_rec(a.recs + tn);
                if (__ldg(a.flags + cur.blk) == 0) {
                    const bool two = two_units(cur);
                    const uint32_t a0 = ut % kPairAcc, a1 = (ut + 1) % kPairAcc;
                    mbar_wait(&acc_empty[a0], ((ut / kPairAcc) & 1u) ^ 1u);          // both CTAs' epilogues have drained these accumulators
                    if (two) mbar_wait(&acc_empty[a1], (((ut + 1) / kPairAcc) & 1u) ^ 1u);
                    tc_fence_after();
                    for (int ks = 0; ks < nk; ++ks, ++it) {
                        const int s = it % kStages;
                        const uint32_t ph = (it / kStages) & 1u;
                        mbar_wait(&full_bar[s], ph);
                        tc_fence_after();
                        const uint32_t st = smem_u32(smem + (size_t)s * 2 * kTileBytes);
                        const uint64_t dJ = make_sw128_kmajor_desc(st), dI0 = make_sw128_kmajor_desc(st + kTileBytes),
                                       dI1 = make_sw128_kmajor_desc(st + kTileBytes + kTileBytes / 2);
                        if (elect_one()) {
#pragma unroll
                            for (int kk = 0; kk < 4; ++kk) {
                                const uint32_t acc = (ks > 0 || kk > 0) ? 1u : 0u;
                                umma_i8_pair(tmem_base + a0 * kTile, dJ + (uint64_t)(kk * 2), dI0 + (uint64_t)(kk * 2), idesc, acc);
                                if (two) umma_i8_pair(tmem_base + a1 * kTile, dJ + (uint64_t)(kk * 2), dI1 + (uint64_t)(kk * 2), idesc, acc);
                            }
                            umma_commit_pair(&empty_bar[s]);
                            if (ks == nk - 1) {
                                umma_commit_pair(&acc_full[a0]);
                                if (two) umma_commit_pair(&acc_full[a1]);
                            }
                        }
                        __syncwarp();
                    }
                    ut += two ? 2u : 1u;
                }
                cur = nxt;
                t = tn;
            }
        }
    } else {
        const int q = warp & 3, half = (warp - 2) >> 2;              // TMEM lane quarter (Sigma columns), 64-row half of a unit
        double2 (*rcb)[128 + 32] = row_consts[warp - 2];
        const double dn = (double)a.n_ref;
        // {S, r} of this warp's rows (64 of unit 0, then 64 of unit 1) and columns of super tile r -> table `buf`
        auto stage = [&](int buf, const TileRec& r) {
            const double2* src = a.rowC + r.goff;
#pragma unroll
            for (int hh = 0; hh < 4; ++hh) {
                const int il = r.ti * kSuper + (hh >> 1) * kTile + half * 64 + 32 * (hh & 1) + lane;
                cp_async16(&rcb[buf][32 * hh + lane], src + (il < r.m ? il : 0), il < r.m);
            }
            const int jl = r.tj * kSuper + (int)rank * kTile + q * 32 + lane;
            cp_async16(&rcb[buf][128 + lane], src + (jl < r.m ? jl : 0), jl < r.m);
        };
        uint32_t ut = 0, n = 0;
        int t = t0;
        TileRec cur = ld_rec(a.recs + min(t, n_tiles - 1)), nxt = cur;
        if (t < n_tiles) stage(0, cur);
        cp_async_commit();
        if (t + tstride < n_tiles) nxt = ld_rec(a.recs + t + tstride);
        while (t < n_tiles) {
            const int tn = t + tstride, tnn = tn + tstride;
            TileRec nn = nxt;
            if (tnn < n_tiles) nn = ld_rec(a.recs + tnn);
            __syncwarp();                                        // every lane is done with the table of tile n - 1
            if (tn < n_tiles) stage((int)((n + 1) & 1u), nxt);
            cp_async_commit();
            if (__ldg(a.flags + cur.blk) == 0) {
                const int jmin = cur.tj * kSuper + (int)rank * kTile + q * 32;      // this warp's first Sigma column
                const int jl = jmin + lane;
                cp_async_wait<1>();                              // this tile's table has landed
                __syncwarp();
                const double2* rc = rcb[n & 1u];
                const double2 cj = rc[128 + lane];
                const double Sj = cj.x, rj = cj.y * dn;
                const int nu = two_units(cur) ? 2 : 1;
#pragma unroll 1
                for (int u = 0; u < nu; ++u, ++ut) {                 // (not unrolled: one copy of the store code)
                    const uint32_t as = ut % kPairAcc;
                    const int i0 = cur.ti * kSuper + u * kTile + half * 64;          // first of this warp's 64 rows of the unit
                    // needed if the rows reach into the block and below (or onto) the diagonal of this warp's columns
                    const bool need = (i0 < cur.mp) && (i0 + 63 >= jmin);
                    mbar_wait(&acc_full[as], (ut / kPairAcc) & 1u);
                    tc_fence_after();
                    const uint32_t tlane = tmem_base + as * kTile + (uint32_t)(half * 64) + ((uint32_t)(q * 32) << 16);
                    uint32_t v[2][32];
                    if (need) {
                        tmem_ld32(tlane, v[0]);
                        tmem_ld32(tlane + 32, v[1]);
                        tmem_ld_wait();
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_rank(&acc_empty[as], 0);          // copied out: the leader's MMA issuer may reuse the accumulator
                    if (need) store_half_tile(a, cur, v, rc + 64 * u, i0 > jmin + 31, i0, jl, Sj, rj);
                }
            }
            cur = nxt;
            nxt = nn;
            t = tn;
            ++n;
        }
        cp_async_wait<0>();
    }
    tc_fence_before();
    cluster_sync_all();          // the peer's shared memory, barriers and TMEM stay alive until both CTAs are done
    if (warp == 1) tmem_dealloc_pair<128 * kPairAcc>(tmem_base);
}

// ------------------------------------------------------------------------------------------
// Fused unpack + Gram for blocks WITHOUT missing calls (the default).  Operands are fetched as 2-BIT rows (packed by
// pack_rows_kernel in plan order, 16-byte aligned pitch) -- [128 rows x 32 B] per 128-sample K step and operand, one 2-D
// TMA load -- and expanded to the int8 SWIZZLE_128B K-major layout in shared memory by four unpack warps (generic-proxy
// stores + fence.proxy.async), so the int8 rows never exist in HBM or L2: a quarter of the operand traffic of the int8-row
// kernel above, which runs at the L2 -> SM bandwidth limit at n_ref = 2,000 (105 int8 op per operand/result byte).
//   warp 0      TMA producer of packed tiles (4-stage ring, 8 KB per stage)
//   warp 1      TMEM allocator + tcgen05.mma issuer (int8 ring of 3 stages, 32 KB each; accumulators double-buffered)
//   warps 2-9   unpack: thread t owns half of operand row t / 2 of the stage: LDS.128 -> 4 x (16 codes -> 16 bytes) -> 4 x STS.128
//               (two unpack warps per SM sub-partition: one alone cannot hide the ALU latency of the expansion chain)
//   warps 10-17 FP64 epilogue (plain_epilogue_tile), overlapping the next tile's main loop
// ------------------------------------------------------------------------------------------
static constexpr int kUThreads = 576;
static constexpr int kUWarps = 8;                         // unpack warps
static constexpr int kUPStages = 4;                       // packed stages
static constexpr int kUIStages = 3;                       // int8 operand stages
static constexpr int kPackedTile = kTile * 32;            // 128 rows x 32 bytes (128 samples)
static constexpr int kUSmem = kUIStages * 2 * kTileBytes + kUPStages * 2 * kPackedTile + 1024;

// sixteen 2-bit codes -> sixteen allele-count bytes (0 -> 2, 2 -> 1, 1 = missing and 3 -> 0), as decode.cu's expand16<false>
__device__ __forceinline__ uint2 gram_expand8(uint32_t h) {
    constexpr uint32_t lut = 0x00010002u;
    uint32_t t = (h | (h << 8)) & 0x00FF00FFu;
    t = (t | (t << 4)) & 0x0F0F0F0Fu;
    t = (t | (t << 2)) & 0x33333333u;
    return make_uint2(__byte_perm(lut, 0u, t), __byte_perm(lut, 0u, t >> 16));
}

__global__ void __launch_bounds__(kUThreads, 1)
gram_packed_kernel(const __grid_constant__ CUtensorMap pmap, const GramArgs a) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t pfull[kUPStages], pempty[kUPStages], ifull[kUIStages], iempty[kUIStages], acc_full[2], acc_empty[2];
    __shared__ __align__(16) double2 row_consts[8][64];
    __shared__ uint32_t tmem_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* pk = smem + kUIStages * 2 * kTileBytes;      // packed ring behind the int8 ring
    const int nk = a.nk;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kUPStages; ++s) { mbar_init(&pfull[s], 1); mbar_init(&pempty[s], kUWarps); }
        for (int s = 0; s < kUIStages; ++s) { mbar_init(&ifull[s], kUWarps); mbar_init(&iempty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 8); }
        mbar_fence_init();
        tma_prefetch_desc(&pmap);
    }
    if (warp == 1) tmem_alloc<256>(&tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t pit = 0;
            for (int tile_i = blockIdx.x; tile_i < a.n_tiles; tile_i += gridDim.x) {
                const GramTile tile = a.tiles[tile_i];
                if (a.flags[tile.blk] != 0) continue;
                const BlockDesc bd = a.blocks[tile.blk];
                const bool diag = (tile.ti == tile.tj);
                const int32_t rowJ = bd.goff + tile.tj * kTile, rowI = bd.goff + tile.ti * kTile;      // packed rows = SNP rows
                for (int ks = 0; ks < nk; ++ks, ++pit) {
                    const int s = pit % kUPStages;
                    mbar_wait(&pempty[s], ((pit / kUPStages) & 1u) ^ 1u);
                    uint8_t* st = pk + (size_t)s * 2 * kPackedTile;
                    mbar_expect_tx(&pfull[s], (uint32_t)((diag ? 1 : 2) * kPackedTile));
                    tma_load_2d(st, &pmap, ks * 32, rowJ, &pfull[s]);
                    if (!diag) tma_load_2d(st + kPackedTile, &pmap, ks * 32, rowI, &pfull[s]);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = make_i8_idesc(kTile, kTile);
            uint32_t iit = 0, lt = 0;
            for (int tile_i = blockIdx.x; tile_i < a.n_tiles; tile_i += gridDim.x) {
                const GramTile tile = a.tiles[tile_i];
                if (a.flags[tile.blk] != 0) continue;
                const bool diag = (tile.ti == tile.tj);
                const uint32_t as = lt & 1u;
                mbar_wait(&acc_empty[as], ((lt >> 1) & 1u) ^ 1u);
                tc_fence_after();
                for (int ks = 0; ks < nk; ++ks, ++iit) {
                    const int s = iit % kUIStages;
                    mbar_wait(&ifull[s], (iit / kUIStages) & 1u);
                    tc_fence_after();
                    const uint32_t st = smem_u32(smem + (size_t)s * 2 * kTileBytes);
                    const uint64_t dJ = make_sw128_kmajor_desc(st), dI = make_sw128_kmajor_desc(diag ? st : st + kTileBytes);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        umma_i8(tmem_base + as * kTile, dJ + (uint64_t)(kk * 2), dI + (uint64_t)(kk * 2), idesc, (ks > 0 || kk > 0) ? 1u : 0u);
                    umma_commit(&iempty[s]);
                }
                umma_commit(&acc_full[as]);
                ++lt;
            }
        }
    } else if (warp < 2 + kUWarps) {
        // ---- unpack: half of operand row `ur` of every stage (16 bytes = 64 samples = four 16-byte output chunks)
        const int ut = threadIdx.x - 64;
        const int ur = ut >> 1, uh = ut & 1;
        const uint32_t src_off = (uint32_t)ur * 32u + (uint32_t)uh * 16u;
        const uint32_t dst_row = (uint32_t)(ur >> 3) * 1024u + (uint32_t)(ur & 7) * 128u;
        const uint32_t sw = (uint32_t)(ur & 7);
        const uint32_t pk_u32 = smem_u32(pk), i8_u32 = smem_u32(smem);
        uint32_t pit = 0;
        for (int tile_i = blockIdx.x; tile_i < a.n_tiles; tile_i += gridDim.x) {
            const GramTile tile = a.tiles[tile_i];
            if (a.flags[tile.blk] != 0) continue;
            const int nop = (tile.ti == tile.tj) ? 1 : 2;
            for (int ks = 0; ks < nk; ++ks, ++pit) {
                const int ps = pit % kUPStages, is = pit % kUIStages;      // one packed stage feeds one int8 stage
                mbar_wait(&pfull[ps], (pit / kUPStages) & 1u);
                mbar_wait(&iempty[is], ((pit / kUIStages) & 1u) ^ 1u);
                uint32_t w[2][4];
#pragma unroll
                for (int op = 0; op < 2; ++op)
                    if (op < nop) {
                        const uint32_t src = pk_u32 + (uint32_t)ps * 2 * kPackedTile + (uint32_t)op * kPackedTile + src_off;
                        asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(w[op][0]), "=r"(w[op][1]), "=r"(w[op][2]), "=r"(w[op][3]) : "r"(src));
                    }
#pragma unroll
                for (int op = 0; op < 2; ++op)
                    if (op < nop) {
                        const uint32_t dst = i8_u32 + (uint32_t)is * 2 * kTileBytes + (uint32_t)op * kTileBytes + dst_row;
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const uint2 lo = gram_expand8(w[op][c] & 0xFFFFu), hi = gram_expand8(w[op][c] >> 16);
                            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(dst + (((uint32_t)(4 * uh + c) ^ sw) << 4)), "r"(lo.x),
                                         "r"(lo.y), "r"(hi.x), "r"(hi.y)
                                         : "memory");
                        }
                    }
                fence_proxy_async();                // the int8 tile was written through the generic proxy, UMMA reads it through the async proxy
                __syncwarp();
                if (lane == 0) { mbar_arrive(&ifull[is]); mbar_arrive(&pempty[ps]); }
            }
        }
    } else {
        const int q = warp & 3, half = (warp - 2 - kUWarps) >> 2;
        double2* rc = row_consts[warp - 2 - kUWarps];
        uint32_t lt = 0;
        for (int tile_i = blockIdx.x; tile_i < a.n_tiles; tile_i += gridDim.x) {
            const GramTile tile = a.tiles[tile_i];
            if (a.flags[tile.blk] != 0) continue;
            const BlockDesc bd = a.blocks[tile.blk];
            const uint32_t my_lt = lt++;
            const uint32_t as = my_lt & 1u;
            plain_epilogue_tile(a, tile, bd, tmem_base + as * kTile, q, half, lane, rc, &acc_full[as], (my_lt >> 1) & 1u, &acc_empty[as]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<256>(tmem_base);
}

// ------------------------------------------------------------------------------------------
// Blocks WITH missing calls: four accumulator planes per tile (Q = g.g, P1 = g_j.M_i, P2 = M_j.g_i, N = M.M) and the
// four-term exact numerator.  Same persistent, warp-specialised shape as above; the output tile is 128 columns (J, the
// A operand, TMEM lanes) x 64 rows (I, the B operand, N = 64), so the four s32 planes take 256 TMEM columns and are
// double-buffered in the 512 the SM has: the FP64 epilogue of one tile overlaps the main loop of the next.
// Stage = J genotype + J mask rows (2 x 16 KB) and I genotype + I mask rows (2 x 8 KB); 4 stages.
// Tile: ti counts 64-row units, tj 128-column units; listed if any entry lies in the lower triangle.
// ------------------------------------------------------------------------------------------
static constexpr int kMStages = 4;
static constexpr int kMStageBytes = 2 * kTileBytes + 2 * (kTileBytes / 2);
static constexpr int kMSmem = kMStages * kMStageBytes + 1024;
static constexpr int kTileI = 64;

__global__ void __launch_bounds__(kPThreads, 1)
gram_missing_kernel(const __grid_constant__ CUtensorMap tmapJ, const __grid_constant__ CUtensorMap tmapI, const GramArgs a) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[kMStages], empty_bar[kMStages], acc_full[2], acc_empty[2];
    __shared__ __align__(16) double4 row_consts[8][32];          // per epilogue warp: {S_i, n_i, r_i} of its 32 rows
    __shared__ uint32_t tmem_slot;
    if (*a.any == 0) return;                                     // no block of this launch has missing calls
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int nk = a.nk;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kMStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 8); }
        mbar_fence_init();
        tma_prefetch_desc(&tmapJ);
        tma_prefetch_desc(&tmapI);
    }
    if (warp == 1) tmem_alloc<512>(&tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        {
            uint32_t it = 0;
            for (int tile_i = blockIdx.x; tile_i < a.n_tiles; tile_i += gridDim.x) {
                const GramTile tile = a.tiles[tile_i];
                if (a.flags[tile.blk] == 0) continue;
                const BlockDesc bd = a.blocks[tile.blk];
                const int32_t rowJ = bd.croff + tile.tj * kTile, rowI = bd.croff + tile.ti * kTileI;
                for (int ks = 0; ks < nk; ++ks, ++it) {
                    const int s = it % kMStages;
                    mbar_wait(&empty_bar[s], ((it / kMStages) & 1u) ^ 1u);
                    uint8_t* st = smem + (size_t)s * kMStageBytes;
                    if (elect_one()) {
                        mbar_expect_tx(&full_bar[s], (uint32_t)kMStageBytes);
                        tma_load_2d(st, &tmapJ, ks * 128, rowJ, &full_bar[s]);
                        tma_load_2d(st + kTileBytes, &tmapJ, ks * 128, rowJ + bd.m, &full_bar[s]);
                        tma_load_2d(st + 2 * kTileBytes, &tmapI, ks * 128, rowI, &full_bar[s]);
                        tma_load_2d(st + 2 * kTileBytes + kTileBytes / 2, &tmapI, ks * 128, rowI + bd.m, &full_bar[s]);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 1) {
        {
            // The I-side genotype rows and mask rows of a stage are adjacent in shared memory (2 x 64 rows), so ONE
            // B descriptor with N = 128 covers both: g_j . [g_i | M_i] fills the Q and P1 planes in one instruction,
            // M_j . [g_i | M_i] the P2 and N planes -- two MMAs per K step instead of four, a third less operand traffic.
            constexpr uint32_t idesc = make_i8_idesc(kTile, 2 * kTileI);
            uint32_t it = 0, lt = 0;
            for (int tile_i = blockIdx.x; tile_i < a.n_tiles; tile_i += gridDim.x) {
                const GramTile tile = a.tiles[tile_i];
                if (a.flags[tile.blk] == 0) continue;
                const uint32_t as = lt & 1u;
                mbar_wait(&acc_empty[as], ((lt >> 1) & 1u) ^ 1u);      // epilogue has drained this accumulator set
                tc_fence_after();
                const uint32_t tm = tmem_base + as * 256;
                for (int ks = 0; ks < nk; ++ks, ++it) {
                    const int s = it % kMStages;
                    mbar_wait(&full_bar[s], (it / kMStages) & 1u);
                    tc_fence_after();
                    const uint32_t st = smem_u32(smem + (size_t)s * kMStageBytes);
                    const uint64_t dgJ = make_sw128_kmajor_desc(st), dmJ = make_sw128_kmajor_desc(st + kTileBytes);
                    const uint64_t dI = make_sw128_kmajor_desc(st + 2 * kTileBytes);      // [g_i (64 rows) | M_i (64 rows)]
                    if (elect_one()) {
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const uint32_t acc = (ks > 0 || kk > 0) ? 1u : 0u;
                            const uint64_t adv = (uint64_t)(kk * 2);   // +32 bytes inside the 128 B swizzle atom
                            umma_i8(tm + 0 * kTileI, dgJ + adv, dI + adv, idesc, acc);        // Q | P1 : g_j . [g_i | M_i]
                            umma_i8(tm + 2 * kTileI, dmJ + adv, dI + adv, idesc, acc);        // P2 | N : M_j . [g_i | M_i]
                        }
                        umma_commit(&empty_bar[s]);
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit(&acc_full[as]);
                __syncwarp();
                ++lt;
            }
        }
    } else {
        const int q = warp & 3, half = (warp - 2) >> 2;              // TMEM lane quarter (columns j), half of the 64 rows
        double4* rc = row_consts[warp - 2];
        uint32_t lt = 0;
        for (int tile_i = blockIdx.x; tile_i < a.n_tiles; tile_i += gridDim.x) {
            const GramTile tile = a.tiles[tile_i];
            if (a.flags[tile.blk] == 0) continue;
            const BlockDesc bd = a.blocks[tile.blk];
            const uint32_t my_lt = lt++;
            const uint32_t as = my_lt & 1u;
            const int jl = tile.tj * kTile + q * 32 + lane;          // Sigma column (block local)
            const int i0 = tile.ti * kTileI + half * 32;             // first row of this warp's 32
            double Sj = 0.0, Nj = 1.0, rj = 0.0;
            if (jl < bd.m) { Sj = (double)a.rowS[bd.goff + jl]; Nj = (double)a.rowN[bd.goff + jl]; rj = a.rowR[bd.goff + jl]; }
            __syncwarp();
            {
                const int il = i0 + lane;
                double4 c = make_double4(0.0, 1.0, 0.0, 0.0);
                if (il < bd.m) c = make_double4((double)a.rowS[bd.goff + il], (double)a.rowN[bd.goff + il], a.rowR[bd.goff + il], 0.0);
                rc[lane] = c;
            }
            __syncwarp();
            mbar_wait(&acc_full[as], (my_lt >> 1) & 1u);
            tc_fence_after();
            const uint32_t tlane = tmem_base + as * 256 + half * 32 + ((uint32_t)(q * 32) << 16);
            double* sig = a.sigma + bd.moff;
            const size_t ld = (size_t)bd.ld;
#pragma unroll 1
            for (int c0 = 0; c0 < 32; c0 += 16) {
                uint32_t v0[16], v1[16], v2[16], v3[16];
                tmem_ld16(tlane + 0 * kTileI + c0, v0);
                tmem_ld16(tlane + 1 * kTileI + c0, v1);
                tmem_ld16(tlane + 2 * kTileI + c0, v2);
                tmem_ld16(tlane + 3 * kTileI + c0, v3);
                tmem_ld_wait();
                if (c0 == 16) {
                    // both chunks are in registers: the MMA issuer may reuse this accumulator set
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty[as]);
                }
                // the values of all 16 rows first, without branches (the FP64 chains of different rows overlap), then the stores
                double vals[16];
#pragma unroll
                for (int r = 0; r < 16; ++r) {
                    const double4 rcv = rc[c0 + r];
                    const double Si = rcv.x, Ni = rcv.y, ri = rcv.z;
                    const double Q = u32_to_f64(v0[r]), P1 = u32_to_f64(v1[r]);      // counts are >= 0
                    const double P2 = u32_to_f64(v2[r]), Nn = u32_to_f64(v3[r]);
                    // A_ij = sum g_i M_j = P2,  A_ji = sum g_j M_i = P1.  num = n_i u - S_i w with u = n_j Q - S_j P2 and
                    // w = n_j P1 - S_j N: u and w are exact (every product and sum below 4 n^2 < 2^53), but n_i u and S_i w
                    // reach 4 n^3 = 2.7e17 at n = 409,344, past 2^53 above n = 2^17.  So n_i u is split into p + pe exactly
                    // (fma gives the low part), p - S_i w is rounded once and pe added: num to within about 2 ulps of itself,
                    // and exact whenever every term is below 2^53 (n <= 2^17).
                    const double u = fma(-Sj, P2, Nj * Q);
                    const double w = fma(-Sj, Nn, Nj * P1);
                    const double p = Ni * u;
                    const double pe = fma(Ni, u, -p);
                    const double num = fma(-Si, w, p) + pe;
                    vals[r] = num * ri * rj;
                }
#pragma unroll
                for (int r = 0; r < 16; ++r) {
                    const int il = i0 + c0 + r;
                    if (il >= bd.mp || jl > il) continue;
                    double val;
                    if (il < bd.m) {
                        val = vals[r];
                        if (il == jl) val += a.one_minus_tau;
                    } else {
                        val = (il == jl) ? 1.0 : 0.0;                 // identity padding rows m..mp-1
                    }
                    sig[(size_t)il * ld + jl] = val;
                    if (a.full && jl < il) sig[(size_t)jl * ld + il] = val;
                    if (a.intQ != nullptr && il < bd.m) {
                        const size_t o = (size_t)bd.moff + (size_t)il * ld + jl, ot = (size_t)bd.moff + (size_t)jl * ld + il;
                        a.intQ[o] = (int32_t)v0[r];
                        a.intQ[ot] = (int32_t)v0[r];
                        a.intA[o] = (int32_t)v2[r];
                        a.intA[ot] = (int32_t)v1[r];
                        a.intN[o] = (int32_t)v3[r];
                        a.intN[ot] = (int32_t)v3[r];
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// One-plane kernel over `a.recs` (128 x 128 tile records; blocks whose flag is set are skipped).
cudaError_t launch_gram(const CUtensorMap& tmap, const GramArgs& a, cudaStream_t st) {
    if (a.n_tiles == 0) return cudaSuccess;
    cudaError_t e;
    int dev = 0, n_sm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    if (a.light) {
        e = cudaFuncSetAttribute(gram_persistent_kernel<3, 2, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, PCfg<3>::kSmem);
        if (e != cudaSuccess) return e;
        gram_persistent_kernel<3, 2, 4><<<std::min(a.n_tiles, n_sm), kPThreads, PCfg<3>::kSmem, st>>>(tmap, a);
    } else {
        e = cudaFuncSetAttribute(gram_persistent_kernel<6, 1, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, PCfg<6>::kSmem);
        if (e != cudaSuccess) return e;
        gram_persistent_kernel<6, 1, 4><<<std::min(a.n_tiles, n_sm), kPThreads, PCfg<6>::kSmem, st>>>(tmap, a);
    }
    return cudaGetLastError();
}

// One-plane CTA-pair kernel over `a.recs` (256 x 256 super-tile records; blocks whose flag is set are skipped).
cudaError_t launch_gram_pair(const CUtensorMap& tmap, const CUtensorMap& tmap64, const GramArgs& a, cudaStream_t st) {
    if (a.n_tiles == 0) return cudaSuccess;
    static int max_pairs[2] = {0, 0};
    const int li = a.light ? 1 : 0;
    constexpr int kFull = 5, kLight = 3;
    const int smem = a.light ? PairCfg<kLight>::kSmem : PairCfg<kFull>::kSmem;
    const void* fn = a.light ? (const void*)gram_pair_kernel<kLight, 2> : (const void*)gram_pair_kernel<kFull, 1>;
    if (max_pairs[li] == 0) {
        cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        int dev = 0, n_sm = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(n_sm & ~1));
        cfg.blockDim = dim3(kPThreads);
        cfg.dynamicSmemBytes = (size_t)smem;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, fn, &cfg) != cudaSuccess || n <= 0) { cudaGetLastError(); n = n_sm / 2; }
        max_pairs[li] = std::min(n, n_sm / 2);
    }
    const int npairs = std::min(a.n_tiles, max_pairs[li]);
    if (a.light) gram_pair_kernel<kLight, 2><<<2 * npairs, kPThreads, smem, st>>>(tmap, tmap64, a);
    else gram_pair_kernel<kFull, 1><<<2 * npairs, kPThreads, smem, st>>>(tmap, tmap64, a);
    return cudaGetLastError();
}

// Fused unpack + one-plane Gram over `a.tiles` from the packed 2-bit rows (pmap: 2-D map over the packed buffer, box
// 32 bytes x 128 rows, no swizzle).
cudaError_t launch_gram_packed(const CUtensorMap& pmap, const GramArgs& a, cudaStream_t st) {
    if (a.n_tiles == 0) return cudaSuccess;
    int dev = 0, n_sm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    cudaError_t e = cudaFuncSetAttribute(gram_packed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kUSmem);
    if (e != cudaSuccess) return e;
    gram_packed_kernel<<<std::min(a.n_tiles, n_sm), kUThreads, kUSmem, st>>>(pmap, a);
    return cudaGetLastError();
}

// Four-plane kernel over `a.tiles` (64-row x 128-column tiles; blocks whose flag is clear are skipped, and the whole
// launch returns at once when *a.any == 0).  tmapI: the same code array with a 64-row box.
cudaError_t launch_gram_missing(const CUtensorMap& tmapJ, const CUtensorMap& tmapI, const GramArgs& a, cudaStream_t st) {
    if (a.n_tiles == 0) return cudaSuccess;
    int dev = 0, n_sm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    cudaError_t e = cudaFuncSetAttribute(gram_missing_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMSmem);
    if (e != cudaSuccess) return e;
    gram_missing_kernel<<<std::min(a.n_tiles, n_sm), kPThreads, kMSmem, st>>>(tmapJ, tmapI, a);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Plain dp4a Gram of consecutive code rows: a cross-check for the tcgen05 path used by the
// test-suite only (dbslmm_b200_debug_gram_simt); never part of a fit.
// ------------------------------------------------------------------------------------------
__global__ void gram_simt_kernel(const int8_t* __restrict__ codes, int32_t n_pad, int64_t row0, int32_t m,
                                 int32_t* __restrict__ q) {
    const int i = blockIdx.y * blockDim.y + threadIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m || j >= m) return;
    const int* a = reinterpret_cast<const int*>(codes + (size_t)(row0 + i) * n_pad);
    const int* b = reinterpret_cast<const int*>(codes + (size_t)(row0 + j) * n_pad);
    int acc = 0;
    for (int k = 0; k < n_pad / 4; ++k) acc = __dp4a(a[k], b[k], acc);
    q[(size_t)i * m + j] = acc;
}
cudaError_t launch_gram_simt(const int8_t* codes, int32_t n_pad, int64_t row0, int32_t m, int32_t* q_out,
                             cudaStream_t st) {
    dim3 blk(16, 16), grd((m + 15) / 16, (m + 15) / 16);
    gram_simt_kernel<<<grd, blk, 0, st>>>(codes, n_pad, row0, m, q_out);
    return cudaGetLastError();
}

// z-score row of every block matrix: row mp <- [z_s ; z_l ; 0...], rows mp+1..mp+7 <- 0.
// Appending z as one more row makes the left-looking factorisation produce y = L^-1 z
// in that row, i.e. the forward substitution comes for free (chol.cu).
__global__ void fill_z_kernel(const BlockDesc* __restrict__ blocks, const int32_t* __restrict__ list,
                              const double* __restrict__ z, double* __restrict__ sigma) {
    const BlockDesc bd = blocks[list ? list[blockIdx.x] : (int)blockIdx.x];
    double* base = sigma + bd.moff + (size_t)bd.mp * bd.ld;
    for (int t = threadIdx.x; t < 8 * bd.ld; t += blockDim.x) {
        const int r = t / bd.ld, c = t - r * bd.ld;
        base[t] = (r == 0 && c < bd.m) ? z[bd.goff + c] : 0.0;
    }
}
// `list` (device, or nullptr = all blocks 0..n_blocks-1) selects the blocks.
cudaError_t launch_fill_z(const BlockDesc* blocks, const int32_t* list, int32_t n_blocks, const double* z, double* sigma,
                          cudaStream_t st) {
    if (n_blocks == 0) return cudaSuccess;
    fill_z_kernel<<<n_blocks, 256, 0, st>>>(blocks, list, z, sigma);
    return cudaGetLastError();
}

}  // namespace dbslmm
