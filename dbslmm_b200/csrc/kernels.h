// kernels.h -- host-callable launchers of the sm_100a kernels (internal to the library).
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>
#include "common.cuh"

namespace dbslmm {

// decode.cu
cudaError_t launch_snp_stats(const uint8_t* bed, int64_t n_snp, int32_t n_ref, SnpStat* stats, int n_sm,
                             cudaStream_t st);
// SNP rows [g0, g0 + n_rows) of the plan: genotype code rows always, mask code rows where needed (see decode.cu)
cudaError_t launch_decode_rows(const uint8_t* bed, int32_t n_ref, int32_t n_pad, const uint32_t* row_src,
                               const int32_t* row_crow, const int32_t* row_mrow, int64_t g0, int64_t n_rows, double tau,
                               int8_t* codes, uint8_t* dirty, int32_t* rowN, int32_t* rowS, double* rowR, double2* rowC, const int32_t* gate,
                               int n_sm, cudaStream_t st);
// the same rows as 2-bit codes in plan order with an aligned pitch (n_pad / 4 bytes) + the per-SNP statistics: the input of
// the fused unpack + Gram kernel
cudaError_t launch_pack_rows(const uint8_t* bed, int32_t n_ref, int32_t n_pad, const uint32_t* row_src, int64_t g0, int64_t n_rows,
                             double tau, uint32_t* packed, int32_t* rowN, int32_t* rowS, double* rowR, double2* rowC, int n_sm, cudaStream_t st);
// row_crow[g] / row_mrow[g] of every SNP row of every block: croff + j and croff + m + j
cudaError_t launch_fill_rowmaps(const BlockDesc* blocks, int32_t n_blocks, int32_t* row_crow, int32_t* row_mrow, cudaStream_t st);
int32_t decode_max_n_ref();          // largest n_ref the row-staging kernels (decoder, statistics) can take
// flags[b] = block b has missing calls (from the decoder's counts), for the blocks in `list` (nullptr: 0..n_list-1);
// *any |= flags
cudaError_t launch_block_flags(const BlockDesc* blocks, const int32_t* list, int32_t n_list, const int32_t* rowN,
                               int32_t n_ref, int32_t* flags, int32_t* any, cudaStream_t st);

// gram.cu
struct GramArgs {
    const GramTile* tiles;      // device (four-plane and packed-row kernels)
    int32_t n_tiles;
    const BlockDesc* blocks;    // device
    int32_t nk;                 // n_pad / 128
    int32_t n_ref;
    double one_minus_tau;
    const int32_t* rowN;
    const int32_t* rowS;
    const double* rowR;
    const double2* rowC;        // {S_i (as double), r_i} per SNP row
    const TileRec* recs;        // self-contained tile records of the one-plane kernels (128 x 128 tiles or 256 x 256 super tiles)
    double* sigma;
    int32_t* intQ;              // optional raw planes (same offsets/ld as sigma)
    int32_t* intA;
    int32_t* intN;
    int32_t full;               // also write the upper triangle
    int32_t light;              // persistent kernel with a 3-stage ring (97 KB: co-resident with a Cholesky panel CTA)
    const int32_t* flags;       // per block: has missing calls (device, written by block_flags_kernel)
    const int32_t* any;         // some block of this launch has missing calls
    int32_t hint;               // tuning bits (DBSLMM_B200_GRAM_HINT): 1 = operand loads with L2 evict-last priority, 2 = streaming (evict-first) Sigma stores; measured, no effect: off
};
cudaError_t launch_gram(const CUtensorMap& tmap, const GramArgs& a, cudaStream_t st);
// CTA-pair kernel: `a.tiles` = 256 x 256 super tiles of the lower triangles
cudaError_t launch_gram_pair(const CUtensorMap& tmap, const CUtensorMap& tmap64, const GramArgs& a, cudaStream_t st);
cudaError_t launch_gram_packed(const CUtensorMap& pmap, const GramArgs& a, cudaStream_t st);
cudaError_t launch_gram_missing(const CUtensorMap& tmapJ, const CUtensorMap& tmapI, const GramArgs& a, cudaStream_t st);
cudaError_t launch_gram_simt(const int8_t* codes, int32_t n_pad, int64_t row0, int32_t m, int32_t* q_out,
                             cudaStream_t st);
cudaError_t launch_fill_z(const BlockDesc* blocks, const int32_t* list, int32_t n_blocks, const double* z, double* sigma,
                          cudaStream_t st);

// chol.cu
// Work lists of one panel step (device pointers): `items` of launch_chol_diag / `diag_items` = blocks active at the step;
// `items` of launch_chol_panel = int4 (block, row macro tile, slice | nslices << 8, split-K group) per CTA, macro tile 0
// of every block first.
cudaError_t launch_chol_diag(const BlockDesc* blocks, const int32_t* items, int32_t n_items, int32_t k,
                             const double* sigma, double* L, double* wbuf, int64_t wstride, double ridge,
                             int32_t* status, cudaStream_t st);
cudaError_t launch_chol_panel(const BlockDesc* blocks, const int4* items, int32_t n_items, const int32_t* diag_items,
                              int32_t n_diag_first, int32_t k, const double* sigma, double* L, double* wbuf, int64_t wstride,
                              bool fuse_end, double ridge, double* scratch, int32_t* counters, int32_t group_base,
                              int32_t* status, int32_t* dflag, bool pdl, cudaStream_t st);
// TMA/mbarrier version of the panel step (default).  tile_rows: rows per item of the list (128: 256-thread CTAs, two per
// SM; 64: 128-thread CTAs, three per SM).  lmaps: one tensor map per block over its matrix in L (device array, see
// engine.cu encode_lmaps); perm: the maps permute rows inside 8-row groups (4-D form); pf: L2 prefetch distance (chunks).
cudaError_t launch_chol_panel_tma(int32_t tile_rows, const BlockDesc* blocks, const int4* items, int32_t n_items, int32_t n_single,
                                  int32_t tpc, const int32_t* diag_items, int32_t n_diag_first, int32_t k, const CUtensorMap* lmaps,
                                  int32_t perm, int32_t pf, const double* sigma, double* L, double* wbuf, int64_t wstride,
                                  bool fuse_end, double ridge, double* scratch, int32_t* counters, int32_t group_base,
                                  int32_t* status, int32_t* dflag, bool pdl, cudaStream_t st);
int chol_panel_ctas_per_sm(int32_t tile_rows);
cudaError_t launch_backsolve(const BlockDesc* blocks, const int32_t* order, int32_t n_blocks, bool big,
                             const double* L, double inv_sqrt_n, double* beta_s, double* beta_l, int32_t max_mp,
                             cudaStream_t st);
cudaError_t chol_configure();

// variance.cu
cudaError_t launch_test_rows(const BlockDesc* blocks, int32_t n_blocks, const uint8_t* tbed, int32_t n_test_total,
                             const int32_t* sel, int32_t n_test, const int32_t* tpos, int64_t n_rows, double* tmu,
                             double* tisd, double* sigma, cudaStream_t st);
cudaError_t launch_variance(const BlockDesc* blocks, int32_t n_blocks, int32_t n_test, const double* sigma,
                            const double* Lbuf, double sigma_s, double n_obs, double* out, cudaStream_t st);

// z' Sigma z per block from the lower triangle of Sigma (variance.cu); z = the plan's z array (block-ordered SNP rows)
cudaError_t launch_quadform(const BlockDesc* blocks, int32_t n_blocks, const double* sigma, const double* z, double* out,
                            cudaStream_t st);

// score.cu
cudaError_t launch_prs(const uint8_t* bed, int32_t n_val, const SnpStat* stats, const int32_t* pos, const uint8_t* flip,
                       const double* beta, int64_t beta_stride, int32_t n_scored, int32_t nf, int32_t n_chunks,
                       double* partial, double* scores, cudaStream_t st);
// the streaming path: a compact chunk (row k = scored SNP j0 + k, pitch ceil(n_val / 4)) with its own row statistics, flip
// and beta slices (beta[f * beta_stride + k]); adds into scores[nf][n_val]
cudaError_t launch_prs_chunk(const uint8_t* chunk, int32_t n_val, const SnpStat* stats, const uint8_t* flip, const double* beta,
                             int64_t beta_stride, int32_t n_rows, int32_t nf, int32_t n_slices, double* partial, double* scores,
                             cudaStream_t st);
// row slices of one scoring launch over n_rows rows (the grid's y extent; partial holds n_slices * nf * n_val doubles)
int32_t prs_slices(int n_sm, int32_t n_val, int64_t n_rows);
// per-row statistics of a compact chunk, any n_val <= kScoreMaxNVal (no shared-memory staging); *n_empty (or NULL) += rows
// without a called genotype
constexpr int32_t kScoreMaxNVal = 536870911;     // INT32_MAX / 4: the int32 sum of squares of a row
cudaError_t launch_chunk_stats(const uint8_t* chunk, int32_t n_rows, int32_t n_val, SnpStat* stats, int32_t* n_empty, int n_sm,
                               cudaStream_t st);
// cnt[i] += 2 x called genotypes, cnt2[i] += copies of the scored allele, over the chunk's rows
cudaError_t launch_score_counts(const uint8_t* chunk, int32_t n_val, const uint8_t* flip, int32_t n_rows, int32_t n_slices,
                                int32_t* cnt, int32_t* cnt2, cudaStream_t st);

// ldscore.cu
struct LdRow {              // one padded row of an LD-score segment (32 bytes); a padding row: w = NaN, N = 0, lo > hi, g = -1
    double S;               // allele sum over the called genotypes
    double w;               // 1 / sqrt(N d), d = N sum g^2 - S^2
    int32_t N;              // called genotypes
    int32_t lo, hi;         // window: padded rows lo..hi of the segment (inclusive)
    int32_t g;              // decoder row of this SNP (index into rowN), -1 for padding
};
struct LdTile {             // one 128 x 128 tile (t, c) of the band (32 bytes)
    int32_t ti, tj;         // row tile t (B operand, TMEM columns) and column tile c >= t (A operand, TMEM lanes), segment-local
    int32_t sr_stride, sc_stride;
    int64_t sr, sc;         // slot of row i of t: sr + i * sr_stride; of row j of c: sc + j * sc_stride (off the diagonal)
};
struct LdArgs {
    const LdTile* tiles;
    int32_t n_tiles;
    int32_t nk;                 // n_pad / 128
    int32_t n_ref;
    int32_t mask_off;           // code row of the mask of code row r: r + mask_off
    const LdRow* rows;          // per padded row of the segment
    const int32_t* gflags;      // per 128-row group of the segment: has a missing call (device, ld_group_flags_kernel)
    const int32_t* any;         // some group has
    double* slots;
    // the annotated band only (ld_band_kernel<kMiss, true>)
    const double* annot;        // per padded row of the segment: n_annot values (0 for padding rows)
    int32_t n_annot;
    double alpha;               // r2adj = (1 + alpha) r^2 - alpha
};
// The pair passes (ld_pairs_kernel, dbslmm_b200_ld_pairs).  A row that never forms a pair has LdRow hi = -1 and g = -1.
struct LdPairArgs {
    double r2_min;
    int32_t* cnt;               // per (row of T, tile, half): passing partners (written by the count pass)
    const int64_t* off;         // emit: per slot, its first pair among its row's pairs
    const int64_t* rowoff;      // emit: per padded row, its first pair in the segment
    int64_t base;               // emit: first pair of the range being emitted
    const int32_t* rid;         // emit: the caller's row index of every padded row
    int32_t* b;                 // emit: b of each pair
    double* r;                  // emit: r of each pair
    int32_t* err;               // emit: set when a slot emits other than it counted
    unsigned long long* nmiss;  // emit: += pairs with a row with missing calls
};
cudaError_t launch_ld_group_flags(const LdRow* rows, int32_t n_groups, const int32_t* rowN, int32_t n_ref, int32_t* gflags,
                                  int32_t* any, cudaStream_t st);
cudaError_t launch_ld_band(const CUtensorMap& tmap, const LdArgs& a, int n_sm, cudaStream_t st);
// the annotated band: tiles (t, c) of the full band, c the scored row tile (TMEM lanes, tj) and t a tile its windows
// reach (ti); the slot of annotation k of row j of c, half h of t's rows: sr + j * sr_stride + h * n_annot + k
cudaError_t launch_ld_band_annot(const CUtensorMap& tmap, const LdArgs& a, int n_sm, cudaStream_t st);
cudaError_t launch_ld_annot_reduce(const double* slots, const int64_t* sbase, const int32_t* nslot, const LdRow* rows, int64_t row0,
                                   int64_t n_rows, int32_t n_annot, double* l2, cudaStream_t st);
// pairs: the count (emit = false) or emit pass over the upper-band tiles (T, P >= T) of a.tiles, T on the TMEM lanes (tj)
cudaError_t launch_ld_pairs(const CUtensorMap& tmap, const LdArgs& a, const LdPairArgs& p, bool emit, int n_sm, cudaStream_t st);
// the count slots of a segment's n_rows padded rows -> off (per slot, within its row) and rowoff[0..n_rows] (per row, from 0)
cudaError_t launch_ld_pair_scan(const int32_t* cnt, const int64_t* sbase, const int32_t* nslot, int64_t n_rows, int64_t* off,
                                int64_t* rowoff, cudaStream_t st);
cudaError_t launch_ld_reduce(const double* slots, const int64_t* tbase, const int32_t* tnslot, const int32_t* wcount,
                             int64_t n_prows, double a, double* l2, cudaStream_t st);

// pcg.cu
struct PcgArgs {
    const BlockDesc* blocks;
    const int32_t* order;       // blocks sorted by descending size
    int32_t n_blocks;
    const double* sigma;        // full symmetric
    double* work;               // per-block scratch (see pcg.cu)
    const int64_t* work_off;
    double ridge;               // 1 / (sigma_s * n_obs)
    double sigma_s;
    double n_obs;
    double* beta_s;
    double* beta_l;
    int32_t* status;
    int32_t* iters;
};
cudaError_t launch_pcg(const PcgArgs& a, int32_t max_ms, cudaStream_t st);

}  // namespace dbslmm
