/* dbslmm_b200.h -- C ABI of the B200-native DBSLMM per-LD-block fit.
 *
 * This is the drop-in boundary for ONE path of fboehm/DBSLMM: the block estimation
 * DBSLMMFIT::est -> calcBlock -> estBlock -> PCG (scr/dbslmmfit.cpp:56-770) fed by
 * IO::readSNPIm + SNPPROC::nomalizeVec (scr/dtpr.cpp:285-380).  Every entry point
 * takes plain host pointers and sizes (caller-owned), returns an int status and never
 * throws.  One handle drives one GPU; LD blocks are independent, so multi-GPU use is
 * "one handle per GPU, each given its own shard of blocks" (dbslmm_b200_plan_shards).
 * There is no CPU fallback: without a CUDA device every call fails with
 * DBSLMM_B200_ERR_CUDA.
 *
 * Reference interface each entry point replaces (paths relative to the reference):
 *   dbslmm_b200_load_bed     the per-block `ifstream bed_in(bed_str)` opens and per-byte
 *                            reads of IO::readSNPIm          scr/dbslmmfit.cpp:384, scr/dtpr.cpp:302-315
 *   dbslmm_b200_snp_stats    the MAF pre-pass of IO::readBim  scr/dtpr.cpp:93-102
 *   dbslmm_b200_plan_shards  the batch-of-60 OpenMP scheduler scr/dbslmmfit.cpp:92-96,189-193
 *   dbslmm_b200_fit          both DBSLMMFIT::est overloads    scr/dbslmmfit.hpp:38-67
 *                            (calcBlock/estBlock/PCGv/PCGm inside)
 */
#ifndef DBSLMM_B200_H
#define DBSLMM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DBSLMM_B200_ABI_VERSION 6

#if defined(__GNUC__)
#define DBSLMM_B200_API __attribute__((visibility("default")))
#else
#define DBSLMM_B200_API
#endif

/* status codes: 0 ok; <0 failure; >0 (fit only) number of blocks whose status != 0 */
#define DBSLMM_B200_OK            0
#define DBSLMM_B200_ERR_CUDA     (-1)   /* no device / CUDA runtime error (see last_error) */
#define DBSLMM_B200_ERR_ARG      (-2)   /* bad argument                                    */
#define DBSLMM_B200_ERR_STATE    (-3)   /* call order (e.g. fit before load_bed)           */
#define DBSLMM_B200_ERR_NOMEM    (-4)   /* device or host allocation failed                */
#define DBSLMM_B200_ERR_SINK     (-5)   /* a caller's sink returned nonzero (dbslmm_b200_ld_pairs) */

/* per-block status bits written to block_status_out */
#define DBSLMM_B200_BLK_OK          0
#define DBSLMM_B200_BLK_NOT_SPD     1   /* Cholesky pivot <= 0 or NaN (monomorphic SNP => NaN column,
                                           the reference poisons the whole block the same way)      */
#define DBSLMM_B200_BLK_PCG_MAXITER 2   /* PCG hit maxiter ("Matrix is Singular", dbslmmfit.cpp:664) */
#define DBSLMM_B200_BLK_SYNC_TIMEOUT 4  /* an in-launch wait of the block solver gave up after ~5 s (never observed; the block's
                                           betas are invalid) */

/* solver selection */
#define DBSLMM_B200_SOLVER_CHOLESKY 0   /* exact: batched FP64 Cholesky of the bordered block system  */
#define DBSLMM_B200_SOLVER_PCG      1   /* reference-faithful Jacobi-PCG, tol 1e-7, maxiter 1000       */

typedef struct dbslmm_b200_handle dbslmm_b200_handle;

/* Device-side phase times of the last fit, CUDA events on the library's own stream (ms). */
typedef struct dbslmm_b200_timing {
    float h2d_ms;        /* plan + z upload                                   */
    float decode_ms;     /* genotype decoder kernel(s)                        */
    float gram_ms;       /* correlation builder kernel(s)                     */
    float solve_ms;      /* block solver (all folds): factor + substitutions  */
    float d2h_ms;        /* beta download                                     */
    float total_ms;      /* first event to last event                         */
    int32_t n_launches;  /* kernels launched by this library in the fit       */
    int32_t n_chol_launches;
    double gram_ops;     /* algorithmic int8 ops  (2*n_pad*m*(m+1)/2 per plain block, x4 planes if missing) */
    double solve_flops;  /* algorithmic FP64 flop (m^3/3 + 2 m^2 per block and fold)                       */
    double decode_bytes; /* algorithmic bytes read + written by the decoder                                */
    double chol_ms;      /* factorisation kernels only (subset of solve_ms), summed over folds             */
    float class_ms[4];   /* last fold: fork -> end of each Cholesky size class (streams run concurrently)  */
    int32_t streamed;    /* 1: the panel came with the call (fit_args.bed) and its upload overlapped the fit;
                            0: the fit ran on a panel that was already complete on the device                 */
    int32_t n_blocks_missing; /* blocks that had missing calls (four-plane Gram), decided on the device      */
} dbslmm_b200_timing;

typedef struct dbslmm_b200_fit_args {
    int32_t  n_blocks;        /* blocks in this call (an m==0 block is a legal no-op)               */
    const int32_t* s_off;     /* [n_blocks+1] CSR offsets of small-effect SNPs                       */
    const int32_t* s_pos;     /* [s_off[n_blocks]] .bed row (INFO::pos) of each small SNP            */
    const double*  s_z;       /* [..] z-score (INFO::z)                                              */
    const int32_t* l_off;     /* NULL => small-only overload (LMM mode) for every block              */
    const int32_t* l_pos;
    const double*  l_z;
    int32_t  n_folds;         /* >=1: heritability folds sharing one Gram per block                  */
    const double* sigma_s;    /* [n_folds] h2/nsnp per fold (dbslmm.cpp:332)                          */
    int64_t  n_obs;           /* GWAS sample size (-n)                                               */
    double   tau;             /* LD shrinkage, 0.8 in the reference (dbslmmfit.cpp:697)              */
    int32_t  solver;          /* DBSLMM_B200_SOLVER_*                                                */
    int32_t  flags;           /* DBSLMM_B200_FLAG_*                                                  */
    double*  beta_s_out;      /* [n_folds][s_off[n_blocks]]                                          */
    double*  beta_l_out;      /* [n_folds][l_off[n_blocks]] or NULL                                  */
    int32_t* block_status_out;/* [n_blocks] or NULL                                                  */
    dbslmm_b200_timing* timing; /* or NULL                                                           */
    /* ---- optional: the fork's asymptotic-variance side channel (scr/calc_asymptotic_variance.cpp:22-57,
     * called from calcBlock, scr/dbslmmfit.cpp:484-490 / 516-519).  All NULL/0 => not computed.
     * For every block and every selected test individual i: variance_out[f][b][i] =
     * (X_l var_bl X_l' + X_s var_bs X_s')_ii with the test genotypes standardised within the selected
     * subset (dbslmmfit.cpp:427-429).  Cholesky solver only. */
    const uint8_t* test_bed;        /* host SNP-major .bed payload (after the magic bytes) of the test data    */
    int64_t  test_n_snp;            /* rows of test_bed                                                        */
    int32_t  test_n_total;          /* individuals in test_bed                                                 */
    const int32_t* test_indicator;  /* [test_n_total] != 0 => individual belongs to the test set              */
    const int32_t* s_tpos;          /* [s_off[n_blocks]] test .bed row of every small SNP                      */
    const int32_t* l_tpos;          /* [l_off[n_blocks]] or NULL                                               */
    double*  variance_out;          /* [n_folds][n_blocks][n_test], n_test = #selected individuals             */
    /* ---- optional: the reference panel travels WITH the fit, as DBSLMMFIT::est receives it (its bed_str argument,
     * scr/dbslmmfit.hpp:38-67, read row by row inside calcBlock).  bed != NULL replaces a prior load_bed: the SNP-major
     * payload (after the 3 magic bytes; pinned host memory for full PCIe speed) is uploaded INSIDE the call, the rows of
     * the biggest blocks first, and every batch of blocks is decoded and factored as soon as its rows have landed, so
     * the upload overlaps the fit.  The panel stays resident afterwards (later calls may pass bed = NULL).          */
    const uint8_t* bed;             /* or NULL: use the panel loaded by dbslmm_b200_load_bed                   */
    int64_t  bed_n_snp;
    int32_t  bed_n_ref;
    /* ---- optional: the quadratic form of the reference's external-validation tool `valid` (scr/validate.cpp:225-259,
     * SURVEY 8f-4) INSTEAD of the solve: quadform_out[b] = z_b' Sigma_b z_b with Sigma_b = tau X'X/n + (1-tau) I of the
     * block's SNPs (s_pos, s_z; `valid` uses the un-shrunk tau = 1: deno = z1' (X'X/n) z1).  Same decoder and integer
     * Gram as the fit; no factorisation.  beta_s_out may then be NULL; l_off must be NULL.                            */
    double*  quadform_out;          /* [n_blocks] or NULL                                                      */
} dbslmm_b200_fit_args;

#define DBSLMM_B200_FLAG_KEEP_INT_GRAM 1  /* also keep raw int32 Gram planes for dbslmm_b200_get_block_gram */
#define DBSLMM_B200_FLAG_FULL_SIGMA    2  /* write both triangles of Sigma (implied by the PCG solver)       */
#define DBSLMM_B200_FLAG_PLAN_CACHED   4  /* reuse the device plan of the previous fit (same CSR arrays)     */
#define DBSLMM_B200_FLAG_PANEL_SUBSET  8  /* with fit_args.bed: upload only the .bed rows this call's blocks use (one GPU of
                                             several, each given the whole host panel and its own blocks); the handle
                                             does NOT keep the panel for later calls                                */

DBSLMM_B200_API int  dbslmm_b200_abi_version(void);
DBSLMM_B200_API int  dbslmm_b200_device_count(void);

DBSLMM_B200_API int  dbslmm_b200_create(int device, dbslmm_b200_handle** out);
DBSLMM_B200_API void dbslmm_b200_destroy(dbslmm_b200_handle* h);
DBSLMM_B200_API const char* dbslmm_b200_last_error(const dbslmm_b200_handle* h);

/* Reference panel.  `bed` points just after the 3 magic bytes of a SNP-major PLINK .bed
 * (pitch = ceil(n_ref/4) bytes per SNP).  Copies to the device and runs the statistics
 * kernel (per-SNP allele sum, sum of squares, non-missing count).  ASYNCHRONOUS: the call
 * returns while the copy is in flight (the caller's next step -- building the block lists,
 * dbslmm_b200_fit planning -- overlaps it), so `bed` must stay valid and unchanged until the
 * next dbslmm_b200_snp_stats / dbslmm_b200_fit / dbslmm_b200_load_bed / dbslmm_b200_destroy
 * on this handle has returned.  (fit_args.bed, by contrast, is no longer needed once that
 * fit call returns.)
 * Limit: n_ref <= 409,344 individuals (the decoder stages two whole .bed rows of ceil(n_ref/4) bytes per warp in 200 KB
 * of shared memory; the reference, which reads byte by byte, has none).  Larger panels are refused with
 * DBSLMM_B200_ERR_ARG and a message naming the limit, here and in dbslmm_b200_fit(fit_args.bed). */
DBSLMM_B200_API int  dbslmm_b200_load_bed(dbslmm_b200_handle* h, const uint8_t* bed, int64_t n_snp, int32_t n_ref);

/* MAF pre-pass product (dtpr.cpp:93-102, 361-362): maf after mean imputation; optional
 * non-missing counts.  Both arrays have n_snp entries. */
DBSLMM_B200_API int  dbslmm_b200_snp_stats(dbslmm_b200_handle* h, double* maf_out, int32_t* n_nonmiss_out);

/* Block scheduler: O(n m^2 + m^3) cost model, longest-processing-time-first onto n_ranks.
 * m_s/m_l are per-block SNP counts (m_l may be NULL).  owner_out[b] in [0, n_ranks). */
DBSLMM_B200_API int  dbslmm_b200_plan_shards(int32_t n_blocks, const int32_t* m_s, const int32_t* m_l,
                             int32_t n_ref, int32_t n_ranks, int32_t* owner_out, double* rank_cost_out);

DBSLMM_B200_API int  dbslmm_b200_fit(dbslmm_b200_handle* h, const dbslmm_b200_fit_args* args);

/* The same fit fanned out over several GPUs of one box: hs[0..n_handles) are handles created on different devices.  The
 * blocks are assigned by dbslmm_b200_plan_shards, every GPU uploads only the panel rows its blocks use (args->bed is required;
 * one host thread per GPU inside the call), and the betas / block statuses land in the caller's block-major arrays as in
 * dbslmm_b200_fit.  This is the multi-GPU shape of DBSLMMFIT::est (one call, scr/dbslmmfit.hpp:38-67; its `thread` argument
 * becomes the handle list).  Not available with the variance side channel, quadform_out or FLAG_PLAN_CACHED.  timing: the
 * slowest GPU's phase times, work counters summed.  Errors are reported on hs[0] (dbslmm_b200_last_error(hs[0])). */
DBSLMM_B200_API int  dbslmm_b200_fit_multi(dbslmm_b200_handle* const* hs, int32_t n_handles, const dbslmm_b200_fit_args* args);

/* Page-locked host memory for the panel (`bed` of load_bed / fit_args.bed): uploads from it run at full PCIe speed and
 * truly asynchronously; ordinary memory works too, but is staged by the driver.  The reference has no counterpart (it
 * reads the .bed through an ifstream, scr/dtpr.cpp:302-315); the `dbslmm` command line reads its .bed files straight
 * into such a buffer.  Needs a created handle (a CUDA context); free with dbslmm_b200_host_free before destroy. */
DBSLMM_B200_API int  dbslmm_b200_host_alloc(dbslmm_b200_handle* h, uint64_t bytes, void** out);
DBSLMM_B200_API void dbslmm_b200_host_free(dbslmm_b200_handle* h, void* p);

/* Polygenic scores over a validation panel (BASELINE config 4; replaces the per-fold
 * `plink --score <eff>.txt 1 2 4 sum` of DBSLMM_script.sh:87): score[f][i] = sum_j beta[f][j] * dosage_ij,
 * dosage = copies of A1 (or of A2 where flip[j] != 0) of validation .bed row pos[j], missing calls
 * mean-imputed.  `bed_val` is a host SNP-major .bed payload (after the magic bytes) of n_snp_val rows and
 * n_val individuals; it is uploaded, scored for all n_folds in one pass and left resident until the next
 * call (bed_val = NULL: score the panel that is already there -- announced by dbslmm_b200_score_prefetch or left by the
 * previous call; n_snp_val / n_val are then ignored).  flip may be NULL.  scores_out is [n_folds][n_val]. */
/* Announce the validation panel of the NEXT dbslmm_b200_score call: its upload (2.75 GB at config 4) is queued behind the
 * panel copies of the next dbslmm_b200_fit on this handle and overlaps that fit's kernels; score is then called with
 * bed_val = NULL.  `bed_val` (pinned for full speed) must stay valid until that score call has returned. */
DBSLMM_B200_API int  dbslmm_b200_score_prefetch(dbslmm_b200_handle* h, const uint8_t* bed_val, int64_t n_snp_val, int32_t n_val);
DBSLMM_B200_API int  dbslmm_b200_score(dbslmm_b200_handle* h, const uint8_t* bed_val, int64_t n_snp_val, int32_t n_val,
                       const int32_t* pos, const uint8_t* flip, int64_t n_scored,
                       const double* beta, int32_t n_folds, double* scores_out, float* kernel_ms_out);

/* Polygenic scores over a target panel of any size, streamed through the GPU: the `plink --bfile <target> --score <eff>.txt
 * 1 2 4 sum` of DBSLMM_script.sh:87 for every fold in one pass.  Same semantics as dbslmm_b200_score (mean imputation from
 * the row's called genotypes, flip[j] != 0 scores A2), plus PLINK's .profile counts:
 *   cnt_out[i]  = 2 x the genotypes of individual i called on the scored rows  (CNT),
 *   cnt2_out[i] = copies of the scored allele among them                      (CNT2);
 * either may be NULL.  A row without a called genotype adds nothing to scores, CNT or CNT2; n_empty_rows_out (or NULL)
 * receives the number of such scored rows.
 * `bed_val` is the SNP-major payload (after the magic bytes) in ORDINARY host memory -- an mmap of the .bed is fine -- and
 * only the rows named by pos are read (pos may be unsorted and may repeat).  The call gathers the scored rows chunk by
 * chunk into pinned staging buffers on the host worker pool and copies each chunk (rows, beta and flip slices) with one
 * asynchronous copy; gather, copy and kernels of consecutive chunks overlap.  A chunk holds
 *   R = max(1, floor(chunk_bytes / (ceil(n_val / 4) + 1)))
 * scored rows (chunk_bytes = 0: 64 MB), i.e. R x (ceil(n_val / 4) + 1 + 8 n_folds) bytes with their beta slices.  Device and
 * pinned memory are five such chunks plus O(n_val x n_folds), whatever n_snp_val.  R does not depend on n_folds, so fold f of
 * an F-fold call is bit-identical to the 1-fold call with beta[f].
 * Deterministic: the same arguments give the same bits; when one chunk holds every scored row the scores are bit-identical
 * to dbslmm_b200_score.  Limits: n_val <= 536,870,911 (int32 row sums), n_scored <= INT32_MAX / 2 (CNT in int32).
 * kernel_ms_out (or NULL): the summed device time of the chunks' kernels.  Synchronous. */
DBSLMM_B200_API int  dbslmm_b200_score_stream(dbslmm_b200_handle* h, const uint8_t* bed_val, int64_t n_snp_val, int32_t n_val,
                              const int32_t* pos, const uint8_t* flip, int64_t n_scored, const double* beta, int32_t n_folds,
                              uint64_t chunk_bytes, double* scores_out, int32_t* cnt_out, int32_t* cnt2_out,
                              int32_t* n_empty_rows_out, float* kernel_ms_out);

/* LD Scores of a reference panel, as `ldsc.py --bfile <panel> --l2` computes them (ldsc 1.0.1's ldscore.py restated):
 *   l_j = sum_{k in W(j)} r2adj(j, k),   r2adj = r^2 - (1 - r^2) / (n - 2)   (denominator n_ref when n_ref <= 2),
 * r = the Pearson correlation of the mean-imputed genotypes of kept SNPs j and k (r_jj = 1), formed from the exact integer
 * Gram of the decoded rows on the tensor cores.
 * rows[0..n_rows) are .bed rows, chromosome-major and in coordinate order within a chromosome; chromosome c is
 * rows[chr_off[c] .. chr_off[c + 1]).  A row is KEPT iff min(f, 1 - f) > maf_min and missing + heterozygous calls < n_ref
 * (f = allele frequency among the called genotypes, 0 when none is called): every kept SNP has nonzero variance.  W(j) is
 * the set of kept SNPs k of j's chromosome with |c_k - c_j| <= max_dist, where c is coord[row] (wind_kind = COORD: cM or
 * base pairs, non-decreasing within a chromosome) or the index among the chromosome's kept SNPs (wind_kind = SNPS, coord
 * NULL, max_dist a whole number).  Windows never cross a chromosome.
 * Outputs, each [n_rows] and each may be NULL: kept_out 0/1, maf_out min(f, 1 - f), l2_out the LD Score (NaN where not
 * kept); guard_out [n_chr]: 1 where the window of the chromosome's last kept SNP reaches its first one (ldsc refuses such a
 * chromosome unless told otherwise; reported here, not enforced).  With l2_out NULL the call stops after the statistics
 * pass: kept_out, maf_out and guard_out only, one pass over the rows (a caller can check the guard before the LD pass).
 * Two passes stream the requested rows from ORDINARY host memory (an mmap of the .bed is fine; only these rows are read)
 * through pinned staging buffers, as dbslmm_b200_score_stream does: per-row statistics, then segments of consecutive
 * 128-row tiles with the halo of rows their windows reach.  Device memory: O(segment + halo) x 2 x n_pad bytes plus one
 * double per (SNP, 128-row tile its window reaches).  segment_rows = 0 sizes the segments from free device memory; a
 * nonzero multiple of 128 fixes them.  Deterministic: the result does not depend on the segment size, on which other
 * chromosomes are in the call, or on the run.  Limits: n_ref <= 409,344, n_rows <= INT32_MAX.  kernel_ms_out (or NULL):
 * the summed device time of the call's kernels.  Synchronous. */
/* Inspection hook (the tests check the window rule through it): the window rule of dbslmm_b200_ldscore over the m kept
 * SNPs of one chromosome, the library's own host code (needs no GPU): W(k) = [lo_out[k],
 * hi_out[k]] = the k' with |c_k' - c_k| <= max_dist, c = coord (non-decreasing) or, with coord NULL, the index k.  The
 * chromosome's guard is lo_out[m - 1] == 0. */
DBSLMM_B200_API int  dbslmm_b200_ld_windows(const double* coord, int64_t m, double max_dist, int32_t* lo_out, int32_t* hi_out);
#define DBSLMM_B200_LD_WIND_COORD 0
#define DBSLMM_B200_LD_WIND_SNPS  1
DBSLMM_B200_API int  dbslmm_b200_ldscore(dbslmm_b200_handle* h, const uint8_t* bed, int64_t n_snp, int32_t n_ref,
                         const int32_t* rows, int64_t n_rows, const int32_t* chr_off, int32_t n_chr,
                         int32_t wind_kind, const double* coord, double max_dist, double maf_min, int64_t segment_rows,
                         uint8_t* kept_out, double* maf_out, double* l2_out, int32_t* guard_out, float* kernel_ms_out);

/* Partitioned LD Scores (`ldsc.py --l2 --annot`): one LD Score per annotation column c,
 *   L_c(j) = sum_{k in W(j)} r2adj(j, k) a_kc,
 * with dbslmm_b200_ldscore's kept set, windows, guard, r and r2adj.  As ldsc does, the unbiased map is applied per term:
 * r2adj = fma(1 + 1/denominator, r^2, -1/denominator) once per pair, then acc_c = fma(r2adj, a_kc, acc_c), the partners k
 * in ascending order within each 128-SNP tile and the tiles in ascending order.  annot is row-major [n_rows][n_annot],
 * aligned with rows, every value finite; 1 <= n_annot <= DBSLMM_B200_LD_MAX_ANNOT.  l2_out is [n_rows][n_annot] (NaN rows
 * where a SNP is not kept); l2_out NULL stops after the statistics pass, as in dbslmm_b200_ldscore.  The other arguments
 * and outputs are dbslmm_b200_ldscore's.  Column c does not depend on the other columns of the call: computed alone or
 * among others it has the same bits.  Deterministic as dbslmm_b200_ldscore.  Device memory: O(segment + halo) x (2 x n_pad
 * + 8 n_annot) bytes, 2 x n_annot doubles per (SNP of the segment, 128-row tile its window reaches), and the result,
 * n_annot doubles per row.  Synchronous. */
#define DBSLMM_B200_LD_MAX_ANNOT 4096
DBSLMM_B200_API int  dbslmm_b200_ldscore_annot(dbslmm_b200_handle* h, const uint8_t* bed, int64_t n_snp, int32_t n_ref,
                         const int32_t* rows, int64_t n_rows, const int32_t* chr_off, int32_t n_chr,
                         int32_t wind_kind, const double* coord, double max_dist, double maf_min, int64_t segment_rows,
                         const double* annot, int32_t n_annot,
                         uint8_t* kept_out, double* maf_out, double* l2_out, int32_t* guard_out, float* kernel_ms_out);

/* Windowed r between SNP pairs of a reference panel, as `plink --r2 --ld-window N --ld-window-kb K --ld-window-r2 R` selects
 * them.  rows, chr_off and coord work as in dbslmm_b200_ldscore (coord: base pairs, non-decreasing within a chromosome,
 * required).  A pair (a, b), a < b positions in rows, is written when both lie in one chromosome, b - a <= max_snps - 1
 * (--ld-window N), coord[b] - coord[a] <= max_dist (--ld-window-kb K as K x 1000, edges included) and r^2 >= r2_min
 * (--ld-window-r2).  Windows never cross a chromosome.  r is dbslmm_b200_ldscore's: the Pearson r of the mean-imputed
 * allele counts, num / sqrt(n_a n_b d_a d_b) from the exact integer numerator; without missing calls in either SNP it is
 * the Pearson r of the allele counts.  A row with no called genotype or with zero variance is not USABLE: it never forms a
 * pair, but it still counts toward the max_snps distance.
 * The pairs are delivered in ascending (a, b) order through `sink`, called on the calling thread with CSR slices: rows
 * a0 .. a1 - 1 (consecutive slices cover every row exactly once), off[0 .. a1 - a0] (off[0] = 0), and for the pairs of row
 * a = a0 + i, entries off[i] .. off[i + 1] - 1 of b (the partner's position in rows) and r (signed).  The arrays are valid
 * during the call only.  A nonzero return from the sink stops the call with DBSLMM_B200_ERR_SINK; the sink is not called
 * again.  Outputs (each may be NULL): usable_out [n_rows] 0/1, n_pairs_out the number of pairs written, n_miss_pairs_out
 * the number of those with a SNP with missing calls, kernel_ms_out the summed device time of the call's kernels.
 * Two passes over the rows as dbslmm_b200_ldscore, segment_rows as there; each segment is counted on the device, then
 * emitted in ranges of row tiles whose pairs fit a fixed device buffer (8 Mi pairs, or the most pairs one 128-row tile can
 * have, whichever is more) and copied to two pinned buffers in turn, so the sink of one range runs while the device
 * emits the next.  Device and pinned memory do not grow with the number of pairs.  Deterministic: the bits and the order
 * of the output depend neither on the segment size, nor on the other chromosomes of the call, nor on the run.
 * Limits: n_ref <= 409,344, n_rows <= INT32_MAX, max_snps >= 1, max_dist >= 0 (may be +inf), r2_min not NaN.
 * Synchronous. */
typedef int (*dbslmm_b200_ld_sink)(void* user, int64_t a0, int64_t a1, const int64_t* off, const int32_t* b, const double* r);
DBSLMM_B200_API int  dbslmm_b200_ld_pairs(dbslmm_b200_handle* h, const uint8_t* bed, int64_t n_snp, int32_t n_ref,
                         const int32_t* rows, int64_t n_rows, const int32_t* chr_off, int32_t n_chr, const double* coord,
                         int32_t max_snps, double max_dist, double r2_min, int64_t segment_rows,
                         dbslmm_b200_ld_sink sink, void* user, uint8_t* usable_out, int64_t* n_pairs_out,
                         int64_t* n_miss_pairs_out, float* kernel_ms_out);

/* ---- inspection hooks used by the parity tests (operate on the state of the last fit) ---- */
/* int8 codes of one decoded row of the last fit: SNP j of block `block` (its small SNPs first, then its large ones),
 * plane 0 = allele counts (missing -> 0), plane 1 = call mask (1 = called; holds the last mask written at that position,
 * which is the current one whenever the block has missing calls); n_out <= n_pad bytes. */
DBSLMM_B200_API int  dbslmm_b200_get_row_codes(dbslmm_b200_handle* h, int32_t block, int32_t j, int32_t plane, int8_t* codes_out, int32_t n_out);
/* Sigma of block b as dense row-major m x m (m = m_s + m_l, small SNPs first).  Lower triangle is
 * always valid; the upper one only with FLAG_FULL_SIGMA / PCG solver (else mirrored on the host). */
DBSLMM_B200_API int  dbslmm_b200_get_block_sigma(dbslmm_b200_handle* h, int32_t block, double* sigma_out);
/* The Cholesky factor of block b's bordered system K = Sigma + c diag(1_small, 0_large) from the LAST fold of the last
 * Cholesky fit: l_out = m x m row-major, the lower triangle of L with its diagonal, zeros above (the W_kk^T the solver
 * keeps in the upper triangles of the diagonal tiles is not returned); y_out = the m entries of y = L^-1 z (matrix row mp).
 * Either may be NULL.  DBSLMM_B200_ERR_STATE after a PCG or quadform fit.  tools/l_diff.py uses it to show where the
 * factors of two fits differ (block, panel, rows). */
DBSLMM_B200_API int  dbslmm_b200_get_block_factor(dbslmm_b200_handle* h, int32_t block, double* l_out, double* y_out);
/* raw integer Gram planes (needs FLAG_KEEP_INT_GRAM): Q = G G^T, A_ij = sum g_i M_j, N = M M^T;
 * A and N may be NULL; for blocks without missing calls A_ij = S_i and N = n_ref. */
DBSLMM_B200_API int  dbslmm_b200_get_block_gram(dbslmm_b200_handle* h, int32_t block, int32_t* q_out, int32_t* a_out, int32_t* n_out);
/* PCG iteration count of block b in the last PCG-solver fit (max over its right-hand sides). */
DBSLMM_B200_API int  dbslmm_b200_get_block_iters(dbslmm_b200_handle* h, int32_t block);

#ifdef __cplusplus
}
#endif
#endif /* DBSLMM_B200_H */
