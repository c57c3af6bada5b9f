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
