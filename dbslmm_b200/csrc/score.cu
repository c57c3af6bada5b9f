// score.cu -- polygenic-score accumulation over a validation panel (SURVEY.md 8f-3, BASELINE config 4).
//
// Replaces the `plink --bfile val --score <eff>.txt 1 2 4 sum` step that the reference's driver runs
// once per heritability fold (DBSLMM_script.sh:87, scored column 4 = beta / sqrt(2 maf (1-maf)) written
// by scr/dbslmm.cpp:354-362): score_i = sum_j beta_j * dosage_ij, dosage = copies of the scored
// allele, missing calls mean-imputed (PLINK's default), all folds in ONE pass over the 2-bit .bed.
// PLINK is external to the reference, so this path's parity is pinned only against a numpy
// restatement of those documented semantics (tests/test_gpu_score.py).
//
// Every .bed byte is read once (coalesced, 4 bytes = 16 individuals per thread); per-chunk partial sums are written to
// a scratch buffer and reduced in a fixed order (deterministic).  The work is one FP64 multiply-add per genotype and
// fold (3.3e10 at config 4), so the FP64 pipe, not HBM, bounds it.
//
// The streaming path (dbslmm_b200_score_stream) feeds the same kernel COMPACT chunks instead of a resident panel: row k
// of a chunk is scored SNP j0 + k, so the pos indirection is gone and the chunk's own row statistics (chunk_stats_kernel,
// no limit on the row length) sit beside it.  score_counts_kernel adds PLINK's CNT / CNT2 columns.
#include <algorithm>
#include "common.cuh"
#include "kernels.h"

namespace dbslmm {

static constexpr int kScoreThreads = 256;
static constexpr int kMaxFolds = 3;          // folds per pass (more folds => several passes): 16 individuals x 3 folds of FP64 accumulators per thread

// One thread = FOUR consecutive .bed bytes = 16 individuals (a warp reads 128 contiguous bytes of a row per load), 64
// scored SNPs per shared-memory batch.  Per SNP the four possible dosages {code 0, 1 = missing -> mean, 2, 3} are put
// in shared memory once (allele flip and mean imputation folded in), so the inner loop is: extract the 2-bit code,
// load the dosage it selects (one LDS.64), NF fused multiply-adds.
// COMPACT = false: rows pos[s] of a resident panel (dbslmm_b200_score).  COMPACT = true: row s of a compact chunk, and a
// row without a called genotype (mean 0/0) contributes nothing instead of NaN.
template <int NF, bool COMPACT>
__global__ void __launch_bounds__(kScoreThreads, 2)
prs_partial_kernel(const uint8_t* __restrict__ bed, int32_t pitch, int32_t n_val, const SnpStat* __restrict__ stats,
                   const int32_t* __restrict__ pos, const uint8_t* __restrict__ flip, const double* __restrict__ beta,
                   int64_t beta_stride, int32_t n_scored, int32_t rows_per_chunk, double* __restrict__ partial) {
    __shared__ double s_beta[64][NF];
    __shared__ __align__(16) double s_dos[64][4];            // dosage of code 0, 1, 2, 3
    __shared__ int32_t s_row[64];
    const int tid = threadIdx.x;
    const int word_col = blockIdx.x * kScoreThreads + tid;   // 4-byte column of the row
    const int byte0 = word_col * 4;
    const bool in_range = byte0 < pitch;
    const bool full_word = byte0 + 4 <= pitch && (pitch & 3) == 0;     // rows stay 4-byte aligned only if the pitch is
    const int s_begin = blockIdx.y * rows_per_chunk;
    const int s_end = min(n_scored, s_begin + rows_per_chunk);
    double acc[16][NF];
#pragma unroll
    for (int q = 0; q < 16; ++q)
#pragma unroll
        for (int f = 0; f < NF; ++f) acc[q][f] = 0.0;
    for (int s0 = s_begin; s0 < s_end; s0 += 64) {
        const int nb = min(64, s_end - s0);
        __syncthreads();
        if (tid < nb) {
            const int row = COMPACT ? s0 + tid : pos[s0 + tid];
            const SnpStat st = stats[row];
            const bool fl = flip != nullptr && flip[s0 + tid] != 0;
            const double mu = (double)st.sum / (double)st.n_nonmiss;        // mean A1 dosage of called genotypes
            s_row[tid] = row;
            // A1 copies: code 0 -> 2, 2 -> 1, 3 -> 0, 1 -> missing (dtpr.cpp:329-350)
            s_dos[tid][0] = fl ? 0.0 : 2.0;
            s_dos[tid][1] = fl ? 2.0 - mu : mu;
            s_dos[tid][2] = 1.0;
            s_dos[tid][3] = fl ? 2.0 : 0.0;
#pragma unroll
            for (int f = 0; f < NF; ++f) s_beta[tid][f] = beta[(int64_t)f * beta_stride + s0 + tid];
            if constexpr (COMPACT) {
                if (st.n_nonmiss == 0) {
                    s_dos[tid][0] = s_dos[tid][1] = s_dos[tid][2] = s_dos[tid][3] = 0.0;
#pragma unroll
                    for (int f = 0; f < NF; ++f) s_beta[tid][f] = 0.0;
                }
            }
        }
        __syncthreads();
        if (!in_range) continue;
        // software pipeline: the four row words of the NEXT group are in flight while this group is accumulated
        auto load_word = [&](int j) -> uint32_t {
            if (j >= nb) return 0xFFFFFFFFu;
            const uint8_t* p = bed + (size_t)s_row[j] * pitch + byte0;
            if (full_word) return __ldg(reinterpret_cast<const uint32_t*>(p));
            uint32_t w = 0;
            for (int bq = 0; bq < 4; ++bq) w |= (uint32_t)((byte0 + bq < pitch) ? p[bq] : 0xFF) << (8 * bq);
            return w;
        };
        uint32_t words[4], next[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) next[u] = load_word(u);
        for (int j0 = 0; j0 < nb; j0 += 4) {
#pragma unroll
            for (int u = 0; u < 4; ++u) words[u] = next[u];
#pragma unroll
            for (int u = 0; u < 4; ++u) next[u] = load_word(j0 + 4 + u);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (j0 + u >= nb) break;
                const uint32_t w = words[u];
                // the SNP's four dosages sit in 32 contiguous bytes of shared memory: one broadcast-class LDS.64 indexed
                // by the 2-bit code replaces the compare/select chain
                const char* dos = reinterpret_cast<const char*>(&s_dos[j0 + u][0]);
                double bf[NF];
#pragma unroll
                for (int f = 0; f < NF; ++f) bf[f] = s_beta[j0 + u][f];
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const uint32_t c8 = (q < 15) ? ((w >> (2 * q)) & 3u) << 3 : (w >> 30) << 3;     // code * 8 bytes
                    const double d = *reinterpret_cast<const double*>(dos + c8);
#pragma unroll
                    for (int f = 0; f < NF; ++f) acc[q][f] = fma(bf[f], d, acc[q][f]);
                }
            }
        }
    }
    if (!in_range) return;
#pragma unroll
    for (int f = 0; f < NF; ++f)
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int ind = byte0 * 4 + q;
            if (ind < n_val) partial[((size_t)blockIdx.y * NF + f) * n_val + ind] = acc[q][f];
        }
}

// ACC = false: scores = the fixed-order sum of the slices (dbslmm_b200_score); ACC = true: scores += that sum (one chunk of
// the streaming path into zeroed accumulators, so a single chunk gives the same bits as the resident path)
template <bool ACC>
__global__ void prs_reduce_kernel(const double* __restrict__ partial, int32_t n_chunks, int32_t nf, int32_t n_val,
                                  double* __restrict__ scores) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int f = blockIdx.y;
    if (i >= n_val) return;
    double s = 0.0;
    for (int c = 0; c < n_chunks; ++c) s += partial[((size_t)c * nf + f) * n_val + i];
    if (ACC) scores[(size_t)f * n_val + i] += s;
    else scores[(size_t)f * n_val + i] = s;
}

template <bool COMPACT>
static cudaError_t launch_prs_t(const uint8_t* bed, int32_t n_val, const SnpStat* stats, const int32_t* pos, const uint8_t* flip,
                                const double* beta, int64_t beta_stride, int32_t n_scored, int32_t nf, int32_t n_chunks,
                                double* partial, double* scores, cudaStream_t st) {
    if (n_scored == 0 || nf == 0) return cudaSuccess;
    const int32_t pitch = (n_val + 3) / 4;
    const int rows_per_chunk = (n_scored + n_chunks - 1) / n_chunks;
    dim3 grid(((pitch + 3) / 4 + kScoreThreads - 1) / kScoreThreads, n_chunks);
    switch (nf) {
        case 1: prs_partial_kernel<1, COMPACT><<<grid, kScoreThreads, 0, st>>>(bed, pitch, n_val, stats, pos, flip, beta, beta_stride, n_scored, rows_per_chunk, partial); break;
        case 2: prs_partial_kernel<2, COMPACT><<<grid, kScoreThreads, 0, st>>>(bed, pitch, n_val, stats, pos, flip, beta, beta_stride, n_scored, rows_per_chunk, partial); break;
        case 3: prs_partial_kernel<3, COMPACT><<<grid, kScoreThreads, 0, st>>>(bed, pitch, n_val, stats, pos, flip, beta, beta_stride, n_scored, rows_per_chunk, partial); break;
        default: return cudaErrorInvalidValue;
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    dim3 rgrid((n_val + 255) / 256, nf);
    prs_reduce_kernel<COMPACT><<<rgrid, 256, 0, st>>>(partial, n_chunks, nf, n_val, scores);
    return cudaGetLastError();
}

cudaError_t launch_prs(const uint8_t* bed, int32_t n_val, const SnpStat* stats, const int32_t* pos, const uint8_t* flip,
                       const double* beta, int64_t beta_stride, int32_t n_scored, int32_t nf, int32_t n_chunks,
                       double* partial, double* scores, cudaStream_t st) {
    return launch_prs_t<false>(bed, n_val, stats, pos, flip, beta, beta_stride, n_scored, nf, n_chunks, partial, scores, st);
}

cudaError_t launch_prs_chunk(const uint8_t* chunk, int32_t n_val, const SnpStat* stats, const uint8_t* flip, const double* beta,
                             int64_t beta_stride, int32_t n_rows, int32_t nf, int32_t n_slices, double* partial, double* scores,
                             cudaStream_t st) {
    return launch_prs_t<true>(chunk, n_val, stats, nullptr, flip, beta, beta_stride, n_rows, nf, n_slices, partial, scores, st);
}

int32_t prs_slices(int n_sm, int32_t n_val, int64_t n_rows) {
    const int32_t pitch = (n_val + 3) / 4;
    return std::max(1, std::min<int>(4 * n_sm / std::max(1, ((pitch + 3) / 4 + 255) / 256), (int)((n_rows + 63) / 64)));
}

// ------------------------------------------------------------------------------------------
// Per-row statistics of a compact chunk (called count, allele sum, sum of squares) for the mean imputation of the
// streaming path.  One CTA per row at a time: every thread reads whole 4-byte words of the row straight from global
// memory (coalesced; the words that straddle the row's ends are masked), then warp shuffles and a fixed-order sum over
// the warps.  Nothing is staged in shared memory, so the row length is limited only by the int32 sums: n_val <=
// kScoreMaxNVal (sum of squares <= 4 n_val).  The chunk needs 3 readable bytes past its last row.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kScoreThreads)
chunk_stats_kernel(const uint8_t* __restrict__ chunk, int32_t n_rows, int32_t pitch, int32_t n_val, SnpStat* __restrict__ stats,
                   int32_t* __restrict__ n_empty) {
    __shared__ int32_t red[3][kScoreThreads / 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int32_t r = blockIdx.x; r < n_rows; r += gridDim.x) {
        const int64_t s = (int64_t)r * pitch;
        const int64_t a0 = s & ~(int64_t)3;
        const int64_t nw = (s + pitch - a0 + 3) >> 2;
        const uint32_t* w32 = reinterpret_cast<const uint32_t*>(chunk + a0);
        int32_t c0 = 0, c1 = 0, c2 = 0;
        for (int64_t i = threadIdx.x; i < nw; i += kScoreThreads) {
            uint32_t w = __ldg(w32 + i);
            // byte k of the word is byte b of the row; it holds min(4, n_val - 4 b) genotypes of the row (none outside it)
            uint32_t valid = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int64_t b = a0 - s + 4 * i + k;
                const int64_t g = (b < 0 || b >= pitch) ? 0 : min((int64_t)4, (int64_t)n_val - 4 * b);
                valid |= ((1u << (2 * g)) - 1u) << (8 * k);
            }
            w |= ~valid;                               // outside the row -> code 3 (counts nothing below)
            const uint32_t lo = w & 0x55555555u, hi = (w >> 1) & 0x55555555u;
            c0 += __popc(~(lo | hi) & 0x55555555u);    // code 0 -> allele count 2
            c1 += __popc(lo & ~hi);                    // code 1 -> missing
            c2 += __popc(hi & ~lo);                    // code 2 -> allele count 1
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            c0 += __shfl_xor_sync(0xffffffffu, c0, o);
            c1 += __shfl_xor_sync(0xffffffffu, c1, o);
            c2 += __shfl_xor_sync(0xffffffffu, c2, o);
        }
        if (lane == 0) { red[0][warp] = c0; red[1][warp] = c1; red[2][warp] = c2; }
        __syncthreads();
        if (threadIdx.x == 0) {
            int32_t t0 = 0, t1 = 0, t2 = 0;
            for (int k = 0; k < kScoreThreads / 32; ++k) { t0 += red[0][k]; t1 += red[1][k]; t2 += red[2][k]; }
            SnpStat o;
            o.n_nonmiss = n_val - t1;
            o.sum = 2 * t0 + t2;
            o.sumsq = 4 * t0 + t2;
            o.pad = 0;
            stats[r] = o;
            if (o.n_nonmiss == 0 && n_empty) atomicAdd(n_empty, 1);
        }
        __syncthreads();
    }
}

cudaError_t launch_chunk_stats(const uint8_t* chunk, int32_t n_rows, int32_t n_val, SnpStat* stats, int32_t* n_empty, int n_sm,
                               cudaStream_t st) {
    if (n_rows == 0) return cudaSuccess;
    const int ctas = std::max(1, std::min(n_rows, 8 * n_sm));
    chunk_stats_kernel<<<ctas, kScoreThreads, 0, st>>>(chunk, n_rows, (n_val + 3) / 4, n_val, stats, n_empty);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// PLINK's CNT / CNT2 over the rows of a compact chunk: per individual, 2 x the called genotypes and the copies of the
// scored allele among them (A1, or A2 where flip[k] != 0).  Same thread layout as the scoring kernel (4 bytes = 16
// individuals per thread, rows sliced over blockIdx.y); each slice adds its integer counts with atomics -- integer sums
// are exact, so the order of the slices does not change the result.  A row without a called genotype adds nothing.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kScoreThreads)
score_counts_kernel(const uint8_t* __restrict__ chunk, int32_t pitch, int32_t n_val, const uint8_t* __restrict__ flip,
                    int32_t n_rows, int32_t rows_per_slice, int32_t* __restrict__ cnt, int32_t* __restrict__ cnt2) {
    const int byte0 = (blockIdx.x * kScoreThreads + threadIdx.x) * 4;
    if (byte0 >= pitch) return;
    const bool full_word = byte0 + 4 <= pitch && (pitch & 3) == 0;
    const int r_begin = blockIdx.y * rows_per_slice;
    const int r_end = min(n_rows, r_begin + rows_per_slice);
    int32_t called[16], copies[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) called[q] = copies[q] = 0;
    for (int r = r_begin; r < r_end; ++r) {
        const uint8_t* p = chunk + (size_t)r * pitch + byte0;
        uint32_t w;
        if (full_word) w = __ldg(reinterpret_cast<const uint32_t*>(p));
        else {
            w = 0;
            for (int bq = 0; bq < 4; ++bq) w |= (uint32_t)((byte0 + bq < pitch) ? p[bq] : 0x55) << (8 * bq);   // past the row: missing
        }
        const bool fl = flip != nullptr && flip[r] != 0;
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const uint32_t c = (w >> (2 * q)) & 3u;
            const int32_t ok = c != 1u;                                   // code 1 = missing
            const int32_t a1 = 2 - (int32_t)(c & 1u) - (int32_t)(c >> 1); // copies of A1: code 0 -> 2, 2 -> 1, 3 -> 0
            called[q] += ok;
            copies[q] += ok ? (fl ? 2 - a1 : a1) : 0;
        }
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int ind = byte0 * 4 + q;
        if (ind < n_val && called[q] != 0) {
            atomicAdd(cnt + ind, 2 * called[q]);
            atomicAdd(cnt2 + ind, copies[q]);
        }
    }
}

cudaError_t launch_score_counts(const uint8_t* chunk, int32_t n_val, const uint8_t* flip, int32_t n_rows, int32_t n_slices,
                                int32_t* cnt, int32_t* cnt2, cudaStream_t st) {
    if (n_rows == 0) return cudaSuccess;
    const int32_t pitch = (n_val + 3) / 4;
    const int rows_per_slice = (n_rows + n_slices - 1) / n_slices;
    dim3 grid(((pitch + 3) / 4 + kScoreThreads - 1) / kScoreThreads, (n_rows + rows_per_slice - 1) / rows_per_slice);
    score_counts_kernel<<<grid, kScoreThreads, 0, st>>>(chunk, pitch, n_val, flip, n_rows, rows_per_slice, cnt, cnt2);
    return cudaGetLastError();
}

}  // namespace dbslmm
