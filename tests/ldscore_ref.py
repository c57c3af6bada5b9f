"""CPU restatement of `ldsc.py --l2` (ldsc 1.0.1's ldscore.py, as dbslmm_b200_ldscore states it), two ways:

  * ldscore_exact: the correlations from the exact integer numerators of the code base's planes
        num_jk = n_j n_k Q_jk - n_j S_k A_jk - n_k S_j A_kj + S_j S_k N_jk,   r_jk^2 = num_jk^2 / (n_j n_k d_j d_k)
    evaluated in x86 extended precision (np.longdouble), r_jj = 1, and r2adj = r^2 - (1 - r^2) / (n - 2) summed per
    term over the window;
  * ldscore_ldsc64: ldsc's own float64 recipe -- mean-impute, standardise (np.std, ddof 0), r = Y^T Y / n, l2_unbiased,
    window sums.

Genotypes are int8 [n_snp, n] copies of the .bim A1 allele, -1 for a missing call."""
import numpy as np

LD = np.longdouble


def ld_panel(rng, m, n, miss, copy=0.7):
    """m rows of A1 copies with LD along the rows; polymorphic and not all-heterozygous (kept at maf_min = 0) when n >= 4."""
    G = rng.binomial(2, rng.uniform(0.05, 0.5, m)[:, None], size=(m, n)).astype(np.int8)
    for k in range(1, m):
        c = rng.random(n) < copy
        G[k, c] = G[k - 1, c]
    if miss > 0:
        G[rng.random(G.shape) < miss] = -1
    if n >= 4:
        G[:, 0], G[:, 1] = 0, 2
    return G


def snp_filter(G, maf_min=0.0):
    """ldsc's __filter_snps_maf__: (kept, maf) per row."""
    n = G.shape[1]
    called = G >= 0
    nn = called.sum(1)
    S = np.where(called, G, 0).astype(np.int64).sum(1)
    het = (G == 1).sum(1)
    f = np.divide(S, 2.0 * nn, out=np.zeros(G.shape[0]), where=nn > 0)
    maf = np.minimum(f, 1.0 - f)
    kept = (maf > maf_min) & ((n - nn) + het < n)
    return kept, maf


def windows(x, max_dist):
    """ldsc's getBlockLefts, both ends: W(k) = lo[k]..hi[k] over coordinates x (non-decreasing)."""
    m = len(x)
    lo = np.zeros(m, np.int64)
    hi = np.zeros(m, np.int64)
    j = 0
    for k in range(m):
        while abs(x[j] - x[k]) > max_dist:
            j += 1
        lo[k] = j
    j = m - 1
    for k in range(m - 1, -1, -1):
        while abs(x[j] - x[k]) > max_dist:
            j -= 1
        hi[k] = j
    return lo, hi


def _chrom_windows(kept_idx, coord, max_dist):
    x = np.arange(len(kept_idx), dtype=np.float64) if coord is None else np.asarray(coord, np.float64)[kept_idx]
    return windows(x, max_dist)


def _int_planes(Gk, block=65536):
    """Q, A (A_jk = g_j . M_k), N of the kept rows in int64; exact: float64 products of small integers, summed in blocks."""
    m, n = Gk.shape
    Q = np.zeros((m, m), np.int64)
    A = np.zeros((m, m), np.int64)
    N = np.zeros((m, m), np.int64)
    for c0 in range(0, n, block):
        X = Gk[:, c0:c0 + block]
        M = (X >= 0).astype(np.float64)
        g = np.where(X >= 0, X, 0).astype(np.float64)
        Q += np.rint(g @ g.T).astype(np.int64)
        A += np.rint(g @ M.T).astype(np.int64)
        N += np.rint(M @ M.T).astype(np.int64)
    return Q, A, N


def ldscore_exact(G, chr_off, coord=None, max_dist=1.0, maf_min=0.0):
    """The contract in extended precision.  Returns dict(l2, kept, maf, guard, s, wcount): l2 / s float64[n_rows]
    (NaN where not kept; s_j = sum_k r^2 + (1 - r^2) / denom, the magnitudes of both parts), wcount = |W(j)|."""
    n_rows, n = G.shape
    kept, maf = snp_filter(G, maf_min)
    denom = LD(n - 2) if n > 2 else LD(n)
    l2 = np.full(n_rows, np.nan)
    s = np.full(n_rows, np.nan)
    wcount = np.zeros(n_rows, np.int64)
    guard = np.zeros(len(chr_off) - 1, bool)
    for c in range(len(chr_off) - 1):
        idx = np.arange(chr_off[c], chr_off[c + 1])
        idx = idx[kept[idx]]
        m = idx.size
        if m == 0:
            continue
        lo, hi = _chrom_windows(idx, coord, max_dist)
        guard[c] = lo[-1] == 0
        Gk = G[idx]
        Q, A, N = _int_planes(Gk)
        # every term is an exact integer below 4 n^3 (< 2^63 for n <= 409,344): int64, converted exactly to longdouble
        nn = np.diag(N)
        S = np.where(Gk >= 0, Gk, 0).astype(np.int64).sum(1)
        d = nn * np.diag(Q) - S * S
        num = (nn[:, None] * nn[None, :]) * Q - (nn[:, None] * S[None, :]) * A - (nn[None, :] * S[:, None]) * A.T + \
              (S[:, None] * S[None, :]) * N
        num2 = np.square(num.astype(LD))
        nd = (nn * d).astype(LD)
        den = nd[:, None] * nd[None, :]
        r2 = num2 / den
        np.fill_diagonal(r2, LD(1))
        adj = r2 - (LD(1) - r2) / denom
        mag = r2 + (LD(1) - r2) / denom
        for k in range(m):
            w = slice(lo[k], hi[k] + 1)
            l2[idx[k]] = float(adj[k, w].sum())
            s[idx[k]] = float(mag[k, w].sum())
            wcount[idx[k]] = hi[k] - lo[k] + 1
    return {"l2": l2, "kept": kept, "maf": maf, "guard": guard, "s": s, "wcount": wcount}


def ldscore_ldsc64(G, chr_off, coord=None, max_dist=1.0, maf_min=0.0):
    """ldsc's float64 path: standardised mean-imputed genotypes, r = Y^T Y / n, l2_unbiased, window sums."""
    n_rows, n = G.shape
    kept, _ = snp_filter(G, maf_min)
    denom = n - 2 if n > 2 else n
    l2 = np.full(n_rows, np.nan)
    for c in range(len(chr_off) - 1):
        idx = np.arange(chr_off[c], chr_off[c + 1])
        idx = idx[kept[idx]]
        if idx.size == 0:
            continue
        lo, hi = _chrom_windows(idx, coord, max_dist)
        X = G[idx].astype(np.float64)
        miss = G[idx] < 0
        mu = np.array([X[k][~miss[k]].mean() for k in range(idx.size)])
        Y = np.where(miss, mu[:, None], X)
        Y = (Y - Y.mean(1, keepdims=True)) / Y.std(1, keepdims=True)
        r = Y @ Y.T / n
        sq = r * r
        adj = sq - (1 - sq) / denom
        for k in range(idx.size):
            l2[idx[k]] = adj[k, lo[k]:hi[k] + 1].sum()
    return l2


def format_ldscore(chrom, snp, bp, l2, kept, print_ids=None):
    """The text of <out>.l2.ldscore (before gzip): CHR SNP BP L2, tab-separated, kept SNPs in .bim order, L2 as %.3f."""
    lines = ["CHR\tSNP\tBP\tL2"]
    for c, v, b, x, k in zip(chrom, snp, bp, l2, kept):
        if k and (print_ids is None or v in print_ids):
            lines.append(f"{c}\t{v}\t{b}\t{x:.3f}")
    return "\n".join(lines) + "\n"


def format_counts(kept, maf):
    """(<out>.l2.M, <out>.l2.M_5_50): kept SNPs, and kept SNPs with MAF > 0.05."""
    kept = np.asarray(kept, bool)
    return f"{int(kept.sum())}\n", f"{int((kept & (np.asarray(maf) > 0.05)).sum())}\n"
