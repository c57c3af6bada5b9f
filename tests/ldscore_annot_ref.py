"""CPU restatement of partitioned LD Scores (`ldsc.py --l2 --annot`, ldsc 1.0.1), two ways:

  * ldscore_annot_exact: L_c(j) = sum_{k in W(j)} r2adj(j, k) a_kc from the exact integer numerators of
    tests/ldscore_ref.py, in x86 extended precision (np.longdouble), r_jj = 1;
  * ldscore_annot_ldsc64: ldsc's own float64 recipe, ldscore.py's __corSumVarBlocks__ -- standardised genotypes taken c
    SNPs at a time, rfunc = l2_unbiased(A^T B / n) per chunk, cor_sum += np.dot(rfunc, annot) -- over the block lefts of
    the window rule.  ldsc rounds each block up to a multiple of c, so its chunks also pair SNPs up to c - 1 places
    beyond the window; like tests/ldscore_ref.py (and the library) this restatement keeps the exact window, by zeroing
    those pairs of rfunc.

Annotation rows are aligned with the rows of G (one per .bim line); both keep ldsc's SNPs, as ldscore_ref does."""
import numpy as np

import ldscore_ref as R

LD = np.longdouble


def ldscore_annot_exact(G, chr_off, annot, coord=None, max_dist=1.0, maf_min=0.0):
    """Returns dict(l2, kept, maf, guard, s, wcount): l2 / s float64[n_rows, C] (NaN rows where not kept;
    s_jc = sum_{k in W(j)} (r^2 + (1 - r^2) / denom) |a_kc|), wcount = |W(j)|."""
    annot = np.asarray(annot, np.float64)
    n_rows, n = G.shape
    C = annot.shape[1]
    kept, maf = R.snp_filter(G, maf_min)
    denom = LD(n - 2) if n > 2 else LD(n)
    l2 = np.full((n_rows, C), np.nan)
    s = np.full((n_rows, C), np.nan)
    wcount = np.zeros(n_rows, np.int64)
    guard = np.zeros(len(chr_off) - 1, bool)
    for c in range(len(chr_off) - 1):
        idx = np.arange(chr_off[c], chr_off[c + 1])
        idx = idx[kept[idx]]
        m = idx.size
        if m == 0:
            continue
        lo, hi = R._chrom_windows(idx, coord, max_dist)
        guard[c] = lo[-1] == 0
        Gk = G[idx]
        Q, A, N = R._int_planes(Gk)
        nn = np.diag(N)
        S = np.where(Gk >= 0, Gk, 0).astype(np.int64).sum(1)
        d = nn * np.diag(Q) - S * S
        num = (nn[:, None] * nn[None, :]) * Q - (nn[:, None] * S[None, :]) * A - (nn[None, :] * S[:, None]) * A.T + \
              (S[:, None] * S[None, :]) * N
        nd = (nn * d).astype(LD)
        r2 = np.square(num.astype(LD)) / (nd[:, None] * nd[None, :])
        np.fill_diagonal(r2, LD(1))
        k = np.arange(m)
        inw = (k[None, :] >= lo[:, None]) & (k[None, :] <= hi[:, None])
        adj = np.where(inw, r2 - (LD(1) - r2) / denom, LD(0))
        mag = np.where(inw, r2 + (LD(1) - r2) / denom, LD(0))
        a = annot[idx].astype(LD)
        l2[idx] = (adj @ a).astype(np.float64)
        s[idx] = (mag @ np.abs(a)).astype(np.float64)
        wcount[idx] = hi - lo + 1
    return {"l2": l2, "kept": kept, "maf": maf, "guard": guard, "s": s, "wcount": wcount}


def _cor_sum_var_blocks(Y, block_left, c, annot):
    """ldsc 1.0.1 ldscore.py __corSumVarBlocks__ with func = l2_unbiased; Y [n, m] standardised genotypes.  rfunc(I, J)
    of columns I (first index i0) and J (j0) is zeroed outside the exact window (pair i < j inside iff block_left[j] <= i)."""
    n, m = Y.shape

    def func(x, i0, j0):
        i = np.arange(i0, i0 + x.shape[0])[:, None]
        j = np.arange(j0, j0 + x.shape[1])[None, :]
        inw = np.where(i <= j, block_left[j] <= i, block_left[i] <= j)
        return np.where(inw, x * x - (1 - x * x) / (n - 2 if n > 2 else n), 0.0)          # ldsc's l2_unbiased
    pos = [0]

    def snp_getter(k):
        X = Y[:, pos[0]:pos[0] + k]
        pos[0] += k
        return X

    block_sizes = np.ceil((np.arange(m) - block_left) / c) * c
    cor_sum = np.zeros((m, annot.shape[1]))
    b = np.nonzero(block_left > 0)
    b = b[0][0] if np.any(b) else m
    b = int(np.ceil(b / c) * c)
    if b > m:
        c = 1
        b = m
    l_A = 0
    A = snp_getter(b)
    for l_B in range(0, b, c):
        B = A[:, l_B:l_B + c]
        rfuncAB = func(np.dot(A.T, B / n), l_A, l_B)
        cor_sum[l_A:l_A + b, :] += np.dot(rfuncAB, annot[l_B:l_B + c, :])
    b0 = b
    md = int(c * np.floor(m / c))
    end = md + 1 if md != m else md
    for l_B in range(b0, end, c):
        old_b = b
        b = int(block_sizes[l_B])
        if l_B > b0 and b > 0:
            A = np.hstack((A[:, old_b - b + c:old_b], B))
            l_A += old_b - b + c
        elif l_B == b0 and b > 0:
            A = A[:, b0 - b:b0]
            l_A = b0 - b
        elif b == 0:
            A = np.array(()).reshape((n, 0))
            l_A = l_B
        if l_B == md:
            c = m - md
        B = snp_getter(c)
        if np.all(annot[l_A:l_A + b, :] == 0) and np.all(annot[l_B:l_B + c, :] == 0):
            continue
        rfuncAB = func(np.dot(A.T, B / n), l_A, l_B)
        cor_sum[l_A:l_A + b, :] += np.dot(rfuncAB, annot[l_B:l_B + c, :])
        cor_sum[l_B:l_B + c, :] += np.dot(annot[l_A:l_A + b, :].T, rfuncAB).T
        rfuncBB = func(np.dot(B.T, B / n), l_B, l_B)
        cor_sum[l_B:l_B + c, :] += np.dot(rfuncBB, annot[l_B:l_B + c, :])
    return cor_sum


def ldscore_annot_ldsc64(G, chr_off, annot, coord=None, max_dist=1.0, maf_min=0.0, chunk=50):
    """ldsc's float64 path, one chromosome at a time (ldsc's --chunk-size default is 50)."""
    annot = np.asarray(annot, np.float64)
    n_rows, n = G.shape
    kept, _ = R.snp_filter(G, maf_min)
    l2 = np.full((n_rows, annot.shape[1]), np.nan)
    for c in range(len(chr_off) - 1):
        idx = np.arange(chr_off[c], chr_off[c + 1])
        idx = idx[kept[idx]]
        if idx.size == 0:
            continue
        lo, _ = R._chrom_windows(idx, coord, max_dist)
        X = G[idx].astype(np.float64)
        miss = G[idx] < 0
        mu = np.array([X[k][~miss[k]].mean() for k in range(idx.size)])
        Y = np.where(miss, mu[:, None], X)
        Y = (Y - Y.mean(1, keepdims=True)) / Y.std(1, keepdims=True)
        l2[idx] = _cor_sum_var_blocks(np.ascontiguousarray(Y.T), lo, chunk, annot[idx])
    return l2


def annot_columns(rng, n_rows, kinds):
    """Annotation columns by kind: 'bin' (0/1), 'cont' (signed continuous), 'zero', 'one'."""
    cols = []
    for k in kinds:
        if k == "bin":
            cols.append((rng.random(n_rows) < 0.3).astype(np.float64))
        elif k == "cont":
            cols.append(rng.standard_normal(n_rows) * rng.uniform(0.1, 10.0))
        elif k == "zero":
            cols.append(np.zeros(n_rows))
        else:
            cols.append(np.ones(n_rows))
    return np.stack(cols, 1)


def format_annot_ldscore(chrom, snp, bp, l2, kept, names, print_ids=None):
    """The text of <out>.l2.ldscore with annotations: CHR SNP BP <name>L2 ... (plain L2 for one column), %.3f."""
    head = ["L2"] if len(names) == 1 else [f"{v}L2" for v in names]
    lines = ["\t".join(["CHR", "SNP", "BP"] + head)]
    for i, (c, v, b, k) in enumerate(zip(chrom, snp, bp, kept)):
        if k and (print_ids is None or v in print_ids):
            lines.append("\t".join([c, v, b] + [f"{x:.3f}" for x in l2[i]]))
    return "\n".join(lines) + "\n"


def format_m(x):
    """A value of <out>.l2.M: whole numbers as integers, others as %.17g."""
    return str(int(x)) if float(x).is_integer() else f"{x:.17g}"


def format_annot_counts(kept, maf, annot):
    """(<out>.l2.M, <out>.l2.M_5_50): per column, the sum of a_kc over kept SNPs, and over kept SNPs with MAF > 0.05,
    added in .bim order."""
    kept = np.asarray(kept, bool)
    common = kept & (np.asarray(maf) > 0.05)
    out = []
    for sel in (kept, common):
        sums = np.zeros(annot.shape[1])
        for i in np.nonzero(sel)[0]:
            sums = sums + annot[i]
        out.append("\t".join(format_m(v) for v in sums) + "\n")
    return tuple(out)
