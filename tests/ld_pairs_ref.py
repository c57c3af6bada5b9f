"""CPU restatement of dbslmm_b200_ld_pairs (`plink --r2 --ld-window N --ld-window-kb K --ld-window-r2 R`, with the code
base's r).  A pair (a, b), a < b positions in the row list, is written when both lie in one chromosome, both rows are
USABLE (a called genotype and nonzero variance), b - a <= max_snps - 1, coord[b] - coord[a] <= max_dist and r^2 >= r2_min.
Unusable rows count toward the max_snps distance.  r is formed from the exact integer numerator

    num_ab = n_a n_b Q_ab - n_a S_b A_ab - n_b S_a A_ba + S_a S_b N_ab,   r_ab = num_ab / sqrt(n_a n_b d_a d_b)

(Q = g.g, A_ab = g_a.M_b, N = M.M over the called genotypes; d = n sum g^2 - S^2) in x86 extended precision: the Pearson
r of the mean-imputed allele counts.  Genotypes are int8 [n_snp, n], -1 for a missing call."""
import numpy as np

from ldscore_ref import LD, _int_planes, ld_panel  # noqa: F401  (ld_panel: the tests' panels)


def usable_rows(G):
    called = G >= 0
    nn = called.sum(1).astype(np.int64)
    g = np.where(called, G, 0).astype(np.int64)
    S = g.sum(1)
    d = nn * (g * g).sum(1) - S * S
    return (nn > 0) & (d > 0)


def window_hi(coord, max_snps, max_dist):
    """Per row of one chromosome: the last position b >= a with b - a <= max_snps - 1 and coord[b] - coord[a] <= max_dist."""
    x = np.asarray(coord, np.float64)
    m = x.size
    hi = np.zeros(m, np.int64)
    j = 0
    for k in range(m):
        j = max(j, k)
        while j + 1 < m and j + 1 - k <= max_snps - 1 and x[j + 1] - x[k] <= max_dist:
            j += 1
        hi[k] = j
    return hi


def exact_r(G):
    """r of every pair of rows of G (longdouble [m, m]; NaN where a row is not usable)."""
    Q, A, N = _int_planes(G)
    called = G >= 0
    n = called.sum(1).astype(np.int64)
    g = np.where(called, G, 0).astype(np.int64)
    S = g.sum(1)
    d = n * (g * g).sum(1) - S * S
    num = (n[:, None] * n[None, :] * Q).astype(LD) - (n[:, None] * S[None, :] * A).astype(LD) \
        - (n[None, :] * S[:, None] * A.T).astype(LD) + (S[:, None] * S[None, :] * N).astype(LD)
    den = np.sqrt(n.astype(LD)[:, None] * n.astype(LD)[None, :] * d.astype(LD)[:, None] * d.astype(LD)[None, :])
    with np.errstate(divide="ignore", invalid="ignore"):
        r = num / den
    ok = (n > 0) & (d > 0)
    r[~ok, :] = np.nan
    r[:, ~ok] = np.nan
    return r


def ld_pairs_exact(G, chr_off, coord, max_snps, max_dist, r2_min=None):
    """Every pair inside the windows (r2_min None) or those with r^2 >= r2_min: dict of a, b (int64, ascending (a, b)),
    r and r2 (longdouble), miss (a SNP of the pair has a missing call) and usable (per row)."""
    use = usable_rows(G)
    nmiss = (G < 0).any(1)
    A_, B_, R_ = [], [], []
    for c in range(len(chr_off) - 1):
        i0, i1 = int(chr_off[c]), int(chr_off[c + 1])
        if i1 == i0:
            continue
        hi = window_hi(coord[i0:i1], max_snps, max_dist)
        r = exact_r(G[i0:i1])
        for k in range(i1 - i0):
            if not use[i0 + k]:
                continue
            bs = np.arange(k + 1, hi[k] + 1)
            bs = bs[use[i0 + bs]]
            A_.append(np.full(bs.size, i0 + k, np.int64))
            B_.append(i0 + bs)
            R_.append(r[k, bs])
    cat = lambda p, t: np.concatenate(p) if p else np.zeros(0, t)
    a, b, r = cat(A_, np.int64), cat(B_, np.int64), cat(R_, LD)
    r2 = r * r
    if r2_min is not None:
        k = r2 >= r2_min
        a, b, r, r2 = a[k], b[k], r[k], r2[k]
    return dict(a=a, b=b, r=r, r2=r2, miss=nmiss[a] | nmiss[b], usable=use)
