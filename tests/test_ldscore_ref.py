"""CPU: the two restatements of `ldsc.py --l2` in tests/ldscore_ref.py agree -- the extended-precision one built from the
exact integer numerators of the Gram planes (what the GPU results are checked against) and ldsc's own float64 recipe
(mean-impute, standardise, Y^T Y / n, unbiased r^2, window sums), which shares no formula with the kernels.  Grid: panel
widths from 2 to 2,000, no and 2 % missing calls, windows in SNPs (none, narrow, whole chromosome) and in coordinates with
duplicate positions and distances exactly equal to the window, and a one-SNP chromosome."""
import numpy as np
import pytest

import ldscore_ref as R


def windows_for(kind, m, rng):
    if kind == "snps0":
        return None, 0.0
    if kind == "snps5":
        return None, 5.0
    if kind == "whole":
        return None, 1e9
    bp = 1000.0 * np.cumsum(rng.choice([0, 1, 2, 5], size=m))              # duplicate positions, steps of whole kb
    return (bp, 10000.0) if kind == "kb_ties" else (bp * 1e-6, 0.01)


@pytest.mark.parametrize("n", [2, 3, 4, 127, 403, 2000])
@pytest.mark.parametrize("miss", [0.0, 0.02])
@pytest.mark.parametrize("kind", ["snps0", "snps5", "whole", "kb_ties", "cm"])
def test_exact_restatement_agrees_with_ldsc_float64(n, miss, kind):
    rng = np.random.default_rng(n * 7 + int(miss * 100) + len(kind))
    G = R.ld_panel(rng, 181, n, miss)
    off = [0, 150, 151, 181]                              # the middle chromosome holds one SNP
    coord, d = windows_for(kind, G.shape[0], rng)
    e = R.ldscore_exact(G, off, coord, d)
    f = R.ldscore_ldsc64(G, off, coord, d)
    k = e["kept"]
    assert np.array_equal(np.isnan(f), ~k)
    if n >= 4:
        assert k.sum() == G.shape[0]
    assert np.all(np.abs(e["l2"][k] - f[k]) <= 1e-12 * np.maximum(1.0, np.abs(e["l2"][k])))
