"""The CPU restatement of `ld --r2` (tests/ld_pairs_ref.py): r against numpy.corrcoef of the mean-imputed genotypes, and
the window rule on hand-built cases."""
import numpy as np

import ld_pairs_ref as P


def mean_imputed(G):
    X = G.astype(np.float64)
    for k in range(X.shape[0]):
        c = G[k] >= 0
        X[k, ~c] = X[k, c].mean()
    return X


def test_r_against_corrcoef():
    rng = np.random.default_rng(5)
    for miss in (0.0, 0.02, 0.2):
        G = P.ld_panel(rng, 60, 301, miss)
        G[7] = G[3]                                              # r = 1
        G[9] = np.where(G[4] >= 0, 2 - G[4], -1)                  # r = -1
        r = P.exact_r(G).astype(np.float64)
        ref = np.corrcoef(mean_imputed(G))
        assert np.abs(r - ref).max() < 1e-12, miss


def test_unusable_rows():
    G = np.array([[0, 1, 2, 1], [1, 1, 1, 1], [-1, -1, -1, -1], [2, 2, -1, 2], [0, 2, 1, -1]], np.int8)
    assert P.usable_rows(G).tolist() == [True, False, False, False, True]
    e = P.ld_pairs_exact(G, [0, 5], np.arange(5.0), 10, 1e9)
    assert e["a"].tolist() == [0] and e["b"].tolist() == [4]      # the unusable rows form no pair
    e = P.ld_pairs_exact(G, [0, 5], np.arange(5.0), 4, 1e9)
    assert e["a"].size == 0                                       # ... but count toward the distance: 4 - 0 > 4 - 1


def test_window_rule():
    # ties in bp: a window of K bp includes every SNP at the edge and every SNP at the same position
    assert P.window_hi([100, 100, 100, 200, 300], 99999, 100).tolist() == [3, 3, 3, 4, 4]
    # both windows binding: the SNP window stops row 0, the kb window row 3
    assert P.window_hi([0, 1, 2, 3, 500, 501], 3, 100).tolist() == [2, 3, 3, 3, 5, 5]
    # N = 2: adjacent rows only
    assert P.window_hi([0, 10, 20], 2, 1e9).tolist() == [1, 2, 2]
    # K = 0: only SNPs at the same position
    assert P.window_hi([5, 5, 6, 7, 7, 7], 99999, 0).tolist() == [1, 1, 2, 5, 5, 5]
    # N = 1: no pair
    assert P.window_hi([0, 1], 1, 1e9).tolist() == [0, 1]


def test_pairs_are_ordered_and_windowed():
    rng = np.random.default_rng(2)
    G = P.ld_panel(rng, 50, 101, 0.0)
    coord = np.cumsum(rng.choice([0, 1000, 2000], 50)).astype(np.float64)
    e = P.ld_pairs_exact(G, [0, 20, 50], coord, 7, 5000, 0.0)
    key = e["a"] * 100 + e["b"]
    assert np.all(np.diff(key) > 0)
    assert np.all(e["b"] - e["a"] <= 6) and np.all(coord[e["b"]] - coord[e["a"]] <= 5000)
    assert not np.any((e["a"] < 20) & (e["b"] >= 20))                   # never across a chromosome
    n_all = sum(min(a + 6, 19 if a < 20 else 49) - a for a in range(50))
    assert e["a"].size <= n_all
