"""CPU: the two restatements of partitioned LD Scores in tests/ldscore_annot_ref.py agree -- the extended-precision one from
the exact integer numerators (what the GPU results are checked against) and ldsc's own float64 __corSumVarBlocks__ recipe
(chunks of standardised genotypes, np.dot(rfunc, annot)) -- and an all-ones column is the unannotated LD Score of
tests/ldscore_ref.py."""
import numpy as np
import pytest

import ldscore_annot_ref as A
import ldscore_ref as R

KINDS = ["bin", "cont", "zero", "one", "cont"]


def windows_for(kind, m, rng):
    if kind == "snps0":
        return None, 0.0
    if kind == "snps5":
        return None, 5.0
    if kind == "whole":
        return None, 1e9
    bp = 1000.0 * np.cumsum(rng.choice([0, 1, 2, 5], size=m))
    return (bp, 10000.0) if kind == "kb_ties" else (bp * 1e-6, 0.01)


@pytest.mark.parametrize("n", [2, 3, 4, 127, 403, 2000])
@pytest.mark.parametrize("miss", [0.0, 0.02])
@pytest.mark.parametrize("kind", ["snps0", "snps5", "whole", "kb_ties", "cm"])
def test_exact_restatement_agrees_with_ldsc_float64(n, miss, kind):
    rng = np.random.default_rng(n * 11 + int(miss * 100) + len(kind))
    G = R.ld_panel(rng, 181, n, miss)
    off = [0, 150, 151, 181]
    coord, d = windows_for(kind, G.shape[0], rng)
    a = A.annot_columns(rng, G.shape[0], KINDS)
    a[40:100, 0] = 0.0                                    # a stretch where ldsc skips chunks with all-zero annotations
    e = A.ldscore_annot_exact(G, off, a, coord, d)
    f = A.ldscore_annot_ldsc64(G, off, a, coord, d, chunk=7)
    k = e["kept"]
    assert np.array_equal(np.isnan(f).all(1), ~k)
    err = np.abs(e["l2"][k] - f[k])
    assert np.all(err <= 1e-12 * np.maximum(1.0, e["s"][k])), float((err / np.maximum(1.0, e["s"][k])).max())


@pytest.mark.parametrize("chunk", [1, 7, 50])
def test_ldsc_recipe_does_not_depend_on_its_chunk_size(chunk):
    rng = np.random.default_rng(chunk)
    G = R.ld_panel(rng, 120, 403, 0.02)
    a = A.annot_columns(rng, 120, KINDS)
    e = A.ldscore_annot_exact(G, [0, 120], a, None, 17)
    f = A.ldscore_annot_ldsc64(G, [0, 120], a, None, 17, chunk=chunk)
    assert np.all(np.abs(e["l2"] - f) <= 1e-12 * np.maximum(1.0, e["s"]))


@pytest.mark.parametrize("n", [3, 403])
def test_all_ones_column_is_the_unannotated_ld_score(n):
    rng = np.random.default_rng(n)
    G = R.ld_panel(rng, 200, n, 0.02)
    G[9] = 1                                              # dropped
    off = [0, 130, 200]
    a = A.annot_columns(rng, 200, ["one", "bin"])
    e = A.ldscore_annot_exact(G, off, a, None, 40)
    u = R.ldscore_exact(G, off, None, 40)
    k = u["kept"]
    assert np.array_equal(e["kept"], k) and np.array_equal(e["guard"], u["guard"]) and np.array_equal(e["wcount"], u["wcount"])
    assert np.all(np.isnan(e["l2"][~k]))
    assert np.all(np.abs(e["l2"][k, 0] - u["l2"][k]) <= 1e-15 * u["s"][k])
    assert np.allclose(e["s"][k, 0], u["s"][k], rtol=1e-15, atol=0)


def test_annotated_formatting():
    chrom, snp, bp = ["1", "1", "2"], ["a", "b", "c"], ["10", "20", "5"]
    l2 = np.array([[1.0, -0.0004], [np.nan, np.nan], [12.3456, 2.0]])
    kept = np.array([True, False, True])
    assert A.format_annot_ldscore(chrom, snp, bp, l2, kept, ["x", "y"]) == \
        "CHR\tSNP\tBP\txL2\tyL2\n1\ta\t10\t1.000\t-0.000\n2\tc\t5\t12.346\t2.000\n"
    assert A.format_annot_ldscore(chrom, snp, bp, l2[:, :1], kept, ["x"]) == "CHR\tSNP\tBP\tL2\n1\ta\t10\t1.000\n2\tc\t5\t12.346\n"
    a = np.array([[1.0, 0.5], [1.0, 0.25], [0.0, 0.1]])
    assert A.format_annot_counts(kept, np.array([0.3, 0.3, 0.01]), a) == ("1\t0.59999999999999998\n", "1\t0.5\n")
