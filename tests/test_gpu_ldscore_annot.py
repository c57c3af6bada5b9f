"""GPU: partitioned LD Scores (dbslmm_b200_ldscore_annot, Engine.ldscore(annot=...)) against the extended-precision
restatement of tests/ldscore_annot_ref.py.  For every kept SNP j and annotation column c the bar is

    |L - L*| <= 8 (|W(j)| + 4) u sum_{k in W(j)} (r^2 + (1 - r^2) / (n - 2)) |a_kc|,   u = 2^-53,

the magnitudes of both parts of every term.  The columns mix binary, signed continuous, all-zero and all-ones
annotations; the numbers of columns straddle the kernel's register group of 16 annotations."""

import numpy as np
import pytest

from dbslmm_b200 import _abi, synth

import ldscore_annot_ref as A
import ldscore_ref as R

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
GROUP = 16                                             # ldscore.cu kLdGroup
WIDTHS = [1, 2, GROUP - 1, GROUP, GROUP + 1, 97]
WORST = {}


def columns(rng, n_rows, C):
    kinds = (["one", "cont", "bin", "zero"] * C)[:C]
    return A.annot_columns(rng, n_rows, kinds)


def check(engine, G, chr_off, annot, coord=None, max_dist=1.0, maf_min=0.0, segment_rows=0, what=""):
    bed = synth.pack_bed(G)
    rows = np.arange(G.shape[0], dtype=np.int32)
    l2, kept, maf, guard = engine.ldscore(bed, G.shape[1], rows, chr_off, coord, max_dist=max_dist, maf_min=maf_min,
                                          segment_rows=segment_rows, annot=annot)
    e = A.ldscore_annot_exact(G, chr_off, annot, coord, max_dist, maf_min)
    assert l2.shape == annot.shape, what
    assert np.array_equal(kept, e["kept"]) and np.array_equal(maf, e["maf"]) and np.array_equal(guard, e["guard"]), what
    assert np.all(np.isnan(l2[~kept])), what
    k = e["kept"]
    err = np.abs(l2[k] - e["l2"][k])
    bar = 8.0 * (e["wcount"][k] + 4)[:, None] * U * e["s"][k]
    ratio = float(np.max(np.where(bar > 0, err / np.where(bar > 0, bar, 1.0), np.where(err > 0, np.inf, 0.0)))) if k.any() else 0.0
    WORST[what] = ratio
    assert np.all(err <= bar), (what, ratio)
    return l2, e


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        w = max(WORST, key=WORST.get)
        print(f"\nldscore_annot: largest |L - L*| / bar = {WORST[w]:.3g} ({w}) over {len(WORST)} cases")


@pytest.mark.parametrize("n", [2, 3, 127, 128, 129, 403, 2000])
@pytest.mark.parametrize("miss", [0.0, 0.02])
def test_n_ref_grid(engine, n, miss):
    rng = np.random.default_rng(n * 10 + int(miss * 100) + 1)
    G = R.ld_panel(rng, 429, n, miss)
    check(engine, G, [0, 129, 429], columns(rng, 429, GROUP + 1), None, 128, segment_rows=256, what=f"n={n} miss={miss}")


WINDOWS = ["snps0", "snps1", "snps127", "snps128", "snps129", "whole", "kb_ties", "cm"]


def window_args(kind, m, rng):
    if kind.startswith("snps"):
        return None, float(kind[4:])
    if kind == "whole":
        return None, 1e9
    bp = 1000.0 * np.cumsum(rng.choice([0, 1, 2, 5], size=m))
    if kind == "kb_ties":
        return bp, 1000.0 * 10
    return bp * 1e-6, 0.01


@pytest.mark.parametrize("m", [1, 127, 128, 129, 300, 1000])
@pytest.mark.parametrize("kind", WINDOWS)
@pytest.mark.parametrize("miss", [0.0, 0.02])
def test_kept_counts_and_windows(engine, m, kind, miss):
    rng = np.random.default_rng(m * 31 + WINDOWS.index(kind) + int(miss * 100) + 1)
    G = R.ld_panel(rng, m + 3, 403, miss)
    coord, d = window_args(kind, m + 3, rng)
    C = WIDTHS[(m + WINDOWS.index(kind)) % len(WIDTHS)]
    check(engine, G, [0, m, m + 3], columns(rng, m + 3, C), coord, d, segment_rows=128 if m > 500 else 0,
          what=f"m={m} {kind} miss={miss} C={C}")


@pytest.mark.parametrize("C", WIDTHS)
@pytest.mark.parametrize("miss", [0.0, 0.02])
def test_annotation_counts(engine, C, miss):
    rng = np.random.default_rng(C * 3 + int(miss * 100))
    G = R.ld_panel(rng, 700, 403, miss)
    check(engine, G, [0, 500, 700], columns(rng, 700, C), None, 150, segment_rows=256, what=f"C={C} miss={miss}")


def test_max_n_ref(engine):
    rng = np.random.default_rng(409344)
    G = R.ld_panel(rng, 300, 409344, 0.02)
    check(engine, G, [0, 300], columns(rng, 300, 5), None, 129, what="n=409344 miss=0.02")


def test_dropped_rows(engine):
    rng = np.random.default_rng(5)
    G = R.ld_panel(rng, 200, 2000, 0.02)
    G[10] = 1
    G[20] = 2
    G[30] = -1
    G[40] = 0
    G[40, :100] = 2
    G[50] = -1
    G[50, :3] = [0, 1, 2]
    _, e = check(engine, G, [0, 200], columns(rng, 200, 3), None, 50, maf_min=0.05, what="dropped rows")
    assert not e["kept"][[10, 20, 30, 40]].any() and e["kept"][50]


def bits(x):
    return np.ascontiguousarray(x).view(np.int64)


def test_deterministic_and_columns_independent(engine, tmp_path):
    rng = np.random.default_rng(77)
    n = 403
    G = np.concatenate([R.ld_panel(rng, 1000, n, 0.0), R.ld_panel(rng, 300, n, 0.02), R.ld_panel(rng, 129, n, 0.0)])
    off = [0, 1000, 1300, 1429]
    path = tmp_path / "panel.bed"
    with open(path, "wb") as f:
        f.write(bytes([0x6C, 0x1B, 0x01]) + synth.pack_bed(G).tobytes())
    bed = np.memmap(path, dtype=np.uint8, mode="r", offset=3)
    rows = np.arange(G.shape[0], dtype=np.int32)
    a = columns(rng, G.shape[0], GROUP + 3)
    ref, _, _, _ = engine.ldscore(bed, n, rows, off, None, max_dist=200, segment_rows=128 * 64, annot=a)
    for seg in (128, 256, 1024, 0):
        l2, _, _, _ = engine.ldscore(bed, n, rows, off, None, max_dist=200, segment_rows=seg, annot=a)
        assert np.array_equal(bits(l2), bits(ref)), seg
    again, _, _, _ = engine.ldscore(bed, n, rows, off, None, max_dist=200, segment_rows=128 * 64, annot=a)
    assert np.array_equal(bits(again), bits(ref))
    for c in range(3):                                   # each chromosome alone
        sub = rows[off[c]:off[c + 1]]
        l2, _, _, _ = engine.ldscore(bed, n, sub, [0, sub.size], None, max_dist=200, segment_rows=256, annot=a[off[c]:off[c + 1]])
        assert np.array_equal(bits(l2), bits(ref[off[c]:off[c + 1]])), c
    for cols in ([0], [1], [GROUP], [GROUP + 2], [3, 1], list(range(GROUP + 3))[::-1]):   # alone or among others
        l2, _, _, _ = engine.ldscore(bed, n, rows, off, None, max_dist=200, segment_rows=256, annot=a[:, cols])
        assert np.array_equal(bits(l2), bits(ref[:, cols])), cols


def test_all_ones_column_matches_the_unannotated_call(engine):
    rng = np.random.default_rng(12)
    n = 403
    G = R.ld_panel(rng, 600, n, 0.02)
    off = [0, 400, 600]
    rows = np.arange(600, dtype=np.int32)
    bed = synth.pack_bed(G)
    a = columns(rng, 600, 4)                             # column 0 is all ones
    la, kept, _, _ = engine.ldscore(bed, n, rows, off, None, max_dist=90, annot=a)
    lu, _, _, _ = engine.ldscore(bed, n, rows, off, None, max_dist=90)
    u = R.ldscore_exact(G, off, None, 90)
    k = kept
    bar_u = 8.0 * (u["wcount"][k] + 4) * U * u["s"][k]
    assert np.all(np.abs(la[k, 0] - u["l2"][k]) <= bar_u)
    assert np.all(np.abs(lu[k] - u["l2"][k]) <= bar_u)
    assert np.all(np.abs(la[k, 0] - lu[k]) <= 2 * bar_u)
    assert np.all(np.isnan(la[~k])) and np.all(np.isnan(lu[~k]))


def test_statistics_pass_only(engine):
    rng = np.random.default_rng(8)
    G = R.ld_panel(rng, 300, 403, 0.02)
    G[5] = 1
    rows = np.arange(300, dtype=np.int32)
    a = columns(rng, 300, 3)
    full = engine.ldscore(synth.pack_bed(G), 403, rows, [0, 100, 300], None, max_dist=150, annot=a)
    l2, kept, maf, guard = engine.ldscore(synth.pack_bed(G), 403, rows, [0, 100, 300], None, max_dist=150, stats_only=True, annot=a)
    assert l2 is None and np.array_equal(kept, full[1]) and np.array_equal(maf, full[2]) and np.array_equal(guard, full[3])


def test_errors(engine):
    rng = np.random.default_rng(3)
    G = R.ld_panel(rng, 10, 50, 0.0)
    bed = synth.pack_bed(G)
    rows = np.arange(10, dtype=np.int32)
    a = np.ones((10, 2))
    lib, h = engine.lib, engine.h
    chr_off = np.array([0, 10], np.int32)
    out = np.zeros((10, _abi.LD_MAX_ANNOT + 1))

    def call(annot_ptr, n_annot):
        return lib.dbslmm_b200_ldscore_annot(h, bed.ctypes.data, 10, 50, rows.ctypes.data, 10, chr_off.ctypes.data, 1,
                                             _abi.LD_WIND_SNPS, None, 1.0, 0.0, 0, annot_ptr, n_annot, None, None,
                                             out.ctypes.data, None, None)

    big = np.ones((10, _abi.LD_MAX_ANNOT + 1))
    for ptr, na, msg in ((a.ctypes.data, 0, "n_annot"), (big.ctypes.data, _abi.LD_MAX_ANNOT + 1, "n_annot"), (None, 2, "NULL")):
        assert call(ptr, na) != 0
        assert msg in lib.dbslmm_b200_last_error(h).decode()
    assert call(big.ctypes.data, _abi.LD_MAX_ANNOT) == 0            # the documented limit itself is accepted
    for bad in (np.nan, np.inf, -np.inf):
        b = a.copy()
        b[7, 1] = bad
        with pytest.raises(_abi.EngineError, match=r"annot\[7\]\[1\] is not finite"):
            engine.ldscore(bed, 50, rows, [0, 10], None, max_dist=1, annot=b)
    with pytest.raises(ValueError, match="annot"):
        engine.ldscore(bed, 50, rows, [0, 10], None, max_dist=1, annot=np.ones((9, 2)))
    for off in ([0, 11], [1, 10]):                       # the unannotated entry's checks still apply
        with pytest.raises(_abi.EngineError, match="offsets"):
            engine.ldscore(bed, 50, rows, off, None, max_dist=1, annot=a)
    with pytest.raises(_abi.EngineError, match="segment_rows"):
        engine.ldscore(bed, 50, rows, [0, 10], None, max_dist=1, segment_rows=100, annot=a)
