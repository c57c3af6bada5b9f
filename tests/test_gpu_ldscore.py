"""GPU: LD Scores (dbslmm_b200_ldscore, Engine.ldscore) against the extended-precision restatement of `ldsc.py --l2` in
tests/ldscore_ref.py.  For every kept SNP j the bar is

    |l_j - l*_j| <= 8 (|W(j)| + 4) u s_j,   u = 2^-53,   s_j = sum_{k in W(j)} r^2(j,k) + (1 - r^2(j,k)) / (n - 2),

the magnitudes of both parts of every term (r2adj of unlinked SNPs is a cancellation near zero).  The panels have LD (each
row copies most of its predecessor), so windows hold both strongly and weakly linked pairs."""

import numpy as np
import pytest

from dbslmm_b200 import _abi, synth

import ldscore_ref as R

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
WORST = {}


ld_panel = R.ld_panel


def check(engine, G, chr_off, coord=None, max_dist=1.0, maf_min=0.0, segment_rows=0, what=""):
    bed = synth.pack_bed(G)
    rows = np.arange(G.shape[0], dtype=np.int32)
    l2, kept, maf, guard = engine.ldscore(bed, G.shape[1], rows, chr_off, coord, max_dist=max_dist, maf_min=maf_min,
                                          segment_rows=segment_rows)
    e = R.ldscore_exact(G, chr_off, coord, max_dist, maf_min)
    assert np.array_equal(kept, e["kept"]), what
    assert np.array_equal(maf, e["maf"]), what
    assert np.array_equal(guard, e["guard"]), what
    assert np.all(np.isnan(l2[~kept])), what
    k = e["kept"]
    err = np.abs(l2[k] - e["l2"][k])
    bar = 8.0 * (e["wcount"][k] + 4) * U * e["s"][k]
    ratio = float((err / bar).max()) if k.any() else 0.0
    WORST[what] = ratio
    assert np.all(err <= bar), (what, ratio)
    return l2, e


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        w = max(WORST, key=WORST.get)
        print(f"\nldscore: largest |l - l*| / bar = {WORST[w]:.3g} ({w}) over {len(WORST)} cases")


@pytest.mark.parametrize("n", [2, 3, 127, 128, 129, 403, 2000])
@pytest.mark.parametrize("miss", [0.0, 0.02])
def test_n_ref_grid(engine, n, miss):
    rng = np.random.default_rng(n * 10 + int(miss * 100))
    G = ld_panel(rng, 429, n, miss)
    check(engine, G, [0, 129, 429], None, 128, segment_rows=256, what=f"n={n} miss={miss}")


WINDOWS = ["snps0", "snps1", "snps127", "snps128", "snps129", "whole", "kb_ties", "cm"]


def window_args(kind, m, rng):
    if kind.startswith("snps"):
        return None, float(kind[4:])
    if kind == "whole":
        return None, 1e9
    bp = 1000.0 * np.cumsum(rng.choice([0, 1, 2, 5], size=m))              # duplicate positions, steps of whole kb
    if kind == "kb_ties":
        return bp, 1000.0 * 10                                             # --ld-wind-kb 10: many pairs exactly 10 kb apart
    return bp * 1e-6, 0.01                                                 # cM = bp x 1e-6, --ld-wind-cm 0.01


@pytest.mark.parametrize("m", [1, 127, 128, 129, 300, 1000])
@pytest.mark.parametrize("kind", WINDOWS)
@pytest.mark.parametrize("miss", [0.0, 0.02])
def test_kept_counts_and_windows(engine, m, kind, miss):
    rng = np.random.default_rng(m * 31 + WINDOWS.index(kind) + int(miss * 100))
    G = ld_panel(rng, m + 3, 403, miss)
    coord, d = window_args(kind, m + 3, rng)
    # a short second chromosome of three SNPs after the one under test
    check(engine, G, [0, m, m + 3], coord, d, segment_rows=128 if m > 500 else 0, what=f"m={m} {kind} miss={miss}")


def test_dropped_rows(engine):
    rng = np.random.default_rng(5)
    n = 2000
    G = ld_panel(rng, 200, n, 0.02)
    G[10] = 1                                            # all heterozygous
    G[20] = 2                                            # monomorphic
    G[30] = -1                                           # all missing
    G[40] = 0
    G[40, :100] = 2                                      # f = 200 / 4000 = 0.05 exactly: MAF equals --maf 0.05
    G[50] = -1
    G[50, :3] = [0, 1, 2]                                # three calls, MAF 0.5: kept
    _, e = check(engine, G, [0, 200], None, 50, maf_min=0.05, what="dropped rows")
    assert not e["kept"][[10, 20, 30, 40]].any() and e["kept"][50]


def test_statistics_pass_only(engine):
    """l2_out NULL: kept, MAF and the guard of the statistics pass, the same as a full call's."""
    rng = np.random.default_rng(8)
    G = ld_panel(rng, 300, 403, 0.02)
    G[5] = 1
    rows = np.arange(300, dtype=np.int32)
    full = engine.ldscore(synth.pack_bed(G), 403, rows, [0, 100, 300], None, max_dist=150)
    l2, kept, maf, guard = engine.ldscore(synth.pack_bed(G), 403, rows, [0, 100, 300], None, max_dist=150, stats_only=True)
    assert l2 is None and np.array_equal(kept, full[1]) and np.array_equal(maf, full[2]) and np.array_equal(guard, full[3])
    assert guard.tolist() == [True, False] and not kept[5]


def test_int64_numerator_at_max_n_ref(engine):
    rng = np.random.default_rng(409344)
    n = 409344
    G = ld_panel(rng, 300, n, 0.02)
    check(engine, G, [0, 300], None, 129, what="n=409344 miss=0.02")


def bits(x):
    return np.ascontiguousarray(x).view(np.int64)


def test_deterministic(engine, tmp_path):
    rng = np.random.default_rng(77)
    n = 403
    G = np.concatenate([ld_panel(rng, 1000, n, 0.0), ld_panel(rng, 300, n, 0.02), ld_panel(rng, 129, n, 0.0)])
    off = [0, 1000, 1300, 1429]
    path = tmp_path / "panel.bed"
    with open(path, "wb") as f:
        f.write(bytes([0x6C, 0x1B, 0x01]) + synth.pack_bed(G).tobytes())
    bed = np.memmap(path, dtype=np.uint8, mode="r", offset=3)
    rows = np.arange(G.shape[0], dtype=np.int32)
    ref, _, _, _ = engine.ldscore(bed, n, rows, off, None, max_dist=200, segment_rows=128 * 64)       # one segment
    e = R.ldscore_exact(G, off, None, 200)
    assert np.all(np.abs(ref - e["l2"])[e["kept"]] <= 8.0 * (e["wcount"] + 4)[e["kept"]] * U * e["s"][e["kept"]])
    for seg in (128, 256, 1024, 0):
        l2, _, _, _ = engine.ldscore(bed, n, rows, off, None, max_dist=200, segment_rows=seg)
        assert np.array_equal(bits(l2), bits(ref)), seg
    again, _, _, _ = engine.ldscore(bed, n, rows, off, None, max_dist=200, segment_rows=128 * 64)
    assert np.array_equal(bits(again), bits(ref))
    for c in range(3):                                   # each chromosome alone
        sub = rows[off[c]:off[c + 1]]
        l2, _, _, _ = engine.ldscore(bed, n, sub, [0, sub.size], None, max_dist=200, segment_rows=256)
        assert np.array_equal(bits(l2), bits(ref[off[c]:off[c + 1]])), c


def test_errors(engine):
    rng = np.random.default_rng(3)
    G = ld_panel(rng, 10, 50, 0.0)
    bed = synth.pack_bed(G)
    rows = np.arange(10, dtype=np.int32)
    with pytest.raises(_abi.EngineError, match="409,344|409344"):
        big = np.zeros((2, (409345 + 3) // 4), np.uint8)
        engine.ldscore(big, 409345, [0, 1], [0, 2], None, max_dist=1)
    for off in ([0, 11], [1, 10], [0, 6, 4, 10]):
        with pytest.raises(_abi.EngineError, match="offsets"):
            engine.ldscore(bed, 50, rows, off, None, max_dist=1)
    coord = np.arange(10, dtype=np.float64)
    coord[4] = 2.5
    with pytest.raises(_abi.EngineError, match="not sorted"):
        engine.ldscore(bed, 50, rows, [0, 10], coord, max_dist=1)
    with pytest.raises(_abi.EngineError, match="out of range"):
        engine.ldscore(bed, 50, np.array([0, 10], np.int32), [0, 2], None, max_dist=1)
    with pytest.raises(_abi.EngineError, match="segment_rows"):
        engine.ldscore(bed, 50, rows, [0, 10], None, max_dist=1, segment_rows=100)
