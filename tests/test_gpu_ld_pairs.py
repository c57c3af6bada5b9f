"""GPU: SNP pairs (dbslmm_b200_ld_pairs, Engine.ld_pairs) against the extended-precision restatement in tests/ld_pairs_ref.py.
Every written r must lie within 8 u of the reference (u = 2^-53, |r| <= 1), and the written set must equal the reference
set except for pairs whose reference r^2 lies within 24 u of r2_min (r^2 of an r within 8 u moves by up to 2 x 8 u, plus
its own rounding)."""
import ctypes as C

import numpy as np
import pytest

from dbslmm_b200 import _abi, synth

import ld_pairs_ref as P
import ldscore_ref as R

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
WORST = {}


def run(engine, G, chr_off, coord, max_snps, max_dist, r2_min, segment_rows=0):
    bed = synth.pack_bed(G)
    rows = np.arange(G.shape[0], dtype=np.int32)
    return engine.ld_pairs(bed, G.shape[1], rows, chr_off, coord, max_snps=max_snps, max_dist=max_dist, r2_min=r2_min,
                           segment_rows=segment_rows)


def check(engine, G, chr_off, coord, max_snps, max_dist, r2_min, segment_rows=0, what=""):
    a, b, r = run(engine, G, chr_off, coord, max_snps, max_dist, r2_min, segment_rows)
    e = P.ld_pairs_exact(G, chr_off, coord, max_snps, max_dist, None)
    assert np.array_equal(engine.last_usable, e["usable"]), what
    key = a * G.shape[0] + b
    assert np.all(np.diff(key) > 0), what                                  # ascending (a, b), no duplicate
    ekey = e["a"] * G.shape[0] + e["b"]
    near = np.abs(e["r2"] - r2_min) <= 24 * U
    want = ekey[(e["r2"] >= r2_min) & ~near]
    assert np.isin(want, key).all(), (what, "missing pairs")
    allowed = ekey[(e["r2"] >= r2_min) | near]
    assert np.isin(key, allowed).all(), (what, "extra pairs")
    idx = np.searchsorted(ekey, key)
    err = np.abs(r.astype(P.LD) - e["r"][idx]).astype(np.float64)
    ratio = float(err.max() / (8 * U)) if err.size else 0.0
    WORST[what] = ratio
    assert ratio <= 1.0, (what, ratio)
    assert engine.last_n_miss_pairs == int(e["miss"][idx].sum()), what
    return a, b, r


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        w = max(WORST, key=WORST.get)
        print(f"\nld_pairs: largest |r - r*| / 8u = {WORST[w]:.3g} ({w}) over {len(WORST)} cases")


@pytest.mark.parametrize("n", [2, 3, 127, 128, 129, 2000, 409344])
@pytest.mark.parametrize("miss", [0.0, 0.02])
def test_n_ref_grid(engine, n, miss):
    rng = np.random.default_rng(n * 10 + int(miss * 100))
    m = 40 if n > 10000 else 300
    G = R.ld_panel(rng, m, n, miss)
    coord = 1000.0 * np.cumsum(rng.choice([0, 1, 2, 5], size=m)).astype(np.float64)
    off = [0, 29, m] if m == 40 else [0, 129, m]
    check(engine, G, off, coord, 99999, 60000.0, 0.0, what=f"n={n} miss={miss}")


@pytest.mark.parametrize("m", [1, 2, 127, 128, 129, 1000])
@pytest.mark.parametrize("max_snps", [2, 10, 99999])
@pytest.mark.parametrize("miss", [0.0, 0.02])
def test_chromosomes_and_windows(engine, m, max_snps, miss):
    rng = np.random.default_rng(m * 7 + max_snps + int(miss * 100))
    G = R.ld_panel(rng, m + 5, 403, miss)
    coord = np.concatenate([1000.0 * np.cumsum(rng.choice([0, 1, 2, 5], size=m)), [100.0, 100.0, 200.0, 200.0, 5000.0]])
    # kb window with ties: many pairs exactly 10 kb apart, several SNPs at one position
    check(engine, G, [0, m, m + 5], coord, max_snps, 10000.0, 0.2, what=f"m={m} N={max_snps} miss={miss}")


@pytest.mark.parametrize("r2_min", [0.0, 0.2, 1.0, 1.5])
def test_thresholds_duplicates_and_unusable_rows(engine, r2_min):
    rng = np.random.default_rng(11)
    G = R.ld_panel(rng, 260, 517, 0.02)
    G[5] = G[4]                                                      # r = 1
    G[9] = np.where(G[8] >= 0, 2 - G[8], -1)                         # r = -1
    G[140] = G[139]
    G[20] = 1                                                        # monomorphic
    G[21] = -1                                                       # no called genotype
    G[150, :] = 0
    G[150, 3] = -1                                                   # monomorphic with a missing call
    coord = 1000.0 * np.arange(260, dtype=np.float64)
    a, b, r = check(engine, G, [0, 130, 260], coord, 99999, 1e9, r2_min, what=f"r2_min={r2_min}")
    assert not np.isin([20, 21, 150], a).any() and not np.isin([20, 21, 150], b).any()
    if r2_min < 1.0:
        k = (a == 4) & (b == 5)
        assert k.sum() == 1 and abs(r[k][0] - 1.0) <= 8 * U
        k = (a == 8) & (b == 9)
        assert k.sum() == 1 and abs(r[k][0] + 1.0) <= 8 * U
    if r2_min > 1.0:
        assert a.size <= 3                                           # only r^2 that rounds above 1 can pass


def test_unusable_rows_count_toward_the_window(engine):
    rng = np.random.default_rng(3)
    G = R.ld_panel(rng, 12, 200, 0.0)
    G[1] = 1
    a, b, r = run(engine, G, [0, 12], np.arange(12.0), 3, 1e9, 0.0)
    assert not ((a == 0) & (b == 3)).any() and ((a == 0) & (b == 2)).any()


def test_consistency_with_ldscore(engine):
    """r2_min = 0, an unbounded SNP window and a kb window: sum over each SNP's pairs of r2adj, plus 1, is its LD Score."""
    rng = np.random.default_rng(8)
    G = R.ld_panel(rng, 700, 611, 0.02)
    coord = 1000.0 * np.cumsum(rng.choice([0, 1, 2, 5], size=700)).astype(np.float64)
    off = [0, 300, 700]
    a, b, r = run(engine, G, off, coord, 2 ** 31 - 1, 20000.0, 0.0)
    rows = np.arange(700, dtype=np.int32)
    l2, kept, _, _ = engine.ldscore(synth.pack_bed(G), G.shape[1], rows, off, coord, max_dist=20000.0)
    assert kept.all()
    n = G.shape[1]
    adj = r * r - (1 - r * r) / (n - 2)
    s = np.ones(700) + np.bincount(a, adj, 700) + np.bincount(b, adj, 700)
    e = R.ldscore_exact(G, off, coord, 20000.0, 0.0)
    bar = 8.0 * (e["wcount"] + 4) * U * e["s"]
    assert np.all(np.abs(s - l2) <= 2 * bar)


def test_bit_identity(engine):
    rng = np.random.default_rng(21)
    G = R.ld_panel(rng, 900, 300, 0.02)
    coord = 1000.0 * np.cumsum(rng.choice([0, 1, 2, 5], size=900)).astype(np.float64)
    off = [0, 200, 333, 900]
    base = run(engine, G, off, coord, 300, 150000.0, 0.1)
    for seg in (128, 256, 1024):
        x = run(engine, G, off, coord, 300, 150000.0, 0.1, segment_rows=seg)
        assert all(np.array_equal(u, v) for u, v in zip(base, x)), seg
    again = run(engine, G, off, coord, 300, 150000.0, 0.1)
    assert all(np.array_equal(u, v) for u, v in zip(base, again))
    # chromosome 1 alone (rows 200..332)
    sub = run(engine, G[200:333], [0, 133], coord[200:333], 300, 150000.0, 0.1)
    k = (base[0] >= 200) & (base[0] < 333)
    assert np.array_equal(sub[0] + 200, base[0][k]) and np.array_equal(sub[1] + 200, base[1][k])
    assert np.array_equal(sub[2], base[2][k])


def test_sink_stop_and_counts(engine):
    rng = np.random.default_rng(4)
    G = R.ld_panel(rng, 1500, 256, 0.0)
    bed = synth.pack_bed(G)
    rows = np.arange(1500, dtype=np.int32)
    off = np.array([0, 1500], np.int32)
    coord = np.arange(1500, dtype=np.float64)
    lib = engine.lib
    calls = []

    def stop_after(k):
        def f(user, a0, a1, o, b, r):
            calls.append((a0, a1, o[a1 - a0]))
            return 1 if len(calls) == k else 0
        return _abi.LD_SINK(f)

    n_pairs, n_miss, ms = C.c_int64(0), C.c_int64(0), C.c_float(0)
    args = (engine.h, bed.ctypes.data, 1500, 256, rows.ctypes.data, 1500, off.ctypes.data, 1, coord.ctypes.data, 1000, 1e9, 0.0, 128)
    sink = stop_after(10 ** 9)
    assert lib.dbslmm_b200_ld_pairs(*args, sink, None, None, C.byref(n_pairs), C.byref(n_miss), C.byref(ms)) == 0
    assert sum(c[2] for c in calls) == n_pairs.value > 0
    assert calls[0][0] == 0 and calls[-1][1] == 1500 and all(calls[i][1] == calls[i + 1][0] for i in range(len(calls) - 1))
    total = len(calls)
    assert total >= 3
    calls.clear()
    sink = stop_after(2)
    assert lib.dbslmm_b200_ld_pairs(*args, sink, None, None, None, None, None) == _abi.ERR_SINK
    assert len(calls) == 2
    calls.clear()
    a, b, r = engine.ld_pairs(bed, 256, rows, off, coord, max_snps=1000, max_dist=1e9, r2_min=0.0)   # the handle still works
    assert a.size == n_pairs.value


def test_segment_split_into_ranges(engine):
    """More pairs in one segment than the 8 Mi-pair buffer holds: the default segment (all 40,000 rows) is emitted in
    several ranges, the later ones starting inside it, through both pinned buffers in turn.  The result must equal, bit for
    bit, a run with 128-row segments, where every segment is one range."""
    rng = np.random.default_rng(31)
    m, n, N = 40000, 32, 256
    G = R.ld_panel(rng, m, n, 0.0)
    bed = synth.pack_bed(G)
    rows = np.arange(m, dtype=np.int32)
    off = np.array([0, m], np.int32)
    coord = np.arange(m, dtype=np.float64)

    def collect(segment_rows):
        calls, A, B, Rr = [], [], [], []

        def f(user, a0, a1, o, b, r):
            oo = np.ctypeslib.as_array(o, (a1 - a0 + 1,)).copy()
            k = int(oo[-1])
            calls.append((a0, a1, k))
            A.append(np.repeat(np.arange(a0, a1, dtype=np.int64), np.diff(oo)))
            B.append(np.ctypeslib.as_array(b, (k,)).copy() if k else np.zeros(0, np.int32))
            Rr.append(np.ctypeslib.as_array(r, (k,)).copy() if k else np.zeros(0, np.float64))
            return 0

        sink = _abi.LD_SINK(f)
        n_pairs = C.c_int64(0)
        rc = engine.lib.dbslmm_b200_ld_pairs(engine.h, bed.ctypes.data, m, n, rows.ctypes.data, m, off.ctypes.data, 1,
                                             coord.ctypes.data, N, 1e12, 0.0, segment_rows, sink, None, None, C.byref(n_pairs),
                                             None, None)
        assert rc == 0, engine.lib.dbslmm_b200_last_error(engine.h)
        return calls, np.concatenate(A), np.concatenate(B), np.concatenate(Rr), n_pairs.value

    calls, a, b, r, n_pairs = collect(0)
    want = int(np.minimum(N - 1, m - 1 - np.arange(m)).sum())         # r2_min = 0: every pair of the window
    assert n_pairs == a.size == want > 8 * 2 ** 20
    assert len(calls) >= 2 and calls[1][0] > 0 and calls[0][2] > 0 and calls[1][2] > 0
    assert calls[0][0] == 0 and calls[-1][1] == m and all(calls[i][1] == calls[i + 1][0] for i in range(len(calls) - 1))
    calls128, a128, b128, r128, _ = collect(128)
    assert len(calls128) == (m + 127) // 128
    assert np.array_equal(a, a128) and np.array_equal(b, b128)
    assert np.array_equal(r.view(np.int64), r128.view(np.int64))
    key = a * m + b
    assert np.all(np.diff(key) > 0) and np.all(b - a <= N - 1)
    # r of the pairs of rows 0..599 and of the rows around the range boundary, against the reference
    for lo in (0, calls[1][0] - 300):
        e = P.ld_pairs_exact(G[lo:lo + 600], [0, 600], coord[lo:lo + 600], N, 1e12, None)
        k = (a >= lo) & (a < lo + 600) & (b < lo + 600)
        assert np.array_equal(a[k] - lo, e["a"]) and np.array_equal(b[k] - lo, e["b"])
        assert np.abs(r[k].astype(P.LD) - e["r"]).max() <= 8 * U


def test_errors(engine):
    G = R.ld_panel(np.random.default_rng(0), 10, 50, 0.0)
    bed = synth.pack_bed(G)
    rows = np.arange(10, dtype=np.int32)
    coord = np.arange(10, dtype=np.float64)
    ok = dict(max_snps=10, max_dist=1e6, r2_min=0.2)
    for kw, msg in ((dict(max_snps=0), "max_snps"), (dict(max_dist=-1.0), "max_dist"), (dict(max_dist=float("nan")), "max_dist"),
                    (dict(r2_min=float("nan")), "r2_min"), (dict(segment_rows=100), "segment_rows")):
        with pytest.raises(_abi.EngineError, match=msg):
            engine.ld_pairs(bed, 50, rows, [0, 10], coord, **{**ok, **kw})
    with pytest.raises(_abi.EngineError, match="not sorted"):
        engine.ld_pairs(bed, 50, rows, [0, 10], coord[::-1].copy(), **ok)
    with pytest.raises(_abi.EngineError, match="out of range"):
        engine.ld_pairs(bed, 50, rows + 5, [0, 10], coord, **ok)
    with pytest.raises(_abi.EngineError, match="chromosome offsets"):
        engine.ld_pairs(bed, 50, rows, [0, 9], coord, **ok)
    with pytest.raises(_abi.EngineError, match="limit"):
        engine.ld_pairs(np.zeros(10 * 102337, np.uint8), 409345, rows, [0, 10], coord, **ok)
