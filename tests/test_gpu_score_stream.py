"""GPU: the streaming scorer (dbslmm_b200_score_stream, Engine.score_stream) against a numpy restatement of PLINK's
`--score ... sum` with its CNT / CNT2 columns: score_i = sum_j beta_j * dosage_ij, dosage = copies of the scored allele,
a missing call replaced by the row's mean dosage over its called genotypes; CNT_i = 2 x calls of i, CNT2_i = copies of the
scored allele among them; a row without a called genotype adds nothing.  The panel is a numpy.memmap of a .bed file, so only
the scored rows are read from it, chunk by chunk."""
import numpy as np
import pytest

from dbslmm_b200 import _abi, synth

pytestmark = pytest.mark.gpu


def restate(G, pos, beta, flip):
    """G int8 [n_snp, n] A1 copies (-1 missing) -> (scores [n_folds, n], cnt [n], cnt2 [n])."""
    X = G[pos]
    miss = X < 0
    called = (~miss).sum(1)
    D = np.where(miss, 0, X).astype(np.float64)
    mu = np.divide(D.sum(1), called, out=np.zeros(len(pos)), where=called > 0)
    fl = flip.astype(bool)
    D = np.where(fl[:, None], 2.0 - D, D)
    mu = np.where(fl, 2.0 - mu, mu)
    D = np.where(miss, mu[:, None], D)
    D[called == 0] = 0.0
    dose_called = np.where(miss, 0, np.where(fl[:, None], 2 - X, X)).astype(np.int64)
    return beta @ D, 2 * (~miss).sum(0).astype(np.int64), dose_called.sum(0)


def make_panel(rng, n_snp, n, miss):
    """Random genotypes with a monomorphic row (1) and an all-missing row (2)."""
    p = rng.uniform(0.05, 0.5, n_snp)
    G = rng.binomial(2, p[:, None], size=(n_snp, n)).astype(np.int8)
    if miss > 0:
        G[rng.random((n_snp, n)) < miss] = -1
    G[1] = 1
    G[2] = -1
    return G


def memmap_bed(tmp_path, G):
    path = tmp_path / "panel.bed"
    with open(path, "wb") as f:
        f.write(bytes([0x6C, 0x1B, 0x01]) + synth.pack_bed(G).tobytes())
    return np.memmap(path, dtype=np.uint8, mode="r", offset=3)


def check(got, exp, what):
    s, c, c2 = got
    es, ec, ec2 = exp
    scale = max(1.0, np.abs(es).max())
    assert np.abs(s - es).max() <= 1e-12 * scale, what
    assert np.array_equal(c, ec) and np.array_equal(c2, ec2), what


@pytest.mark.parametrize("n_val,n_snp,n_scored", [(1, 30, 41), (3, 30, 41), (5, 60, 83), (17, 60, 83), (1003, 200, 301),
                                                  (4097, 120, 150), (409345, 12, 23)])
@pytest.mark.parametrize("miss", [0.0, 0.02])
def test_stream_matches_restatement_at_every_chunk_size(engine, tmp_path, n_val, n_snp, n_scored, miss):
    rng = np.random.default_rng(n_val * 7 + int(miss * 100))
    G = make_panel(rng, n_snp, n_val, miss)
    bed = memmap_bed(tmp_path, G)
    pos = rng.integers(0, n_snp, n_scored).astype(np.int32)          # unsorted, with repeats
    pos[:3] = [2, 1, pos[5]]                                          # the all-missing and the monomorphic row, a repeat
    beta = rng.standard_normal((3, n_scored)) * 1e-2
    flip = (rng.random(n_scored) < 0.4).astype(np.uint8)
    exp = restate(G, pos, beta, flip)
    pitch = (n_val + 3) // 4
    rows_odd = next(r for r in (4, 5, 6, 8, 9, 11) if n_scored % r)  # a chunk size that does not divide n_scored
    runs = {}
    for rows in (1, 7, rows_odd, None):
        cb = 0 if rows is None else rows * (pitch + 1)
        got = engine.score_stream(bed, n_val, pos, beta, flip, chunk_bytes=cb)
        check(got, exp, f"rows per chunk {rows}")
        assert engine.last_empty_rows == int((G[pos] < 0).all(1).sum())
        runs[rows] = got
    again = engine.score_stream(bed, n_val, pos, beta, flip, chunk_bytes=7 * (pitch + 1))
    assert all(np.array_equal(a, b) for a, b in zip(again, runs[7]))                # deterministic
    for rows in (1, rows_odd, None):
        assert np.abs(runs[rows][0] - runs[7][0]).max() <= 1e-12 * max(1.0, np.abs(exp[0]).max())
    s, c, c2 = engine.score_stream(bed, n_val, pos, beta, None, chunk_bytes=7 * (pitch + 1))      # no flip array
    check((s, c, c2), restate(G, pos, beta, np.zeros(n_scored, np.uint8)), "flip = None")


@pytest.mark.parametrize("n_folds", [1, 3, 4, 7])
def test_fold_k_equals_the_one_fold_call(engine, tmp_path, n_folds):
    rng = np.random.default_rng(40 + n_folds)
    n_val, n_snp = 2051, 90
    G = make_panel(rng, n_snp, n_val, 0.02)
    bed = memmap_bed(tmp_path, G)
    pos = rng.permutation(n_snp).astype(np.int32)
    beta = rng.standard_normal((n_folds, n_snp))
    flip = (rng.random(n_snp) < 0.5).astype(np.uint8)
    for cb in (0, 7 * ((n_val + 3) // 4 + 1)):
        s, c, c2 = engine.score_stream(bed, n_val, pos, beta, flip, chunk_bytes=cb)
        check((s, c, c2), restate(G, pos, beta, flip), f"{n_folds} folds")
        for k in range(n_folds):
            s1, c1, c21 = engine.score_stream(bed, n_val, pos, beta[k:k + 1], flip, chunk_bytes=cb)
            assert np.array_equal(s1[0], s[k]) and np.array_equal(c1, c) and np.array_equal(c21, c2)


@pytest.mark.parametrize("n_val,n_folds", [(17, 1), (1003, 3), (4097, 4)])
def test_single_chunk_is_bit_identical_to_the_resident_scorer(engine, tmp_path, n_val, n_folds):
    rng = np.random.default_rng(n_val + n_folds)
    G = make_panel(rng, 150, n_val, 0.02)
    G[2] = G[3]                                  # the resident scorer turns an all-missing row into NaN: leave it out here
    bed = memmap_bed(tmp_path, G)
    pos = rng.integers(0, 150, 230).astype(np.int32)
    beta = rng.standard_normal((n_folds, pos.size)) * 1e-2
    flip = (rng.random(pos.size) < 0.3).astype(np.uint8)
    ref, _ = engine.score(np.array(bed), n_val, pos, beta, flip)
    s, _, _ = engine.score_stream(bed, n_val, pos, beta, flip)
    assert np.array_equal(s, ref)


def test_argument_errors(engine, tmp_path):
    G = make_panel(np.random.default_rng(3), 20, 100, 0.0)
    bed = memmap_bed(tmp_path, G)
    ok_pos = np.arange(20, dtype=np.int32)
    with pytest.raises(_abi.EngineError, match="pos out of range"):
        engine.score_stream(bed, 100, np.array([25], np.int32), np.ones((1, 1)))
    with pytest.raises(_abi.EngineError, match="pos out of range"):
        engine.score_stream(bed, 100, np.array([-1], np.int32), np.ones((1, 1)))
    with pytest.raises(_abi.EngineError, match="bad arguments"):
        engine.score_stream(bed, 100, ok_pos, np.ones((0, 20)))                     # n_folds < 1
    lib, h = engine.lib, engine.h
    beta = np.ones(20)
    out = np.zeros(100)
    args = lambda **kw: dict(dict(bed=bed.ctypes.data, n_snp=20, n=100, pos=ok_pos.ctypes.data, n_scored=20, out=out.ctypes.data), **kw)
    def call(a):
        return lib.dbslmm_b200_score_stream(h, a["bed"], a["n_snp"], a["n"], a["pos"], None, a["n_scored"], beta.ctypes.data, 1, 0,
                                            a["out"], None, None, None, None)
    assert call(args()) == 0                                                         # counts and timing may be NULL
    exp = restate(G, ok_pos, beta[None], np.zeros(20, np.uint8))[0][0]
    assert np.abs(out - exp).max() <= 1e-12 * max(1.0, np.abs(exp).max())
    assert call(args(out=None)) == -2                                                # NULL scores
    assert call(args(bed=None)) == -2                                                # NULL panel
    assert call(args(pos=None)) == -2
    assert call(args(n_scored=2**31 // 2)) == -2 and "too many SNPs" in lib.dbslmm_b200_last_error(h).decode()
    assert call(args(n=536870912)) == -2 and "limit" in lib.dbslmm_b200_last_error(h).decode()
    assert call(args(n_snp=0)) == -2
