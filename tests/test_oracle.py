"""CPU: the oracle against the golden vectors produced by the UNMODIFIED reference
(tools/make_golden.py) and against independent numpy restatements."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from parity_bars import bar
from oracle import refharness as R

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def c1():
    return np.load(os.path.join(GOLD, "c1_testdat.npz"), allow_pickle=False)


@pytest.fixture(scope="module")
def ragged():
    return np.load(os.path.join(GOLD, "synth_ragged.npz"), allow_pickle=False)


def relmax(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def test_decode_matches_numpy_twin(ragged):
    bed, G, n = ragged["bed"], ragged["G"], int(ragged["n_ref"])
    for pos in (0, 17, G.shape[0] - 1):
        g, maf = O.read_snp_im(bed, pos, n)
        row = G[pos].astype(np.float64)
        miss = row < 0
        mu = row[~miss].mean()
        exp = np.where(miss, mu, row)
        assert np.allclose(g, exp, rtol=0, atol=1e-15)
        af = 0.5 * exp.sum() / n
        assert maf == pytest.approx(min(af, 1 - af), abs=1e-15)


def test_decode_indicator_and_padding(ragged):
    bed, G, n = ragged["bed"], ragged["G"], int(ragged["n_ref"])   # n = 403: last byte has one padding sample
    ind = (np.arange(n) % 4 != 1).astype(np.int32)
    g, _ = O.read_snp_im(bed, 5, n, ind)
    assert g.size == int(ind.sum())
    row = G[5][ind != 0].astype(np.float64)
    miss = row < 0
    assert np.allclose(g[~miss], row[~miss])


def test_ref_maf_golden(ragged, c1):
    for d in (ragged, c1):
        maf = O.snp_maf(d["bed"], d["bed"].shape[0], int(d["n_ref"]))
        assert np.abs(maf - d["ref_maf"]).max() < 1e-15


def test_normalize_is_n_minus_one(c1):
    g, _ = O.read_snp_im(c1["bed"], 10, int(c1["n_ref"]))
    x = O.normalize(g)
    n = x.size
    assert abs(x.mean()) < 1e-14
    assert float(x @ x) == pytest.approx(n - 1, rel=1e-12)        # diag(X'X/n) = (n-1)/n


def test_integer_gram_formula_equals_float_path(ragged):
    """The exact-integer restatement the CUDA Gram epilogue implements (SURVEY 8a K3)."""
    bed, n = ragged["bed"], int(ragged["n_ref"])
    pos = np.arange(150, dtype=np.int32)                            # block 0: has missing calls
    Q, A, N = O.gram_int(bed, n, pos)
    Q, A, N = Q.astype(np.float64), A.astype(np.float64), N.astype(np.float64)
    S = np.diag(A).copy()        # A_ii = sum g_i M_i = S_i
    ni = np.diag(N).copy()
    tau = 0.8
    d = ni * np.diag(Q) - S * S
    r = np.sqrt(tau * (n - 1.0) / (n * ni * d))
    num = np.outer(ni, ni) * Q - (ni[:, None] * S[None, :]) * A - (ni[None, :] * S[:, None]) * A.T + np.outer(S, S) * N
    sigma = num * np.outer(r, r) + (1 - tau) * np.eye(pos.size)
    assert np.abs(sigma - O.sigma(bed, n, pos, tau)).max() < 1e-13


def test_pcg_against_direct_solve(c1):
    pos = c1["lmm_pos"][:200]
    S = O.sigma(c1["bed"], int(c1["n_ref"]), pos)
    A = S + np.eye(200) / (float(c1["sigma_s"]) * int(c1["n_obs"]))
    b = c1["lmm_z"][:200]
    x, it = O.pcgv(A, b)
    assert 0 < it < 1000
    assert np.linalg.norm(A @ x - b) <= 1.1e-7


def test_oracle_ref_mode_matches_reference_golden_c1(c1):
    n_ref, n_obs, sig = int(c1["n_ref"]), int(c1["n_obs"]), float(c1["sigma_s"])
    b, _, sing, it = O.est(c1["bed"], n_ref, n_obs, sig, c1["lmm_off"], c1["lmm_pos"], c1["lmm_z"], mode=O.MODE_REF)
    assert sing == 0 and 30 <= it <= 60
    assert relmax(b, c1["lmm_beta"]) < 1e-9
    bs, bl, sing, _ = O.est(c1["bed"], n_ref, n_obs, sig, c1["s_off"], c1["s_pos"], c1["s_z"], c1["l_off"], c1["l_pos"],
                            c1["l_z"], mode=O.MODE_REF)
    # (m_l + 2) chained PCG solves: two faithful PCG implementations differ by the CG recurrence's sensitivity
    # to summation order near the 1e-7 stopping threshold (iteration counts flip by one on some columns),
    # so agreement here is bounded by the truncation error itself, not by rounding.
    assert relmax(bs, c1["beta_s"]) <= bar("c1_testdat", "beta_s", "pcg") and relmax(bl, c1["beta_l"]) <= bar("c1_testdat", "beta_l", "pcg")


def test_oracle_ref_mode_matches_reference_golden_ragged(ragged):
    d = ragged
    n_ref, n_obs, sig = int(d["n_ref"]), int(d["n_obs"]), float(d["sigma_s"])
    bs, bl, sing, _ = O.est(d["bed"], n_ref, n_obs, sig, d["s_off"], d["s_pos"], d["s_z"], d["l_off"], d["l_pos"], d["l_z"],
                            threads=2, mode=O.MODE_REF)
    assert sing == 0
    assert relmax(bs, d["beta_s"]) <= bar("synth_ragged", "beta_s", "pcg") and relmax(bl, d["beta_l"]) <= bar("synth_ragged", "beta_l", "pcg")
    # the single-block entry point on block 5: the stored betas of that block are what the reference's estBlock returned
    # for it (oracle/ref_harness.cpp's ref_est_path calls ref_est_block once per block)
    s0, s1, l0, l1 = d["s_off"][5], d["s_off"][6], d["l_off"][5], d["l_off"][6]
    assert l1 > l0
    o_s, o_l, _, _ = O.est_block(d["bed"], n_ref, n_obs, sig, d["s_pos"][s0:s1], d["s_z"][s0:s1], d["l_pos"][l0:l1], d["l_z"][l0:l1],
                                 mode=O.MODE_REF)
    assert relmax(o_s, d["beta_s"][s0:s1]) < 1e-9 and relmax(o_l, d["beta_l"][l0:l1]) < 1e-9
    b, _, _, _ = O.est(d["bed"], n_ref, n_obs, sig, d["lmm_off"], np.arange(d["lmm_z"].size, dtype=np.int32), d["lmm_z"],
                       threads=2, mode=O.MODE_REF)
    assert relmax(b, d["lmm_beta"]) < 1e-9


def test_exact_mode_gap_to_reference_is_the_pcg_truncation(c1):
    """Cholesky/direct form vs the reference's PCG: the gap is the reference's own truncation error
    (SURVEY 7 hard part 1): ~3e-9 in LMM mode, a few 1e-8 in DBSLMM mode on test_dat."""
    n_ref, n_obs, sig = int(c1["n_ref"]), int(c1["n_obs"]), float(c1["sigma_s"])
    b, _, _, _ = O.est(c1["bed"], n_ref, n_obs, sig, c1["lmm_off"], c1["lmm_pos"], c1["lmm_z"], mode=O.MODE_EXACT)
    assert relmax(b, c1["lmm_beta"]) <= bar("c1_testdat", "lmm_beta")
    bs, bl, _, _ = O.est(c1["bed"], n_ref, n_obs, sig, c1["s_off"], c1["s_pos"], c1["s_z"], c1["l_off"], c1["l_pos"],
                         c1["l_z"], mode=O.MODE_EXACT)
    assert relmax(bs, c1["beta_s"]) <= bar("c1_testdat", "beta_s") and relmax(bl, c1["beta_l"]) <= bar("c1_testdat", "beta_l")


def test_bordered_system_identity(ragged):
    """beta = K^-1 z / sqrt(N) with K = Sigma + c diag(1_small, 0_large) reproduces estBlock's
    Schur-complement algebra (what chol.cu factorises)."""
    d = ragged
    n_ref, n_obs, sig = int(d["n_ref"]), int(d["n_obs"]), float(d["sigma_s"])
    b = 0
    ps = d["s_pos"][d["s_off"][b]:d["s_off"][b + 1]]
    pl = d["l_pos"][d["l_off"][b]:d["l_off"][b + 1]]
    zs = d["s_z"][d["s_off"][b]:d["s_off"][b + 1]]
    zl = d["l_z"][d["l_off"][b]:d["l_off"][b + 1]]
    assert pl.size > 0
    S = O.sigma(d["bed"], n_ref, np.concatenate([ps, pl]))
    K = S.copy()
    K[np.arange(ps.size), np.arange(ps.size)] += 1.0 / (sig * n_obs)
    x = np.linalg.solve(K, np.concatenate([zs, zl])) / np.sqrt(n_obs)
    bs, bl, _, _ = O.est_block(d["bed"], n_ref, n_obs, sig, ps, zs, pl, zl, mode=O.MODE_EXACT)
    assert relmax(x[:ps.size], bs) < 1e-11 and relmax(x[ps.size:], bl) < 1e-11


def test_est_handles_empty_blocks(ragged):
    d = ragged
    off = d["lmm_off"]
    assert (np.diff(off) == 0).any()
    b, _, sing, _ = O.est(d["bed"], int(d["n_ref"]), int(d["n_obs"]), float(d["sigma_s"]), off,
                          np.arange(d["lmm_z"].size, dtype=np.int32), d["lmm_z"], mode=O.MODE_EXACT)
    assert sing == 0 and np.isfinite(b).all()


@pytest.mark.skipif(not R.available(), reason="oracle/_ref (unmodified reference build) not present")
def test_oracle_against_live_reference_build(ragged):
    d = ragged
    n = int(d["n_ref"])
    with R.BedFile(d["bed"]) as bf:
        for pos in (0, 33, 424):
            g1, m1 = O.read_snp_im(d["bed"], pos, n)
            g2, m2 = R.read_snp_im(bf.path, pos, n)
            assert np.array_equal(g1, g2) and m1 == m2
            assert np.abs(O.normalize(g1) - R.normalize(g2)).max() < 1e-14
        ps = d["s_pos"][d["s_off"][5]:d["s_off"][6]]
        zs = d["s_z"][d["s_off"][5]:d["s_off"][6]]
        pl = d["l_pos"][d["l_off"][5]:d["l_off"][6]]
        zl = d["l_z"][d["l_off"][5]:d["l_off"][6]]
        r_s, r_l = R.est_block(bf.path, n, int(d["n_obs"]), float(d["sigma_s"]), ps, zs, pl, zl)
        o_s, o_l, _, _ = O.est_block(d["bed"], n, int(d["n_obs"]), float(d["sigma_s"]), ps, zs, pl, zl, mode=O.MODE_REF)
        assert relmax(o_s, r_s) < 1e-9 and relmax(o_l, r_l) < 1e-9      # live: oracle vs the unmodified estBlock on one block (measured 1e-11)


@pytest.mark.skipif(not R.available(), reason="oracle/_ref (unmodified reference build) not present")
@pytest.mark.parametrize("with_large", [True, False])
def test_variance_oracle_against_live_reference_build(ragged, with_large):
    """calc_nt_by_nt_matrix(...).diag() through the reference's own functions vs the oracle restatement."""
    d = ragged
    n = int(d["n_ref"])
    rng = np.random.default_rng(9)
    from dbslmm_b200 import synth
    Gt = synth.make_genotypes(rng, [int(d["sizes"].sum())], 57, missing_rate=0.02)
    tbed = synth.pack_bed(Gt)
    ind = (rng.random(57) < 0.6).astype(np.int32)
    b = 0
    ps = d["s_pos"][d["s_off"][b]:d["s_off"][b + 1]]
    pl = d["l_pos"][d["l_off"][b]:d["l_off"][b + 1]] if with_large else None
    with R.BedFile(d["bed"]) as b1, R.BedFile(tbed) as b2:
        ref = R.variance_block(b1.path, n, b2.path, 57, ind, int(d["n_obs"]), float(d["sigma_s"]), ps, ps, pl, pl)
    got = O.variance_block(d["bed"], n, tbed, 57, ind, int(d["n_obs"]), float(d["sigma_s"]), ps, ps, pl, pl)
    assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max()


def test_valid_tool_restatement_matches_the_reference_binary():
    """SURVEY 8f-4: oracle.valid_run against <r2>.txt written by the UNMODIFIED scr/main_valid.cpp + scr/validate.cpp
    (oracle/_ref/valid_ref, tools/make_golden.py valid_synth), with and without the MAF constraint."""
    g = np.load(os.path.join(GOLD, "synth_cli.npz"))
    v = np.load(os.path.join(GOLD, "valid_synth.npz"))
    for key, maf_max in (("r2_c", 0.2), ("r2_u", 1.0)):
        nume, deno = O.valid_run(str(g["cli_txt"]), str(v["ext_txt"]), str(g["bim_txt"]), str(g["block_txt"]), g["bed"], int(g["n_ref"]), maf_max)
        ref = np.array([[float(x) for x in ln.split()] for ln in str(v[key]).strip().split("\n")])
        assert ref.shape == (3, 2)
        assert np.abs(nume - ref[:, 0]).max() <= 5e-6 * np.abs(ref[:, 0]).max()       # 6 printed digits
        assert np.abs(deno - ref[:, 1]).max() <= 5e-6 * np.abs(ref[:, 1]).max()
    assert str(v["r2_c"]) != str(v["r2_u"])                                              # the MAF filter really removed SNPs
