"""CPU: the extended-precision reference and the stage checks of tests/solver_ref.py are themselves right.  LAPACK's
own factor and solves pass every bar with margin at the block solver's edge shapes, and each injected defect fails the
stage it belongs to (the tile check also names the tile)."""
import numpy as np
import pytest
import scipy.linalg as sla

from dbslmm_b200 import synth
from oracle import oracle as O

import solver_ref as R

N_REF, TAU, N_OBS = 403, 0.8, 20_000
RIDGES = (1e-4, 1.0, 1e3)                                    # sigma_s = 5e-1, 5e-5, 5e-8 at N = 20,000


def z_scores(rng, ms, ml):
    zl = rng.choice([-1.0, 1.0], size=ml) * (6.0 + rng.exponential(2.0, size=ml))
    return np.concatenate([1.3 * rng.standard_normal(ms), zl])


_GENO = {}


def genotypes(m, seed=7):
    key = (m, seed)
    if key not in _GENO:
        rng = np.random.default_rng(seed + m)
        _GENO[key] = synth.pack_bed(synth.make_genotypes(rng, [m], N_REF))
    return _GENO[key]


def lapack_block(m, ms, c, seed=7):
    """One block solved by LAPACK from a correctly rounded Sigma: what a perfect library would return."""
    bed = genotypes(m, seed)
    pos = np.arange(m, dtype=np.int32)
    sstar = R.exact_sigma(bed, N_REF, pos, TAU)
    slib = sstar.astype(np.float64)
    K = R.k_matrix(slib, ms, c)
    L = sla.cholesky(K, lower=True)
    z = z_scores(np.random.default_rng(seed * 31 + m), ms, m - ms)
    y = sla.solve_triangular(L, z, lower=True)
    x = sla.solve_triangular(L.T, y, lower=False)
    xstar, kappa = R.refined_solve(R.k_matrix(sstar, ms, c), z)
    return dict(bed=bed, pos=pos, sstar=sstar, slib=slib, K=K, L=L, z=z, y=y, x=x, xstar=xstar, kappa=kappa, ms=ms, c=c)


def run_checks(b, **over):
    a = dict(ms=b["ms"], c=b["c"], z=b["z"], sigma_lib=b["slib"], sigma_star=b["sstar"], L=b["L"], y=b["y"], x=b["x"],
             xstar=b["xstar"], kappa=b["kappa"])
    a.update(over)
    return R.check_block("test", **a)


def test_exact_sigma_agrees_with_the_float_path_and_is_symmetric():
    g = np.load(R.__file__.replace("solver_ref.py", "golden/synth_ragged.npz"))
    n = int(g["n_ref"])
    # every block of the fixture has missing calls (four-plane formula); the same genotypes with the missing calls set
    # to 0 take the one-plane formula (A_ij = S_i, N = n)
    G = g["G"]
    for bed, missing in ((g["bed"], True), (synth.pack_bed(np.where(G < 0, 0, G).astype(np.int8)), False)):
        off = 0
        for m in g["sizes"]:
            pos = np.arange(off, off + m, dtype=np.int32)
            off += m
            S = R.exact_sigma(bed, n, pos, TAU)
            assert S.dtype == np.longdouble and S.shape == (m, m)
            assert np.array_equal(S, S.T)
            if m:
                assert np.abs(S.astype(np.float64) - O.sigma(bed, n, pos, TAU)).max() < 1e-13
                assert (O.gram_int(bed, n, pos)[2] == n).all() != missing


def test_refined_solve_is_exact_to_far_below_u():
    b = lapack_block(300, 290, 1e-4)
    Ks = R.k_matrix(b["sstar"], 290, 1e-4)
    xs = b["xstar"]
    # componentwise backward error of x* at the level of the extended residual, a hundredth of FP64's unit roundoff
    res = np.abs(b["z"].astype(np.longdouble) - Ks @ xs)
    scale = np.abs(Ks) @ np.abs(xs) + np.abs(b["z"])
    assert float((res / scale).max()) < 1e-2 * R.U
    assert 1.0 <= b["kappa"] < 1e8


EDGE = [(1, 1), (1, 0), (8, 0), (8, 5), (64, 64), (64, 0), (65, 64), (1024, 1023), (1025, 1024), (2049, 1985)]


@pytest.mark.parametrize("c", RIDGES)
@pytest.mark.parametrize("m,ms", EDGE)
def test_lapack_passes_every_bar_with_margin(m, ms, c):
    r = run_checks(lapack_block(m, ms, c))
    assert set(r) == set(R.STAGES)
    for s, v in r.items():
        assert v < R.BARS[s] / 4, (s, v)


def first_failure(b, **over):
    with pytest.raises(R.SolverCheckError) as e:
        run_checks(b, **over)
    return e.value


@pytest.fixture(scope="module")
def big():
    return lapack_block(1025, 960, 1e-4)


def test_scaled_offdiagonal_tile_fails_the_factor_and_is_located(big):
    L = big["L"].copy()
    L[640:704, 192:256] *= 1 + 1e-9                           # tile (10, 3)
    e = first_failure(big, L=L)
    assert e.failed[0] in ("factor", "tiles") and "tiles" in e.failed
    assert (e.tiles[0][0], e.tiles[0][1]) == (10, 3)


@pytest.mark.parametrize("where", ["missing_on_small", "added_on_large"])
def test_misplaced_ridge_fails_the_factor(big, where):
    K = big["K"].copy()
    j = 959 if where == "missing_on_small" else 960          # last small SNP, first large one (a panel edge: 960 = 15*64)
    K[j, j] += -big["c"] if where == "missing_on_small" else big["c"]
    L = sla.cholesky(K, lower=True)
    e = first_failure(big, L=L, y=sla.solve_triangular(L, big["z"], lower=True))
    assert e.failed[0] in ("factor", "tiles")
    assert (e.tiles[0][0], e.tiles[0][1]) == (15 if where == "added_on_large" else 14, j // 64)


def test_forward_substitution_from_a_neighbouring_ridge_fails_forward(big):
    L2 = sla.cholesky(R.k_matrix(big["slib"], big["ms"], 1.0), lower=True)
    y = sla.solve_triangular(L2, big["z"], lower=True)
    x = sla.solve_triangular(big["L"].T, y, lower=False)
    e = first_failure(big, y=y, x=x)
    assert e.failed[0] == "forward"


def test_stale_panel_in_back_substitution_fails_back(big):
    x = big["x"].copy()
    x[512:576] = x[576:640]                                  # panel 8 holds what panel 9 (solved just before it) got
    e = first_failure(big, x=x)
    assert e.failed[0] == "back"


def test_sigma_entry_off_by_64_ulps_fails_sigma(big):
    s = big["slib"].copy()
    s[700, 300] = s[300, 700] = s[700, 300] * (1 + 64 * R.U)
    e = first_failure(big, sigma_lib=s)
    assert e.failed[0] == "sigma"
    s = big["slib"].copy()
    s[700, 300] = s[300, 700] = s[700, 300] * (1 + 6 * R.U)   # a few roundings more than the library spends still pass
    run_checks(big, sigma_lib=s)


# The detection floors quoted in solver_ref.py (strictly lower part of tile (last row tile, panel 0), tile (0, 0) at
# m = 64), asserted at ten times the floor
FLOORS = {64: 3.0e-15, 1025: 3.0e-15, 2049: 3.4e-15}


def scaled_tile_rho(b, delta):
    m = b["L"].shape[0]
    L = b["L"].copy()
    I = (m - 1) // R.TILE
    blk = L[I * R.TILE:(I + 1) * R.TILE, 0:R.TILE]
    blk[...] = np.where(np.tri(*blk.shape, I * R.TILE - 1, dtype=bool), blk * (1 + delta), blk)
    return float(np.nanmax(R.tile_ratios(b["K"], L)))


@pytest.mark.parametrize("m", sorted(FLOORS))
def test_tile_check_detects_ten_times_its_floor(m):
    b = lapack_block(m, m - m // 32, 1e-4)
    assert scaled_tile_rho(b, 0.0) < R.BARS["tiles"] / 4
    assert scaled_tile_rho(b, 10 * FLOORS[m]) >= R.BARS["tiles"]
    assert scaled_tile_rho(b, FLOORS[m] / 10) < R.BARS["tiles"]


# ---- the integer Gram planes by BLAS, and the Sigma bar against the four-plane epilogue's numerator ----------------
@pytest.mark.parametrize("n,missing", [(403, 0.0), (403, 0.02), (125 * 4 - 3, 0.01), (5, 0.1)])
def test_blas_planes_equal_the_oracle_bit_for_bit(n, missing):
    rng = np.random.default_rng(n + int(missing * 100))
    G = synth.make_genotypes(rng, [40, 23], n, missing_rate=missing)
    bed = synth.pack_bed(G)
    pos = np.array([0, 5, 5, 62, 17, 40, 3, 61, 22], np.int32)           # out of order, one row twice
    assert np.array_equal(R.bed_genotypes(bed, n, pos), G[pos])
    for chunk in (256 << 20, 4 * pos.size * 7):                            # one chunk; chunks of 7 samples
        for got, want in zip(R.gram_planes(R.bed_genotypes(bed, n, pos), chunk_bytes=chunk), O.gram_int(bed, n, pos)):
            assert got.dtype == np.int64 and np.array_equal(got, want)


def decoder_r(S, ni, sq, n, tau):
    """r_i as the decoder computes it in FP64 (decode.cu): sqrt(tau (n - 1) / (n n_i d)), d = n_i sum g^2 - S^2."""
    d = ni.astype(np.float64) * sq.astype(np.float64) - S.astype(np.float64) ** 2
    return np.sqrt(tau * (float(n) - 1.0) / (float(n) * ni.astype(np.float64) * d))


def epilogue_sigma(Q, A, N, n, tau, numerator):
    """The four-plane epilogue's Sigma, replayed on the host with exactly rounded fma, then (num r_i) r_j and 1 - tau added
    on the diagonal.  The numerator is
      "exact"  the exact integer, rounded once to FP64;
      "chain"  num = (n_i n_j) Q; num = fma(-(n_i S_j), A_ij, num); num = fma(-(n_j S_i), A_ji, num);
               num = fma(S_i S_j, N_ij, num) -- what gram.cu computed before, exact only while every term is below 2^53;
      "split"  u = fma(-S_j, A_ij, n_j Q); w = fma(-S_j, N, n_j A_ji); p = n_i u; pe = fma(n_i, u, -p);
               num = fma(-S_i, w, p) + pe -- what gram.cu computes."""
    from fractions import Fraction

    def fma(a, b, c):
        return float(Fraction(a) * Fraction(b) + Fraction(c))
    S, ni = np.diag(A).astype(np.int64), np.diag(N).astype(np.int64)
    r = decoder_r(S, ni, np.diag(Q), n, tau)
    m = Q.shape[0]
    out = np.zeros((m, m))
    for i in range(m):
        for j in range(i + 1):
            Ni, Nj, Si, Sj = (int(x) for x in (ni[i], ni[j], S[i], S[j]))
            if numerator == "exact":
                num = float(Ni * Nj * int(Q[i, j]) - Ni * Sj * int(A[i, j]) - Nj * Si * int(A[j, i]) + Si * Sj * int(N[i, j]))
            elif numerator == "split":
                u = fma(-float(Sj), float(A[i, j]), float(Nj) * float(Q[i, j]))
                w = fma(-float(Sj), float(N[i, j]), float(Nj) * float(A[j, i]))
                p = float(Ni) * u
                num = fma(-float(Si), w, p) + fma(float(Ni), u, -p)
            else:
                num = (float(Ni) * float(Nj)) * float(Q[i, j])
                num = fma(-(float(Ni) * float(Sj)), float(A[i, j]), num)
                num = fma(-(float(Nj) * float(Si)), float(A[j, i]), num)
                num = fma(float(Si) * float(Sj), float(N[i, j]), num)
            v = num * r[i] * r[j]
            out[i, j] = out[j, i] = v + (1.0 - tau) if i == j else v
    return out


def test_sigma_bar_detects_an_fp64_numerator_at_max_n_ref():
    """At n = 409,344 with 1 % missing calls and half the SNPs counting the major allele, the terms of the four-plane
    numerator reach 4 n^3 = 2.7e17 > 2^53: the FP64 chain rounds them and misses the 16-ulp Sigma bar; the exact numerator
    and the split form meet it.  Below n = 2^17 every term is exact and the three agree bit for bit."""
    for n, fails in ((409_344, True), (2_000, False)):
        rng = np.random.default_rng(1)
        G = synth.make_genotypes(rng, [24], n)
        flip = rng.random(24) < 0.5
        G[flip] = 2 - G[flip]
        G = np.where(rng.random(G.shape) < 0.01, np.int8(-1), G)
        Q, A, N = R.gram_planes(G)
        sstar = R.sigma_from_planes(Q, A, N, n, TAU)
        chain, exact, split = (epilogue_sigma(Q, A, N, n, TAU, k) for k in ("chain", "exact", "split"))
        for S in (exact, split):
            assert R.sigma_ratio(S, sstar) <= R.BARS["sigma"], (n, R.sigma_ratio(S, sstar))
        assert (R.sigma_ratio(chain, sstar) > R.BARS["sigma"]) == fails, (n, R.sigma_ratio(chain, sstar))
        if not fails:
            assert np.array_equal(chain, exact) and np.array_equal(split, exact)
