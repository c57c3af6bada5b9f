"""Extended-precision reference of the block solver and per-stage checks of one block's GPU outputs (host only).

The block solver (dbslmm_b200/csrc/chol.cu) factors, per LD block, the bordered system
    K = Sigma + c diag(1_small, 0_large),   c = 1 / (sigma_s N),   K x = z,   beta = x / sqrt(N)
with the small-effect SNPs first.  Its outputs are checked stage by stage against the ratios of LAPACK's testing
programs (xPOT01 for the factor, xTRT02 for the triangular solves, xGET04 for the forward error), u = 2^-53:

  sigma       max |Sigma_lib - Sigma*|_ij / (u |Sigma*|_ij) over the lower triangle;
              Sigma*_ij = 0 must come out exactly 0                                                      bar 16
  factor      ||K - L L^T||_1 / (m ||K||_1 u), K from the library's own Sigma and c                        bar 30
  tiles       rho_IJ = max over the 64 x 64 tile (I, J) of
              |K - L L^T|_ij / (u (min(i, j) + 1) (|L| |L|^T)_ij)                                          bar 30
              (the localiser: a failure names the worst tiles as (row tile, panel step))
  forward     ||L y - z||_1 / (m ||L||_1 ||y||_1 u), y = L^-1 z (the z row the solver carries as row mp)   bar 30
  back        ||L^T x - y||_1 / (m ||L^T||_1 ||x||_1 u), x = beta sqrt(N)                                 bar 30
  end_to_end  ||x - x*||_inf / (||x*||_inf kappa_inf(K*) u), x* solving the EXACT K* = Sigma* + c diag(..)  bar 30

Sigma* is formed in x86 extended precision (64-bit significand) from the integer Gram planes, and x* by iterative
refinement with the residual in that precision, so both are exact to far below u.  The host forms L L^T with FP64 BLAS,
whose own error is of the order of the componentwise bound: that is why the bars are 30, as in LAPACK, and not 1.

The Sigma bar is twice the roundings the library spends on an entry: r_i = sqrt(tau (n-1) / (n n_i d_i)) costs three
(the quotient, the root, and tau (n-1)), the numerator is an exact integer, then r_i and r_j are multiplied in (two),
n_i folded into r_i on the fast path (one), and (1 - tau) added on the diagonal (one, exact itself for tau >= 1/2):
about 7-8 roundings, 16 ulps.

LAPACK's own factor of such a block gives factor ~ 1e-3 - 2e-2, forward and back below 1e-2, end_to_end below 0.04
and tiles ~ 2.0: the tile ratio's largest entry is (0, 0), where L_00 = sqrt(K_00) is rounded once and L_00^2 once more.

Detection floor of the tile check (measured on the host: the LAPACK factor of K of a synthetic block, n_ref = 403,
tau = 0.8, c = 1e-4, m_s = m - m // 32; the strictly lower part of tile (last row tile, panel 0) -- tile (0, 0) at m = 64
-- scaled by (1 + delta); the smallest delta whose rho reaches 30, by bisection):
    m = 64:   delta = 3.0e-15
    m = 1025: delta = 3.0e-15
    m = 2049: delta = 3.4e-15
The floor is low because the scaled entries lie in the first panel, where min(i, j) + 1 is small.
tests/test_solver_ref.py asserts detection at ten times these floors.
"""
import numpy as np
import scipy.linalg as sla

U = 2.0 ** -53
BARS = {"sigma": 16.0, "factor": 30.0, "tiles": 30.0, "forward": 30.0, "back": 30.0, "end_to_end": 30.0}
STAGES = ("sigma", "factor", "tiles", "forward", "back", "end_to_end")
TILE = 64


def _require_extended():
    # the reference needs a significand well beyond FP64's; x86 long double has 64 bits (eps = 2^-63)
    if not np.finfo(np.longdouble).eps < 1.1e-19:
        raise RuntimeError("solver_ref needs an extended-precision np.longdouble (x86 80-bit); this platform's is "
                           f"eps = {np.finfo(np.longdouble).eps}: a double-double residual would be needed here")


def ridge(sigma_s, n_obs):
    """c exactly as the library computes it: 1.0 / (sigma_s * n_obs) in FP64."""
    return 1.0 / (float(sigma_s) * float(n_obs))


def exact_sigma(bed, n_ref, pos, tau):
    """Sigma* of the SNPs `pos` in np.longdouble from the integer Gram planes Q = G G^T, A_ij = sum g_i M_j, N = M M^T:
    num_ij = n_i n_j Q_ij - n_i S_j A_ij - n_j S_i A_ji + S_i S_j N_ij (an exact int64),
    Sigma_ij = num_ij r_i r_j + (1 - tau) delta_ij,  r_i = sqrt(tau (n - 1) / (n n_i d_i)),  d_i = n_i Q_ii - S_i^2."""
    _require_extended()
    from oracle import oracle as O
    pos = np.ascontiguousarray(pos, np.int32)
    m = pos.size
    if m == 0:
        return np.zeros((0, 0), np.longdouble)
    Q, A, N = (x.astype(np.int64) for x in O.gram_int(bed, int(n_ref), pos))
    S = np.diag(A).copy()
    ni = np.diag(N).copy()
    num = np.outer(ni, ni) * Q - (ni[:, None] * S[None, :]) * A - (ni[None, :] * S[:, None]) * A.T + np.outer(S, S) * N
    d = ni * np.diag(Q) - S * S
    LD = np.longdouble
    n = LD(int(n_ref))
    t = LD(float(tau))
    r = np.sqrt(t * (n - LD(1)) / (n * ni.astype(LD) * d.astype(LD)))
    sig = num.astype(LD) * r[:, None] * r[None, :]
    sig[np.arange(m), np.arange(m)] += LD(1) - t
    return np.tril(sig) + np.tril(sig, -1).T                   # exactly symmetric


def k_matrix(sigma, ms, c):
    """K = Sigma + c diag(1_small, 0_large) in Sigma's own precision (the ridge on the first ms diagonal entries)."""
    K = np.array(sigma, copy=True)
    i = np.arange(int(ms))
    K[i, i] += K.dtype.type(c)
    return K


def refined_solve(Kstar, z, max_iter=40):
    """x* of Kstar x = z: FP64 solve plus iterative refinement, the residual in np.longdouble, until the correction is
    below 1e-3 u ||x||_inf.  A residual in extended precision limits x* to about kappa 2^-64 relative, which is above
    1e-3 u once kappa exceeds a few units; the refinement then stops when the correction no longer halves, provided it is
    below 1e-3 u kappa ||x||_inf: x*'s own error is then under a thousandth of the end-to-end ratio's unit.
    Returns (x* as np.longdouble, kappa_inf(K*) from the FP64 inverse)."""
    _require_extended()
    m = Kstar.shape[0]
    if m == 0:
        return np.zeros(0, np.longdouble), 1.0
    K64 = np.asarray(Kstar, np.float64)
    Kinv = sla.inv(K64)
    kappa = float(np.abs(K64).sum(axis=1).max() * np.abs(Kinv).sum(axis=1).max())
    lu = sla.lu_factor(K64)
    Kl = np.asarray(Kstar).astype(np.longdouble)
    zl = np.asarray(z, np.float64).astype(np.longdouble)
    x = sla.lu_solve(lu, zl.astype(np.float64)).astype(np.longdouble)
    prev = np.inf
    for _ in range(max_iter):
        dx = sla.lu_solve(lu, (zl - Kl @ x).astype(np.float64))
        x += dx.astype(np.longdouble)
        step = float(np.abs(dx).max()) / max(float(np.abs(x).max()), 1e-300)
        if step <= 1e-3 * U or (step > 0.5 * prev and step <= 1e-3 * U * kappa):
            break
        prev = step
    else:
        raise RuntimeError("iterative refinement did not converge: K* is too ill-conditioned for an FP64 solve")
    return x, kappa


# ---- stage ratios (one block each) --------------------------------------------------------------------------------
def sigma_ratio(sigma_lib, sigma_star):
    """max |Sigma_lib - Sigma*|_ij / (u |Sigma*|_ij) over the lower triangle; inf if a zero Sigma*_ij is not exactly 0."""
    m = sigma_star.shape[0]
    if m == 0:
        return 0.0
    il = np.tril_indices(m)
    s = np.asarray(sigma_star)[il]
    d = np.abs(np.asarray(sigma_lib, np.longdouble)[il] - s)
    zero = (s == 0)
    if np.any(d[zero] != 0):
        return float("inf")
    return float((d[~zero] / (U * np.abs(s[~zero]))).max(initial=0.0))


def factor_residual(K, L):
    R = K - L @ L.T
    return R


def factor_ratio(K, L, R=None):
    m = K.shape[0]
    if m == 0:
        return 0.0
    R = factor_residual(K, L) if R is None else R
    nk = np.abs(K).sum(axis=0).max()
    return float(np.abs(R).sum(axis=0).max() / (m * nk * U))


def tile_ratios(K, L, R=None):
    """rho[I, J] for the 64 x 64 tiles on and below the diagonal (nan above)."""
    m = K.shape[0]
    nt = (m + TILE - 1) // TILE
    if m == 0:
        return np.zeros((0, 0))
    R = factor_residual(K, L) if R is None else R
    A = np.abs(L)
    D = A @ A.T
    i = np.arange(m)
    mn = np.minimum(i[:, None], i[None, :]) + 1.0
    num = np.abs(R)
    den = U * mn * D
    with np.errstate(divide="ignore", invalid="ignore"):
        rho = np.where(num == 0, 0.0, num / den)
    rho = np.tril(rho)
    out = np.full((nt, nt), np.nan)
    for I in range(nt):
        for J in range(I + 1):
            out[I, J] = rho[I * TILE:(I + 1) * TILE, J * TILE:(J + 1) * TILE].max()
    return out


def worst_tiles(rho, n=5):
    flat = np.where(np.isnan(rho), -1.0, rho).ravel()
    idx = np.argsort(-flat, kind="stable")[:n]
    return [(int(k // rho.shape[1]), int(k % rho.shape[1]), float(flat[k])) for k in idx if flat[k] >= 0]


def forward_ratio(L, y, z):
    m = L.shape[0]
    if m == 0:
        return 0.0
    r = np.abs(L @ y - z).sum()
    den = m * np.abs(L).sum(axis=0).max() * np.abs(y).sum() * U
    return float(r / den) if den > 0 else (0.0 if r == 0 else float("inf"))


def back_ratio(L, x, y):
    m = L.shape[0]
    if m == 0:
        return 0.0
    r = np.abs(L.T @ x - y).sum()
    den = m * np.abs(L).sum(axis=1).max() * np.abs(x).sum() * U         # ||L^T||_1 = ||L||_inf (xTRT02)
    return float(r / den) if den > 0 else (0.0 if r == 0 else float("inf"))


def end_to_end_ratio(x, xstar, kappa):
    if xstar.size == 0:
        return 0.0
    xs = np.asarray(xstar, np.longdouble)
    err = float(np.abs(np.asarray(x, np.longdouble) - xs).max())
    nx = float(np.abs(xs).max())
    if nx == 0:
        return 0.0 if err == 0 else float("inf")
    return err / (nx * kappa * U)


class SolverCheckError(AssertionError):
    def __init__(self, block, failed, ratios, tiles):
        self.block, self.failed, self.ratios, self.tiles = block, failed, ratios, tiles
        shown = {k: f"{v:.3g}" for k, v in ratios.items()}
        msg = f"block {block}: stage {failed[0]} fails (all failing: {', '.join(failed)}); ratios {shown}"
        if tiles:
            msg += "; worst tiles (row tile, panel step, rho): " + ", ".join(f"({I}, {J}, {r:.3g})" for I, J, r in tiles)
        super().__init__(msg)


def check_block(block, *, ms, c, z, sigma_lib=None, sigma_star=None, L=None, y=None, x=None, xstar=None, kappa=None,
                bars=BARS):
    """Every check whose inputs are given, for one block (z, y, x in block order: small SNPs, then large).  Returns
    {stage: ratio}; raises SolverCheckError naming the block, the first failing stage in solver order (sigma, factor,
    tiles, forward, back, end_to_end) and, if the factor fails, its five worst tiles."""
    z = np.asarray(z, np.float64)
    out, tiles = {}, []
    if sigma_lib is not None and sigma_star is not None:
        out["sigma"] = sigma_ratio(sigma_lib, sigma_star)
    if L is not None:
        K = k_matrix(np.asarray(sigma_lib, np.float64), ms, c)
        R = factor_residual(K, L)
        out["factor"] = factor_ratio(K, L, R)
        rho = tile_ratios(K, L, R)
        out["tiles"] = float(np.nanmax(rho)) if rho.size else 0.0
        if out["factor"] >= bars["factor"] or out["tiles"] >= bars["tiles"]:
            tiles = worst_tiles(rho)
        if y is not None:
            out["forward"] = forward_ratio(L, y, z)
        if x is not None and y is not None:
            out["back"] = back_ratio(L, np.asarray(x, np.float64), y)
    if x is not None and xstar is not None:
        out["end_to_end"] = end_to_end_ratio(x, xstar, kappa)
    failed = [s for s in STAGES if s in out and not out[s] < bars[s]]
    if failed:
        raise SolverCheckError(block, failed, out, tiles)
    return out
