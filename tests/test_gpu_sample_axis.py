"""The correlation builder along the sample axis, from 2 to 409,344 individuals (the decoder's limit), against the
extended-precision reference of tests/solver_ref.py.

The decoder stages whole .bed rows in shared memory, so its ring of staging buffers and its warps per CTA change with the
row length (decode.cu: stage_bytes, stage_warps):
    n_ref <= 25,412      4 buffers x 8 warps        102,213 .. 204,612   2 x 2
    25,413 .. 51,012     2 x 8                      204,613 .. 409,344   2 x 1
    51,013 .. 102,212    2 x 4
snp_stats_kernel (always 2 buffers) and pack_rows_kernel switch at the same points.  The four-plane epilogue's numerator
n_i n_j Q - n_i S_j A_ij - n_j S_i A_ji + S_i S_j N has terms up to 4 n^3, past 2^53 above n = 2^17 = 131,072.

Every case has one block of each size around the four-plane tiles (64 x 128) and the one-plane tiles (128 x 128), at least
a quarter of the SNPs count the major allele (large Q entries), and with missing calls one block has none, so both Gram
kernels run in one fit.  Checked: per-SNP counts and maf, the decoder's code and mask rows with their zero padding, the
integer planes bit for bit, Sigma entry by entry within 16 ulps (with and without the debug planes, which select another
epilogue path in the one-plane kernel), the end-to-end forward error, and streaming betas bit-identical to resident ones.
"""
import functools
import os
from fractions import Fraction

import numpy as np
import pytest

from dbslmm_b200 import _abi
from oracle import oracle as O

import parity_bars
import solver_ref as R

pytestmark = pytest.mark.gpu

TAU, N_OBS, SIGMA_S = 0.8, 20_000, [5e-5]
MAX_N = 409_344
BLOCKS = [1, 63, 65, 129, 200]
CLEAN_BLOCK = 2                                    # never has a missing call
N_GRID = [2, 3, 4, 5, 127, 128, 129, 403, 25_412, 25_413, 51_012, 51_013, 102_212, 102_213, 131_072, 131_073,
          204_612, 204_613, MAX_N]
_LUT = np.array([3, 2, 0, 1], np.uint8)            # allele count & 3 (missing = -1 -> 3) -> PLINK 2-bit code


def pack_bed(G):
    """synth.pack_bed without its int64 temporaries (panels here reach 190 M genotypes)."""
    m, n = G.shape
    pitch = (n + 3) // 4
    c = np.zeros((m, pitch * 4), np.uint8)
    c[:, :n] = _LUT[G.view(np.uint8) & 3]
    c = c.reshape(m, pitch, 4)
    return c[:, :, 0] | (c[:, :, 1] << 2) | (c[:, :, 2] << 4) | (c[:, :, 3] << 6)


def make_genotypes(rng, blocks, n, missing, clean=(), flip_frac=0.34):
    """int8 [sum(blocks), n] (-1 = missing): binomial rows with A1 frequency ~ U(0.05, 0.5), each row after the first of a
    block copying half its samples from the row before (LD); a third of the rows flipped (g -> 2 - g: A1 the major allele);
    missing calls at `missing` except in the blocks `clean`.  A row monomorphic among its calls is redrawn."""
    m = int(sum(blocks))
    G = np.empty((m, n), np.int8)
    flip = np.zeros(m, bool)
    flip[rng.choice(m, size=int(np.ceil(flip_frac * m)), replace=False)] = True
    starts = set(np.cumsum([0] + list(blocks))[:-1].tolist())
    ends = np.cumsum(blocks)
    for j in range(m):
        b = int(np.searchsorted(ends, j, side="right"))
        miss = 0.0 if b in clean else missing
        p = np.float32(rng.uniform(0.05, 0.5))
        for attempt in range(1000):
            g = (rng.random(n, dtype=np.float32) < p).astype(np.int8) + (rng.random(n, dtype=np.float32) < p)
            if j not in starts and attempt == 0:
                keep = rng.random(n, dtype=np.float32) < 0.5
                prev = np.where(G[j - 1] < 0, g, 2 - G[j - 1] if flip[j - 1] else G[j - 1])
                g = np.where(keep, prev, g).astype(np.int8)
            if flip[j]:
                g = (2 - g).astype(np.int8)
            if miss > 0:
                g = np.where(rng.random(n, dtype=np.float32) < miss, np.int8(-1), g)
            calls = g[g >= 0]
            if calls.size and calls.min() != calls.max():
                break
            p = np.float32(0.5)
        else:
            raise RuntimeError("no polymorphic row drawn")
        G[j] = g
    return G, flip


def make_csr(rng, blocks):
    """Explicit CSR over consecutive .bed rows: about one SNP in twenty of a block (at random) is a large one."""
    s_off, l_off, s_pos, l_pos = [0], [0], [], []
    row = 0
    for m in blocks:
        rows = np.arange(row, row + m)
        row += m
        large = np.zeros(m, bool)
        large[rng.choice(m, size=m // 20, replace=False)] = True
        s_pos.append(rows[~large]); l_pos.append(rows[large])
        s_off.append(s_off[-1] + int((~large).sum())); l_off.append(l_off[-1] + int(large.sum()))
    s_pos, l_pos = np.concatenate(s_pos).astype(np.int32), np.concatenate(l_pos).astype(np.int32)
    s_z = 1.3 * rng.standard_normal(s_pos.size)
    l_z = rng.choice([-1.0, 1.0], size=l_pos.size) * (6.0 + rng.exponential(2.0, size=l_pos.size))
    return (np.asarray(s_off, np.int32), s_pos, s_z, np.asarray(l_off, np.int32), l_pos, l_z)


@functools.lru_cache(maxsize=2)
def panel(n, missing, blocks=tuple(BLOCKS), seed=0):
    rng = np.random.default_rng(seed * 1_000_003 + n * 7 + int(missing * 1000))
    G, flip = make_genotypes(rng, blocks, n, missing, clean=(CLEAN_BLOCK,) if missing > 0 else ())
    return {"G": G, "bed": pack_bed(G), "n": n, "blocks": list(blocks), "csr": make_csr(rng, blocks), "flip": flip}


def exact_maf(G):
    """min(f, 1 - f) of f = S / (2 n_i), the mean-imputed allele frequency, rounded once from the exact rational."""
    S, ni = np.maximum(G, 0).sum(axis=1, dtype=np.int64), (G >= 0).sum(axis=1)
    return np.array([float(min(Fraction(int(s), 2 * int(k)), 1 - Fraction(int(s), 2 * int(k)))) for s, k in zip(S, ni)])


def block_pos(csr, b):
    s_off, s_pos, s_z, l_off, l_pos, l_z = csr
    return (np.concatenate([s_pos[s_off[b]:s_off[b + 1]], l_pos[l_off[b]:l_off[b + 1]]]).astype(np.int32),
            np.concatenate([s_z[s_off[b]:s_off[b + 1]], l_z[l_off[b]:l_off[b + 1]]]), int(s_off[b + 1] - s_off[b]))


def x_hat(csr, r, b):
    s_off, _, _, l_off, _, _ = csr
    return np.concatenate([r["beta_s"][0][s_off[b]:s_off[b + 1]], r["beta_l"][0][l_off[b]:l_off[b + 1]]]) * np.sqrt(N_OBS)


def reference(p, tau=TAU):
    """Per block: its rows, z, m_s, the integer planes (BLAS), Sigma* and x*, kappa."""
    out = []
    for b in range(len(p["blocks"])):
        pos, z, ms = block_pos(p["csr"], b)
        planes = R.gram_planes(p["G"][pos])
        sstar = R.sigma_from_planes(*planes, p["n"], tau)
        xstar, kappa = R.refined_solve(R.k_matrix(sstar, ms, R.ridge(SIGMA_S[0], N_OBS)), z)
        out.append({"pos": pos, "z": z, "ms": ms, "planes": planes, "sstar": sstar, "xstar": xstar, "kappa": kappa,
                    "missing": bool((p["G"][pos] < 0).any())})
    return out


class Maxima:
    def __init__(self):
        self.v = {}

    def add(self, ratios):
        for k, x in ratios.items():
            self.v[k] = max(self.v.get(k, 0.0), x)

    def record(self, prefix):
        for k, x in self.v.items():
            parity_bars.record(f"{prefix}/{k}", x)


def check_fit(eng, p, ref, r, what, mx, planes=False, codes=False):
    """Sigma of every block within 16 ulps and the end-to-end ratio below 30 -- all blocks first, so a failure lists every
    block's ratios -- then, on request, the integer planes and the decoder's rows."""
    n, G = p["n"], p["G"]
    n_pad = (n + 127) // 128 * 128
    assert r["n_bad"] == 0 and not r["status"].any(), (what, r["status"])
    assert r["timing"]["n_blocks_missing"] == sum(rb["missing"] for rb in ref), what
    ratios, failed = [], []
    for b, rb in enumerate(ref):
        m = rb["pos"].size
        try:
            rt = R.check_block(b, ms=rb["ms"], c=R.ridge(SIGMA_S[0], N_OBS), z=rb["z"], sigma_lib=eng.block_sigma(b, m),
                               sigma_star=rb["sstar"], x=x_hat(p["csr"], r, b), xstar=rb["xstar"], kappa=rb["kappa"])
        except R.SolverCheckError as e:
            rt = e.ratios
            failed.append(b)
        ratios.append(rt)
        mx.add({f"{k}_{'missing' if rb['missing'] else 'plain'}": v for k, v in rt.items()})
    shown = ", ".join(f"block {b} (m={rb['pos'].size}, {'missing' if rb['missing'] else 'no missing'}): "
                      f"sigma {rt['sigma']:.3g} end_to_end {rt['end_to_end']:.3g}" for b, (rb, rt) in enumerate(zip(ref, ratios)))
    assert not failed, f"{what}, n = {n}: blocks {failed} fail; {shown}"
    for b, rb in enumerate(ref):
        m = rb["pos"].size
        if planes:
            Q, A, N = eng.block_gram(b, m)
            Qo, Ao, No = rb["planes"]
            assert np.array_equal(Q, Qo) and np.array_equal(A, Ao) and np.array_equal(N, No), (what, n, b)
        if codes:
            for j in sorted({0, m // 2, m - 1}):
                g = G[rb["pos"][j]]
                c, k = eng.row_codes(b, j, n_pad), eng.row_codes(b, j, n_pad, plane=1)
                assert np.array_equal(c[:n], np.maximum(g, 0)) and not c[n:].any(), (what, n, b, j)
                assert np.array_equal(k[:n], (g >= 0).astype(np.int8)) and not k[n:].any(), (what, n, b, j)


@pytest.fixture(scope="module")
def eng():
    e = _abi.Engine(0)
    yield e
    e.close()


_MX = Maxima()


@pytest.mark.parametrize("missing", [0.0, 0.01])
@pytest.mark.parametrize("n", N_GRID)
def test_sample_axis(eng, n, missing):
    p = panel(n, missing)
    assert p["flip"].mean() >= 0.25
    ref = reference(p)
    csr = p["csr"]
    eng.load_bed(p["bed"], n)
    maf, nn = eng.snp_stats()
    assert np.array_equal(nn, (p["G"] >= 0).sum(axis=1))
    assert np.abs(maf - exact_maf(p["G"])).max() <= 1e-15
    # the oracle restates readSNPIm: a running FP64 sum over the n mean-imputed genotypes, whose own rounding grows with n
    assert np.abs(maf - O.snp_maf(p["bed"], p["G"].shape[0], n)).max() <= 1e-15 + n * 2.0 ** -52
    r = eng.fit(*csr, sigma_s=SIGMA_S, n_obs=N_OBS, flags=_abi.FLAG_KEEP_INT_GRAM)
    check_fit(eng, p, ref, r, "resident, debug planes", _MX, planes=True, codes=True)
    res = eng.fit(*csr, sigma_s=SIGMA_S, n_obs=N_OBS)
    check_fit(eng, p, ref, res, "resident", _MX)
    r = eng.fit(*csr, sigma_s=SIGMA_S, n_obs=N_OBS, flags=_abi.FLAG_KEEP_INT_GRAM, bed=p["bed"], n_ref=n)
    check_fit(eng, p, ref, r, "streaming, debug planes", _MX, planes=True, codes=True)
    st = eng.fit(*csr, sigma_s=SIGMA_S, n_obs=N_OBS, bed=p["bed"], n_ref=n)
    check_fit(eng, p, ref, st, "streaming", _MX)
    # every block is in size class 0, so the streaming batch is the resident one: the same launches, the same bits
    assert np.array_equal(st["beta_s"], res["beta_s"]) and np.array_equal(st["beta_l"], res["beta_l"])
    _MX.record("sample_axis/grid")


def test_above_the_limit_is_refused_and_the_handle_still_fits(eng):
    G, _ = make_genotypes(np.random.default_rng(5), [3], MAX_N + 1, 0.0)
    bed = pack_bed(G)
    off, pos, z = np.array([0, 3], np.int32), np.arange(3, dtype=np.int32), np.ones(3)
    with pytest.raises(_abi.EngineError, match=str(MAX_N)):
        eng.load_bed(bed, MAX_N + 1)
    with pytest.raises(_abi.EngineError, match=str(MAX_N)):
        eng.fit(off, pos, z, sigma_s=SIGMA_S, n_obs=N_OBS, bed=bed, n_ref=MAX_N + 1)
    p = panel(403, 0.01)
    ref = reference(p)
    eng.load_bed(p["bed"], 403)
    r = eng.fit(*p["csr"], sigma_s=SIGMA_S, n_obs=N_OBS, flags=_abi.FLAG_KEEP_INT_GRAM)
    check_fit(eng, p, ref, r, "after the refusals", Maxima(), planes=True, codes=True)


def test_changing_panel_width_on_one_handle():
    """403 -> 400 -> 403 individuals (both n_pad = 512) with missing calls in only some rows of a block: the mask rows of
    the rows without missing calls must follow the panel width (the decoder's dirty map is reset when it changes)."""
    e = _abi.Engine(0)
    mx = Maxima()
    try:
        for n in (403, 400, 403):
            p = panel(n, 0.002, blocks=(64, 129), seed=1)
            ref = reference(p)
            some = [(p["G"][rb["pos"]] < 0).any(axis=1) for rb in ref]
            assert any(s.any() and not s.all() for s in some)
            e.load_bed(p["bed"], n)
            r = e.fit(*p["csr"], sigma_s=SIGMA_S, n_obs=N_OBS, flags=_abi.FLAG_KEEP_INT_GRAM)
            check_fit(e, p, ref, r, f"width {n}", mx, planes=True, codes=True)
    finally:
        e.close()


def test_changing_block_layout_on_one_handle():
    """Same width, other block layouts: a code row that held a mask in one fit and a genotype row in the next must not be
    taken for a default mask row in a third fit whose block has missing calls in other rows only."""
    n = 403
    rng = np.random.default_rng(11)
    G, _ = make_genotypes(rng, [128, 64], n, 0.0)
    some = rng.random(64) < 0.5                                    # rows 128 .. 191: missing calls in about half of them
    G[128:][some] = np.where(rng.random((int(some.sum()), n)) < 0.01, np.int8(-1), G[128:][some])
    calls_ok = [(lambda c: c.size and c.min() != c.max())(g[g >= 0]) for g in G]
    assert all(calls_ok) and (G[128:] < 0).any(axis=1).any() and not (G[128:] < 0).any(axis=1).all()
    bed = pack_bed(G)
    e = _abi.Engine(0)
    mx = Maxima()
    try:
        e.load_bed(bed, n)
        # fit 1 sizes the code buffer; fit 2 writes default mask rows 64 .. 127; fit 3 writes genotypes over them;
        # fit 4 has its mask rows there again
        for rows in (np.arange(192), np.arange(64), np.arange(128), np.arange(128, 192)):
            off, z = np.array([0, rows.size], np.int32), np.random.default_rng(rows.size).standard_normal(rows.size)
            r = e.fit(off, rows.astype(np.int32), z, sigma_s=SIGMA_S, n_obs=N_OBS, flags=_abi.FLAG_KEEP_INT_GRAM)
            assert r["n_bad"] == 0
            Q, A, N = e.block_gram(0, rows.size)
            Qo, Ao, No = R.gram_planes(G[rows])
            assert np.array_equal(Q, Qo) and np.array_equal(A, Ao) and np.array_equal(N, No), rows[0]
            k = np.stack([e.row_codes(0, j, 512, plane=1)[:n] for j in range(rows.size)])
            assert np.array_equal(k, (G[rows] >= 0).astype(np.int8)), rows[0]
            s = R.sigma_ratio(e.block_sigma(0, rows.size), R.sigma_from_planes(Qo, Ao, No, n, TAU))
            mx.add({"sigma": s})
            assert s <= R.BARS["sigma"], (rows[0], s)
    finally:
        e.close()


def test_valid_quadform_at_max_n_ref(eng):
    """z^T Sigma z per block (tau = 1, the `valid` tool's deno) at 409,344 individuals with missing calls, against the
    componentwise bound |q - q*| <= (16 + m) u |z|^T |Sigma*| |z|, q* in extended precision."""
    p = panel(MAX_N, 0.01)
    eng.load_bed(p["bed"], MAX_N)
    s_off, s_pos, s_z, l_off, l_pos, l_z = p["csr"]
    off = (s_off + l_off).astype(np.int32)
    pos = np.concatenate([block_pos(p["csr"], b)[0] for b in range(len(p["blocks"]))])
    z = np.concatenate([block_pos(p["csr"], b)[1] for b in range(len(p["blocks"]))])
    q = eng.quadform(off, pos, z)
    worst = 0.0
    for b in range(len(p["blocks"])):
        bp, bz, _ = block_pos(p["csr"], b)
        S = R.sigma_from_planes(*R.gram_planes(p["G"][bp]), MAX_N, 1.0)
        zl = bz.astype(np.longdouble)
        qstar = zl @ S @ zl
        bound = (16 + bp.size) * R.U * (np.abs(zl) @ np.abs(S) @ np.abs(zl))
        ratio = float(abs(np.longdouble(q[b]) - qstar) / bound)
        worst = max(worst, ratio)
        assert ratio <= 1.0, (b, ratio)
    parity_bars.record("sample_axis/quadform_max_n/err_over_bound", worst)


@pytest.mark.parametrize("variant", ["packed", "pair"])
def test_gram_variants_with_two_staging_buffers(variant):
    """DBSLMM_B200_GRAM=packed and =pair at 60,000 individuals (2 staging buffers x 4 warps: pack_rows_kernel<2>)."""
    n = 60_000
    p = panel(n, 0.01)
    ref = reference(p)
    os.environ["DBSLMM_B200_GRAM"] = variant
    try:
        e = _abi.Engine(0)
    finally:
        os.environ.pop("DBSLMM_B200_GRAM", None)
    mx = Maxima()
    try:
        e.load_bed(p["bed"], n)
        r = e.fit(*p["csr"], sigma_s=SIGMA_S, n_obs=N_OBS, flags=_abi.FLAG_KEEP_INT_GRAM)
        check_fit(e, p, ref, r, variant + ", debug planes", mx, planes=True)
        r = e.fit(*p["csr"], sigma_s=SIGMA_S, n_obs=N_OBS)
        check_fit(e, p, ref, r, variant, mx)
        r = e.fit(*p["csr"], sigma_s=SIGMA_S, n_obs=N_OBS, flags=_abi.FLAG_KEEP_INT_GRAM, bed=p["bed"], n_ref=n)
        check_fit(e, p, ref, r, variant + ", streaming", mx, planes=True)
    finally:
        e.close()
    mx.record(f"sample_axis/gram_{variant}")
