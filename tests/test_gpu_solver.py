"""The block solver, stage by stage, against the extended-precision reference of tests/solver_ref.py.

Every scheduling mode of tests/test_gpu_modes.py runs on an EDGE workload: blocks at the panel (64), macro-tile (128) and
padding (8) edges, at the default size-class bounds (8 / 16 / 32 panels), on both sides of the switch between the
one-CTA and the cluster back substitution (m = 1024 / 1025), blocks without small SNPs, small/large borders on and next
to a panel edge, a duplicated .bed row and empty blocks; n_ref = 403 (a 101-byte pitch with padding samples), so above
m ~ 400 the pre-shrinkage part of Sigma is rank-deficient and lambda_min(Sigma) = 1 - tau, the worst tau = 0.8 allows.
Three folds put the ridge c at 1e-4, 1 and 1e3.  For every block the Sigma entries, the factor (normwise and per 64 x 64
tile), the forward and the back substitution and the end-to-end forward error are checked against their bars; a fold
of a multi-fold fit must equal the one-fold fit with its sigma_s bit for bit, and a NaN column must stay in its block.
"""
import os

import numpy as np
import pytest

from dbslmm_b200 import _abi, synth
from oracle import oracle as O

import parity_bars
import solver_ref as R
import test_gpu_modes as TM

pytestmark = pytest.mark.gpu

N_REF, TAU, N_OBS = 403, 0.8, 20_000
SIGMA_S = [5e-1, 5e-5, 5e-8]                       # c = 1e-4, 1, 1e3
EDGE_BLOCKS = ([(0, 0), (1, 1), (1, 0), (7, 7), (8, 0), (9, 4), (63, 63), (64, 0), (65, 64), (127, 63), (128, 128),
                (129, 65), (200, 199), (0, 0), (511, 448), (512, 512), (513, 0), (1024, 1023), (1025, 1024),
                (2048, 2047), (2049, 1985)] + [(300, 290)] * 6 + [(0, 0)])
DUP_BLOCK = 12                                      # (200, 199): one .bed row listed twice among its small SNPs


def make_edge_workload(seed, blocks, n_ref, missing_rate=0.0, dup=()):
    """Explicit CSR: block b has m rows of its own in the .bed, m - m_s of them (at random) are its large SNPs.  For a
    block in `dup`, its last small SNP reads the .bed row of its first one instead (the own row goes unused)."""
    rng = np.random.default_rng(seed)
    G = synth.make_genotypes(rng, [m for m, _ in blocks], n_ref, missing_rate=missing_rate)
    s_off, l_off = [0], [0]
    s_pos, l_pos, s_z, l_z = [], [], [], []
    row = 0
    for b, (m, ms) in enumerate(blocks):
        rows = np.arange(row, row + m)
        row += m
        large = np.zeros(m, bool)
        large[rng.choice(m, size=m - ms, replace=False)] = True
        sp, lp = rows[~large], rows[large]
        for k in dup:
            if k == b and sp.size >= 2:
                sp = sp.copy()
                sp[-1] = sp[0]
        s_pos.append(sp); l_pos.append(lp)
        s_z.append(1.3 * rng.standard_normal(ms))
        l_z.append(rng.choice([-1.0, 1.0], size=m - ms) * (6.0 + rng.exponential(2.0, size=m - ms)))
        s_off.append(s_off[-1] + ms); l_off.append(l_off[-1] + m - ms)
    cat = lambda xs, t: np.concatenate(xs).astype(t) if xs else np.zeros(0, t)
    return {"bed": synth.pack_bed(G), "n_ref": n_ref, "blocks": list(blocks),
            "s_off": np.asarray(s_off, np.int32), "s_pos": cat(s_pos, np.int32), "s_z": cat(s_z, np.float64),
            "l_off": np.asarray(l_off, np.int32), "l_pos": cat(l_pos, np.int32), "l_z": cat(l_z, np.float64)}


def csr(w, lmm=False):
    if not lmm:
        return (w["s_off"], w["s_pos"], w["s_z"], w["l_off"], w["l_pos"], w["l_z"])
    # LMM mode: every SNP of a block is a small one, in the same block order (small, then large)
    off = w["s_off"] + w["l_off"]
    pos = np.concatenate([np.concatenate([w["s_pos"][w["s_off"][b]:w["s_off"][b + 1]], w["l_pos"][w["l_off"][b]:w["l_off"][b + 1]]])
                          for b in range(len(w["blocks"]))]).astype(np.int32)
    z = np.concatenate([np.concatenate([w["s_z"][w["s_off"][b]:w["s_off"][b + 1]], w["l_z"][w["l_off"][b]:w["l_off"][b + 1]]])
                        for b in range(len(w["blocks"]))])
    return (off.astype(np.int32), pos, z)


def block_view(w, b, lmm=False):
    """(m, m_s, .bed rows, z) of block b in the solver's order."""
    so, lo = w["s_off"], w["l_off"]
    pos = np.concatenate([w["s_pos"][so[b]:so[b + 1]], w["l_pos"][lo[b]:lo[b + 1]]]).astype(np.int32)
    z = np.concatenate([w["s_z"][so[b]:so[b + 1]], w["l_z"][lo[b]:lo[b + 1]]])
    m = pos.size
    return m, (m if lmm else int(so[b + 1] - so[b])), pos, z


def x_hat(w, r, b, f, lmm=False):
    """beta * sqrt(N) of block b, fold f, in block order."""
    if lmm:
        o = w["s_off"] + w["l_off"]
        return r["beta_s"][f][o[b]:o[b + 1]] * np.sqrt(N_OBS)
    so, lo = w["s_off"], w["l_off"]
    return np.concatenate([r["beta_s"][f][so[b]:so[b + 1]], r["beta_l"][f][lo[b]:lo[b + 1]]]) * np.sqrt(N_OBS)


def reference(w, sigma_s, tau=TAU, lmm=False):
    """Sigma*, and x*, kappa per fold, of every block (independent of the scheduling mode)."""
    ref = []
    for b in range(len(w["blocks"])):
        m, ms, pos, z = block_view(w, b, lmm)
        sstar = R.exact_sigma(w["bed"], w["n_ref"], pos, tau)
        folds = [R.refined_solve(R.k_matrix(sstar, ms, R.ridge(s, N_OBS)), z) for s in sigma_s]
        ref.append({"m": m, "ms": ms, "z": z, "sstar": sstar, "folds": folds})
    return ref


@pytest.fixture(scope="module")
def edge():
    w = make_edge_workload(4031, EDGE_BLOCKS, N_REF, dup=(DUP_BLOCK,))
    assert w["blocks"][DUP_BLOCK] == (200, 199)
    return w, reference(w, SIGMA_S)


def engine_for(mode):
    saved = {k: os.environ.pop(k, None) for k in TM.KEYS}
    os.environ.update(TM.MODES[mode])
    try:
        return _abi.Engine(0)                                  # the switches are read at create
    finally:
        for k in TM.KEYS:
            os.environ.pop(k, None)
            if saved[k] is not None:
                os.environ[k] = saved[k]


class Maxima:
    def __init__(self):
        self.v = {}

    def add(self, ratios):
        for k, x in ratios.items():
            self.v[k] = max(self.v.get(k, 0.0), x)

    def record(self, prefix):
        for k, x in self.v.items():
            parity_bars.record(f"{prefix}/{k}", x)


def end_to_end(w, ref, r, folds, mx, lmm=False, what=""):
    for b, rb in enumerate(ref):
        if rb["m"] == 0:
            continue
        for f in folds:
            xstar, kappa = rb["folds"][f]
            mx.add(R.check_block(f"{b} (m={rb['m']}, fold {f}{what})", ms=rb["ms"], c=R.ridge(SIGMA_S[f], N_OBS),
                                 z=rb["z"], x=x_hat(w, r, b, f, lmm), xstar=xstar, kappa=kappa))


def stage_checks(eng, w, ref, r, f, f_ref, mx, lmm=False, sigma_s=SIGMA_S, what=""):
    """All stages of every block, from the LAST fold of the last fit (r), which used sigma_s[f_ref]; r's fold f."""
    for b, rb in enumerate(ref):
        m = rb["m"]
        if m == 0:
            continue
        L, y = eng.block_factor(b, m)
        xstar, kappa = rb["folds"][f_ref]
        mx.add(R.check_block(f"{b} (m={m}, m_s={rb['ms']}, fold {f_ref}{what})", ms=rb["ms"], c=R.ridge(sigma_s[f_ref], N_OBS),
                             z=rb["z"], sigma_lib=eng.block_sigma(b, m), sigma_star=rb["sstar"], L=L, y=y,
                             x=x_hat(w, r, b, f, lmm), xstar=xstar, kappa=kappa))


def same_bits(a, b):
    return all(np.array_equal(a[k], b[k]) for k in ("beta_s", "beta_l") if a[k] is not None)


MODES = list(TM.MODES)


@pytest.mark.parametrize("mode", MODES)
def test_every_mode_every_block_every_stage(edge, mode):
    w, ref = edge
    eng = engine_for(mode)
    mx = Maxima()
    try:
        eng.load_bed(w["bed"], N_REF)
        r3 = eng.fit(*csr(w), sigma_s=SIGMA_S, n_obs=N_OBS)
        assert r3["n_bad"] == 0 and not r3["status"].any()
        end_to_end(w, ref, r3, range(3), mx)
        for f, s in enumerate(SIGMA_S):
            r1 = eng.fit(*csr(w), sigma_s=[s], n_obs=N_OBS)
            assert r1["n_bad"] == 0
            stage_checks(eng, w, ref, r1, 0, f, mx)
            # the plan does not depend on n_folds: a difference here is state carried from fold to fold
            # (split-K counters, deferred-diagonal flags, the parity of the W buffer)
            assert np.array_equal(r1["beta_s"][0], r3["beta_s"][f]) and np.array_equal(r1["beta_l"][0], r3["beta_l"][f]), \
                f"fold {f} of the 3-fold fit differs from the 1-fold fit with sigma_s = {s}"
        # streaming: its bulk is ONE batch (size classes 0 and 1 together) where the resident fit has one per class, so
        # the batches -- and with them the split-K groups and the step launches -- need not coincide: 1e-12 per block,
        # not bit equality
        rs = eng.fit(*csr(w), sigma_s=SIGMA_S, n_obs=N_OBS, bed=w["bed"], n_ref=N_REF)
        assert rs["n_bad"] == 0
        end_to_end(w, ref, rs, range(3), mx, what=", streaming")
        for b, rb in enumerate(ref):
            for f in range(3):
                a, e = x_hat(w, rs, b, f), x_hat(w, r3, b, f)
                if a.size:
                    assert np.abs(a - e).max() <= 1e-12 * np.abs(e).max(), (b, f)
        r3b = eng.fit(*csr(w), sigma_s=SIGMA_S, n_obs=N_OBS)
        assert same_bits(r3b, r3), "a second resident fit is not bit-identical"
    finally:
        eng.close()
    mx.record(f"solver/{mode}")


NAN_SNPS = [(20, 700), (18, 1023), (8, 64)]          # (block, SNP in block order): see the test


@pytest.mark.parametrize("mode", MODES)
def test_nan_column_stays_in_its_block(edge, mode):
    """Monomorphic .bed rows (legal input; the reference poisons the whole block the same way) of: column 700 of the
    (2049, 1985) block -- panel 10, a split-K class; the last small SNP (1023) of the (1025, 1024) block -- its own
    partial panel; the one large SNP of the (65, 64) block.  Exactly those blocks are flagged NOT_SPD, none SYNC_TIMEOUT,
    and every other block is bit-identical to the fit of the clean panel."""
    w, _ = edge
    bad = sorted(b for b, _ in NAN_SNPS)
    bed = w["bed"].copy()
    for b, j in NAN_SNPS:
        assert w["blocks"][b][0] > j
        _, _, pos, _ = block_view(w, b)
        bed[pos[j]] = 0xFF                                  # every sample homozygous: allele count 0 ...
        bed[pos[j], -1] = 0x3F                              # ... and the padding slot of the last byte 00, as PLINK writes
    eng = engine_for(mode)
    try:
        eng.load_bed(w["bed"], N_REF)
        clean = eng.fit(*csr(w), sigma_s=SIGMA_S, n_obs=N_OBS)
        eng.load_bed(bed, N_REF)
        r = eng.fit(*csr(w), sigma_s=SIGMA_S, n_obs=N_OBS)
    finally:
        eng.close()
    assert not (r["status"] & 4).any(), f"SYNC_TIMEOUT in blocks {np.flatnonzero(r['status'] & 4)}"
    assert sorted(np.flatnonzero(r["status"] & 1).tolist()) == bad
    assert r["n_bad"] == len(bad)
    for b in range(len(w["blocks"])):
        for f in range(3):
            x, e = x_hat(w, r, b, f), x_hat(w, clean, b, f)
            if b in bad:
                assert not np.isfinite(x).all(), (b, f)
            else:
                assert np.array_equal(x, e), (b, f)


def test_harder_conditioning():
    """tau = 0.98 (lambda_min(Sigma) = 0.02), n_ref = 150, two duplicated rows: all stages, and the exact oracle (an FP64
    Cholesky of its float-path Sigma) passes the same end-to-end bar."""
    blocks = [(600, 0), (1100, 550), (300, 300)]
    w = make_edge_workload(98, blocks, 150)
    # two SNPs of the (600, 0) block read the .bed rows of two others
    lp = w["l_pos"]
    lp[10], lp[400] = lp[11], lp[401]
    sig = [0.5]                                                       # c = 1e-4
    ref = reference(w, sig, tau=0.98)
    eng = _abi.Engine(0)
    mx = Maxima()
    try:
        eng.load_bed(w["bed"], 150)
        r = eng.fit(*csr(w), sigma_s=sig, n_obs=N_OBS, tau=0.98)
        assert r["n_bad"] == 0
        stage_checks(eng, w, ref, r, 0, 0, mx, sigma_s=sig)
    finally:
        eng.close()
    bs, bl, sing, _ = O.est(w["bed"], 150, N_OBS, sig[0], *csr(w), threads=8, mode=O.MODE_EXACT, tau=0.98)
    assert sing == 0
    orc = {"beta_s": bs[None], "beta_l": bl[None]}
    for b, rb in enumerate(ref):
        xstar, kappa = rb["folds"][0]
        parity_bars.record(f"solver/harder_conditioning/kappa_inf_block{b}", kappa)
        if rb["ms"] == 0:
            # the oracle, like the reference's block loop, leaves a block without small SNPs unsolved (betas 0); the
            # library solves K = Sigma there, which the stage checks above cover
            assert not x_hat(w, orc, b, 0).any()
            continue
        mx.add({"oracle_end_to_end": R.end_to_end_ratio(x_hat(w, orc, b, 0), xstar, kappa)})
        R.check_block(f"{b} (exact oracle)", ms=rb["ms"], c=R.ridge(sig[0], N_OBS), z=rb["z"], x=x_hat(w, orc, b, 0),
                      xstar=xstar, kappa=kappa)
    mx.record("solver/harder_conditioning")


def test_missing_calls_resident_and_streaming():
    """The four-plane Gram (its numerator through the fma chain) under every check, the Sigma ulps included."""
    w = make_edge_workload(4032, EDGE_BLOCKS, N_REF, missing_rate=0.01, dup=(DUP_BLOCK,))
    ref = reference(w, SIGMA_S)
    eng = _abi.Engine(0)
    mx = Maxima()
    try:
        eng.load_bed(w["bed"], N_REF)
        r3 = eng.fit(*csr(w), sigma_s=SIGMA_S, n_obs=N_OBS)
        assert r3["n_bad"] == 0 and r3["timing"]["n_blocks_missing"] > 0
        end_to_end(w, ref, r3, range(3), mx)
        for f, s in enumerate(SIGMA_S):
            r1 = eng.fit(*csr(w), sigma_s=[s], n_obs=N_OBS)
            stage_checks(eng, w, ref, r1, 0, f, mx)
        rs = eng.fit(*csr(w), sigma_s=SIGMA_S, n_obs=N_OBS, bed=w["bed"], n_ref=N_REF)
        assert rs["n_bad"] == 0
        end_to_end(w, ref, rs, range(3), mx, what=", streaming")
        stage_checks(eng, w, ref, rs, 2, 2, mx, what=", streaming")
    finally:
        eng.close()
    mx.record("solver/missing_calls")


def test_lmm_mode():
    w = make_edge_workload(4031, EDGE_BLOCKS, N_REF, dup=(DUP_BLOCK,))
    ref = reference(w, SIGMA_S, lmm=True)
    eng = _abi.Engine(0)
    mx = Maxima()
    try:
        eng.load_bed(w["bed"], N_REF)
        r3 = eng.fit(*csr(w, lmm=True), sigma_s=SIGMA_S, n_obs=N_OBS)
        assert r3["n_bad"] == 0
        end_to_end(w, ref, r3, range(3), mx, lmm=True)
        for f, s in enumerate(SIGMA_S):
            r1 = eng.fit(*csr(w, lmm=True), sigma_s=[s], n_obs=N_OBS)
            stage_checks(eng, w, ref, r1, 0, f, mx, lmm=True)
    finally:
        eng.close()
    mx.record("solver/lmm")


def test_block_factor_refuses_after_a_quadform_fit(edge):
    w, _ = edge
    eng = _abi.Engine(0)
    try:
        eng.load_bed(w["bed"], N_REF)
        eng.fit(*csr(w), sigma_s=SIGMA_S[:1], n_obs=N_OBS)
        L, y = eng.block_factor(1, 1)
        assert L.shape == (1, 1) and L[0, 0] > 0 and y.shape == (1,)
        eng.quadform(w["s_off"], w["s_pos"], w["s_z"])
        with pytest.raises(_abi.EngineError):
            eng.block_factor(1, 1)
    finally:
        eng.close()
