"""Every scheduling mode of the block solver must give the same betas (they only differ in which CTA factors a diagonal
tile when, how K is sliced, and how launches depend on each other); and the genome-wide workload -- the only one big
enough to take the 'diagonal tile factored by macro tile 0 at the END of a multi-wave step' path by default -- is checked
through the residual of K x = z on sampled blocks."""
import os

import numpy as np
import pytest

from dbslmm_b200 import _abi, synth
from oracle import oracle as O

import solver_ref as R

pytestmark = pytest.mark.gpu

MODES = {
    "default": {},
    "diag_at_end_of_step": {"DBSLMM_B200_DEFER_CTAS": "0"},           # every diagonal tile fused into the previous step
    "diag_first_in_step": {"DBSLMM_B200_DEFER_CTAS": "1000000"},      # every diagonal tile deferred to its own step
    "separate_diag_launches": {"DBSLMM_B200_FUSE_DIAG": "0"},
    "no_split_k": {"DBSLMM_B200_SPLITK": "1,1"},
    "deep_split_k": {"DBSLMM_B200_SPLITK": "32,1"},
    "programmatic_dependent_launch": {"DBSLMM_B200_PDL": "0.000001"},
    "seven_size_classes": {"DBSLMM_B200_CLASSES": "2,4,8,12,16,24"},
    # the panel step kernel: TMA/mbarrier pipeline (default) with several items per CTA, one item per CTA, plain 2-D
    # tensor maps (no row permutation), and the cp.async kernel of round 1
    "tma_many_items_per_cta": {"DBSLMM_B200_TPC": "8,0"},
    "tma_three_items_per_cta_diag_first": {"DBSLMM_B200_TPC": "3,0", "DBSLMM_B200_DEFER_CTAS": "1000000"},
    "tma_one_item_per_cta": {"DBSLMM_B200_TPC": "1"},
    "tma_plain_2d_tensor_maps": {"DBSLMM_B200_TMAP_PERM": "0", "DBSLMM_B200_TPC": "2,0"},
    "legacy_cp_async_panel_kernel": {"DBSLMM_B200_PANEL": "legacy"},
    # macro-tile height of the TMA panel kernel: 64 rows / 128-thread CTAs everywhere (default), only for the bulk
    # batches, or 128 rows / 256-thread CTAs everywhere; with the L2 tensor prefetch on
    "tile64_bulk_only": {"DBSLMM_B200_TILE64": "1"},
    "tile128_everywhere_many_items_per_cta": {"DBSLMM_B200_TILE64": "0", "DBSLMM_B200_TPC": "8,0"},
    "tile128_diag_at_end_of_step": {"DBSLMM_B200_TILE64": "0", "DBSLMM_B200_DEFER_CTAS": "0"},
    "tile64_l2_prefetch": {"DBSLMM_B200_L2_PF": "3"},
    # the correlation builder of blocks without missing calls: the int8-row kernel fed by the decoder (default) or the
    # experimental fused unpack + Gram from packed 2-bit rows
    "fused_unpack_gram_from_packed_rows": {"DBSLMM_B200_GRAM": "packed"},
    # ... or by CTA pairs (tcgen05 cta_group::2, 256 x 256 super tiles as two N = 128 MMAs), with and without the L2 hints
    "gram_by_cta_pairs": {"DBSLMM_B200_GRAM": "pair"},
    "gram_by_cta_pairs_l2_hints": {"DBSLMM_B200_GRAM": "pair", "DBSLMM_B200_GRAM_HINT": "3"},
    "gram_single_cta_l2_hints": {"DBSLMM_B200_GRAM": "single", "DBSLMM_B200_GRAM_HINT": "3"},
    # the panel kernel without the next item's first chunk issued during the epilogue
    "no_next_item_prefetch": {"DBSLMM_B200_NEXT_PF": "0", "DBSLMM_B200_TPC": "8,0"},
    # the cluster back substitution (chosen per batch from its largest block) on blocks of 5-16 panels, and on every
    # block, 1-SNP and empty ones included
    "cluster_backsolve_on_bulk_sizes": {"DBSLMM_B200_CLASSES": "4,20"},
    "one_size_class": {"DBSLMM_B200_CLASSES": "40"},
}
KEYS = sorted({k for m in MODES.values() for k in m})


def relmax(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


@pytest.fixture(scope="module")
def problem():
    sizes = [520, 40, 1100, 70, 2100, 600, 9, 700, 0, 1300]
    w = synth.make_workload(2024, sizes, 500, missing_rate=0.0, frac_large=0.02)
    csr = (w["s_off"], w["s_pos"], w["s_z"], w["l_off"], w["l_pos"], w["l_z"])
    bs, bl, _, _ = O.est(w["bed"], 500, 20_000, 2e-4, *csr, threads=8, mode=O.MODE_EXACT)
    return w, csr, bs, bl


@pytest.mark.parametrize("mode", list(MODES))
def test_solver_modes_agree_with_the_oracle(problem, mode):
    w, csr, bs, bl = problem
    saved = {k: os.environ.pop(k, None) for k in KEYS}
    os.environ.update(MODES[mode])
    try:
        eng = _abi.Engine(0)                                      # the switches are read at create
    finally:
        for k in KEYS:
            os.environ.pop(k, None)
            if saved[k] is not None:
                os.environ[k] = saved[k]
    try:
        eng.load_bed(w["bed"], 500)
        r = eng.fit(*csr, sigma_s=[2e-4], n_obs=20_000)
        assert r["n_bad"] == 0
        assert relmax(r["beta_s"][0], bs) <= 1e-10 and relmax(r["beta_l"][0], bl) <= 1e-10
        rs = eng.fit(*csr, sigma_s=[2e-4], n_obs=20_000, bed=w["bed"], n_ref=500)
        assert relmax(rs["beta_s"][0], bs) <= 1e-10 and relmax(rs["beta_l"][0], bl) <= 1e-10
    finally:
        eng.close()


def test_genome_wide_residuals_and_streaming_equality(engine):
    """BASELINE.json configs[2] at full size (1,703 blocks, 1.1 M SNPs, n_ref 2,000): K x = z residual from the library's
    own Sigma and every stage check of tests/solver_ref.py on sampled blocks (largest, smallest, spread), all block
    statuses clean, streaming fit == resident fit."""
    from test_gpu_solver import Maxima
    torch = pytest.importorskip("torch")
    import bench
    import argparse
    ns = argparse.Namespace(config="c3", missing=0.0, seed=20240003)
    dev = torch.device("cuda", 0)
    w = bench.build_workload(ns, torch, dev, ns.seed)
    sz = w["z"][w["s_pos"]]
    lz = w["z"][w["l_pos"]]
    csr = (w["s_off"], w["s_pos"], sz, w["l_off"], w["l_pos"], lz)
    sig, n_obs = 0.5 / w["nsnp_total"], w["n_obs"]
    engine.load_bed(w["bed"], w["n_ref"])
    r = engine.fit(*csr, sigma_s=[sig], n_obs=n_obs, flags=_abi.FLAG_FULL_SIGMA)
    assert r["n_bad"] == 0 and np.isfinite(r["beta_s"]).all() and np.isfinite(r["beta_l"]).all()
    sizes = w["sizes"]
    order = np.argsort(sizes)
    sample = sorted(set(order[:3].tolist() + order[-4:].tolist() + order[:: max(1, order.size // 16)].tolist()))
    mx = Maxima()
    for b in sample:
        ms = int(w["s_off"][b + 1] - w["s_off"][b]); ml = int(w["l_off"][b + 1] - w["l_off"][b])
        m = ms + ml
        if m == 0:
            continue
        S = engine.block_sigma(b, m)
        K = S.copy()
        K[np.arange(ms), np.arange(ms)] += 1.0 / (sig * n_obs)                      # ridge on the small SNPs only
        x = np.concatenate([r["beta_s"][0][w["s_off"][b]:w["s_off"][b + 1]], r["beta_l"][0][w["l_off"][b]:w["l_off"][b + 1]]]) * np.sqrt(n_obs)
        z = np.concatenate([sz[w["s_off"][b]:w["s_off"][b + 1]], lz[w["l_off"][b]:w["l_off"][b + 1]]])
        res = np.abs(K @ x - z).max() / max(np.abs(z).max(), 1e-300)
        assert res < 1e-10, (b, m, res)
        # every stage of the block against the extended-precision reference (tests/solver_ref.py)
        pos = np.concatenate([w["s_pos"][w["s_off"][b]:w["s_off"][b + 1]], w["l_pos"][w["l_off"][b]:w["l_off"][b + 1]]])
        sstar = R.exact_sigma(w["bed"], w["n_ref"], pos, 0.8)
        c = R.ridge(sig, n_obs)
        xstar, kappa = R.refined_solve(R.k_matrix(sstar, ms, c), z)
        L, y = engine.block_factor(b, m)
        mx.add(R.check_block(f"{b} (m={m}, genome-wide)", ms=ms, c=c, z=z, sigma_lib=S, sigma_star=sstar, L=L, y=y, x=x,
                             xstar=xstar, kappa=kappa))
    mx.record("solver/genome_wide")
    rs = engine.fit(*csr, sigma_s=[sig], n_obs=n_obs, bed=w["bed"], n_ref=w["n_ref"])
    assert relmax(rs["beta_s"], r["beta_s"]) <= 1e-11 and relmax(rs["beta_l"], r["beta_l"]) <= 1e-11
    # run-to-run determinism at full load (every reduction order is fixed): a second resident fit is bit-identical.  This
    # is the check that exposed a ring stage handed back to the TMA producer before its shared-memory loads had returned.
    for _ in range(2):
        r2 = engine.fit(*csr, sigma_s=[sig], n_obs=n_obs, flags=_abi.FLAG_FULL_SIGMA)
        assert np.array_equal(r2["beta_s"], r["beta_s"]) and np.array_equal(r2["beta_l"], r["beta_l"])
