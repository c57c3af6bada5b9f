"""Two identical resident fits: where do the factors L differ? (debugging aid; reads L through Engine.block_factor)"""
import argparse, sys, os
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, bench
from dbslmm_b200 import _abi
ns = argparse.Namespace(config="c3", missing=0.0, seed=20240003)
w = bench.build_workload(ns, torch, torch.device("cuda", 0), ns.seed)
sz = w["z"][w["s_pos"]]; lz = w["z"][w["l_pos"]]
csr = (w["s_off"], w["s_pos"], sz, w["l_off"], w["l_pos"], lz)
sig, n_obs = 0.5 / w["nsnp_total"], w["n_obs"]
eng = _abi.Engine(0); eng.load_bed(w["bed"], w["n_ref"])
sizes = w["sizes"]
cand = [b for b in range(len(sizes)) if 700 <= sizes[b] <= 1300][:160]
def run():
    r = eng.fit(*csr, sigma_s=[sig], n_obs=n_obs)
    return r, {b: eng.block_factor(b, int(sizes[b])) for b in cand}
r1, L1 = run(); r2, L2 = run()
nb = 0
for b in cand:
    (A, ya), (B, yb) = L1[b], L2[b]
    d = np.abs(A - B)
    if d.max() > 0 or not np.array_equal(ya, yb):
        nb += 1
        if d.max() == 0:
            print(f"block {b} m {sizes[b]}: L identical, y = L^-1 z differs at {np.flatnonzero(ya != yb)[:12]}", flush=True)
            continue
        ij = np.argwhere(d > 0)
        cols = np.unique(ij[:, 1])
        fc = cols[0]; rows_fc = ij[ij[:, 1] == fc][:, 0]
        print(f"block {b} m {sizes[b]}: {len(ij)} entries differ; first col {fc} (panel {fc//64}, col-in-panel {fc%64}), rows in that col {rows_fc[:12]} (n={len(rows_fc)}); maxdiff {d.max():.3e}; "
              f"in first differing panel: rows {np.unique(ij[(ij[:,1]//64)==(fc//64)][:,0])[:20]} cols {np.unique(ij[(ij[:,1]//64)==(fc//64)][:,1])[:20]}", flush=True)
        if nb >= 8: break
print("blocks differing:", nb, "of", len(cand))
