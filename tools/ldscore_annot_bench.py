"""Measure partitioned LD Scores (dbslmm_b200_ldscore_annot) and the unannotated call on one B200; write JSON.

    python tools/ldscore_annot_bench.py [--out profiles/r10_ldscore_annot.json] [--parent-tree DIR]

Panels (tools/ldscore_bench.py's: synthesised on the GPU by bench.py's AR(1) haplotype model, no missing calls, held in
pageable host memory):
  * the C3 shape, 1.1 M SNPs over chromosomes 1-22 at n_ref 2,000, --ld-wind-cm 1;
  * one chromosome of 500,000 SNPs at n_ref 489, --ld-wind-snps 2000.
Each panel is timed without annotations and with C = 1, 8 and 97 columns (binary and continuous).  Reported per case:
wall and summed kernel time, the FP64 FMAs of the annotated epilogue, C x sum_j |W(j)|, and the int8 operations of the
band (2 x 128 x 128 x n_pad per tile: the half band without annotations, the full band with them), both from shapes; the
FP64 FMA rate against a DGEMM (torch.matmul, float64) measured in the same run; and the copy/kernel overlap of one traced
call.  With --parent-tree (a checkout of the parent commit with its library built) the unannotated C3 call is also timed
against that tree's package, alternating the two in child processes.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from ldscore_bench import c3_layout, panel  # noqa: E402
from score_stream_bench import card, overlap_summary  # noqa: E402


def dgemm_rate(n=8192, reps=5):
    import torch
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return {"shape": [n, n, n], "best_ms": min(ts), "fma_per_s_best": float(n) ** 3 / (min(ts) * 1e-3)}


def shapes(kept, off, coord, max_dist, n_ref):
    """sum_j |W(j)| over kept SNPs, and the tiles of the half and of the full band."""
    from dbslmm_b200 import _abi
    w = half = full = 0
    for c in range(len(off) - 1):
        k = np.where(kept[off[c]:off[c + 1]])[0]
        if k.size == 0:
            continue
        x = None if coord is None else coord[off[c]:off[c + 1]][k]
        lo, hi = _abi.ld_windows(x, max_dist, m=k.size)
        w += int((hi.astype(np.int64) - lo + 1).sum())
        for t in range((k.size + 127) // 128):
            tl, th = int(lo[128 * t]) // 128, int(hi[min(k.size, 128 * t + 128) - 1]) // 128
            half += th - t + 1
            full += th - tl + 1
    return w, half, full


def traced(eng, *a, **kw):
    os.environ["DBSLMM_B200_TRACE"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tf:
        os.dup2(tf.fileno(), 2)
        try:
            eng.ldscore(*a, **kw)
        finally:
            sys.stderr.flush()
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["DBSLMM_B200_TRACE"]
        tf.seek(0)
        lines = [ln for ln in tf.read().split("\n") if " pass2 chunk " in ln]
    out = []
    for ln in lines:
        t = ln.split()
        i = t.index("chunk")
        out.append({"chunk": int(t[i + 1]), "rows": int(t[i + 3]), "bytes": int(t[i + 5]),
                    "copy": [float(t[i + 7]), float(t[i + 8])], "kernels": [float(t[i + 10]), float(t[i + 11])]})
    return overlap_summary(out)


def case(eng, bed, n_ref, off, coord, max_dist, annot, reps, dgemm):
    rows = np.arange(off[-1], dtype=np.int32)
    kw = dict(max_dist=max_dist) if annot is None else dict(max_dist=max_dist, annot=annot)
    eng.ldscore(bed, n_ref, rows, off, coord, **kw)                       # warm-up
    walls, kms = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        l2, kept, _, _ = eng.ldscore(bed, n_ref, rows, off, coord, **kw)
        walls.append(time.perf_counter() - t0)
        kms.append(eng.last_kernel_ms)
    C = 0 if annot is None else annot.shape[1]
    w, half, full = shapes(kept, off, coord, max_dist, n_ref)
    n_pad = (n_ref + 127) // 128 * 128
    k = float(np.median(kms))
    fma = float(C) * w
    r = {"n_ref": n_ref, "n_snp": int(off[-1]), "n_kept": int(kept.sum()), "max_dist": max_dist, "n_annot": C,
         "wall_s": walls, "wall_s_median": float(np.median(walls)), "kernel_ms": kms, "kernel_ms_median": k,
         "sum_window": w, "fp64_fma": fma, "band_tiles": full if C else half,
         "band_int8_ops": 2.0 * 128 * 128 * n_pad * (full if C else half), "pass2_overlap": traced(eng, bed, n_ref, rows, off, coord, **kw)}
    if C:
        r["fp64_fma_per_s_over_all_kernels"] = fma / (k * 1e-3)
        r["share_of_dgemm_fma_rate"] = fma / (k * 1e-3) / dgemm["fma_per_s_best"]
    return r


def columns(rng, n, C):
    a = np.empty((n, C))
    for c in range(C):
        a[:, c] = (rng.random(n) < 0.2) if c % 2 == 0 else rng.standard_normal(n)
    return a


def child(reps, tree):
    """Time the unannotated C3 call with the dbslmm_b200 package of `tree` (this tree if empty); print one JSON line."""
    if tree:
        sys.path.insert(0, os.path.abspath(tree))
    from dbslmm_b200 import _abi
    per = c3_layout()
    bed, off, bp = panel(per, 2000, 1)
    eng = _abi.Engine(0)
    try:
        r = case(eng, bed, 2000, off, bp * 1e-6, 1.0, None, reps, None)
    finally:
        eng.close()
    print(json.dumps({"kernel_ms": r["kernel_ms"], "wall_s": r["wall_s"]}))


def ab(parent_tree, rounds, reps):
    out = {"parent": [], "this": []}
    for _ in range(rounds):
        for tag, tree in (("parent", parent_tree), ("this", "")):
            env = dict(os.environ)
            env.pop("DBSLMM_B200_LIB", None)
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--reps", str(reps), "--parent-tree", tree],
                               env=env, stdout=subprocess.PIPE, text=True, check=True)
            out[tag].append(json.loads(p.stdout.strip().splitlines()[-1]))
    for tag in ("parent", "this"):
        ks = [x for r in out[tag] for x in r["kernel_ms"]]
        ws = [x for r in out[tag] for x in r["wall_s"]]
        out[tag + "_kernel_ms_median"] = float(np.median(ks))
        out[tag + "_wall_s_median"] = float(np.median(ws))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_ldscore_annot.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parent-tree", default="")
    ap.add_argument("--child", action="store_true")
    args = ap.parse_args()
    if args.child:
        return child(args.reps, args.parent_tree)
    from dbslmm_b200 import _abi
    info = {"card": card(), "dgemm": dgemm_rate()}
    rng = np.random.default_rng(0)
    eng = _abi.Engine(0)
    try:
        bed, off, bp = panel(c3_layout(), 2000, 1)
        for C in (0, 1, 8, 97):
            a = None if C == 0 else columns(rng, int(off[-1]), C)
            info[f"c3_2000_cm1_C{C}"] = case(eng, bed, 2000, off, bp * 1e-6, 1.0, a, args.reps, info["dgemm"])
        del bed
        bed, off, _ = panel([(1, 500_000, 2.5e8)], 489, 2)
        for C in (0, 1, 8, 97):
            a = None if C == 0 else columns(rng, int(off[-1]), C)
            info[f"chr500k_489_snps2000_C{C}"] = case(eng, bed, 489, off, None, 2000, a, args.reps, info["dgemm"])
        del bed
    finally:
        eng.close()
    if args.parent_tree:
        info["unannotated_c3_vs_parent"] = ab(args.parent_tree, 2, args.reps)
    info["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(info, f, indent=1)
    brief = {k: {kk: v[kk] for kk in ("wall_s_median", "kernel_ms_median", "fp64_fma", "share_of_dgemm_fma_rate") if kk in v}
             for k, v in info.items() if isinstance(v, dict) and "kernel_ms" in v}
    if "unannotated_c3_vs_parent" in info:
        brief["vs_parent"] = {k: v for k, v in info["unannotated_c3_vs_parent"].items() if k.endswith("median")}
    print(json.dumps({"card": info["card"], **brief}))


if __name__ == "__main__":
    main()
