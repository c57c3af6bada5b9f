"""Measure the LD-score call (dbslmm_b200_ldscore) on one B200 and write the figures as JSON.

    python tools/ldscore_bench.py [--out profiles/r09_ldscore.json]

Panels (synthesised on the GPU by bench.py's AR(1) haplotype model, no missing calls, then held in host memory):
  * the C3 shape: 1.1 M SNPs over chromosomes 1-22 (synth.eur_block_sizes, per chromosome), n_ref 2,000, positions spread
    uniformly over each chromosome's length, cM = bp x 1e-6; windows --ld-wind-cm 1 and --ld-wind-kb 1000;
  * chromosome 1 of that shape at n_ref 20,000, --ld-wind-cm 1.
Reported per case: wall time of the call from pageable memory and from an mmap of a .bed file (page cache warm), the
summed kernel time, the band's tiles and int8 operations (computed from the shapes: 2 x 128 x 128 x n_pad per tile), the
int8 rate that implies against torch._int_mm measured in the same run, and the per-chunk timeline of one traced call
(copy and kernel intervals from CUDA events): the share of the device span the copy engine is busy, and the share of
chunks whose kernels end before the next chunk's copy ends.  The CPU restatement (tests/ldscore_ref.py, ldsc's float64
recipe) is timed on chromosome 22 for scale.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from score_stream_bench import card, overlap_summary  # noqa: E402


def int8_rate(n=16384, reps=10):
    import torch
    a = torch.randint(-8, 8, (n, n), dtype=torch.int8, device="cuda")
    b = torch.randint(-8, 8, (n, n), dtype=torch.int8, device="cuda")
    torch._int_mm(a, b)
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch._int_mm(a, b); e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return {"shape": [n, n, n], "best_ms": min(ts), "ops_per_s_best": 2.0 * n ** 3 / (min(ts) * 1e-3)}


def c3_layout(n_snp_total=1_100_000, cap=3000):
    from dbslmm_b200 import synth
    lens = json.load(open(os.path.join(ROOT, "dbslmm_b200", "data", "eur_ld_block_lengths.json")))
    sizes = synth.eur_block_sizes(n_snp_total, cap)
    per, b0 = [], 0
    for c in range(1, 23):
        nb = len(lens[str(c)])
        per.append((c, int(sizes[b0:b0 + nb].sum()), float(np.sum(lens[str(c)]))))
        b0 += nb
    return per


def panel(per, n_ref, seed):
    import torch
    import bench
    n_snp = sum(m for _, m, _ in per)
    bed = bench.make_bed_cuda(torch, torch.device("cuda"), n_snp, n_ref, seed).numpy()
    bp = np.concatenate([np.linspace(1.0, length, m) for _, m, length in per])
    off = np.concatenate([[0], np.cumsum([m for _, m, _ in per])]).astype(np.int32)
    return np.array(bed), off, bp                       # np.array: a pageable copy


def traced_call(eng, *a, **kw):
    os.environ["DBSLMM_B200_TRACE"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tf:
        os.dup2(tf.fileno(), 2)
        try:
            res = eng.ldscore(*a, **kw)
        finally:
            sys.stderr.flush()
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["DBSLMM_B200_TRACE"]
        tf.seek(0)
        lines = [ln for ln in tf.read().split("\n") if "ldscore pass" in ln]
    out = {"pass1": [], "pass2": []}
    for ln in lines:
        t = ln.split()
        i = t.index("chunk")
        out[t[i - 1]].append({"chunk": int(t[i + 1]), "rows": int(t[i + 3]), "bytes": int(t[i + 5]),
                              "copy": [float(t[i + 7]), float(t[i + 8])], "kernels": [float(t[i + 10]), float(t[i + 11])]})
    return res, out


def band_shape(kept, off, coord, max_dist, n_ref):
    """Tiles of the band and their int8 operations (one plane), from the kept SNPs and the window rule."""
    from dbslmm_b200 import _abi
    n_pad = (n_ref + 127) // 128 * 128
    tiles = 0
    for c in range(len(off) - 1):
        k = np.where(kept[off[c]:off[c + 1]])[0]
        if k.size == 0:
            continue
        lo, hi = _abi.ld_windows(coord[off[c]:off[c + 1]][k], max_dist)
        for t in range((k.size + 127) // 128):
            tiles += int(hi[min(k.size, 128 * t + 128) - 1]) // 128 - t + 1
    return tiles, 2.0 * 128 * 128 * n_pad * tiles


def case(eng, bed, n_ref, off, coord, max_dist, reps, int8):
    rows = np.arange(off[-1], dtype=np.int32)
    eng.ldscore(bed, n_ref, rows, off, coord, max_dist=max_dist)                                     # warm-up
    walls, kms = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        l2, kept, _, _ = eng.ldscore(bed, n_ref, rows, off, coord, max_dist=max_dist)
        walls.append(time.perf_counter() - t0)
        kms.append(eng.last_kernel_ms)
    with tempfile.NamedTemporaryFile(suffix=".bed", dir=tempfile.gettempdir()) as f:
        f.write(bytes([0x6C, 0x1B, 0x01]))
        f.write(bed.tobytes())
        f.flush()
        mm = np.memmap(f.name, dtype=np.uint8, mode="r", offset=3)
        eng.ldscore(mm, n_ref, rows, off, coord, max_dist=max_dist)
        mwalls = []
        for _ in range(reps):
            t0 = time.perf_counter()
            l2m, _, _, _ = eng.ldscore(mm, n_ref, rows, off, coord, max_dist=max_dist)
            mwalls.append(time.perf_counter() - t0)
        same = bool(np.array_equal(l2m.view(np.int64), l2.view(np.int64)))
        del mm
    _, tr = traced_call(eng, bed, n_ref, rows, off, coord, max_dist=max_dist)
    tiles, ops = band_shape(kept, off, coord, max_dist, n_ref)
    k = float(np.median(kms))
    span = tr["pass2"][-1]["kernels"][1] - tr["pass1"][0]["copy"][0] if tr["pass2"] else None
    copy_ms = sum(c["copy"][1] - c["copy"][0] for c in tr["pass1"] + tr["pass2"])
    return {"n_ref": n_ref, "n_snp": int(off[-1]), "n_kept": int(kept.sum()), "max_dist": max_dist,
            "bed_bytes": int(bed.size), "wall_s_pageable": walls, "wall_s_pageable_median": float(np.median(walls)),
            "wall_s_mmap": mwalls, "wall_s_mmap_median": float(np.median(mwalls)), "mmap_bit_identical": same,
            "kernel_ms": kms, "kernel_ms_median": k, "band_tiles": tiles, "band_int8_ops": ops,
            "int8_ops_per_s_over_all_kernels": ops / (k * 1e-3), "share_of_int_mm_rate": ops / (k * 1e-3) / int8["ops_per_s_best"],
            "pcie_bytes_two_passes": 2 * int(bed.size),
            "device_span_ms": span, "copy_ms_sum": copy_ms, "copy_share_of_span": copy_ms / span if span else None,
            "pass1": overlap_summary(tr["pass1"]), "pass2": overlap_summary(tr["pass2"])}


def cpu_restatement_chr22(bed, n_ref, off, coord, max_dist):
    import ldscore_ref as R
    c = 21
    sub = bed[off[c]:off[c + 1]]
    codes = np.stack([(sub >> s) & 3 for s in (0, 2, 4, 6)], axis=2).reshape(sub.shape[0], -1)[:, :n_ref]
    G = np.array([2, -1, 1, 0], np.int8)[codes]
    t0 = time.perf_counter()
    R.ldscore_ldsc64(G, [0, G.shape[0]], coord[off[c]:off[c + 1]], max_dist)
    return {"n_snp": int(G.shape[0]), "n_ref": n_ref, "wall_s": time.perf_counter() - t0,
            "what": "tests/ldscore_ref.ldscore_ldsc64 (numpy float64, dense per chromosome): for scale only"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_ldscore.json"))
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    from dbslmm_b200 import _abi
    info = {"card": card(), "int8_int_mm": int8_rate()}
    per = c3_layout()
    eng = _abi.Engine(0)
    try:
        bed, off, bp = panel(per, 2000, 1)
        info["c3_2000_cm1"] = case(eng, bed, 2000, off, bp * 1e-6, 1.0, args.reps, info["int8_int_mm"])
        info["c3_2000_kb1000"] = case(eng, bed, 2000, off, bp, 1000.0 * 1000, args.reps, info["int8_int_mm"])
        info["cpu_restatement_chr22"] = cpu_restatement_chr22(bed, 2000, off, bp * 1e-6, 1.0)
        del bed
        bed, off, bp = panel(per[:1], 20000, 2)
        info["chr1_20000_cm1"] = case(eng, bed, 20000, off, bp * 1e-6, 1.0, args.reps, info["int8_int_mm"])
        del bed
    finally:
        eng.close()
    info["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(info, f, indent=1)
    brief = {k: {kk: v[kk] for kk in ("wall_s_pageable_median", "wall_s_mmap_median", "kernel_ms_median", "band_int8_ops",
                                      "share_of_int_mm_rate", "copy_share_of_span") if kk in v}
             for k, v in info.items() if isinstance(v, dict) and "kernel_ms" in v}
    print(json.dumps({"card": info["card"], **brief}))


if __name__ == "__main__":
    main()
