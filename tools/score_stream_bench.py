"""Measure the streaming scorer (dbslmm_b200_score_stream) on one B200 and write the figures as JSON.

    python tools/score_stream_bench.py [--out profiles/r08_score_stream.json]

Synthetic target panels live in ordinary (pageable) host memory, as an mmap of a .bed would:
  * 100,000 individuals x 200,000 SNPs (5.0 GB), every SNP scored in file order, 3 folds;
  * 500,000 individuals x 40,000 SNPs (5.0 GB): above the 409,344-individual limit of the resident scorer.
Reported per panel: wall time of the call, streamed rate (scored row bytes / wall time), summed kernel time and the FP64
FMA rate it implies (n_scored x n_val x n_folds FMAs), and the per-chunk timeline of one traced call (copy and kernel
intervals from CUDA events): the share of chunks whose kernels end before the next chunk's copy ends, i.e. hide behind
the copies.  The pinned host-to-device copy rate is measured in the same run (torch, 256 MB, CUDA events), and the
resident scorer dbslmm_b200_score is timed on a panel that fits (100,000 x 20,000), alternated with the streaming call.
The card's name and power limit are read in the same run."""
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


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().split("\n")[0] if q.returncode == 0 else None}


def pinned_h2d_rate(mb=256, reps=10):
    import torch
    n = mb << 20
    h = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    h.fill_(7)
    d = torch.empty(n, dtype=torch.uint8, device="cuda")
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); d.copy_(h, non_blocking=True); e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    del h, d
    torch.cuda.empty_cache()
    return {"bytes": n, "best_ms": min(ts), "median_ms": float(np.median(ts)), "GB_per_s_best": n / min(ts) / 1e6,
            "GB_per_s_median": n / float(np.median(ts)) / 1e6}


def make_panel(n_val, n_snp, seed):
    rng = np.random.default_rng(seed)
    pitch = (n_val + 3) // 4
    bed = np.frombuffer(rng.bytes(n_snp * pitch), np.uint8).reshape(n_snp, pitch)
    return bed


def traced_call(eng, *a, **kw):
    """One call with the library's per-chunk trace on; returns (result, chunk list) parsed from stderr."""
    os.environ["DBSLMM_B200_TRACE"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tf:
        os.dup2(tf.fileno(), 2)
        try:
            res = eng.score_stream(*a, **kw)
        finally:
            sys.stderr.flush()
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["DBSLMM_B200_TRACE"]
        tf.seek(0)
        lines = [ln for ln in tf.read().split("\n") if "score_stream chunk" in ln]
    chunks = []
    for ln in lines:
        t = ln.split()
        i = t.index("chunk")
        chunks.append({"chunk": int(t[i + 1]), "rows": int(t[i + 3]), "bytes": int(t[i + 5]),
                       "copy": [float(t[i + 7]), float(t[i + 8])], "kernels": [float(t[i + 10]), float(t[i + 11])]})
    return res, chunks


def overlap_summary(chunks):
    if not chunks:
        return {}
    copy = np.array([c["copy"][1] - c["copy"][0] for c in chunks])
    kern = np.array([c["kernels"][1] - c["kernels"][0] for c in chunks])
    # chunk k's kernels are hidden if they end before the copy of chunk k+1 ends (the copy engine stays the bottleneck)
    hidden = [chunks[k]["kernels"][1] <= chunks[k + 1]["copy"][1] for k in range(len(chunks) - 1)]
    span = chunks[-1]["kernels"][1] - chunks[0]["copy"][0]
    return {"n_chunks": len(chunks), "chunk_bytes": chunks[0]["bytes"], "rows_per_chunk": chunks[0]["rows"],
            "copy_ms_median": float(np.median(copy)), "kernel_ms_median": float(np.median(kern)),
            "copy_ms_sum": float(copy.sum()), "kernel_ms_sum": float(kern.sum()),
            "device_span_ms": span, "kernels_hidden_share": float(np.mean(hidden)) if hidden else None,
            "copy_engine_busy_share": float(copy.sum() / span) if span > 0 else None,
            "first_chunks": chunks[:3], "last_chunks": chunks[-2:]}


def stream_case(eng, n_val, n_snp, n_folds, reps, seed):
    bed = make_panel(n_val, n_snp, seed)
    rng = np.random.default_rng(seed + 1)
    pos = np.arange(n_snp, dtype=np.int32)
    beta = rng.standard_normal((n_folds, n_snp)) * 1e-3
    flip = (rng.random(n_snp) < 0.3).astype(np.uint8)
    pitch = bed.shape[1]
    eng.score_stream(bed, n_val, pos, beta, flip)                                    # warm-up: buffers, modules
    walls, kms = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        eng.score_stream(bed, n_val, pos, beta, flip)
        walls.append(time.perf_counter() - t0)
        kms.append(eng.last_kernel_ms)
    _, chunks = traced_call(eng, bed, n_val, pos, beta, flip)
    scored_bytes = n_snp * pitch
    fma = float(n_snp) * n_val * n_folds
    w = float(np.median(walls))
    k = float(np.median(kms))
    out = {"n_val": n_val, "n_snp": n_snp, "n_scored": n_snp, "n_folds": n_folds, "scored_row_bytes": scored_bytes,
           "wall_s": walls, "wall_s_median": w, "streamed_GB_per_s": scored_bytes / w / 1e9,
           "kernel_ms": kms, "kernel_ms_median": k, "fp64_fma_per_s": fma / (k * 1e-3),
           "overlap": overlap_summary(chunks)}
    del bed
    return out


def resident_vs_stream(eng, n_val, n_snp, n_folds, reps, seed):
    bed = make_panel(n_val, n_snp, seed)
    rng = np.random.default_rng(seed + 1)
    pos = np.arange(n_snp, dtype=np.int32)
    beta = rng.standard_normal((n_folds, n_snp)) * 1e-3
    flip = (rng.random(n_snp) < 0.3).astype(np.uint8)
    one_chunk = n_snp * (bed.shape[1] + 1)
    eng.score(bed, n_val, pos, beta, flip)
    eng.score_stream(bed, n_val, pos, beta, flip)
    res = {"score_wall_s": [], "score_kernel_ms": [], "stream_wall_s": [], "stream_kernel_ms": []}
    for _ in range(reps):
        t0 = time.perf_counter()
        s_res, kms = eng.score(bed, n_val, pos, beta, flip)
        res["score_wall_s"].append(time.perf_counter() - t0)
        res["score_kernel_ms"].append(kms)
        t0 = time.perf_counter()
        s_str, _, _ = eng.score_stream(bed, n_val, pos, beta, flip)
        res["stream_wall_s"].append(time.perf_counter() - t0)
        res["stream_kernel_ms"].append(eng.last_kernel_ms)
    s_one, _, _ = eng.score_stream(bed, n_val, pos, beta, flip, chunk_bytes=one_chunk)
    scale = float(np.abs(s_res).max())
    res.update({"n_val": n_val, "n_snp": n_snp, "n_folds": n_folds,
                "score_wall_s_median": float(np.median(res["score_wall_s"])),
                "stream_wall_s_median": float(np.median(res["stream_wall_s"])),
                "stream_default_chunks_max_rel_diff": float(np.abs(s_str - s_res).max() / scale),
                "stream_one_chunk_bit_identical": bool(np.array_equal(s_one, s_res))})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_score_stream.json"))
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    from dbslmm_b200 import _abi
    info = {"card": card(), "pinned_h2d": pinned_h2d_rate()}
    eng = _abi.Engine(0)
    try:
        info["stream_100k_x_200k"] = stream_case(eng, 100_000, 200_000, 3, args.reps, 1)
        info["stream_500k_x_40k"] = stream_case(eng, 500_000, 40_000, 3, args.reps, 2)
        info["resident_vs_stream_100k_x_20k"] = resident_vs_stream(eng, 100_000, 20_000, 3, args.reps, 3)
    finally:
        eng.close()
    info["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(info, f, indent=1)
    brief = {k: {kk: v[kk] for kk in ("wall_s_median", "streamed_GB_per_s", "kernel_ms_median", "fp64_fma_per_s") if kk in v}
             for k, v in info.items() if k.startswith("stream_")}
    print(json.dumps({"card": info["card"], "pinned_h2d_GB_per_s": info["pinned_h2d"]["GB_per_s_median"], **brief}))


if __name__ == "__main__":
    main()
