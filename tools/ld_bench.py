"""Measure the SNP-pair call (dbslmm_b200_ld_pairs) and the `ld` command line on one B200 and write the figures as JSON.

    python tools/ld_bench.py [--out profiles/r11_ld_pairs.json]

Panel: the C3 shape of tools/ldscore_bench.py (1.1 M SNPs over chromosomes 1-22, n_ref 2,000, bench.py's AR(1) haplotype
model, positions spread uniformly over each chromosome).  Cases:
  * PLINK's defaults: --ld-window 10 --ld-window-kb 1000 --ld-window-r2 0.2;
  * --ld-window 99999 --ld-window-kb 1000 --ld-window-r2 0.2.
Per case: the call through the C ABI with a sink that only counts (wall time, summed kernel time, pairs, bytes delivered
to the sink: 12 per pair plus 8 per row offset), then `build/ld --r2 gz` on a .bed/.bim/.fam written to a temporary
directory, whose log gives the wall split (kernels, time inside the sink, formatting and gzip CPU time).  Engine.ldscore
(--ld-wind-kb 1000) runs before and after each case, alternating, to show the unannotated LD-score call unchanged.  The
card's name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from ldscore_bench import c3_layout, panel  # noqa: E402
from score_stream_bench import card  # noqa: E402

CASES = {"defaults": (10, 1000.0, 0.2), "window99999": (99999, 1000.0, 0.2)}


def api_call(eng, bed, n_ref, off, bp, n, kb, r2):
    from dbslmm_b200 import _abi
    rows = np.arange(off[-1], dtype=np.int32)
    got = {"calls": 0, "pairs": 0, "rows": 0}

    def f(user, a0, a1, o, b, r):
        got["calls"] += 1
        got["pairs"] += o[a1 - a0]
        got["rows"] += a1 - a0
        return 0

    sink = _abi.LD_SINK(f)
    n_pairs, n_miss, ms = C.c_int64(0), C.c_int64(0), C.c_float(0)
    t0 = time.perf_counter()
    rc = eng.lib.dbslmm_b200_ld_pairs(eng.h, bed.ctypes.data, bed.shape[0], n_ref, rows.ctypes.data, rows.size, off.ctypes.data,
                                      off.size - 1, bp.ctypes.data, n, kb * 1000.0, r2, 0, sink, None, None, C.byref(n_pairs),
                                      C.byref(n_miss), C.byref(ms))
    wall = time.perf_counter() - t0
    eng._check(rc, "ld_pairs")
    assert got["pairs"] == n_pairs.value
    return {"wall_s": wall, "kernel_ms": ms.value, "pairs": n_pairs.value, "sink_calls": got["calls"],
            "bytes_delivered": 12 * got["pairs"] + 8 * (got["rows"] + got["calls"])}


def ldscore_ms(eng, bed, n_ref, off, bp):
    rows = np.arange(off[-1], dtype=np.int32)
    t0 = time.perf_counter()
    eng.ldscore(bed, n_ref, rows, off, bp, max_dist=1000.0 * 1000)
    return {"wall_s": time.perf_counter() - t0, "kernel_ms": eng.last_kernel_ms}


def cli(d, prefix, n, kb, r2):
    t0 = time.perf_counter()
    r = subprocess.run([os.path.join(ROOT, "build", "ld"), "--bfile", prefix, "--r2", "gz", "--ld-window", str(n), "--ld-window-kb",
                        str(kb), "--ld-window-r2", str(r2), "--out", os.path.join(d, "o")], capture_output=True, text=True)
    wall = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError(r.stderr)
    log = open(os.path.join(d, "o.log")).read()
    num = lambda pat: float(re.search(pat, log).group(1))
    out = {"wall_s": wall, "kernel_ms": num(r"GPU kernel time ([0-9.e+-]+) ms"), "call_s": num(r"ld_pairs call ([0-9.e+-]+) s"),
           "sink_s": num(r"of which sink ([0-9.e+-]+) s"), "format_cpu_s": num(r"formatting ([0-9.e+-]+) s"),
           "gzip_cpu_s": num(r"gzip ([0-9.e+-]+) s"), "threads": int(num(r"on ([0-9]+) threads")),
           "bytes_written": int(num(r"([0-9]+) bytes written")), "pairs": int(num(r"([0-9]+) pairs written")), "log": log}
    os.remove(os.path.join(d, "o.ld.gz"))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_ld_pairs.json"))
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    from dbslmm_b200 import _abi
    info = {"card": card()}
    per = c3_layout()
    bed, off, bp = panel(per, 2000, 1)
    bp = np.floor(bp)
    chrom = np.repeat(np.arange(1, 23), np.diff(off))
    eng = _abi.Engine(0)
    with tempfile.TemporaryDirectory() as d:
        prefix = os.path.join(d, "c3")
        with open(prefix + ".bed", "wb") as f:
            f.write(bytes([0x6C, 0x1B, 0x01]))
            f.write(bed.tobytes())
        with open(prefix + ".bim", "w") as f:
            f.writelines(f"{c}\trs{i}\t0\t{int(x)}\tA\tG\n" for i, (c, x) in enumerate(zip(chrom, bp)))
        with open(prefix + ".fam", "w") as f:
            f.writelines(f"F{i} I{i} 0 0 1 -9\n" for i in range(2000))
        try:
            ldscore_ms(eng, bed, 2000, off, bp)                                              # warm-up
            for name, (n, kb, r2) in CASES.items():
                api_call(eng, bed, 2000, off, bp, n, kb, r2)                                 # warm-up
                res = {"ld_window": n, "ld_window_kb": kb, "ld_window_r2": r2, "api": [], "ldscore_kb1000": []}
                for _ in range(args.reps):                                                   # alternating with ldscore
                    res["ldscore_kb1000"].append(ldscore_ms(eng, bed, 2000, off, bp))
                    res["api"].append(api_call(eng, bed, 2000, off, bp, n, kb, r2))
                res["ldscore_kb1000"].append(ldscore_ms(eng, bed, 2000, off, bp))
                res["cli_gz"] = cli(d, prefix, n, kb, r2)
                info[name] = res
        finally:
            eng.close()
    info["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(info, f, indent=1)
    brief = {k: {"pairs": v["api"][-1]["pairs"], "kernel_ms": [x["kernel_ms"] for x in v["api"]],
                 "wall_s": [x["wall_s"] for x in v["api"]], "ldscore_kernel_ms": [x["kernel_ms"] for x in v["ldscore_kb1000"]],
                 "cli": {kk: v["cli_gz"][kk] for kk in ("wall_s", "kernel_ms", "sink_s", "format_cpu_s", "gzip_cpu_s", "bytes_written")}}
             for k, v in info.items() if k in CASES}
    print(json.dumps({"card": info["card"], **brief}))


if __name__ == "__main__":
    main()
