#!/usr/bin/env python
"""bench.py -- headline benchmark: LD blocks fitted / second, genome-wide DBSLMM fit.

One "step" = one pass of the hot path (decode -> Gram -> block solve -> betas on the host) over the whole
synthetic genome (BASELINE.json configs[2]: 22 chromosomes, ~1.1 M SNPs, 1,703 EUR LD blocks, n_ref = 2,000,
clumped large-effect SNPs).  With N GPUs the blocks are sharded by the library's LPT cost model (no collective
on the data path), so the job size is fixed: "strong" scaling as BASELINE.json's config asks ("sharded at
1/2/4/8 GPUs"); `--scaling weak` gives every rank its own genome instead.

  value  : blocks/s from the library's CUDA-event time of one fit with the panel, the plan and the block lists
           resident in HBM: first event (z-score upload) to last event (betas copied back to pinned host memory)
  e2e    : blocks/s through ONE C-ABI call per step from HOST buffers (fit_args.bed: batched panel H2D overlapped with
           the fit, plan/z H2D, kernels, beta D2H), wall clock around the synchronous calls
  parity : after the timed regions, at every N: the betas of the timed fit against the reference's own CPU functions
           on the fixed reference sample, against the exact (Cholesky) oracle on a few of each rank's blocks, the
           integer Gram of two blocks bit for bit, and a checksum of the gathered betas (must not depend on N)
  --impl reference : the reference's CPU path on this box's host cores on the same fixed sample of blocks.
  --config c4 | c5 | --missing 0.005 : BASELINE.json configs[3], configs[4] and the mask path (parity cases, not the
           headline; their lines are kept under profiles/).
  --dump-outputs DIR : the betas of the last timed fit (c4 on one GPU: and its PRS scores) as DIR/beta_s.npy, beta_l.npy[, prs.npy].
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (total_snps, chroms, cap, n_ref, n_obs)
    "c3": (1_100_000, list(range(1, 23)), 3000, 2000, 300_000),
    "c4": (1_100_000, list(range(1, 23)), 3000, 2000, 300_000),      # c3 + 3 heritability folds + PRS over a 10k-sample panel
    "c5": (1_100_000, list(range(1, 23)), 5000, 20_000, 300_000),    # large-reference stress
    "c2": (90_000, [1], 3000, 500, 300_000),
    "chr20_22": (60_000, [20, 21, 22], 3000, 2000, 300_000),         # three real-sized chromosomes at the c3 SNP density (CLI tests)
    "tiny": (6_000, [22], 400, 400, 2400),
}
WORKLOAD_NAME = {
    "c3": "genome-wide synthetic DBSLMM: 22 chr, ~1.1M SNPs, 1,703 EUR LD blocks, n_ref=2000, clumped large-effect SNPs",
    "c4": "tuning version: the c3 genome with h2 folds 0.8/1.0/1.2 sharing one Gram per block + PRS of the 3 folds over a 10k-sample validation .bed",
    "c5": "large-reference stress: 22 chr, ~1.1M SNPs, 1,703 EUR LD blocks of up to 5,000 SNPs, n_ref=20000",
    "c2": "LMM-size synthetic chr1: ~90k SNPs, 133 EUR LD blocks, n_ref=500",
    "chr20_22": "chromosomes 20-22 at the genome-wide SNP density, n_ref=2000",
    "tiny": "tiny synthetic chr22 slice",
}
N_VAL = 10_000          # c4: individuals of the validation panel


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=list(CONFIGS))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--missing", type=float, default=0.0)
    ap.add_argument("--solver", default="cholesky", choices=["cholesky", "pcg"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--seed", type=int, default=20240003)
    ap.add_argument("--emulate-shard", default="", help="R/N: time rank R's shard of an N-GPU run on one GPU (tuning aid)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float64); "
                         "in strong scaling over several GPUs, the betas of all ranks gathered in workload order (no PRS)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: the inputs are seeded, so two builds run with the same arguments can be compared output for output.
    Above DUMP_MAX_BYTES in all, every array keeps the same fraction of its last axis at positions drawn from a fixed seed,
    written beside it as <name>_index.npy."""
    arrays = {k: np.ascontiguousarray(v, np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    frac = 1.0
    if total > DUMP_MAX_BYTES:          # each kept column also costs its 8-byte index; 64 KB left for the .npy headers
        frac = (DUMP_MAX_BYTES - (64 << 10)) / (total + 8.0 * sum(a.shape[-1] for a in arrays.values()))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        if frac < 1.0:
            n = a.shape[-1]
            idx = np.sort(np.random.default_rng(0).choice(n, int(n * frac), replace=False))
            a = a[..., idx]
            np.save(os.path.join(out_dir, k + "_index.npy"), idx.astype(np.float64))
        np.save(os.path.join(out_dir, k + ".npy"), a)


# ---------------------------------------------------------------------------------------------
# synthetic genome on the GPU (torch is plumbing here: RNG + pinned host buffers)
# ---------------------------------------------------------------------------------------------
def make_bed_cuda(torch, dev, n_snp, n_ref, seed, missing_rate=0.0, rho=0.9, chunk=256):
    """uint8 [n_snp, ceil(n_ref/4)] in pinned host memory.  AR(1) latent Gaussian per haplotype
    along the SNP axis (same model as dbslmm_b200.synth.make_genotypes, run as chunked scans)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    pitch = (n_ref + 3) // 4
    n4 = pitch * 4
    host = torch.empty((n_snp, pitch), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
    slab_rows = max(chunk, (1 << 28) // max(pitch, 1) // chunk * chunk)       # ~256 MB of packed rows per device slab
    slab = torch.empty((slab_rows, pitch), dtype=torch.uint8, device=dev)
    s = (1.0 - rho * rho) ** 0.5
    i = torch.arange(chunk, device=dev, dtype=torch.float64)
    T = torch.tril(s * rho ** (i[:, None] - i[None, :]).clamp(min=0)).float()
    pw = (rho ** (i + 1.0)).float()[:, None]
    carry = torch.randn((1, 2 * n_ref), generator=g, device=dev)
    normal = torch.distributions.Normal(0.0, 1.0)
    lut = torch.tensor([3, 2, 0], dtype=torch.uint8, device=dev)       # allele count -> PLINK code
    shifts = torch.tensor([0, 2, 4, 6], dtype=torch.int32, device=dev)
    slab0 = 0
    for c0 in range(0, n_snp, chunk):
        m = min(chunk, n_snp - c0)
        E = torch.randn((chunk, 2 * n_ref), generator=g, device=dev)
        L = T @ E + pw * carry
        carry = L[chunk - 1:chunk].clone()
        p = torch.rand((chunk, 1), generator=g, device=dev) * 0.45 + 0.05
        thr = normal.icdf(p)
        A = (L < thr)
        G = (A[:, :n_ref].to(torch.uint8) + A[:, n_ref:].to(torch.uint8))
        mono = (G.amin(dim=1) == G.amax(dim=1))
        if bool(mono.any()):                                             # re-draw monomorphic rows
            fix = (torch.rand((chunk, n_ref), generator=g, device=dev) < 0.3).to(torch.uint8)
            G = torch.where(mono[:, None], fix, G)
        code = lut[G.long()]
        if missing_rate > 0:
            miss = torch.rand((chunk, n_ref), generator=g, device=dev) < missing_rate
            code = torch.where(miss, torch.ones_like(code), code)
        full = torch.zeros((chunk, n4), dtype=torch.uint8, device=dev)
        full[:, :n_ref] = code
        packed = (full.view(chunk, pitch, 4).to(torch.int32) << shifts).sum(dim=2).to(torch.uint8)
        slab[c0 - slab0:c0 - slab0 + m] = packed[:m]
        if c0 + m - slab0 >= slab_rows or c0 + m == n_snp:
            host[slab0:c0 + m].copy_(slab[:c0 + m - slab0])
            slab0 = c0 + m
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    del slab
    torch.cuda.empty_cache()
    return host


def build_workload(args, torch, dev, rank_seed):
    from dbslmm_b200 import synth
    total, chroms, cap, n_ref, n_obs = CONFIGS[args.config]
    sizes = synth.eur_block_sizes(total, cap, chroms=chroms)
    n_snp = int(sizes.sum())
    bed_t = make_bed_cuda(torch, dev, n_snp, n_ref, rank_seed, missing_rate=args.missing)
    rng = np.random.default_rng(rank_seed + 1)
    z, large = synth.make_sumstats(rng, sizes)
    s_off, s_pos, l_off, l_pos = synth.split_csr(sizes, large)
    return {"sizes": sizes, "n_snp": n_snp, "n_ref": n_ref, "n_obs": n_obs, "bed_t": bed_t,
            "bed": bed_t.numpy(), "z": z, "s_off": s_off, "s_pos": s_pos, "l_off": l_off, "l_pos": l_pos,
            "nsnp_total": n_snp}


def shard_workload(w, owner, rank, torch):
    """Compact per-rank problem (dbslmm_b200.multigpu.shard) with the .bed shard in pinned host memory."""
    from dbslmm_b200 import multigpu
    keep = []

    def pinned(shape):
        t = torch.empty(shape, dtype=torch.uint8, pin_memory=True)
        keep.append(t)
        return t.numpy()
    ww = dict(w)
    ww["s_z"] = w["z"][w["s_pos"]]
    ww["l_z"] = w["z"][w["l_pos"]]
    sh = multigpu.shard(ww, owner, rank, pinned_alloc=pinned)
    sh["_pin"] = keep
    return sh


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []          # (arrival time, text)
        self.proc = None
        self.t_mark = 0.0

    def mark(self):
        """Samples that arrive from now on count (nvidia-smi needs a moment to start: it is launched before the warm-up)."""
        self.t_mark = time.perf_counter()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if ts < self.t_mark:
                continue
            t = [x.strip() for x in ln.split(",")]
            if len(t) < 9:
                continue
            try:
                sm.append(float(t[1])); mx.append(float(t[2]))
            except ValueError:
                continue
            for nm, v in zip(names, t[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measure_fp64_peak(torch, dev):
    """cuBLAS DGEMM 8192^3, best of 5 (TFLOP/s): the FP64 tensor-pipe roofline denominator.
    MEASURED_PEAKS.json has no FP64 figure, so it is measured here, on this box, and labelled so."""
    n = 8192
    a = torch.randn((n, n), dtype=torch.float64, device=dev)
    b = torch.randn((n, n), dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
        best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    del a, b
    torch.cuda.empty_cache()
    return best


def measure_int8_peak(torch, dev):
    """Library int8 GEMM with s32 accumulation (torch._int_mm -> cuBLASLt IGEMM), 8192^3, best of 5 (Pop/s): the int8
    tensor-pipe denominator of the correlation builder.  MEASURED_PEAKS.json has no int8 figure; None if the library
    call is unavailable here."""
    try:
        n = 8192
        a = torch.randint(-2, 3, (n, n), dtype=torch.int8, device=dev)
        b = torch.randint(-2, 3, (n, n), dtype=torch.int8, device=dev)
        torch._int_mm(a, b)
        best = 0.0
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch._int_mm(a, b); e1.record(); torch.cuda.synchronize()
            best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e15)
        del a, b
        torch.cuda.empty_cache()
        return best
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------
# CPU arms (the only place bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------
def block_cost(sizes, n_ref):
    """CPU cost model of one block in the reference (seconds-like units): the FP64 X'X loops dominate (2 n m^2 flop),
    the PCG solves add ~60 iterations of 2 m^2 each."""
    m = np.asarray(sizes, np.float64)
    return 2.0 * n_ref * m * m + 120.0 * m * m + 1e5


def reference_sample(sizes, n_ref):
    """The FIXED block sample both CPU legs time (--impl reference and cpu_baseline): blocks at evenly spaced quantiles
    of the size distribution up to the 97th percentile, in block order.  It depends on the workload only -- not on the
    thread count, not on --steps -- so two runs on equal hosts time the same work.  The sample count is set from the
    cost model so one pass costs ~100 core-seconds (48 blocks at n_ref = 2,000; fewer at n_ref = 20,000).  The
    blocks above the 97th percentile are left out because ONE of them costs 15-20 core-seconds on a single thread
    (blocks are not split across threads in the reference), which would make a pass as long as that block whatever
    the core count; the figure for the whole genome is the cost-weighted extrapolation below."""
    sizes = np.asarray(sizes)
    order = np.argsort(sizes, kind="stable")
    nb = sizes.size
    mean_core_s = float(block_cost(sizes, n_ref).mean()) / 1.9e9
    n_sample = int(min(48, max(8, round(100.0 / max(mean_core_s, 1e-9)))))
    n_sample = min(n_sample, nb)
    qs = (np.arange(n_sample) + 0.5) / n_sample * 0.97
    return np.unique(order[np.minimum((qs * nb).astype(np.int64), nb - 1)])


def sub_csr(w, blocks):
    """CSR lists of a subset of blocks over a compact .bed holding only their rows."""
    s_off = np.zeros(blocks.size + 1, np.int32)
    l_off = np.zeros(blocks.size + 1, np.int32)
    sp, lp = [], []
    for i, b in enumerate(blocks):
        a = w["s_pos"][w["s_off"][b]:w["s_off"][b + 1]]
        c = w["l_pos"][w["l_off"][b]:w["l_off"][b + 1]]
        sp.append(a); lp.append(c)
        s_off[i + 1] = s_off[i] + a.size
        l_off[i + 1] = l_off[i] + c.size
    sp = np.concatenate(sp).astype(np.int64) if sp else np.zeros(0, np.int64)
    lp = np.concatenate(lp).astype(np.int64) if lp else np.zeros(0, np.int64)
    rows = np.unique(np.concatenate([sp, lp]))
    remap = np.full(w["n_snp"], -1, np.int64); remap[rows] = np.arange(rows.size)
    sub = np.ascontiguousarray(w["bed"][rows])
    return {"bed": sub, "s_off": s_off, "s_pos": remap[sp].astype(np.int32), "s_z": w["z"][sp],
            "l_off": l_off, "l_pos": remap[lp].astype(np.int32), "l_z": w["z"][lp], "gs": sp, "gl": lp}


def run_cpu(w, blocks, threads, sigma_s):
    """CPU arm on a block sample.  Prefers the UNMODIFIED reference functions (oracle/_ref: IO::readSNPIm +
    SNPPROC::nomalizeVec + DBSLMMFIT::estBlock/PCG, compiled over oracle/shim) driven by oracle/ref_harness.cpp's
    ref_est_path -- a restatement of DBSLMMFIT::est's batches-of-60 omp-dynamic loop (est() itself drags in the
    fork's variance side channel and its file formats) -- and falls back to the oracle port.
    Returns (seconds, kind, beta_s, beta_l, sub)."""
    from oracle import oracle as O
    from oracle import refharness as R
    sub = sub_csr(w, blocks)
    csr = (sub["s_off"], sub["s_pos"], sub["s_z"], sub["l_off"], sub["l_pos"], sub["l_z"])
    if R.available():
        try:
            tmpdir = "/dev/shm" if os.path.isdir("/dev/shm") else None
            import tempfile
            f = tempfile.NamedTemporaryFile(suffix=".bed", dir=tmpdir, delete=False); f.close()
            R.write_bed(sub["bed"], f.name)
            try:
                t = time.perf_counter()
                bs, bl = R.est_path(f.name, w["n_ref"], w["n_obs"], sigma_s, *csr, threads=threads)
                return time.perf_counter() - t, "reference", bs, bl, sub
            finally:
                os.unlink(f.name)
        except OSError:
            pass
    t = time.perf_counter()
    bs, bl, _, _ = O.est(sub["bed"], w["n_ref"], w["n_obs"], sigma_s, *csr, threads=threads, mode=O.MODE_REF)
    return time.perf_counter() - t, "port", bs, bl, sub


KIND_TEXT = {"reference": "unmodified reference functions (readSNPIm + nomalizeVec + estBlock/PCG) under ref_est_path, the harness's "
                          "restatement of DBSLMMFIT::est's batches-of-60 omp-dynamic loop, over oracle/shim",
             "port": "ref-mode oracle port (PCG tol 1e-7, batches of 60, omp dynamic)"}


def cpu_line(w, blocks, dt, kind, threads):
    """blocks/s of the CPU arm: the sample's time extrapolated to the genome by the cost model."""
    cost_all = float(block_cost(w["sizes"], w["n_ref"]).sum())
    cost_smp = float(block_cost(w["sizes"][blocks], w["n_ref"]).sum())
    genome_s = dt * cost_all / cost_smp
    return {"value": w["sizes"].size / genome_s, "unit": "blocks/s", "cores": threads, "kind": kind,
            "sample": f"fixed sample of {blocks.size} of {w['sizes'].size} LD blocks (size quantiles up to p97, sizes "
                      f"{int(w['sizes'][blocks].min())}-{int(w['sizes'][blocks].max())}), {KIND_TEXT[kind]}; {dt:.2f} s per pass, "
                      f"extrapolated to the genome by the cost model 2 n m^2 + 120 m^2 ({genome_s:.1f} s per genome)",
            "sample_seconds": dt, "sample_blocks_per_s": blocks.size / dt, "genome_seconds": genome_s}


def relmax(a, b):
    a = np.asarray(a); b = np.asarray(b)
    if a.size == 0:
        return 0.0
    return float(np.abs(a - b).max() / max(float(np.abs(b).max()), 1e-300))


def pick(beta, off, blocks):
    return np.concatenate([beta[off[b]:off[b + 1]] for b in blocks]) if len(blocks) else np.zeros(0)


def main():
    args = parse()
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    total, chroms, cap, n_ref, n_obs = CONFIGS[args.config]
    workload_name = WORKLOAD_NAME[args.config]
    folds = [0.8, 1.0, 1.2] if args.config == "c4" else [1.0]

    # ---------------- reference arm: CPU only, rank 0 only
    if args.impl == "reference":
        if rank != 0:
            return
        dev = torch.device("cuda", local) if torch.cuda.is_available() else None
        if dev is None:
            print(json.dumps({"impl": "reference", "unavailable": "needs a CUDA device to synthesise the workload"}))
            return
        torch.cuda.set_device(dev)
        w = build_workload(args, torch, dev, args.seed)
        threads = min(os.cpu_count() or 1, 100)                 # reference caps -t at 100 (dbslmm.cpp:224)
        blocks = reference_sample(w["sizes"], w["n_ref"])
        sigma_s = 0.5 / w["nsnp_total"]
        times = []
        kind = "port"
        for i in range(min(args.warmup, 1) + args.steps):       # one warm-up pass is enough on the CPU
            dt, kind, ref_bs, ref_bl, _ = run_cpu(w, blocks, threads, sigma_s)
            if i >= min(args.warmup, 1):
                times.append(dt)
        dt = float(np.mean(times)) if times else float("nan")
        cl = cpu_line(w, blocks, dt, kind, threads)
        v = cl["value"]
        line = {"metric": "LD blocks fitted/sec genome-wide", "value": v, "unit": "blocks/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
                "config": {"workload": workload_name, "blocks": int(w["sizes"].size), "snps": int(w["n_snp"]), "n_ref": n_ref,
                           "n_obs": n_obs, "missing_rate": args.missing,
                           "sample": f"each step = the fixed {blocks.size}-block sample; value = 1,703-block genome / cost-extrapolated genome time"},
                "cpu_baseline": cl,
                "e2e": {"value": v, "unit": "blocks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"beta_s": ref_bs, "beta_l": ref_bl})
        return

    # ---------------- B200 arm
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback)")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from dbslmm_b200 import _abi
    seed = args.seed if args.scaling == "strong" else args.seed + 1000 * rank
    w = build_workload(args, torch, dev, seed)
    nb_total = int(w["sizes"].size)
    eng = _abi.Engine(local)
    ms_blk = (w["s_off"][1:] - w["s_off"][:-1]).astype(np.int32)
    ml_blk = (w["l_off"][1:] - w["l_off"][:-1]).astype(np.int32)
    if args.emulate_shard:
        er, en = (int(x) for x in args.emulate_shard.split("/"))
        owner, _ = eng.plan_shards(ms_blk, ml_blk, n_ref, en)
        my_rank = er
    elif args.scaling == "strong" and world > 1:
        owner, _ = eng.plan_shards(ms_blk, ml_blk, n_ref, world)
        my_rank = rank
    else:
        my_rank = 0 if args.scaling == "strong" else rank
        owner = np.zeros(nb_total, np.int32) + my_rank
    sh = shard_workload(w, owner, my_rank, torch)
    my_blocks = int(sh["blocks"].size)
    my_snps = int(sh["s_pos"].size + sh["l_pos"].size)
    sigma_s = [0.5 * f / w["nsnp_total"] for f in folds]
    solver = _abi.SOLVER_CHOLESKY if args.solver == "cholesky" else _abi.SOLVER_PCG
    fit_kw = dict(sigma_s=sigma_s, n_obs=n_obs, tau=0.8, solver=solver)
    csr = (sh["s_off"], sh["s_pos"], sh["s_z"], sh["l_off"], sh["l_pos"], sh["l_z"])

    fp64_peak = measure_fp64_peak(torch, dev) if rank == 0 else 0.0
    int8_peak = measure_int8_peak(torch, dev) if rank == 0 else None

    # c4: validation panel + scoring lists (every fitted SNP of this rank is scored; SNP j of the shard = row j of the panel)
    val = None
    if args.config == "c4":
        n_rows = int(sh["bed"].shape[0])
        val_bed = make_bed_cuda(torch, dev, n_rows, N_VAL, seed + 77)
        val = {"bed_t": val_bed, "bed": val_bed.numpy(), "pos": np.concatenate([sh["s_pos"], sh["l_pos"]]).astype(np.int32)}

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def score(r, prefetched=False):
        beta = np.concatenate([r["beta_s"], r["beta_l"]], axis=1)
        return eng.score(None if prefetched else val["bed"], N_VAL, val["pos"], beta)

    # ---- device-resident throughput (value)
    eng.load_bed(sh["bed"], n_ref)
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        r = eng.fit(*csr, **fit_kw)
        if val:
            score(r)
    barrier()
    sampler.mark()
    dev_ms, tms, prs_ms = [], [], []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = eng.fit(*csr, flags=_abi.FLAG_PLAN_CACHED, **fit_kw)
        t = r["timing"]
        tms.append(t)
        step_ms = t["total_ms"]                    # z upload -> decode -> Gram -> solve -> betas in pinned host memory
        if val:
            prs_timed, kms = score(r)
            prs_ms.append(kms)
            step_ms += kms
        dev_ms.append(step_ms)
    barrier()
    wall_resident = time.perf_counter() - t0
    clocks = sampler.stop()
    n_bad = int(r["n_bad"])
    beta_s_timed = r["beta_s"].copy()
    beta_l_timed = r["beta_l"].copy()

    # ---- end to end from host buffers (e2e): ONE C-ABI call per step takes the pinned host .bed shard and the CSR
    # block lists and returns the betas on the host -- the shape of the reference's DBSLMMFIT::est(bed_str, info, ...).
    # Inside the call the panel upload is cut into batches (big blocks first) and overlaps decode/Gram/Cholesky.
    # (c4: the validation panel is announced before the fit, so its 2.75 GB upload queues behind the reference panel's and
    # overlaps the fit's kernels; the scoring call then finds it on the device)
    def e2e_step():
        if val:
            eng.score_prefetch(val["bed"], N_VAL)
        rr = eng.fit(*csr, bed=sh["bed"], n_ref=n_ref, reuse_outputs=True, **fit_kw)
        if val:
            score(rr, prefetched=True)
        return rr
    for _ in range(min(args.warmup, 2)):
        r2 = e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r2 = e2e_step()
    barrier()
    wall_e2e = time.perf_counter() - t0
    stream_vs_resident = relmax(r2["beta_s"], beta_s_timed)
    # the same work as two calls (upload everything, then fit): what the overlap buys
    barrier()
    t0 = time.perf_counter()
    for _ in range(max(1, args.steps // 2)):
        eng.load_bed(sh["bed"], n_ref)
        eng.fit(*csr, **fit_kw)
    barrier()
    wall_two_call = (time.perf_counter() - t0) / max(1, args.steps // 2)

    # ---- parity (outside every timed region): the betas of the timed fit
    parity = None
    cpu_base = None
    if not args.no_parity:
        from oracle import oracle as O
        mine = sh["blocks"]
        # (1) exact oracle on a few of THIS rank's blocks: size quantiles 10/50/90/99 % among blocks of <= m_cap SNPs
        m_cap = int(min(2000, (2e10 / (2.0 * n_ref)) ** 0.5))     # keeps the oracle's FP64 Gram of one block under ~10 core-seconds
        ok = mine[w["sizes"][mine] <= m_cap]
        ok = ok[np.argsort(w["sizes"][ok], kind="stable")]
        chk = np.unique(ok[np.minimum((np.array([0.1, 0.5, 0.9, 0.99]) * ok.size).astype(int), max(ok.size - 1, 0))]) if ok.size else ok
        sub = sub_csr(w, chk)
        pos_in = {int(b): i for i, b in enumerate(mine)}
        local_idx = [pos_in[int(b)] for b in chk]
        ex = 0.0
        for f, sg in enumerate(sigma_s):
            bs, bl, _, _ = O.est(sub["bed"], n_ref, n_obs, sg, sub["s_off"], sub["s_pos"], sub["s_z"], sub["l_off"], sub["l_pos"],
                                 sub["l_z"], threads=min(len(chk), os.cpu_count() or 1), mode=O.MODE_EXACT)
            ex = max(ex, relmax(pick(beta_s_timed[f], sh["s_off"], local_idx), bs))
            if bl.size:
                ex = max(ex, relmax(pick(beta_l_timed[f], sh["l_off"], local_idx), bl))
        # (2) integer Gram of the two smallest checked blocks, bit for bit (a small extra fit that keeps the s32 planes)
        small = chk[np.argsort(w["sizes"][chk], kind="stable")][:2]
        sg2 = sub_csr(w, small)
        eng.load_bed(sg2["bed"], n_ref)
        eng.fit(sg2["s_off"], sg2["s_pos"], sg2["s_z"], sg2["l_off"], sg2["l_pos"], sg2["l_z"], sigma_s=sigma_s[:1], n_obs=n_obs,
                flags=_abi.FLAG_KEEP_INT_GRAM)
        gram_ok = True
        for i in range(small.size):
            pos_b = np.concatenate([sg2["s_pos"][sg2["s_off"][i]:sg2["s_off"][i + 1]], sg2["l_pos"][sg2["l_off"][i]:sg2["l_off"][i + 1]]]).astype(np.int32)
            Q, A, N = eng.block_gram(i, pos_b.size)
            Qo, Ao, No = O.gram_int(sg2["bed"], n_ref, pos_b)
            gram_ok = gram_ok and np.array_equal(Q, Qo) and np.array_equal(A, Ao) and np.array_equal(N, No)
        # (3) checksum of the gathered betas (fold 0): must not depend on the number of GPUs
        if dist is not None and args.scaling == "strong":
            from dbslmm_b200 import multigpu
            ww = {"s_off": w["s_off"], "l_off": w["l_off"]}
            full_s, full_l = multigpu.gather_betas(ww, owner, rank, world, beta_s_timed[0], beta_l_timed[0], dist)
        else:
            full_s, full_l = beta_s_timed[0], beta_l_timed[0]
        wts = np.cos(np.arange(full_s.size, dtype=np.float64) * 0.61803398875)
        checksum = {"sum_beta_s": float(full_s.sum()), "sum_abs_beta_s": float(np.abs(full_s).sum()),
                    "cos_weighted_beta_s": float((full_s * wts).sum()), "sum_abs_beta_l": float(np.abs(full_l).sum()),
                    "n_beta": int(full_s.size + full_l.size)}
        parity = {"max_rel_vs_exact_oracle": ex, "exact_blocks_checked_per_rank": int(chk.size), "gram_bit_exact": bool(gram_ok),
                  "gram_blocks_checked_per_rank": int(small.size), "streaming_vs_resident_max_rel": stream_vs_resident,
                  "beta_checksum": checksum, "blocks_not_spd": n_bad,
                  "norm": "max |beta_gpu - beta_cpu| / max |beta_cpu| over the checked blocks, small and large effects separately (max of the two)"}
        # (4) the reference's own CPU functions on the fixed sample (= the cpu_baseline leg): rank 0, and at N > 1 only
        # the sample blocks that rank 0 owns enter the comparison
        if rank == 0 and not args.no_cpu_baseline and args.config != "c4":
            try:
                threads = min(os.cpu_count() or 1, 100)
                blocks = reference_sample(w["sizes"], n_ref)
                dt, kind, rbs, rbl, rsub = run_cpu(w, blocks, threads, sigma_s[0])
                cpu_base = cpu_line(w, blocks, dt, kind, threads)
                own = [i for i, b in enumerate(blocks) if int(b) in pos_in]
                li = [pos_in[int(blocks[i])] for i in own]
                rv = relmax(pick(beta_s_timed[0], sh["s_off"], li), pick(rbs, rsub["s_off"], own))
                if rsub["l_off"][-1] > 0:
                    rv = max(rv, relmax(pick(beta_l_timed[0], sh["l_off"], li), pick(rbl, rsub["l_off"], own)))
                parity["max_rel_vs_reference"] = rv
                parity["reference_blocks_checked"] = len(own)
                parity["reference_note"] = ("the reference stops its PCG at an absolute residual of 1e-7 (dbslmmfit.cpp:648), so its own "
                                            "truncation error (1e-9 .. 1e-7 of max|beta|) bounds this figure; the exact-oracle figure is the gate")
            except Exception as e:  # the checker must never take the product bench down
                cpu_base = {"value": None, "unit": "blocks/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
        eng.load_bed(sh["bed"], n_ref)          # leave the engine as the timed loops had it
    elif rank == 0 and not args.no_cpu_baseline:
        try:
            threads = min(os.cpu_count() or 1, 100)
            blocks = reference_sample(w["sizes"], n_ref)
            dt, kind, _, _, _ = run_cpu(w, blocks, threads, sigma_s[0])
            cpu_base = cpu_line(w, blocks, dt, kind, threads)
        except Exception as e:
            cpu_base = {"value": None, "unit": "blocks/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}

    # --dump-outputs: with several GPUs in strong scaling the betas are gathered into workload order, so the files do not
    # depend on how the cost model sharded the blocks; the PRS of a rank is over its own validation panel and is left out
    outputs = None
    if args.dump_outputs:
        if dist is not None and args.scaling == "strong":
            from dbslmm_b200 import multigpu
            ww = {"s_off": w["s_off"], "l_off": w["l_off"]}
            full = [multigpu.gather_betas(ww, owner, rank, world, beta_s_timed[f], beta_l_timed[f], dist) for f in range(len(folds))]
            outputs = {"beta_s": np.stack([s for s, _ in full]), "beta_l": np.stack([l for _, l in full])}
        else:
            outputs = {"beta_s": beta_s_timed, "beta_l": beta_l_timed}
            if val:
                outputs["prs"] = prs_timed

    dev_total = float(np.sum(dev_ms))
    par_vec = [parity["max_rel_vs_exact_oracle"], 0.0 if parity["gram_bit_exact"] else 1.0, parity["streaming_vs_resident_max_rel"]] if parity else [0.0, 0.0, 0.0]
    stats = torch.tensor([dev_total, wall_e2e, wall_resident, float(my_blocks), float(my_snps), float(n_bad)] + par_vec, dtype=torch.float64, device=dev)
    if dist is not None:
        mx = stats.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_total, wall_e2e, wall_resident = float(mx[0]), float(mx[1]), float(mx[2])
        blocks_all, snps_all = float(sm[3]), float(sm[4])
        if parity:
            parity["max_rel_vs_exact_oracle"] = float(mx[6])
            parity["gram_bit_exact"] = bool(float(mx[7]) == 0.0)
            parity["streaming_vs_resident_max_rel"] = float(mx[8])
            parity["blocks_not_spd"] = int(sm[5])
            parity["ranks_checked"] = world
    else:
        blocks_all, snps_all = float(my_blocks), float(my_snps)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    K = args.steps
    value = blocks_all * K / (dev_total * 1e-3)
    e2e_v = blocks_all * K / wall_e2e
    avg = lambda k: float(np.mean([t[k] for t in tms]))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    chol_ms = avg("chol_ms")
    chol_flops = float(tms[-1]["solve_flops"])
    ach = chol_flops / (chol_ms * 1e-3) / 1e12 if chol_ms > 0 else 0.0
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "chol_traffic.json")))
        if world == 1 and args.config == "c3" and args.missing == 0.0:
            traffic = tj["dram_bytes_per_fit"]
    except Exception:
        pass
    roofline = {"bound": "tensor", "kernel": "chol_panel_tma_kernel<1> (64-row items, 128-thread CTAs) + chol_diag_kernel (all panel steps of one fit, all folds)",
                "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach / fp64_peak if fp64_peak else None,
                "traffic": traffic,
                "traffic_note": "dram__bytes_read+write summed over all chol_* launches of one fit (ncu, profiles/chol_traffic.json); "
                                "algorithmic flops / traffic = arithmetic intensity of the factorisation",
                "peak_source": "cuBLAS DGEMM 8192^3 measured in this run (MEASURED_PEAKS.json has no FP64 figure)",
                "flops_per_step": chol_flops, "ms_per_step": chol_ms}
    # decoder: algorithmic bytes = the .bed rows it reads (SURVEY 8d); the int8 codes it writes are reported separately
    bed_bytes = float(my_snps) * ((n_ref + 3) // 4)          # every .bed row is staged once, whatever planes it yields
    dec_ms, gram_ms = avg("decode_ms"), avg("gram_ms")
    dec_gbs = bed_bytes / (dec_ms * 1e-3) / 1e9 if dec_ms > 0 else 0.0
    dec_all_gbs = float(tms[-1]["decode_bytes"]) / (dec_ms * 1e-3) / 1e9 if dec_ms > 0 else 0.0
    gram_pops = float(tms[-1]["gram_ops"]) / (gram_ms * 1e-3) / 1e15 if gram_ms > 0 else 0.0
    sigma_bytes = float(np.sum((w["sizes"].astype(np.float64)) ** 2)) * 4.0     # lower triangle, 8 B
    # operand bytes the one-plane kernel pulls from L2 per fit: a 128 x 128 tile loads two [128 rows x n_pad] int8 strips
    # (one on the diagonal)
    _nt = np.ceil(np.ceil(w["sizes"] / 8.0) * 8.0 / 128.0)
    gram_l2_bytes = float(np.sum(_nt + _nt * (_nt - 1.0))) * 128.0 * float(((n_ref + 127) // 128) * 128)
    other = {"decode": {"bound": "hbm", "achieved": dec_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": dec_gbs / hbm_peak,
                        "bytes": ".bed rows read (algorithmic, SURVEY 8d)", "with_int8_codes_written_GBs": dec_all_gbs,
                        "with_int8_codes_written_frac": dec_all_gbs / hbm_peak, "peak_source": hbm_src, "ms": dec_ms},
             "gram": {"bound": "int8 tensor / hbm (Sigma write)", "achieved": gram_pops, "unit": "Pop/s", "peak": int8_peak,
                      "frac": (gram_pops / int8_peak) if int8_peak else None,
                      "peak_source": "torch._int_mm (cuBLASLt IGEMM s8 x s8 -> s32) 8192^3 measured in this run (MEASURED_PEAKS.json has no int8 figure)",
                      "sigma_write_GBs": sigma_bytes / (gram_ms * 1e-3) / 1e9 if world == 1 and gram_ms > 0 else None,
                      "sigma_write_frac_of_hbm": sigma_bytes / (gram_ms * 1e-3) / 1e9 / hbm_peak if world == 1 and gram_ms > 0 else None,
                      "operand_l2_GBs": gram_l2_bytes / (gram_ms * 1e-3) / 1e9 if world == 1 and gram_ms > 0 and args.missing == 0 else None,
                      "operand_l2_note": "128 x 128 tiles pull 32 KB of int8 operands per 128-sample K step and tile from L2 (TMA); ncu l1tex__m_xbar2l1tex_read_bytes agrees (profiles/r03_gram_single_full.txt).  No ceiling is claimed: the same kernel sustains 15.8 TB/s at C5 (157 K steps per tile) against 10.8 TB/s at C3 (16 K steps per tile)",
                      "ms": gram_ms},
             "solve_total_ms": avg("solve_ms"), "h2d_ms": avg("h2d_ms"), "d2h_ms": avg("d2h_ms"),
             "chol_class_ms": [float(np.mean([t["class_ms"][c] for t in tms])) for c in range(4)]}
    if val:
        vb = float(val["bed"].nbytes)
        other["prs"] = {"bound": "hbm", "ms": float(np.mean(prs_ms)), "achieved": vb / (np.mean(prs_ms) * 1e-3) / 1e9, "unit": "GB/s",
                        "peak": hbm_peak, "frac": vb / (np.mean(prs_ms) * 1e-3) / 1e9 / hbm_peak,
                        "bytes": "validation .bed rows read once for all folds", "n_val": N_VAL, "folds": len(folds)}
    h2d = int(sh["bed"].nbytes + 8 * my_snps + 24 * my_snps + (val["bed"].nbytes + 4 * my_snps + 8 * my_snps * len(folds) if val else 0))
    d2h = int(8 * my_snps * len(folds) + 8 * my_blocks + (8 * N_VAL * len(folds) if val else 0))
    line = {"metric": "LD blocks fitted/sec genome-wide", "value": value, "unit": "blocks/s", "n_gpus": world,
            "steps": K, "warmup": args.warmup, "ms_per_step": dev_total / K, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64 (int8 Gram, s32 accumulate)",
            "data": "synthetic", "impl": "b200",
            "config": {"workload": workload_name, "blocks": nb_total, "snps": int(w["n_snp"]), "n_ref": n_ref,
                       "n_obs": n_obs, "missing_rate": args.missing, "solver": args.solver, "h2_folds": folds,
                       "parallelism": f"blocks sharded over {world} GPU(s) by LPT cost model, no collective on the data path",
                       "l2": "inputs larger than L2 (codes 2.2 GB, Sigma 8+ GB per step)",
                       "value_window": "CUDA events, first (z upload) to last (betas in pinned host memory); the panel and the plan are resident"},
            "snps_per_s": snps_all * K / (dev_total * 1e-3),
            "e2e": {"value": e2e_v, "unit": "blocks/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": wall_e2e / K * 1e3,
                    "how": "one dbslmm_b200_fit call per step with fit_args.bed = pinned host .bed: batched H2D of the panel "
                           "overlapped with decode/Gram/Cholesky, plan + z H2D, betas written by the back substitution into pinned host memory (D2H over PCIe, "
                           "counted in d2h_bytes_per_step) and copied to the caller's arrays; wall clock",
                    "upload_then_fit_ms_per_step": wall_two_call * 1e3},
            "resident_wall_ms_per_step": wall_resident / K * 1e3,
            "gpu_launches": int(sum(t["n_launches"] for t in tms)) + (2 * K * ((len(folds) + 2) // 3) if val else 0),
            "clocks": clocks, "roofline": roofline, "rooflines_other": other, "blocks_not_spd": n_bad}
    if parity:
        line["parity"] = parity
    if cpu_base:
        line["cpu_baseline"] = cpu_base
    print(json.dumps(line), flush=True)
    if outputs:
        dump_outputs(args.dump_outputs, outputs)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
