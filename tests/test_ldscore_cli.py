"""The `ldscore` command line (`ldsc.py --bfile <panel> --l2 ...`): option and file checks and the window rule on the CPU;
on the GPU, the written file set (.l2.ldscore.gz, .l2.M, .l2.M_5_50) against the extended-precision restatement of
tests/ldscore_ref.py."""
import gzip
import os
import subprocess

import numpy as np
import pytest

from dbslmm_b200 import _abi, synth

import ldscore_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LDSCORE = os.path.join(ROOT, "build", "ldscore")


@pytest.fixture(scope="module", autouse=True)
def _ldscore_cli():
    from dbslmm_b200 import build
    build.build_lib()
    build.build_cli()
    assert os.path.exists(LDSCORE)


def write_fileset(d, prefix, G, bim_rows, magic=(0x6C, 0x1B, 0x01)):
    """G int8 [n_snp, n]; bim_rows = [(chr, id, cm, bp)]."""
    n = G.shape[1]
    (d / f"{prefix}.fam").write_text("".join(f"F{i} I{i} 0 0 1 -9\n" for i in range(n)))
    (d / f"{prefix}.bim").write_text("".join(f"{c}\t{v}\t{cm}\t{bp}\tA\tG\n" for c, v, cm, bp in bim_rows))
    with open(d / f"{prefix}.bed", "wb") as f:
        f.write(bytes(magic) + synth.pack_bed(G).tobytes())
    return str(d / prefix)


def run(*args, cwd=None):
    return subprocess.run([LDSCORE, *map(str, args)], capture_output=True, text=True, cwd=cwd)


def small_panel(tmp_path, chroms=("1", "1", "1", "2", "2"), bp=(100, 200, 300, 100, 400)):
    rng = np.random.default_rng(0)
    G = rng.integers(0, 3, (len(chroms), 12)).astype(np.int8)
    bim = [(c, f"rs{k}", f"{b * 1e-6:.6f}", b) for k, (c, b) in enumerate(zip(chroms, bp))]
    return write_fileset(tmp_path, "p", G, bim), G, bim


# ---------------------------------------------------------------- CPU: options, files, window rule, formatting
def test_banner_and_help():
    r = run()
    assert r.returncode == 0 and "ldscore" in r.stdout
    r = run("-h")
    assert r.returncode == 0 and "--ld-wind-cm" in r.stdout and "--print-snps" in r.stdout


def test_option_refusals(tmp_path):
    p, _, _ = small_panel(tmp_path)
    base = ["--bfile", p, "--l2", "--out", tmp_path / "o"]
    for extra in (["--annot", "x"], ["--cts-bin", "x"], ["--keep", "k"], ["--extract", "e"], ["--per-allele"],
                  ["--pq-exp", "1"], ["--chunk-size", "50"], ["--h2", "x"]):
        r = run(*base, "--ld-wind-snps", "1", *extra)
        assert r.returncode == 1 and f"'{extra[0]}'" in r.stderr, extra
    r = run(*base)
    assert r.returncode == 1 and "exactly one of" in r.stderr
    r = run(*base, "--ld-wind-snps", "1", "--ld-wind-kb", "1")
    assert r.returncode == 1 and "exactly one of" in r.stderr
    r = run("--bfile", p, "--ld-wind-snps", "1", "--out", tmp_path / "o")
    assert r.returncode == 1 and "--l2 is required" in r.stderr
    r = run("--l2", "--ld-wind-snps", "1", "--out", tmp_path / "o")
    assert r.returncode == 1 and "--bfile is required" in r.stderr
    r = run("--bfile", p, "--l2", "--ld-wind-snps", "1")
    assert r.returncode == 1 and "--out is required" in r.stderr
    r = run(*base, "--ld-wind-snps", "1.5")
    assert r.returncode == 1 and "whole number" in r.stderr
    r = run(*base, "--ld-wind-kb", "-1")
    assert r.returncode == 1 and ">= 0" in r.stderr
    r = run(*base, "--ld-wind-kb", "1", "--maf", "0.5")
    assert r.returncode == 1 and "--maf" in r.stderr
    assert not os.path.exists(tmp_path / "o.l2.ldscore.gz")


def test_bed_checks(tmp_path):
    p, _, _ = small_panel(tmp_path)
    args = ["--bfile", p, "--l2", "--ld-wind-snps", "1", "--out", tmp_path / "o"]
    raw = open(p + ".bed", "rb").read()
    open(p + ".bed", "wb").write(raw[:-1])
    r = run(*args)
    assert r.returncode == 1 and "3 + n_snp x ceil(n/4)" in r.stderr
    open(p + ".bed", "wb").write(bytes([0x6C, 0x1C, 0x01]) + raw[3:])
    r = run(*args)
    assert r.returncode == 1 and "magic" in r.stderr
    open(p + ".bed", "wb").write(bytes([0x6C, 0x1B, 0x00]) + raw[3:])
    r = run(*args)
    assert r.returncode == 1 and "individual-major" in r.stderr
    os.remove(p + ".bed")
    r = run(*args)
    assert r.returncode == 1 and "does not exist" in r.stderr


def test_chromosome_checks(tmp_path):
    p, _, _ = small_panel(tmp_path, chroms=("1", "1", "2", "1", "2"), bp=(100, 200, 300, 400, 500))
    r = run("--bfile", p, "--l2", "--ld-wind-snps", "1", "--out", tmp_path / "o")
    assert r.returncode == 1 and "chromosome 1 is not contiguous" in r.stderr
    p, _, _ = small_panel(tmp_path, bp=(100, 300, 200, 100, 400))
    for w in ("--ld-wind-kb", "--ld-wind-cm"):
        r = run("--bfile", p, "--l2", w, "1", "--out", tmp_path / "o")
        assert r.returncode == 1 and "are not sorted" in r.stderr, w
    p, _, _ = small_panel(tmp_path)
    (tmp_path / "ids.txt").write_text("rs99 x\nrsX\n")
    r = run("--bfile", p, "--l2", "--ld-wind-snps", "1", "--print-snps", tmp_path / "ids.txt", "--out", tmp_path / "o")
    assert r.returncode == 1 and "no SNP of" in r.stderr


def test_window_rule():
    """ldsc's getBlockLefts, both ends, as the library applies it (host code): ties, a distance exactly equal to max_dist,
    duplicate positions, a one-SNP chromosome, the guard."""
    x = np.array([0.0, 0.0, 1.0, 2.0, 2.0, 2.0, 3.5, 5.5, 7.5, 7.5])
    lo, hi = _abi.ld_windows(x, 2.0)
    assert lo.tolist() == [0, 0, 0, 0, 0, 0, 3, 6, 7, 7]
    assert hi.tolist() == [5, 5, 5, 6, 6, 6, 7, 9, 9, 9]
    for d in (0.0, 0.5, 1.0, 2.0, 3.5, 7.5):
        lo, hi = _abi.ld_windows(x, d)
        elo, ehi = R.windows(x, d)
        assert lo.tolist() == elo.tolist() and hi.tolist() == ehi.tolist(), d
    assert _abi.ld_windows(x, 7.5)[0][-1] == 0 and _abi.ld_windows(x, 7.4)[0][-1] != 0       # the guard: last reaches first
    lo, hi = _abi.ld_windows(np.array([12.0]), 0.0)                                              # one SNP: its own window, guard
    assert lo.tolist() == [0] and hi.tolist() == [0]
    lo, hi = _abi.ld_windows(None, 2, m=6)                                                       # --ld-wind-snps 2
    assert lo.tolist() == [0, 0, 0, 1, 2, 3] and hi.tolist() == [2, 3, 4, 5, 5, 5]
    lo, hi = _abi.ld_windows(None, 0, m=3)
    assert lo.tolist() == [0, 1, 2] and hi.tolist() == [0, 1, 2]


def test_formatting_of_a_stub_result():
    chrom, snp, bp = ["1", "1", "1", "2", "2"], ["a", "b", "c", "d", "e"], ["10", "20", "30", "5", "6"]
    l2 = np.array([1.0, np.nan, -0.0004, 12.3456, 0.0005001])
    kept = np.array([True, False, True, True, True])
    maf = np.array([0.3, 0.0, 0.05, 0.0501, 0.2])
    assert R.format_ldscore(chrom, snp, bp, l2, kept) == "CHR\tSNP\tBP\tL2\n1\ta\t10\t1.000\n1\tc\t30\t-0.000\n2\td\t5\t12.346\n2\te\t6\t0.001\n"
    assert R.format_ldscore(chrom, snp, bp, l2, kept, {"d", "b"}) == "CHR\tSNP\tBP\tL2\n2\td\t5\t12.346\n"
    assert R.format_counts(kept, maf) == ("4\n", "3\n")


# ---------------------------------------------------------------- GPU: the written file set
def assert_clear_of_rounding(e):
    """No restated l2 lies within 1e-9 of a %.3f rounding boundary (the text comparison then tests the values, not luck)."""
    x = e["l2"][e["kept"]] * 1000.0
    assert np.all(np.abs(x - np.floor(x) - 0.5) > 1e-6), "a restated l2 lies within 1e-9 of a %.3f rounding boundary"


def two_chromosome_panel(tmp_path, seed):
    rng = np.random.default_rng(seed)
    n, m1, m2 = 403, 300, 200
    G = rng.binomial(2, rng.uniform(0.02, 0.5, m1 + m2)[:, None], size=(m1 + m2, n)).astype(np.int8)
    for k in range(1, m1 + m2):
        c = rng.random(n) < 0.6
        G[k, c] = G[k - 1, c]
    G[rng.random(G.shape) < 0.01] = -1
    G[7] = 1                                                         # dropped: all heterozygous
    G[m1 + 3] = 0                                                    # dropped: monomorphic
    bp = np.concatenate([np.cumsum(rng.choice([0, 1000, 2000, 5000], m1)), np.cumsum(rng.choice([0, 1000, 3000], m2))]) + 10000
    chrom = ["1"] * m1 + ["2"] * m2
    bim = [(c, f"rs{k}", f"{b * 1e-6:.6f}", int(b)) for k, (c, b) in enumerate(zip(chrom, bp))]
    return write_fileset(tmp_path, "ref", G, bim), G, bim, [0, m1, m1 + m2], bp.astype(np.float64)


@pytest.mark.gpu
def test_file_set_matches_restatement(tmp_path):
    p, G, bim, off, bp = two_chromosome_panel(tmp_path, 21)
    e = R.ldscore_exact(G, off, bp, 1000.0 * 20, 0.01)
    assert_clear_of_rounding(e)
    chrom, snp, bps = [b[0] for b in bim], [b[1] for b in bim], [str(b[3]) for b in bim]
    r = run("--bfile", p, "--l2", "--ld-wind-kb", "20", "--maf", "0.01", "--out", tmp_path / "all")
    assert r.returncode == 0, r.stderr
    got = gzip.open(tmp_path / "all.l2.ldscore.gz", "rt").read()
    assert got == R.format_ldscore(chrom, snp, bps, e["l2"], e["kept"])
    m, m550 = R.format_counts(e["kept"], e["maf"])
    assert (tmp_path / "all.l2.M").read_text() == m and (tmp_path / "all.l2.M_5_50").read_text() == m550
    assert "GPU kernel time" in (tmp_path / "all.log").read_text()
    ids = {f"rs{k}" for k in range(0, 500, 7)}
    (tmp_path / "ids.txt").write_text("".join(f"{v}\tx\n" for v in sorted(ids)))
    r = run("--bfile", p, "--l2", "--ld-wind-kb", "20", "--maf", "0.01", "--print-snps", tmp_path / "ids.txt", "--out", tmp_path / "sub")
    assert r.returncode == 0, r.stderr
    assert gzip.open(tmp_path / "sub.l2.ldscore.gz", "rt").read() == R.format_ldscore(chrom, snp, bps, e["l2"], e["kept"], ids)
    assert (tmp_path / "sub.l2.M").read_text() == m and (tmp_path / "sub.l2.M_5_50").read_text() == m550


@pytest.mark.gpu
def test_cm_and_snp_windows_and_the_guard(tmp_path):
    p, G, bim, off, bp = two_chromosome_panel(tmp_path, 22)
    chrom, snp, bps = [b[0] for b in bim], [b[1] for b in bim], [str(b[3]) for b in bim]
    cm = np.array([float(b[2]) for b in bim])
    r = run("--bfile", p, "--l2", "--ld-wind-cm", "0.01", "--out", tmp_path / "cm")
    assert r.returncode == 0, r.stderr
    e = R.ldscore_exact(G, off, cm, 0.01)
    assert_clear_of_rounding(e)
    assert gzip.open(tmp_path / "cm.l2.ldscore.gz", "rt").read() == R.format_ldscore(chrom, snp, bps, e["l2"], e["kept"])
    r = run("--bfile", p, "--l2", "--ld-wind-snps", "250", "--out", tmp_path / "w")               # spans chromosome 2 (199 kept)
    assert r.returncode == 1 and "chromosome 2" in r.stderr and "--yes-really" in r.stderr
    assert "GPU kernel time" not in r.stdout                                                        # refused after the statistics pass
    assert not os.path.exists(tmp_path / "w.l2.ldscore.gz")
    r = run("--bfile", p, "--l2", "--ld-wind-snps", "250", "--yes-really", "--out", tmp_path / "w")
    assert r.returncode == 0, r.stderr
    e = R.ldscore_exact(G, off, None, 250)
    assert_clear_of_rounding(e)
    assert gzip.open(tmp_path / "w.l2.ldscore.gz", "rt").read() == R.format_ldscore(chrom, snp, bps, e["l2"], e["kept"])
