"""The `ld` command line (`plink --r2 [gz] --ld-window N --ld-window-kb K --ld-window-r2 R`): option and file checks on the
CPU; on the GPU, the .ld table against tests/ld_pairs_ref.py at printed precision, gz against the plain file, and the log."""
import gzip
import os
import subprocess

import numpy as np
import pytest

from dbslmm_b200 import synth

import ld_pairs_ref as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LD = os.path.join(ROOT, "build", "ld")


@pytest.fixture(scope="module", autouse=True)
def _ld_cli():
    from dbslmm_b200 import build
    build.build_lib()
    build.build_cli()
    assert os.path.exists(LD)


def write_fileset(d, prefix, G, bim_rows, magic=(0x6C, 0x1B, 0x01)):
    n = G.shape[1]
    (d / f"{prefix}.fam").write_text("".join(f"F{i} I{i} 0 0 1 -9\n" for i in range(n)))
    (d / f"{prefix}.bim").write_text("".join(f"{c}\t{v}\t0\t{bp}\tA\tG\n" for c, v, bp in bim_rows))
    with open(d / f"{prefix}.bed", "wb") as f:
        f.write(bytes(magic) + synth.pack_bed(G).tobytes())
    return str(d / prefix)


def run(*args):
    return subprocess.run([LD, *map(str, args)], capture_output=True, text=True)


def small_panel(tmp_path, chroms=("1", "1", "1", "2", "2"), bp=(100, 200, 300, 100, 400), **kw):
    G = np.random.default_rng(0).integers(0, 3, (len(chroms), 12)).astype(np.int8)
    return write_fileset(tmp_path, "p", G, [(c, f"rs{k}", b) for k, (c, b) in enumerate(zip(chroms, bp))], **kw)


# ---------------------------------------------------------------- CPU: options and files, refused before the GPU
def test_help():
    r = run("-h")
    assert r.returncode == 0 and "--ld-window-kb" in r.stdout


@pytest.mark.parametrize("extra,msg", [
    (["--r"], "--r is not supported"),
    (["--r2", "square"], "modifier 'square'"), (["--r2", "square0"], "modifier"), (["--r2", "triangle"], "modifier"),
    (["--r2", "bin"], "modifier"), (["--r2", "bin4"], "modifier"), (["--r2", "dprime"], "modifier"),
    (["--r2", "with-freqs"], "modifier"), (["--r2", "gz", "inter-chr"], "modifier 'inter-chr'"),
    (["--ld-snp", "rs1"], "unsupported option '--ld-snp'"), (["--ld-snp-list", "x"], "unsupported option"),
    (["--maf", "0.01"], "unsupported option"), (["--keep", "k"], "unsupported option"), (["--extract", "e"], "unsupported option"),
    (["--ld-window", "1"], "--ld-window needs"), (["--ld-window", "2.5"], "--ld-window needs"),
    (["--ld-window-kb", "-1"], "--ld-window-kb needs"), (["--ld-window-r2", "1.5"], "--ld-window-r2 needs"),
    (["--ld-window-r2", "-0.1"], "--ld-window-r2 needs"), (["--ld-window-r2", "x"], "needs a number"),
])
def test_option_refusals(tmp_path, extra, msg):
    p = small_panel(tmp_path)
    base = ["--bfile", p, "--out", tmp_path / "o"]
    args = base + (extra if extra[0] == "--r2" else ["--r2"] + extra)
    r = run(*args)
    assert r.returncode == 1 and msg in r.stderr, (extra, r.stderr)
    assert not os.path.exists(tmp_path / "o.ld")


def test_required_options(tmp_path):
    p = small_panel(tmp_path)
    assert "--r2 is required" in run("--bfile", p, "--out", tmp_path / "o").stderr
    assert "--bfile is required" in run("--r2", "--out", tmp_path / "o").stderr
    assert "--out is required" in run("--bfile", p, "--r2").stderr


def test_bad_files(tmp_path):
    p = small_panel(tmp_path, chroms=("1", "2", "1", "3", "3"))
    assert "not contiguous" in run("--bfile", p, "--r2", "--out", tmp_path / "o").stderr
    d = tmp_path / "s"
    d.mkdir()
    p = small_panel(d, bp=(100, 300, 200, 100, 400))
    assert "not sorted" in run("--bfile", p, "--r2", "--out", d / "o").stderr
    d = tmp_path / "m"
    d.mkdir()
    p = small_panel(d, magic=(0x6C, 0x1B, 0x00))
    assert "individual-major" in run("--bfile", p, "--r2", "--out", d / "o").stderr
    d = tmp_path / "t"
    d.mkdir()
    p = small_panel(d)
    with open(p + ".bed", "ab") as f:
        f.write(b"\0")
    assert "bytes" in run("--bfile", p, "--r2", "--out", d / "o").stderr
    os.remove(p + ".fam")
    assert "does not exist" in run("--bfile", p, "--r2", "--out", d / "o").stderr


# ---------------------------------------------------------------- GPU: the table and the log
@pytest.mark.gpu
def test_table_gz_and_log(tmp_path):
    rng = np.random.default_rng(9)
    m = 400
    G = P.ld_panel(rng, m, 333, 0.02)
    G[50] = 1                                                         # no pair
    bp = np.concatenate([np.cumsum(rng.choice([0, 1000, 3000], 250)), np.cumsum(rng.choice([0, 1000, 3000], 150))]).astype(np.int64)
    chroms = ["1"] * 250 + ["7"] * 150
    p = write_fileset(tmp_path, "q", G, [(c, f"rs{k}", b) for k, (c, b) in enumerate(zip(chroms, bp))])
    args = ["--bfile", p, "--ld-window", 20, "--ld-window-kb", 30, "--ld-window-r2", 0.1]
    r = run(*args, "--r2", "--out", tmp_path / "o")
    assert r.returncode == 0, r.stderr
    r = run(*args, "--r2", "gz", "--out", tmp_path / "z")
    assert r.returncode == 0, r.stderr
    plain = (tmp_path / "o.ld").read_text()
    assert gzip.decompress((tmp_path / "z.ld.gz").read_bytes()).decode() == plain
    lines = plain.splitlines()
    assert lines[0].split() == ["CHR_A", "BP_A", "SNP_A", "CHR_B", "BP_B", "SNP_B", "R2"]
    e = P.ld_pairs_exact(G, [0, 250, 400], bp.astype(np.float64), 20, 30000.0, None)
    want = {(int(a), int(b)): float(r2) for a, b, r2 in zip(e["a"], e["b"], e["r2"])}
    got = []
    for ln in lines[1:]:
        t = ln.split()
        a, b = int(t[2][2:]), int(t[5][2:])
        assert t[0] == chroms[a] and t[3] == chroms[b] and int(t[1]) == bp[a] and int(t[4]) == bp[b]
        assert abs(float(t[6]) - want[(a, b)]) <= 5e-6 * max(want[(a, b)], 1e-300), (a, b)
        got.append((a, b))
    assert got == sorted(got)
    sel = {k for k, v in want.items() if v >= 0.1 + 1e-12}
    assert sel <= set(got) and all(want[k] >= 0.1 - 1e-12 for k in got)
    log = (tmp_path / "o.log").read_text()
    n_miss = int(sum(e["miss"][i] for i, k in enumerate(zip(e["a"], e["b"])) if (int(k[0]), int(k[1])) in set(got)))
    assert f"{len(got)} pairs written" in log and "1 variant(s) with no called genotype or zero variance" in log
    assert f"{n_miss} pair(s) with a SNP with missing calls" in log
