"""`ldscore --annot FILE [--thin-annot]` (`ldsc.py --l2 --annot`): the annotation file checks on the CPU; on the GPU, the
written file set (.l2.ldscore.gz with one <name>L2 column per annotation, .l2.M and .l2.M_5_50 with one sum per
annotation) against the restatement of tests/ldscore_annot_ref.py, for full and thin, plain and gzip files."""
import gzip
import os
import subprocess

import numpy as np
import pytest

import ldscore_annot_ref as A
import ldscore_ref as R
from test_ldscore_cli import LDSCORE, two_chromosome_panel, write_fileset


@pytest.fixture(scope="module", autouse=True)
def _ldscore_cli():
    from dbslmm_b200 import build
    build.build_lib()
    build.build_cli()
    assert os.path.exists(LDSCORE)


def run(*args):
    return subprocess.run([LDSCORE, *map(str, args)], capture_output=True, text=True)


def write_annot(path, bim, names, a, thin=False, gz=False, snp=None):
    lines = ["\t".join(([] if thin else ["CHR", "BP", "SNP", "CM"]) + list(names))]
    for i, (c, v, cm, bp) in enumerate(bim):
        vals = [repr(float(x)) for x in a[i]]
        lines.append("\t".join(vals if thin else [c, str(bp), v if snp is None else snp[i], str(cm)] + vals))
    text = "\n".join(lines) + "\n"
    if gz:
        with gzip.open(path, "wt") as f:
            f.write(text)
    else:
        open(path, "w").write(text)
    return path


def small(tmp_path):
    rng = np.random.default_rng(0)
    G = rng.integers(0, 3, (5, 12)).astype(np.int8)
    bim = [("1", f"rs{k}", f"{k * 1e-6:.6f}", 100 * (k + 1)) for k in range(5)]
    return write_fileset(tmp_path, "p", G, bim), bim


# ---------------------------------------------------------------- CPU: the annotation file checks (before the GPU)
def test_annot_refusals(tmp_path):
    p, bim = small(tmp_path)
    base = ["--bfile", p, "--l2", "--ld-wind-snps", "1", "--out", tmp_path / "o"]
    a = np.arange(10, dtype=np.float64).reshape(5, 2)

    def refused(path, *extra, expect):
        r = run(*base, "--annot", path, *extra)
        assert r.returncode == 1 and expect in r.stderr, (expect, r.stderr)
        assert "cannot initialise the GPU" not in r.stderr

    refused(tmp_path / "missing.annot", expect="'--annot'")
    r = run(*base, "--thin-annot")
    assert r.returncode == 1 and "--thin-annot needs --annot" in r.stderr
    write_annot(tmp_path / "short.annot", bim[:4], ["x", "y"], a[:4])
    refused(tmp_path / "short.annot", expect="has 4 rows; the .bim has 5")
    write_annot(tmp_path / "long.annot", bim + [("1", "rs9", "0", 900)], ["x", "y"], np.vstack([a, a[:1]]))
    refused(tmp_path / "long.annot", expect="more rows than the .bim")
    write_annot(tmp_path / "snp.annot", bim, ["x", "y"], a, snp=["rs0", "rs1", "rsX", "rs3", "rs4"])
    refused(tmp_path / "snp.annot", expect="line 4: SNP rsX is not rs2")
    (tmp_path / "none.annot").write_text("CHR\tBP\tSNP\tCM\n" + "".join(f"1\t{b[3]}\t{b[1]}\t0\n" for b in bim))
    refused(tmp_path / "none.annot", expect="no annotation columns")
    (tmp_path / "empty.annot").write_text("")
    refused(tmp_path / "empty.annot", "--thin-annot", expect="no annotation columns")
    t = write_annot(tmp_path / "ragged.annot", bim, ["x", "y"], a).read_text().splitlines()
    t[3] += "\t7"
    (tmp_path / "ragged.annot").write_text("\n".join(t) + "\n")
    refused(tmp_path / "ragged.annot", expect="line 4: 7 columns, the header has 6")
    for bad in ("abc", "nan", "inf", "1e999", "0x"):
        t = write_annot(tmp_path / "bad.annot", bim, ["x", "y"], a).read_text().splitlines()
        t[2] = t[2].rsplit("\t", 1)[0] + "\t" + bad
        (tmp_path / "bad.annot").write_text("\n".join(t) + "\n")
        refused(tmp_path / "bad.annot", expect=f"line 3: '{bad}' (annotation y) is not a finite number")
    names = [f"a{k}" for k in range(4097)]
    write_annot(tmp_path / "wide.annot", bim, names, np.zeros((5, 4097)), thin=True)
    refused(tmp_path / "wide.annot", "--thin-annot", expect="4097 annotations; ldscore takes at most 4096")
    write_annot(tmp_path / "thin.annot", bim, ["x", "y"], a, thin=True)
    refused(tmp_path / "thin.annot", expect="no annotation columns")        # a thin file read as a full one
    for extra in (["--cts-bin", "x"], ["--per-allele"], ["--pq-exp", "1"]):
        r = run(*base, "--annot", tmp_path / "thin.annot", "--thin-annot", *extra)
        assert r.returncode == 1 and f"'{extra[0]}'" in r.stderr, extra
    assert not os.path.exists(tmp_path / "o.l2.ldscore.gz")


def test_help_lists_annot():
    r = run("-h")
    assert r.returncode == 0 and "--annot" in r.stdout and "--thin-annot" in r.stdout


# ---------------------------------------------------------------- GPU: the written file set
def clear_of_rounding(e):
    x = e["l2"][e["kept"]] * 1000.0
    return bool(np.all(np.abs(x - np.floor(x) - 0.5) > 1e-6))


def panel_and_annot(tmp_path, seed, C):
    """The two-chromosome panel of test_ldscore_cli with C columns: binary, signed multiples of 1/8, zeros, ones (every
    M sum exact in any order)."""
    p, G, bim, off, bp = two_chromosome_panel(tmp_path, seed)
    rng = np.random.default_rng(seed + 100)
    a = A.annot_columns(rng, G.shape[0], (["bin", "cont", "zero", "one"] * C)[:C])
    a[:, 1::4] = np.round(a[:, 1::4] * 8.0) / 8.0
    return p, G, bim, off, bp, a


@pytest.mark.gpu
@pytest.mark.parametrize("thin,gz", [(False, True), (True, False)])
def test_file_set_matches_restatement(tmp_path, thin, gz):
    for seed in range(31, 60):
        p, G, bim, off, bp, a = panel_and_annot(tmp_path, seed, 5)
        e = A.ldscore_annot_exact(G, off, a, bp, 1000.0 * 20, 0.01)
        if clear_of_rounding(e):
            break
    else:
        pytest.fail("no seed gives a panel clear of %.3f rounding edges")
    names = ["base", "cont", "zero", "ones", "bin2"]
    f = write_annot(tmp_path / ("a.annot.gz" if gz else "a.annot"), bim, names, a, thin=thin, gz=gz)
    thin_opt = ["--thin-annot"] if thin else []
    r = run("--bfile", p, "--l2", "--ld-wind-kb", "20", "--maf", "0.01", "--annot", f, *thin_opt, "--out", tmp_path / "all")
    assert r.returncode == 0, r.stderr
    chrom, snp, bps = [b[0] for b in bim], [b[1] for b in bim], [str(b[3]) for b in bim]
    assert gzip.open(tmp_path / "all.l2.ldscore.gz", "rt").read() == A.format_annot_ldscore(chrom, snp, bps, e["l2"], e["kept"], names)
    m, m550 = A.format_annot_counts(e["kept"], e["maf"], a)
    assert (tmp_path / "all.l2.M").read_text() == m and (tmp_path / "all.l2.M_5_50").read_text() == m550
    assert "read 5 annotation(s)" in (tmp_path / "all.log").read_text()
    ids = {f"rs{k}" for k in range(0, 500, 7)}
    (tmp_path / "ids.txt").write_text("".join(f"{v}\tx\n" for v in sorted(ids)))
    r = run("--bfile", p, "--l2", "--ld-wind-kb", "20", "--maf", "0.01", "--annot", f, *thin_opt, "--print-snps", tmp_path / "ids.txt",
            "--out", tmp_path / "sub")
    assert r.returncode == 0, r.stderr
    assert gzip.open(tmp_path / "sub.l2.ldscore.gz", "rt").read() == \
        A.format_annot_ldscore(chrom, snp, bps, e["l2"], e["kept"], names, ids)
    assert (tmp_path / "sub.l2.M").read_text() == m and (tmp_path / "sub.l2.M_5_50").read_text() == m550


@pytest.mark.gpu
def test_single_column_header_and_unannotated_files(tmp_path):
    for seed in range(61, 90):
        p, G, bim, off, bp, a = panel_and_annot(tmp_path, seed, 2)
        a = a[:, 1:2]                                    # one signed column
        e = A.ldscore_annot_exact(G, off, a, None, 40)
        u = R.ldscore_exact(G, off, None, 40)
        if clear_of_rounding(e) and clear_of_rounding(u):
            break
    else:
        pytest.fail("no seed gives a panel clear of %.3f rounding edges")
    f = write_annot(tmp_path / "one.annot", bim, ["only"], a)
    r = run("--bfile", p, "--l2", "--ld-wind-snps", "40", "--annot", f, "--out", tmp_path / "one")
    assert r.returncode == 0, r.stderr
    chrom, snp, bps = [b[0] for b in bim], [b[1] for b in bim], [str(b[3]) for b in bim]
    got = gzip.open(tmp_path / "one.l2.ldscore.gz", "rt").read()
    assert got.splitlines()[0] == "CHR\tSNP\tBP\tL2"
    assert got == A.format_annot_ldscore(chrom, snp, bps, e["l2"], e["kept"], ["only"])
    assert (tmp_path / "one.l2.M").read_text() == A.format_annot_counts(e["kept"], e["maf"], a)[0]
    r = run("--bfile", p, "--l2", "--ld-wind-snps", "40", "--out", tmp_path / "plain")         # without --annot: as before
    assert r.returncode == 0, r.stderr
    assert gzip.open(tmp_path / "plain.l2.ldscore.gz", "rt").read() == R.format_ldscore(chrom, snp, bps, u["l2"], u["kept"])
    assert (tmp_path / "plain.l2.M").read_text() == R.format_counts(u["kept"], u["maf"])[0]
