"""The `score` command line (`plink --bfile <target> --score <eff>.txt 1 2 4 sum`, DBSLMM_script.sh:87): option and file
checks on the CPU (they all run before the GPU is touched); on the GPU, .profile files scored with the <eff>_f<k>.txt of a
real `dbslmm --h2-folds` run against a numpy restatement of PLINK's documented semantics."""
import os
import subprocess

import numpy as np
import pytest

from dbslmm_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCORE = os.path.join(ROOT, "build", "score")
DBSLMM = os.path.join(ROOT, "build", "dbslmm")
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module", autouse=True)
def _score_cli():
    from dbslmm_b200 import build
    build.build_cli()
    assert os.path.exists(SCORE)


def write_fileset(d, prefix, G, bim_rows, fam_rows=None, magic=(0x6C, 0x1B, 0x01)):
    """G int8 [n_snp, n]; bim_rows = [(chr, id, a1, a2)]; fam_rows = [(fid, iid, pat, mat, sex, pheno)]."""
    n = G.shape[1]
    fam_rows = fam_rows or [(f"F{i}", f"I{i}", "0", "0", "1", "-9") for i in range(n)]
    (d / f"{prefix}.fam").write_text("".join(" ".join(r) + "\n" for r in fam_rows))
    (d / f"{prefix}.bim").write_text("".join(f"{c}\t{v}\t0\t{1000 + k}\t{a1}\t{a2}\n" for k, (c, v, a1, a2) in enumerate(bim_rows)))
    with open(d / f"{prefix}.bed", "wb") as f:
        f.write(bytes(magic) + synth.pack_bed(G).tobytes())
    return str(d / prefix)


def run(*args, cwd=None):
    return subprocess.run([SCORE, *map(str, args)], capture_output=True, text=True, cwd=cwd)


def small_target(tmp_path, n=10, m=4):
    rng = np.random.default_rng(0)
    G = rng.integers(0, 3, (m, n)).astype(np.int8)
    bim = [("1", f"rs{k}", "A", "G") for k in range(m)]
    prefix = write_fileset(tmp_path, "t", G, bim)
    (tmp_path / "s.txt").write_text("".join(f"rs{k} A 0.1 {0.01 * (k + 1)} 0\n" for k in range(m)))
    return prefix, G, bim


# ---------------------------------------------------------------- CPU: options and file checks
def test_banner_and_help():
    r = run()
    assert r.returncode == 0 and "score" in r.stdout
    r = run("-h")
    assert r.returncode == 0 and "--bfile" in r.stdout and "--score" in r.stdout and "sum" in r.stdout


def test_option_checks(tmp_path):
    prefix, _, _ = small_target(tmp_path)
    s = tmp_path / "s.txt"
    r = run("--bfile", prefix, "--score", s, "1", "2", "4")
    assert r.returncode == 1 and "`sum`" in r.stderr
    for mod in ("no-mean-imputation", "double-dosage", "center", "include-cnt"):
        r = run("--bfile", prefix, "--score", s, "1", "2", "4", "sum", mod)
        assert r.returncode == 1 and f"'{mod}'" in r.stderr, mod
    r = run("--bfile", prefix, "--score", s, "sum", "--read-freq", "x.frq")
    assert r.returncode == 1 and "'--read-freq'" in r.stderr
    r = run("--bfile", prefix, "--score", s, "1", "2", "sum")
    assert r.returncode == 1 and "three column numbers" in r.stderr
    r = run("--score", s, "sum")
    assert r.returncode == 1 and "--bfile is required" in r.stderr
    r = run("--bfile", prefix, "--score", tmp_path / "nope.txt", "sum")
    assert r.returncode == 1 and "does not exist" in r.stderr


def test_bed_checks(tmp_path):
    prefix, G, bim = small_target(tmp_path)
    s = tmp_path / "s.txt"
    os.rename(prefix + ".bed", prefix + ".bak")
    r = run("--bfile", prefix, "--score", s, "sum")
    assert r.returncode == 1 and "does not exist" in r.stderr
    raw = open(prefix + ".bak", "rb").read()
    open(prefix + ".bed", "wb").write(raw[:-1])                                     # truncated
    r = run("--bfile", prefix, "--score", s, "sum")
    assert r.returncode == 1 and "3 + n_snp x ceil(n/4)" in r.stderr
    open(prefix + ".bed", "wb").write(raw + b"\0")                                  # one byte too many
    assert run("--bfile", prefix, "--score", s, "sum").returncode == 1
    open(prefix + ".bed", "wb").write(bytes([0x6C, 0x1C, 0x01]) + raw[3:])           # wrong magic
    r = run("--bfile", prefix, "--score", s, "sum")
    assert r.returncode == 1 and "magic" in r.stderr
    open(prefix + ".bed", "wb").write(bytes([0x6C, 0x1B, 0x00]) + raw[3:])           # individual-major
    r = run("--bfile", prefix, "--score", s, "sum")
    assert r.returncode == 1 and "individual-major" in r.stderr


def test_score_file_and_fileset_checks(tmp_path):
    prefix, G, bim = small_target(tmp_path)
    s = tmp_path / "s.txt"
    (tmp_path / "dup.txt").write_text("rs0 A 0.1 0.2 0\nrs1 A 0.1 0.2 0\nrs0 A 0.1 0.3 0\n")
    r = run("--bfile", prefix, "--score", tmp_path / "dup.txt", "sum")
    assert r.returncode == 1 and "'rs0' is repeated" in r.stderr
    # several files: same variants and alleles in the same order, or an error
    (tmp_path / "s2.txt").write_text("".join(f"rs{k} A 0.1 0.5 0\n" for k in (0, 1, 3, 2)))
    r = run("--bfile", prefix, "--score", f"{s},{tmp_path / 's2.txt'}", "sum")
    assert r.returncode == 1 and "same variants and alleles in the same order" in r.stderr
    (tmp_path / "s3.txt").write_text("".join(f"rs{k} {'G' if k == 1 else 'A'} 0.1 0.5 0\n" for k in range(4)))
    r = run("--bfile", prefix, "--score", f"{s},{tmp_path / 's3.txt'}", "sum")
    assert r.returncode == 1 and "same variants and alleles in the same order" in r.stderr
    (tmp_path / "s4.txt").write_text("".join(f"rs{k} A 0.1 0.5 0\n" for k in range(3)))
    r = run("--bfile", prefix, "--score", f"{s},{tmp_path / 's4.txt'}", "sum")
    assert r.returncode == 1 and "variants" in r.stderr
    (tmp_path / "short.txt").write_text("rs0 A 0.1\n")
    r = run("--bfile", prefix, "--score", tmp_path / "short.txt", "sum")
    assert r.returncode == 1 and "columns" in r.stderr
    # an ID that names several .bim rows
    write_fileset(tmp_path, "d", G, bim[:3] + [("1", "rs0", "A", "G")])
    r = run("--bfile", tmp_path / "d", "--score", s, "sum")
    assert r.returncode == 1 and "several rows" in r.stderr
    # a scored variant outside chromosomes 1-22
    write_fileset(tmp_path, "x", G, bim[:3] + [("X", "rs3", "A", "G")])
    r = run("--bfile", tmp_path / "x", "--score", s, "sum")
    assert r.returncode == 1 and "chromosome X" in r.stderr
    # a .fam with parents
    fam = [(f"F{i}", f"I{i}", "0", "0", "1", "-9") for i in range(10)]
    fam[4] = ("F4", "I4", "I1", "I2", "1", "-9")
    write_fileset(tmp_path, "p", G, bim, fam)
    r = run("--bfile", tmp_path / "p", "--score", s, "sum")
    assert r.returncode == 1 and "parents" in r.stderr


# ---------------------------------------------------------------- GPU: .profile files
def read_profile(path):
    rows = [ln.split() for ln in open(path).read().strip().split("\n")]
    assert rows[0] == ["FID", "IID", "PHENO", "CNT", "CNT2", "SCORESUM"]
    rows = rows[1:]
    return ([r[0] for r in rows], [r[1] for r in rows], [r[2] for r in rows], np.array([int(r[3]) for r in rows]),
            np.array([int(r[4]) for r in rows]), np.array([float(r[5]) for r in rows]))


def restate_profile(G, bim, score_lines, col=(1, 2, 4)):
    """PLINK 1.9 --score <f> varcol allelecol scorecol sum, restated: G int8 [n_snp, n] copies of bim A1 (-1 missing)."""
    row = {v: k for k, (_, v, _, _) in enumerate(bim)}
    n = G.shape[1]
    s = np.zeros(n)
    cnt = np.zeros(n, np.int64)
    cnt2 = np.zeros(n, np.int64)
    for t in score_lines:
        vid, al, x = t[col[0] - 1], t[col[1] - 1], float(t[col[2] - 1])
        if vid not in row or not np.isfinite(x):
            continue
        r = row[vid]
        if al == bim[r][2]:
            fl = False
        elif al == bim[r][3]:
            fl = True
        else:
            continue
        g = G[r]
        miss = g < 0
        if miss.all():
            continue
        d = np.where(miss, 0, g).astype(np.float64)
        d = 2.0 - d if fl else d
        mu = d[~miss].mean()
        s += x * np.where(miss, mu, d)
        cnt += 2 * (~miss)
        cnt2 += np.where(miss, 0, d).astype(np.int64)
    return s, cnt, cnt2


def _c1_fold_files(tmp_path):
    """<eff>_f<k>.txt of a real `dbslmm --h2-folds 0.8,1,1.2` run on the C1 test fixture."""
    d = np.load(os.path.join(GOLD, "c1_testdat.npz"))
    (tmp_path / "ref.bim").write_text(str(d["bim_txt"]))
    (tmp_path / "ref.fam").write_text("f i 0 0 0 -9\n" * int(d["fam_lines"]))
    with open(tmp_path / "ref.bed", "wb") as f:
        f.write(bytes([0x6C, 0x1B, 0x01]) + d["bed"].tobytes())
    (tmp_path / "summ.txt").write_text(str(d["summary_txt"]))
    (tmp_path / "blocks.bed").write_text(str(d["block_txt"]))
    cmd = [DBSLMM, "-s", tmp_path / "summ.txt", "-r", tmp_path / "ref", "-n", "2400", "-nsnp", "996", "-mafMax", "0.2",
           "-b", tmp_path / "blocks.bed", "-h", "0.5", "-t", "1", "-eff", tmp_path / "eff", "--h2-folds", "0.8,1,1.2"]
    r = subprocess.run(list(map(str, cmd)), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    files = [[ln.split() for ln in (tmp_path / f"eff_f{k}.txt").read_text().strip().split("\n")] for k in range(3)]
    ref_bim = [ln.split() for ln in str(d["bim_txt"]).strip().split("\n")]
    return files, {t[1]: (t[4], t[5]) for t in ref_bim}


@pytest.mark.gpu
def test_profiles_of_h2_folds_match_restatement(tmp_path):
    files, ref_alleles = _c1_fold_files(tmp_path)
    rng = np.random.default_rng(11)
    ids = [t[0] for t in files[0]]
    assert len(ids) > 200
    # target .bim: most scored IDs, some with A1/A2 swapped (flipped dosage), some with other alleles (mismatch), some
    # missing (unmatched), plus variants nobody scores; then a nan score in every file and one more only in the second
    bim = []
    kind = rng.choice(4, size=len(ids), p=[0.7, 0.15, 0.05, 0.10])
    for v, k in zip(ids, kind):
        a1, a2 = ref_alleles[v]
        if k == 0:
            bim.append(("1", v, a1, a2))
        elif k == 1:
            bim.append(("1", v, a2, a1))
        elif k == 2:
            bim.append(("1", v, "C" if "C" not in (a1, a2) else "T", "G" if "G" not in (a1, a2) else "A"))
    bim += [("1", f"extra{k}", "A", "G") for k in range(25)]
    order = rng.permutation(len(bim))
    bim = [bim[i] for i in order]
    n = 1237
    G = rng.binomial(2, rng.uniform(0.05, 0.5, len(bim))[:, None], size=(len(bim), n)).astype(np.int8)
    G[rng.random(G.shape) < 0.02] = -1
    G[5] = -1                                                                        # an all-missing target row
    fam = [(f"FAM{i}", f"ID{i}", "0", "0", str(1 + i % 2), "-9" if i % 3 == 0 else f"{rng.standard_normal():.4f}") for i in range(n)]
    prefix = write_fileset(tmp_path, "target", G, bim, fam)
    for k in range(3):
        files[k][3][3] = "nan"
    files[1][7][3] = "nan"
    paths = []
    for k in range(3):
        p = tmp_path / f"in_f{k}.txt"
        p.write_text("SNP A1 BETA SCORE FLAG\n" + "".join(" ".join(t) + "\n" for t in files[k]))
        paths.append(str(p))
    r = run("--bfile", prefix, "--score", ",".join(paths), "1", "2", "4", "header", "sum", "--out", tmp_path / "all")
    assert r.returncode == 0, r.stderr
    log = (tmp_path / "all.log").read_text()
    assert "with no ID match" in log and "neither A1 nor A2" in log and "non-finite" in log and "GPU kernel time" in log
    assert f"{n} individuals" in log
    for k in range(3):
        fid, iid, pheno, cnt, cnt2, s = read_profile(tmp_path / f"all_f{k}.profile")
        assert fid == [f[0] for f in fam] and iid == [f[1] for f in fam] and pheno == [f[5] for f in fam]
        es, ec, ec2 = restate_profile(G, bim, files[k])
        assert np.array_equal(cnt, ec) and np.array_equal(cnt2, ec2), k
        assert np.all(np.abs(s - es) <= 5e-6 * np.abs(es) + 1e-9 * np.abs(es).max()), k
        # the 3-file run equals a 1-file run of the same file
        r1 = run("--bfile", prefix, "--score", paths[k], "header", "sum", "--out", tmp_path / f"one{k}")
        assert r1.returncode == 0, r1.stderr
        assert (tmp_path / f"one{k}.profile").read_text() == (tmp_path / f"all_f{k}.profile").read_text()


@pytest.mark.gpu
def test_score_columns_and_default_out(tmp_path):
    """Other column numbers (beta in column 3), the default --out prefix `plink`, a single .profile."""
    prefix, G, bim = small_target(tmp_path, n=9, m=4)
    lines = [f"rs{k} {'G' if k == 2 else 'A'} {0.5 * (k + 1)} 0.0 0" for k in range(4)] + ["rs9 A 1.0 1.0 0"]
    (tmp_path / "s.txt").write_text("\n".join(lines) + "\n")
    r = run("--bfile", prefix, "--score", tmp_path / "s.txt", "1", "2", "3", "sum", cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    _, _, pheno, cnt, cnt2, s = read_profile(tmp_path / "plink.profile")
    es, ec, ec2 = restate_profile(G, bim, [ln.split() for ln in lines], col=(1, 2, 3))
    assert np.array_equal(cnt, ec) and np.array_equal(cnt2, ec2) and pheno == ["-9"] * 9
    assert np.all(np.abs(s - es) <= 5e-6 * np.abs(es) + 1e-12)
