"""In-tree build of the sm_100a library and the `dbslmm` CLI (explicit nvcc / g++ calls).

    python -m dbslmm_b200.build            # libdbslmm_b200.so + build/dbslmm, build/valid, build/score, build/ldscore, build/ld
Outputs stay inside the repo (git-ignored) so they travel with a gpurun snapshot.
"""
import concurrent.futures as cf
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
HOST = os.path.join(PKG, "host")
BUILD = os.path.join(ROOT, "build")
LIB = os.path.join(PKG, "libdbslmm_b200.so")
CLI = os.path.join(BUILD, "dbslmm")
VALID_CLI = os.path.join(BUILD, "valid")
SCORE_CLI = os.path.join(BUILD, "score")
LDSCORE_CLI = os.path.join(BUILD, "ldscore")
LD_CLI = os.path.join(BUILD, "ld")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
GXX = "/usr/bin/g++"
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
CU_FLAGS = ["-O3", "-lineinfo", "-std=c++17", "-ccbin", GXX, "-Xcompiler", "-fPIC,-fvisibility=hidden",
            "-Xptxas", "-v"]
CU_SOURCES = ["decode.cu", "gram.cu", "chol.cu", "score.cu", "variance.cu", "pcg.cu", "ldscore.cu", "engine.cu"]
HOST_SOURCES = ["dbslmm_main.cpp", "ingest.cpp"]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _run(cmd, log=None):
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if log:
        with open(log, "w") as f:
            f.write(" ".join(cmd) + "\n" + p.stdout)
    if p.returncode != 0:
        sys.stderr.write(p.stdout)
        raise RuntimeError("build step failed: " + " ".join(cmd))
    return p.stdout


def build_lib(force=False, verbose=False):
    os.makedirs(BUILD, exist_ok=True)
    headers = [os.path.join(CSRC, h) for h in ("common.cuh", "kernels.h")] + [os.path.join(ROOT, "include", "dbslmm_b200.h")]
    srcs = [s for s in CU_SOURCES if os.path.exists(os.path.join(CSRC, s))]
    objs, jobs = [], []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(BUILD, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _newer(obj, [src] + headers):
            jobs.append(([NVCC] + ARCH + CU_FLAGS + ["-c", src, "-o", obj], os.path.join(BUILD, s + ".ptxas.log")))
    with cf.ThreadPoolExecutor(max_workers=max(1, len(jobs))) as ex:
        for out in ex.map(lambda j: _run(*j), jobs):
            if verbose:
                print(out)
    if force or jobs or _newer(LIB, objs):
        _run([NVCC] + ARCH + ["-shared", "-ccbin", GXX, "-o", LIB] + objs + ["-cudart", "static"])
    return LIB


def build_cli(force=False):
    srcs = [os.path.join(HOST, s) for s in HOST_SOURCES if os.path.exists(os.path.join(HOST, s))]
    if not srcs:
        return None
    deps = srcs + [LIB, os.path.join(HOST, "ingest.hpp"), os.path.join(ROOT, "include", "dbslmm_b200.h")]
    if force or _newer(CLI, deps):
        _run([GXX, "-O2", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", CLI] + srcs +
             ["-L", PKG, "-ldbslmm_b200", "-Wl,-rpath,$ORIGIN/../dbslmm_b200", "-Wl,-rpath," + PKG])
    # the reference's second binary, `valid` (external validation; SURVEY 8f-4)
    vsrcs = [os.path.join(HOST, "valid_main.cpp"), os.path.join(HOST, "ingest.cpp")]
    if os.path.exists(vsrcs[0]) and (force or _newer(VALID_CLI, vsrcs + deps)):
        _run([GXX, "-O2", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", VALID_CLI] + vsrcs +
             ["-L", PKG, "-ldbslmm_b200", "-Wl,-rpath,$ORIGIN/../dbslmm_b200", "-Wl,-rpath," + PKG])
    # `score`: plink --score <eff>.txt 1 2 4 sum over a target fileset (DBSLMM_script.sh:87), every fold in one pass
    ssrc = os.path.join(HOST, "score_main.cpp")
    if os.path.exists(ssrc) and (force or _newer(SCORE_CLI, [ssrc, os.path.join(HOST, "plink_bed.hpp")] + deps)):
        _run([GXX, "-O2", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", SCORE_CLI, ssrc] +
             ["-L", PKG, "-ldbslmm_b200", "-Wl,-rpath,$ORIGIN/../dbslmm_b200", "-Wl,-rpath," + PKG])
    # `ldscore`: ldsc.py --bfile <panel> --l2 (LD Scores of the reference panel, the input of LDSC's -h / -nsnp)
    lsrc = os.path.join(HOST, "ldscore_main.cpp")
    ldeps = [lsrc, os.path.join(HOST, "plink_bed.hpp")] + deps
    if os.path.exists(lsrc) and (force or _newer(LDSCORE_CLI, ldeps)):
        _run([GXX, "-O2", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", LDSCORE_CLI, lsrc] +
             ["-L", PKG, "-ldbslmm_b200", "-Wl,-rpath,$ORIGIN/../dbslmm_b200", "-Wl,-rpath," + PKG, "-lz"])
    # `ld`: plink --r2 (the table of SNP pairs within a window and their r^2)
    dsrc = os.path.join(HOST, "ld_main.cpp")
    ddeps = [dsrc, os.path.join(HOST, "plink_bed.hpp"), os.path.join(CSRC, "hostpool.hpp")] + deps
    if os.path.exists(dsrc) and (force or _newer(LD_CLI, ddeps)):
        _run([GXX, "-O2", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", LD_CLI, dsrc] +
             ["-L", PKG, "-ldbslmm_b200", "-Wl,-rpath,$ORIGIN/../dbslmm_b200", "-Wl,-rpath," + PKG, "-lz"])
    return CLI


def main():
    force = "--force" in sys.argv
    print(build_lib(force=force, verbose="-v" in sys.argv))
    print(build_cli(force=force))


if __name__ == "__main__":
    main()
