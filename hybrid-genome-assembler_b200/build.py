"""Builds libhga_b200.so (CUDA kernels + C-ABI, sm_100a only) and the `categorization` / `jf_occurrences` host executables, in-tree.

    python hybrid-genome-assembler_b200/build.py [--force] [--verbose]

nvcc cross-compiles without a GPU. Objects are cached under hybrid-genome-assembler_b200/build/ by source mtime.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
CLI = os.path.join(HERE, "cli")
BUILD = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libhga_b200.so")
EXE = os.path.join(HERE, "categorization")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-Xptxas", "-v",
              "--expt-relaxed-constexpr", "-I", os.path.join(ROOT, "include")]
CPP_SOURCES = ["hga_spectral.cpp", "hga_tails.cpp", "hga_sdk.cpp", "hga_pack.cpp"]        # host-only translation units (g++)
CU_SOURCES = ["hga_capi.cu", "hga_table.cu", "hga_scan.cu", "hga_index.cu", "hga_pairs.cu", "hga_select.cu", "hga_cc.cu", "hga_enrich.cu", "hga_comm.cu", "hga_count.cu"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _run(cmd, verbose):
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        raise RuntimeError("build failed: " + " ".join(cmd[:3]))
    if verbose:
        sys.stderr.write(r.stderr)
    return r.stderr


def build(force=False, verbose=False):
    os.makedirs(BUILD, exist_ok=True)
    headers = [os.path.join(CSRC, "hga_internal.cuh"), os.path.join(CSRC, "hga_pack.h"), os.path.join(ROOT, "include", "hga_b200.h")]
    objs, jobs = [], []
    for src in CU_SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(BUILD, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            jobs.append([NVCC] + NVCC_FLAGS + ["-c", s, "-o", o])
    for src in CPP_SOURCES:
        sfile = os.path.join(CSRC, src)
        o = os.path.join(BUILD, src.replace(".cpp", ".o"))
        objs.append(o)
        if force or _stale(o, [sfile] + headers):
            jobs.append(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-Wall", "-I", os.path.join(ROOT, "include"), "-c", sfile, "-o", o])
    logs = {}
    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for cmd, log in zip(jobs, ex.map(lambda c: _run(c, verbose), jobs)):
                logs[os.path.basename(cmd[-3])] = log
        with open(os.path.join(BUILD, "ptxas.log"), "a") as f:
            for k, v in logs.items():
                f.write(f"==== {k}\n{v}\n")
    if force or jobs or _stale(LIB, objs):
        _run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs + ["-lcudart", "-ldl"], verbose)
    cli_src = os.path.join(CLI, "categorization.cpp")
    if os.path.exists(cli_src):
        cli_deps = [os.path.join(CLI, f) for f in os.listdir(CLI)] + headers
        if force or _stale(EXE, cli_deps) or _stale(EXE, [LIB]):
            _run(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", CLI, "-o", EXE, cli_src,
                  "-L", HERE, "-lhga_b200", "-Wl,-rpath,$ORIGIN", "-lpthread"], verbose)
    occ_src = os.path.join(CLI, "jf_occurrences.cpp")
    occ_exe = os.path.join(HERE, "jf_occurrences")
    if os.path.exists(occ_src) and (force or _stale(occ_exe, [occ_src, os.path.join(CLI, "hga_host.h")] + headers) or _stale(occ_exe, [LIB])):
        _run(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", CLI, "-o", occ_exe, occ_src,
              "-L", HERE, "-lhga_b200", "-Wl,-rpath,$ORIGIN", "-lpthread"], verbose)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(LIB)
