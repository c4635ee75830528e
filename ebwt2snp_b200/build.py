"""Builds the CUDA library and the CLIs in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m ebwt2snp_b200.build            # library + CLIs
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")
LIB_DIR = os.path.join(HERE, "lib")
BIN_DIR = os.path.join(HERE, "bin")
LIB = os.path.join(LIB_DIR, "libebwt2snp_b200.so")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
CUFLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-cudart", "static"] + ARCH

CU_SOURCES = ["ctx.cu", "shard.cu", "build_host.cu", "phase1.cu", "phase2.cu", "pipeline.cu", "cluster.cu", "scan.cu", "merge.cu", "snp.cu", "unpack.cu", "build_egsa.cu"]
CLI_SOURCES = {"ebwt2clust": ["ebwt2clust_main.cpp"], "clust2snp": ["clust2snp_main.cpp"], "build_gesa": ["build_gesa_main.cpp"],
               "ebwt2snp": ["ebwt2snp_main.cpp"]}
# text post-processors of the .snp format (no GPU work, no library): SURVEY.md 8(f) rank 3
TEXT_TOOLS = {"filter_snp": ["filter_snp_main.cpp"], "snp2fastq": ["snp2fastq_main.cpp"], "snp_vs_vcf": ["snp_vs_vcf_main.cpp"]}


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("build failed: " + " ".join(cmd))
    if verbose and (r.stdout or r.stderr):
        print(r.stdout + r.stderr)


def build_library(force=False, verbose=False, extra=()):
    os.makedirs(LIB_DIR, exist_ok=True)
    srcs = [os.path.join(CSRC, f) for f in CU_SOURCES]
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    deps.append(os.path.join(ROOT, "include", "ebwt2snp_b200.h"))
    if force or _newer(LIB, deps):
        objs = []
        for s in srcs:
            o = os.path.join(LIB_DIR, os.path.basename(s) + ".o")
            if force or _newer(o, deps):
                _run([NVCC, *CUFLAGS, *extra, "-c", s, "-o", o], verbose)
            objs.append(o)
        _run([NVCC, *ARCH, "-shared", "-cudart", "static", "-o", LIB, *objs], verbose)
    return LIB


def build_clis(force=False, verbose=False):
    os.makedirs(BIN_DIR, exist_ok=True)
    out = []
    for name, files in CLI_SOURCES.items():
        srcs = [os.path.join(HOST, f) for f in files]
        if not all(os.path.exists(s) for s in srcs):
            continue
        exe = os.path.join(BIN_DIR, name)
        deps = srcs + [LIB, os.path.join(ROOT, "include", "ebwt2snp_b200.h"), os.path.join(HOST, "host_io.hpp")]
        if force or _newer(exe, deps):
            _run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), *srcs, "-o", exe,
                  "-L", LIB_DIR, "-lebwt2snp_b200", "-Wl,-rpath,$ORIGIN/../lib", "-ldl", "-lpthread", "-lrt"], verbose)
        out.append(exe)
    for name, files in TEXT_TOOLS.items():
        srcs = [os.path.join(HOST, f) for f in files]
        exe = os.path.join(BIN_DIR, name)
        if force or _newer(exe, srcs + [os.path.join(HOST, "snp_text.hpp")]):
            _run(["g++", "-O2", "-std=c++17", "-I", HOST, *srcs, "-o", exe], verbose)
        out.append(exe)
    return out


def build_all(force=False, verbose=False):
    lib = build_library(force, verbose)
    clis = build_clis(force, verbose)
    return lib, clis


if __name__ == "__main__":
    lib, clis = build_all(force="--force" in sys.argv, verbose=True)
    print("built", lib, *clis)
