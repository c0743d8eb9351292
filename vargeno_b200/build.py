"""In-tree build of libvgb200.so (hand-written CUDA for sm_100a + the C ABI of include/vgb200.h).

    python -m vargeno_b200.build            # incremental
    python -m vargeno_b200.build --force

nvcc cross-compiles without a GPU; the .so is git-ignored but travels with the gpurun snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB = os.path.join(HERE, "libvgb200.so")
HOST_BIN = os.path.join(HERE, "vargeno-b200")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

CU = ["vgb_api.cu", "vgb_index.cu", "vgb_fastq.cu", "vgb_geno.cu", "vgb_call.cu", "vgb_bench.cu", "vgb_build.cu", "vgb_gzip.cu", "vgb_bam.cu", "vgb_vcf.cu"]
CPP = ["vgb_tables.cpp", "vgb_nccl.cpp"]
HOST_CPP = ["host/vargeno_main.cpp", "host/geno_host.cpp", "host/index_host.cpp"]
HEADERS = ["vgb_common.cuh", "vgb_internal.h", "vgb_geno8.inl", "vgb_inflate.cuh", "vgb_gzip.cuh", "vgb_bam.cuh", "vgb_deflate.cuh", "vgb_vcf.cuh", os.path.join("..", "..", "include", "vgb200.h"), "host/geno_host.h"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-ffp-contract=off,-Wall", "-ccbin", "g++", "--fmad=false"] + os.environ.get("VGB_NVCC_DEFINES", "").split()   # A/B builds of compile-time variants (tools/sweep_wgs.py, VGB200_LIB)
CXX_FLAGS = ["-O2", "-g", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wall", "-I/usr/local/cuda/include"]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def _run(cmd):
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if p.returncode != 0:
        raise RuntimeError("build step failed: %s\n%s" % (" ".join(cmd), p.stdout))
    return p.stdout


def build(force: bool = False, verbose: bool = False, ptxas_info: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    jobs = []
    objs = []
    for src in CU:
        o = os.path.join(OBJ, src + ".o")
        objs.append(o)
        if force or _newer(o, [os.path.join(CSRC, src)] + hdrs):
            cmd = [NVCC] + NVCC_FLAGS + (["-Xptxas", "-v"] if ptxas_info else []) + ["-c", os.path.join(CSRC, src), "-o", o]
            jobs.append(cmd)
    for src in CPP:
        o = os.path.join(OBJ, src + ".o")
        objs.append(o)
        if force or _newer(o, [os.path.join(CSRC, src)] + hdrs):
            jobs.append(["g++"] + CXX_FLAGS + ["-c", os.path.join(CSRC, src), "-o", o])
    with ThreadPoolExecutor(max_workers=8) as ex:
        outs = list(ex.map(_run, jobs))
    if verbose or ptxas_info:
        for cmd, out in zip(jobs, outs):
            print(" ".join(cmd))
            if out.strip():
                print(out)
    if force or jobs or not os.path.exists(LIB):
        _run([NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static", "-ldl", "-lm", "-lrt", "-lpthread",
                                                   "-Xlinker", "--no-undefined"])
    # the stand-alone C++ host (same CLI as the reference: `vargeno-b200 geno <prefix> <fq> <vcf> <out>`)
    host_srcs = [os.path.join(CSRC, s) for s in HOST_CPP]
    if all(os.path.exists(s) for s in host_srcs):
        if force or _newer(HOST_BIN, host_srcs + hdrs + [LIB]):
            _run(["g++", "-O2", "-g", "-std=c++17", "-ffp-contract=off", "-Wall", "-o", HOST_BIN] + host_srcs +
                 ["-L" + HERE, "-lvgb200", "-Wl,-rpath,$ORIGIN", "-lpthread", "-lz"])
    # stand-alone measurement tool (profiles/r01_sector_probe.md); not linked into anything
    probe_src = os.path.join(HERE, "tools", "probes", "sector_probe.cu")
    probe_bin = os.path.join(HERE, "tools", "probes", "sector_probe")
    if os.path.exists(probe_src) and (force or _newer(probe_bin, [probe_src])):
        _run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-o", probe_bin, probe_src])
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True, ptxas_info="--ptxas" in sys.argv)
    print(LIB)
