"""Builds libofdis_b200.so (CUDA kernels + C-ABI) in-tree with nvcc for sm_100a.

    python -m of_dis_b200.build [--force] [--verbose]

-fmad=false: no FMA contraction -- the results must be bitwise equal to the
reference CPU build (DESIGN.md section 4).  -lineinfo keeps ncu's source page
usable.  The runtime is linked statically so the library only needs the driver.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libofdis_b200.so")
SOURCES = ["ofdis_capi.cu", "patch_kernels.cu", "pyramid_kernels.cu", "varref_kernels.cu"]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "ofdis_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl", "-o", LIB]  # -ldl: NVTX v3 loads its injection library lazily
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode:
        raise RuntimeError("nvcc failed building libofdis_b200.so")
    return LIB


BINDIR = os.path.join(HERE, "bin")
HOST = os.path.join(HERE, "host")
CLI_TARGETS = {"run_OF_INT": (1, 1), "run_OF_RGB": (1, 3), "run_DE_INT": (2, 1), "run_DE_RGB": (2, 3)}


def build_host(force: bool = False) -> str:
    """The reference's four command-line binaries (CMakeLists.txt:25-46) plus the C++
    self-test, g++ against libofdis_b200.so (rpath $ORIGIN/../lib)."""
    build(force=False)
    os.makedirs(BINDIR, exist_ok=True)
    srcs = [os.path.join(HOST, f) for f in ("ofdis_host.cpp", "ofdis_host.h", "run_dense.cpp", "host_selftest.cpp")]
    newest = max(os.path.getmtime(f) for f in srcs + [LIB])
    common = ["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-Wall", os.path.join(HOST, "ofdis_host.cpp")]
    link = ["-L" + LIBDIR, "-lofdis_b200", "-lz", "-Wl,-rpath,$ORIGIN/../lib"]
    jobs = {name: common + [os.path.join(HOST, "run_dense.cpp"), "-DSELECTMODE=%d" % m, "-DSELECTCHANNEL=%d" % c]
            for name, (m, c) in CLI_TARGETS.items()}
    for name, (m, c) in CLI_TARGETS.items():  # batch front-end: list file in, many pairs per launch
        jobs[name + "_batch"] = jobs[name] + ["-DOFDIS_BATCH"]
    jobs["ofdis_host_selftest"] = common + [os.path.join(HOST, "host_selftest.cpp")]
    jobs["ofdis_imgdump"] = common + [os.path.join(HOST, "run_dense.cpp"), "-DOFDIS_IMGDUMP"]  # decoder test tool (no GPU)
    for name, cmd in jobs.items():
        out = os.path.join(BINDIR, name)
        if force or not os.path.exists(out) or os.path.getmtime(out) < newest:
            res = subprocess.run(cmd + ["-o", out] + link, capture_output=True, text=True)
            if res.returncode:
                sys.stderr.write(res.stdout + res.stderr)
                raise RuntimeError("g++ failed building %s" % name)
    return BINDIR


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
    print(build_host(force="--force" in sys.argv))
