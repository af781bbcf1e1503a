"""Builds libnohuman_gpu.so in-tree with nvcc for sm_100a (no JIT cache: the
.so travels to the GPU box with the repo snapshot).

    python -m nohuman_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libnohuman_gpu.so")
CLI = os.path.join(PKG, "bin", "nohuman")

CU_SOURCES = ["nh_kernels.cu", "nh_capi.cu", "nh_synth.cu", "nh_deflate.cu", "nh_inflate.cu", "nh_build.cu", "nh_dust.cu"]
CC_SOURCES = ["nh_pipeline.cc", "nh_pack.cc"]  # host pipeline and the host-side packer, compiled into the same library

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-O3,-Wall,-pthread",
    "-Xptxas", "-v",
]
# experiment hook: NH_NVCC_EXTRA='-DNH_LD_SECTOR_OP="ld.global.L2::64B.v8.u32"' python -m nohuman_b200.build --force
NVCC_FLAGS += [f for f in os.environ.get("NH_NVCC_EXTRA", "").split() if f]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _existing(names):
    return [os.path.join(CSRC, n) for n in names if os.path.exists(os.path.join(CSRC, n))]


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    srcs = _existing(CU_SOURCES) + _existing(CC_SOURCES)
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hdrs.append(os.path.join(PKG, "..", "include", "nohuman_gpu.h"))
    if force or _stale(LIB, srcs + hdrs + [os.path.abspath(__file__)]):
        cmd = [_nvcc(), *NVCC_FLAGS, "-ccbin", "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++",
               "-shared", "-o", LIB, *srcs, "-lz", "-lpthread", "-ldl"]
        if verbose:
            print(" ".join(cmd))
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = r.stdout + r.stderr
        with open(os.path.join(PKG, "build.log"), "w") as f:
            f.write(" ".join(cmd) + "\n" + log)
        if r.returncode != 0:
            sys.stderr.write(log)
            raise RuntimeError("nvcc failed building libnohuman_gpu.so")
        if verbose:
            print(log)
    main_cc = os.path.join(CSRC, "nohuman_main.cc")
    if os.path.exists(main_cc) and (force or _stale(CLI, [main_cc, LIB])):
        os.makedirs(os.path.dirname(CLI), exist_ok=True)
        cmd = ["/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++", "-O2", "-std=c++17", "-Wall",
               "-o", CLI, main_cc, "-L", PKG, "-lnohuman_gpu", "-Wl,-rpath,$ORIGIN/..", "-lpthread"]
        subprocess.check_call(cmd)
        # the same binary under the names nohuman looks for on $PATH (src/main.rs:170), the one that builds
        # a database for it and the masker kraken2-build --add-to-library runs: argv shims
        for name in ("kraken2", "kraken2-build", "dustmasker"):
            shim = os.path.join(os.path.dirname(CLI), name)
            if os.path.lexists(shim):
                os.remove(shim)
            shutil.copy2(CLI, shim)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
