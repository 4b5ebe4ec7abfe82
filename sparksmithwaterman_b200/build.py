"""Builds libswb200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m sparksmithwaterman_b200.build [--force]

nvcc cross-compiles without a GPU; the .so travels to the GPU box with the snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "_lib")
BIN_DIR = os.path.join(HERE, "_bin")
LIB = os.path.join(LIB_DIR, "libswb200.so")
MICROBENCH = os.path.join(BIN_DIR, "dpx_microbench")
PAIR_BENCH = os.path.join(BIN_DIR, "pair_bench")

SOURCES = ["swb_api.cu", "swb_align.cu", "swb_fill.cu", "swb_fill_bias.cu", "swb_trace.cu", "swb_trace_tile.cu", "swb_wide.cu", "swb_wide_host.cu", "swb_multi.cu", "swb_queue.cu", "swb_assemble.cu", "swb_hits.cu", "swb_strands.cu", "dpx_microbench.cu"]
HEADERS = ["swb_internal.h", "swb_device.cuh", "swb_host.h", os.path.join("..", "..", "include", "swb200.h")]
NVCC_FLAGS = ["-std=c++17", "-O3", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a",
              "-Xcompiler", "-fPIC", "-cudart", "static"]


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(d) <= t for d in deps)


def build_native(force: bool = False, verbose: bool = False) -> str:
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS]
    os.makedirs(LIB_DIR, exist_ok=True)
    os.makedirs(BIN_DIR, exist_ok=True)
    if force or not _newer(LIB, deps):
        objs = []
        procs = []
        for s in srcs:
            o = os.path.join(LIB_DIR, os.path.basename(s) + ".o")
            objs.append(o)
            if force or not _newer(o, deps):
                cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", o, s]
                procs.append((cmd, subprocess.Popen(cmd)))
        for cmd, p in procs:
            if p.wait() != 0:
                raise RuntimeError("nvcc failed: " + " ".join(cmd))
        cmd = [nvcc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-ldl"]
        subprocess.check_call(cmd)
    if force or not _newer(MICROBENCH, [os.path.join(CSRC, "dpx_microbench.cu")]):
        subprocess.check_call([nvcc] + NVCC_FLAGS + ["-DSWB_MICROBENCH_MAIN", "-o", MICROBENCH,
                                                      os.path.join(CSRC, "dpx_microbench.cu")])
    # native pairs/s harness of the single-pair (unchanged driver) path: plain C on the ABI
    src = os.path.normpath(os.path.join(HERE, "..", "tools", "pair_bench.c"))
    if os.path.exists(src) and (force or not _newer(PAIR_BENCH, [src, LIB])):
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-Wall", "-pthread", "-I" + os.path.normpath(os.path.join(HERE, "..", "include")),
                               src, "-L" + LIB_DIR, "-lswb200", "-lm", "-Wl,-rpath," + LIB_DIR, "-Wl,-rpath,$ORIGIN/../_lib", "-o", PAIR_BENCH])
    return LIB


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose="-v" in sys.argv))
