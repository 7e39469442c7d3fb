"""Build libort_b200.so (hand-written CUDA for sm_100a + the C++ host side) in-tree with nvcc.

    python -m octree_ray_tracing_b200.build [--force] [--verbose] [--no-experiments]

The library is the product: there is no JIT, no torch extension and no CPU fallback.  nvcc
cross-compiles without a GPU, so this also runs in CPU-only containers.

A second library, libort_b200_exp.so, is the same sources with -DORT_EXPERIMENTS: it additionally carries the kernels
that were measured and not adopted (csrc/ort_experiments.cuh), so that those decisions can be re-measured.  Nothing
loads it unless ORT_B200_EXPERIMENTS=1 is set (tests/test_experiments.py, tools/).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libort_b200.so")
LIB_EXP = os.path.join(HERE, "libort_b200_exp.so")
SOURCES = ["ort_device.cu", "ort_host_tree.cpp", "ort_host_octree.cpp", "ort_fixture.cpp"]
HEADERS = ["ort_internal.h", "ort_trace.cuh", "ort_beam.cuh", "ort_kernels.cuh", "ort_build.cuh", "ort_mg.cuh", "ort_noise.h", "ort_rcp_table.h", os.path.join("..", "..", "include", "ort_b200.h")]
HEADERS_EXP = ["ort_experiments.cuh", "ort_trace_experiments.cuh"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",                      # a*b+c is only ever fused where the source says __fmaf_rn
    "-Xcompiler", "-fPIC,-O2,-ffp-contract=off,-Wall",
    "-Xptxas", "-v",
    "-shared", "-cudart", "static", "-ldl",
]


def kernel_source_hash() -> str:
    """sha256[:16] over the sources and flags that decide the trace kernels' machine code (the per-ray walk and the
    kernels around it).  ncu captures are tied to it (profiles/traffic.json): a number read from a capture of OTHER
    code must not end up in a bench line."""
    import hashlib
    h = hashlib.sha256()
    for name in ("ort_trace.cuh", "ort_beam.cuh", "ort_kernels.cuh"):
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()[:16]


def nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libort_b200.so cannot be built")


def needs_build(lib: str = LIB, extra=()) -> bool:
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS + list(extra)] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(lib: str, defines, log_name: str, verbose: bool) -> None:
    cmd = [nvcc()] + NVCC_FLAGS + list(defines) + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", lib]
    out = subprocess.run(cmd, capture_output=True, text=True)
    log = out.stdout + out.stderr
    # the last build's ptxas -v report (registers, spills, stack per kernel); a build product, kept out of git
    with open(os.path.join(HERE, log_name), "w") as f:
        f.write(" ".join(cmd) + "\n" + log + "\n")
    if verbose or out.returncode:
        print(log)
    if out.returncode:
        raise RuntimeError(f"nvcc failed building {os.path.basename(lib)}")


def build(force: bool = False, verbose: bool = False, experiments: bool = True) -> str:
    if force or needs_build():
        _compile(LIB, [], "build.log", verbose)
    if experiments and (force or needs_build(LIB_EXP, HEADERS_EXP)):
        _compile(LIB_EXP, ["-DORT_EXPERIMENTS"], "build_exp.log", verbose)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv or "-v" in sys.argv, experiments="--no-experiments" not in sys.argv)
    print(LIB)
