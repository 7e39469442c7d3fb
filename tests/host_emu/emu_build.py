"""TEST INFRASTRUCTURE: ctypes wrapper of tests/host_emu/emu_build.cpp -- the dense-grid builder's content hash
(csrc/ort_build.cuh: build_hash) compiled for the host.  Not a product path."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import emu

SO = os.path.join(emu.HERE, "_build", "libort_emu_build.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        deps = [os.path.join(emu.HERE, "emu_build.cpp"), os.path.join(emu.HERE, "cuda_shim.h"), os.path.join(emu.CSRC, "ort_build.cuh")]
        if not (os.path.exists(SO) and all(os.path.getmtime(d) <= os.path.getmtime(SO) for d in deps)):
            os.makedirs(os.path.dirname(SO), exist_ok=True)
            cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unused-function", deps[0], "-o", SO]
            out = subprocess.run(cmd, capture_output=True, text=True)
            if out.returncode:
                raise RuntimeError("host emulation build failed:\n" + out.stderr)
        _lib = C.CDLL(SO)
    return _lib


def build_hash(w8):
    """build_hash of each row of an (n, 8) array of uint32 words, as the device computes it"""
    w8 = np.ascontiguousarray(w8, np.uint32).reshape(-1, 8)
    out = np.empty(w8.shape[0], np.uint32)
    lib().emu_build_hash(emu._p(w8), C.c_size_t(w8.shape[0]), emu._p(out))
    return out
