"""TEST INFRASTRUCTURE: ctypes wrapper of tests/host_emu/emu_query.cpp -- the voxel queries' per-point and per-cell code
(csrc/ort_query.cuh) compiled for the host.  Not a product path."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import emu

SO = os.path.join(emu.HERE, "_build", "libort_emu_query_san.so" if emu.SANITIZE else "libort_emu_query.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        deps = [os.path.join(emu.HERE, "emu_query.cpp"), os.path.join(emu.HERE, "cuda_shim.h"), os.path.join(emu.CSRC, "ort_query.cuh")]
        if not (os.path.exists(SO) and all(os.path.getmtime(d) <= os.path.getmtime(SO) for d in deps)):
            os.makedirs(os.path.dirname(SO), exist_ok=True)
            cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unused-function", deps[0], "-o", SO]
            if emu.SANITIZE:
                cmd[1:2] = ["-O1", "-g", "-fsanitize=address,undefined", "-fno-omit-frame-pointer"]
            out = subprocess.run(cmd, capture_output=True, text=True)
            if out.returncode:
                raise RuntimeError("host emulation build failed:\n" + out.stderr)
        _lib = C.CDLL(SO)
        for f in (_lib.emu_voxels_at, _lib.emu_read_voxels):
            f.restype = C.c_ulonglong
    return _lib


def _layout(pool, root):
    return (0, 0) if pool else (1, int(root))


def voxels_at(nodes8, root, depth, xyz, pool=False):
    """(values, out-of-bounds loads) of at() on a mirror holding nodes8: compact ids from `root` (pool=False, root 0 =
    no tree) or an och::octree pool walked from row 0 (pool=True)."""
    nodes8 = np.ascontiguousarray(nodes8, np.uint32).reshape(-1, 8)
    xyz = np.ascontiguousarray(xyz, np.int64).astype(np.int32).reshape(-1, 3)
    out = np.empty(len(xyz), np.uint32)
    base, r = _layout(pool, root)
    oob = lib().emu_voxels_at(emu._p(nodes8), C.c_size_t(nodes8.shape[0]), base, C.c_uint32(r), depth, emu._p(xyz), C.c_size_t(len(xyz)), emu._p(out))
    return out, int(oob)


def read_voxels(nodes8, root, depth, origin, extent, pool=False, offset=0):
    """(grid [nz, ny, nx], out-of-bounds loads) of the box.  The output starts `offset` uint32 past an 8-byte boundary
    (1: every 8-byte pair of an even-aligned box falls on the 4-byte path), inside a guard band that must stay intact."""
    nodes8 = np.ascontiguousarray(nodes8, np.uint32).reshape(-1, 8)
    nx, ny, nz = (int(v) for v in extent)
    n = nx * ny * nz
    guard = 16
    buf = np.full(n + 2 * guard + 2, 0xDEADBEEF, np.uint32)
    start = guard + (-(buf.ctypes.data // 4) % 2) + offset            # buf + start: 8-byte aligned plus `offset` words
    out = buf[start:start + n]
    base, r = _layout(pool, root)
    oob = lib().emu_read_voxels(emu._p(nodes8), C.c_size_t(nodes8.shape[0]), base, C.c_uint32(r), depth,
                                *(C.c_uint32(int(v)) for v in origin), nx, ny, nz, emu._p(out))
    assert (buf[:start] == 0xDEADBEEF).all() and (buf[start + n:] == 0xDEADBEEF).all(), "read_voxels wrote outside the box"
    return out.reshape(nz, ny, nx).copy(), int(oob)
