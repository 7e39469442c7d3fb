"""TEST INFRASTRUCTURE: ctypes wrapper of tests/host_emu/emu_refine.cpp -- the host emulation (emu.py) plus camera frames
whose tile starts are refined on the level-8 grid (csrc/ort_beam.cuh, item 2).  Not a product path."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import emu

SO = os.path.join(emu.HERE, "_build", "libort_emu_refine.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        deps = [os.path.join(emu.HERE, "emu_refine.cpp"), os.path.join(emu.HERE, "emu.cpp"), os.path.join(emu.HERE, "cuda_shim.h"),
                os.path.join(emu.CSRC, "ort_trace.cuh"), os.path.join(emu.CSRC, "ort_trace_experiments.cuh"), os.path.join(emu.CSRC, "ort_beam.cuh")]
        if not (os.path.exists(SO) and all(os.path.getmtime(d) <= os.path.getmtime(SO) for d in deps)):
            os.makedirs(os.path.dirname(SO), exist_ok=True)
            out = subprocess.run(["g++", "-O2", "-std=c++17", "-fopenmp", "-mfma", "-mavx2", "-ffp-contract=off", "-fPIC", "-shared",
                                  "-Wall", "-Wno-unused-function", deps[0], "-o", SO], capture_output=True, text=True)
            if out.returncode:
                raise RuntimeError("host emulation build failed:\n" + out.stderr)
        _lib = C.CDLL(SO)
        _lib.emu_refine_fine_t.restype = C.c_float
        _lib.emu_stats_words.restype = C.c_int
    return _lib


def beam_fine_t(pos, rot, fov, W, H, depth, rcp_tab=None) -> float:
    """The time limit of the level-8 refinement the library gives this camera (0.0: none)."""
    tab = emu.default_rcp_table() if rcp_tab is None else np.ascontiguousarray(rcp_tab, np.uint32)
    pos = np.ascontiguousarray(pos, np.float32)
    rot = np.ascontiguousarray(rot, np.float32)
    return float(lib().emu_refine_fine_t(emu._p(pos), emu._p(rot), C.c_float(fov), W, H, depth, emu._p(tab), int(np.log2(len(tab)))))


def trace_frame(nodes8, root, depth, pos, rot, fov, W, H, beam, fine, y0=0, rows=None, tile_rows=1, tile_step=1, rcp_tab=None,
                miss_t=np.inf, want_npush=False, nthreads=None):
    """A frame of the compact DAG (walker 13) with the beam start of the level-k grid `beam`, refined on the level-8 grid
    `fine` as the library does for this camera (fine=None: not refined).  Returns (voxel, face, t[, npush], stats, tau)."""
    nodes8 = np.ascontiguousarray(nodes8, np.uint32)
    tab = emu.default_rcp_table() if rcp_tab is None else np.ascontiguousarray(rcp_tab, np.uint32)
    rows = H - y0 if rows is None else rows
    n = rows * W
    beam = np.ascontiguousarray(beam, np.uint8)
    fine_t = 0.0
    if fine is not None:
        fine = np.ascontiguousarray(fine, np.uint8)
        assert fine.shape[0] == 256, "the refinement grid is level 8"
        fine_t = beam_fine_t(pos, rot, fov, W, H, depth, tab)
    pos = np.ascontiguousarray(pos, np.float32); rot = np.ascontiguousarray(rot, np.float32)
    vox = np.empty(n, np.uint32); face = np.empty(n, np.uint8); t = np.empty(n, np.float32); tau = np.empty(n, np.float32)
    npush = np.empty(n, np.uint16) if want_npush else None
    stats = np.zeros(lib().emu_stats_words(), np.uint64)
    oob = lib().emu_refine_trace_frame(emu._p(nodes8), C.c_size_t(nodes8.size // 8), C.c_uint32(root), depth, C.c_float(miss_t), emu._p(tab), int(np.log2(len(tab))),
                                       emu._p(pos), emu._p(rot), C.c_float(fov), W, H, y0, rows, tile_rows, tile_step,
                                       emu._p(vox), emu._p(face), emu._p(t), emu._p(npush), emu._p(stats), nthreads or os.cpu_count() or 1,
                                       emu._p(beam), int(np.log2(beam.shape[0])), emu._p(fine), C.c_float(fine_t), emu._p(tau))
    if oob:
        raise MemoryError("host emulation: the walk loaded from outside the node array / reciprocal table")
    out = [vox, face, t] + ([npush] if want_npush else []) + [emu._stats(stats), tau]
    return tuple(out)
