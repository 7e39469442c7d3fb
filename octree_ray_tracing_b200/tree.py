"""Python mirror of the reference's interface for the trace path.

``HOctree(log2_table_capacity, depth)`` has the members of ``och::h_octree<L,D>``
(och_h_octree.h:17-452): ``register_node``, ``remove_node``, ``set``, ``at``, ``set_root``,
``get_root``, ``get_fillcnt``, ``get_nodecnt``, ``get_max_refcnt``, ``clear`` and ``sse_trace``
(one ray -> (direction, voxel, time)), with the same argument meaning and error behaviour, plus the
batched forms the GPU needs (``trace_rays``, ``trace_frame``).  All tracing runs on the GPU through
``libort_b200.so``; there is no CPU implementation behind these calls.
"""
from __future__ import annotations

import ctypes as C
import enum
import os

import numpy as np

from ._lib import OrtError, check, lib

_vp = C.c_void_p


class Direction(enum.IntEnum):
    """och::direction (och_tree_helper.h:7-18)"""
    x_pos = 0
    y_pos = 1
    z_pos = 2
    x_neg = 3
    y_neg = 4
    z_neg = 5
    exit = 6
    inside = 7
    error = 8


def _p(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(_vp)
    if isinstance(a, int):
        return _vp(a)
    if hasattr(a, "data_ptr"):          # torch tensor (device or pinned host memory)
        return _vp(a.data_ptr())
    raise TypeError(type(a))


def host_rcp_table(log2n: int = 11):
    """(table, mismatches): this host CPU's RCPSS as a table for TraceContext.set_rcp_table (see ort_host_rcp_table)."""
    tab = np.zeros(1 << log2n, np.uint32)
    bad = lib().ort_host_rcp_table(_p(tab), log2n)
    return tab, int(bad)


def camera_coeffs(yaw: float, pitch: float):
    """rot[9], fov_factor as tree_camera::update_position computes them (test_och_h_octree.cpp:95-115)."""
    rot = np.zeros(9, np.float32)
    fov = C.c_float(0)
    lib().ort_camera_coeffs(yaw, pitch, _p(rot), C.byref(fov))
    return rot, float(np.float32(fov.value))


class FrameJob(C.Structure):
    """ort_frame_job (include/ort_b200.h): one frame / strip of a batched launch."""
    _fields_ = [("pos", C.c_float * 3), ("rot", C.c_float * 9), ("fov_factor", C.c_float),
                ("W", C.c_int), ("H", C.c_int), ("y0", C.c_int), ("rows", C.c_int), ("tile_rows", C.c_int), ("tile_step", C.c_int),
                ("voxel", C.c_void_p), ("face", C.c_void_p), ("t", C.c_void_p), ("npush", C.c_void_p)]


def _addr(a):
    if a is None:
        return None
    return a.data_ptr() if hasattr(a, "data_ptr") else int(a)


class TraceContext:
    """One GPU's node mirror + streams (``ort_ctx``)."""

    def __init__(self, depth: int, device: int = 0, node_capacity: int = 1 << 16):
        self.L = lib()
        h = _vp()
        check(self.L.ort_create(C.byref(h), device, depth, node_capacity))
        self.h = h
        self.depth = depth
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.L.ort_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        check(rc, self.h)

    def set_rcp_table(self, tab):
        tab = np.ascontiguousarray(tab, np.uint32)
        log2n = int(tab.size).bit_length() - 1
        assert tab.size == 1 << log2n
        self._ck(self.L.ort_set_rcp_table(self.h, _p(tab), log2n))

    def upload_full(self, nodes8, root: int):
        a = np.ascontiguousarray(nodes8, np.uint32).reshape(-1, 8)
        self._ck(self.L.ort_upload_full(self.h, _p(a), a.shape[0], root))

    def upload_delta(self, ids, nodes8, root: int):
        i = np.ascontiguousarray(ids, np.uint32)
        a = np.ascontiguousarray(nodes8, np.uint32).reshape(-1, 8)
        assert a.shape[0] == i.size
        self._ck(self.L.ort_upload_delta(self.h, _p(i), _p(a), i.size, root))

    def upload_voxels(self, grid):
        """Build the DAG of a dense voxel grid on this context's GPU and install it as the mirror (ort_build_voxels).
        grid: C-contiguous 3-D numpy array or torch tensor (CPU or CUDA) of shape (nz, ny, nx), dtype uint8, int32 or
        uint32 (read as unsigned); grid[z, y, x] is voxel (x, y, z), 0 = empty.  Returns (n_nodes, level_offsets):
        the mirror then holds what HOctree.flatten() gives for a table holding these voxels."""
        if isinstance(grid, np.ndarray):
            if grid.dtype not in (np.uint8, np.int32, np.uint32):
                raise TypeError(f"upload_voxels: dtype {grid.dtype} (uint8, int32 or uint32 required)")
            if grid.ndim != 3 or not grid.flags.c_contiguous:
                raise ValueError("upload_voxels: a C-contiguous 3-D array of shape (nz, ny, nx) is required")
            elem = grid.dtype.itemsize
        elif hasattr(grid, "data_ptr"):
            import torch
            if grid.dtype not in (torch.uint8, torch.int32, torch.uint32):
                raise TypeError(f"upload_voxels: dtype {grid.dtype} (uint8, int32 or uint32 required)")
            if grid.dim() != 3 or not grid.is_contiguous():
                raise ValueError("upload_voxels: a contiguous 3-D tensor of shape (nz, ny, nx) is required")
            if grid.is_cuda:
                if grid.device.index != self.device:
                    raise ValueError(f"upload_voxels: the tensor is on {grid.device}, the context on cuda:{self.device}")
                torch.cuda.current_stream(grid.device).synchronize()      # the builder reads it on its own stream
            elem = grid.element_size()
        else:
            raise TypeError(f"upload_voxels: numpy array or torch tensor required, got {type(grid).__name__}")
        nz, ny, nx = (int(s) for s in grid.shape)
        n = C.c_size_t(0)
        lo = np.zeros(self.depth + 1, np.uint32)
        self._ck(self.L.ort_build_voxels(self.h, _p(grid), elem, nx, ny, nz, C.byref(n), _p(lo)))
        return n.value, lo

    def read_nodes(self, first: int = 1, n: int | None = None) -> np.ndarray:
        """Rows first .. first + n - 1 (compact ids, 1-based) of the device mirror as an (n, 8) uint32 array."""
        if n is None:
            n = max(0, self.node_count - first + 1)
        out = np.zeros((n, 8), np.uint32)
        self._ck(self.L.ort_read_nodes(self.h, first, n, _p(out)))
        return out

    def set_option(self, key: str, value: int):
        self._ck(self.L.ort_set_option(self.h, key.encode(), value))

    @property
    def node_count(self):
        return self.L.ort_node_count(self.h)

    @property
    def root(self):
        return self.L.ort_root(self.h)

    @property
    def launch_count(self):
        return self.L.ort_launch_count(self.h)

    @property
    def stream(self):
        return self.L.ort_stream(self.h)

    def sync(self):
        self._ck(self.L.ort_sync(self.h))

    def measure_gather_peak(self, nbytes: int) -> float:
        """GB/s of random 32-B sector gathers over an nbytes buffer (roofline denominator for L2-resident DAGs)."""
        out = C.c_double(0)
        self._ck(self.L.ort_measure_gather_peak(self.h, nbytes, C.byref(out)))
        return out.value

    def beam_level(self, pos, rot, fov_factor: float, W: int, H: int) -> int:
        """Grid level the beam start of W x H frames with this camera would use (0: none)."""
        pos = np.ascontiguousarray(pos, np.float32)
        rot = np.ascontiguousarray(rot, np.float32)
        return int(self.L.ort_beam_level(self.h, _p(pos), _p(rot), fov_factor, W, H))

    def beam_grid(self, level: int) -> np.ndarray:
        """The level-`level` skip grid of the DAG on the device, (N, N, N) bytes indexed [z, y, x]."""
        n = 1 << level
        out = np.zeros((n, n, n), np.uint8)
        self._ck(self.L.ort_beam_grid(self.h, level, _p(out)))
        return out

    @property
    def build_bytes(self) -> int:
        """Device bytes the last successful upload_voxels allocated (its peak on top of what the context held)."""
        return self.L.ort_build_bytes(self.h)

    @property
    def beam_builds(self) -> int:
        return self.L.ort_beam_builds(self.h)

    @property
    def band_schedules(self) -> int:
        return self.L.ort_band_schedules(self.h)

    def set_stream(self, stream):
        """Queue subsequent work on a caller stream (a cudaStream_t as int, a torch.cuda.Stream, or None)."""
        if stream is not None and hasattr(stream, "cuda_stream"):
            stream = stream.cuda_stream
        self._ck(self.L.ort_set_stream(self.h, _vp(stream) if stream else None))

    # ---- host-buffer calls -------------------------------------------------------------------
    def trace_rays(self, o, d, want_npush=False):
        d = np.ascontiguousarray(d, np.float32).reshape(-1, 3)
        o = np.ascontiguousarray(o, np.float32)
        n = d.shape[0]
        stride = 0 if o.size == 3 else 3
        if stride:
            assert o.size == 3 * n
        vox = np.empty(n, np.uint32)
        face = np.empty(n, np.uint8)
        t = np.empty(n, np.float32)
        npush = np.empty(n, np.uint16) if want_npush else None
        self._ck(self.L.ort_trace_rays(self.h, _p(o), stride, _p(d), n, _p(vox), _p(face), _p(t), _p(npush)))
        return (vox, face, t, npush) if want_npush else (vox, face, t)

    def trace_frame(self, pos, rot, fov_factor, W, H, y0=0, rows=None, tile_rows=1, tile_step=1, want_npush=False, out=None):
        rows = H - y0 if rows is None else rows
        pos = np.ascontiguousarray(pos, np.float32)
        rot = np.ascontiguousarray(rot, np.float32)
        n = rows * W
        if out is None:
            vox = np.empty(n, np.uint32)
            face = np.empty(n, np.uint8)
            t = np.empty(n, np.float32)
            npush = np.empty(n, np.uint16) if want_npush else None
        else:
            vox, face, t, npush = out
        self._ck(self.L.ort_trace_frame(self.h, _p(pos), _p(rot), fov_factor, W, H, y0, rows, tile_rows, tile_step,
                                        _p(vox), _p(face), _p(t), _p(npush)))
        return (vox, face, t, npush) if want_npush else (vox, face, t)

    # ---- shaded frames (trace_pixel's colour lookup fused into the kernel) -------------------------
    def set_palette(self, rgba6, exit_rgba=0xFFFEBF00, inside_rgba=0xFF07193F):
        a = np.ascontiguousarray(rgba6, np.uint32).reshape(-1, 6)
        self._ck(self.L.ort_set_palette(self.h, _p(a), a.shape[0], exit_rgba, inside_rgba))

    def trace_frame_rgba(self, pos, rot, fov_factor, W, H, y0=0, rows=None, tile_rows=1, tile_step=1, out=None):
        """One uint32 pixel per ray (olc::Pixel::n packing).  out: host array / pinned tensor (synchronous) or a
        CUDA tensor (enqueue only)."""
        rows = H - y0 if rows is None else rows
        pos = np.ascontiguousarray(pos, np.float32)
        rot = np.ascontiguousarray(rot, np.float32)
        if out is None:
            out = np.empty(rows * W, np.uint32)
        self._ck(self.L.ort_trace_frame_rgba(self.h, _p(pos), _p(rot), fov_factor, W, H, y0, rows, tile_rows, tile_step, _p(out)))
        return out

    # ---- device-buffer, enqueue-only calls (pointers or torch CUDA tensors) ---------------------
    def trace_frame_async(self, pos, rot, fov_factor, W, H, y0, rows, tile_rows, tile_step, d_vox, d_face, d_t, d_npush=None):
        pos = np.ascontiguousarray(pos, np.float32)
        rot = np.ascontiguousarray(rot, np.float32)
        self._ck(self.L.ort_trace_frame_async(self.h, _p(pos), _p(rot), fov_factor, W, H, y0, rows, tile_rows, tile_step,
                                              _p(d_vox), _p(d_face), _p(d_t), _p(d_npush)))

    def trace_frames_async(self, jobs):
        """jobs: iterable of (pos, rot, fov_factor, W, H, y0, rows, tile_rows, tile_step, d_vox, d_face, d_t[, d_npush]) --
        all of them in one launch (ort_trace_frames_async)."""
        jobs = list(jobs)
        arr = (FrameJob * len(jobs))()
        for k, j in enumerate(jobs):
            pos, rot, fov, W, H, y0, rows, tile_rows, tile_step, dv, df, dt = j[:12]
            dn = j[12] if len(j) > 12 else None
            arr[k].pos[:] = [float(x) for x in pos]
            arr[k].rot[:] = [float(x) for x in rot]
            arr[k].fov_factor = float(fov)
            arr[k].W, arr[k].H, arr[k].y0, arr[k].rows, arr[k].tile_rows, arr[k].tile_step = W, H, y0, rows, tile_rows, tile_step
            arr[k].voxel, arr[k].face, arr[k].t, arr[k].npush = _addr(dv), _addr(df), _addr(dt), _addr(dn)
        self._ck(self.L.ort_trace_frames_async(self.h, C.byref(arr), len(jobs)))

    def trace_rays_async(self, d_o, o_stride, d_d, n, d_vox, d_face, d_t, d_npush=None):
        self._ck(self.L.ort_trace_rays_async(self.h, _p(d_o), o_stride, _p(d_d), n, _p(d_vox), _p(d_face), _p(d_t), _p(d_npush)))


class HOctree:
    """och::h_octree<Log2_table_capacity, Depth> (och_h_octree.h:17-452) with a GPU tracer."""

    def __init__(self, log2_table_capacity: int, depth: int, device: int | None = 0, node_capacity: int = 1 << 16):
        self.L = lib()
        h = _vp()
        check(self.L.ort_tree_create(C.byref(h), log2_table_capacity, depth))
        self.h = h
        self.depth = depth                                   # :24
        self.dim = 1 << depth                                # :25
        self.log2_table_capacity = log2_table_capacity       # :26
        self.table_capacity = 1 << log2_table_capacity       # :27
        self.voxel_dim = np.float32(1.0) / np.float32(self.dim)  # :28
        self.ctx = None
        if device is not None:
            self.attach(TraceContext(depth, device, node_capacity))

    def attach(self, ctx: TraceContext):
        self.ctx = ctx
        check(self.L.ort_tree_attach(self.h, ctx.h))

    def __del__(self):
        try:
            if self.h:
                self.L.ort_tree_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # ---- node store ------------------------------------------------------------------------------
    def register_node(self, children) -> int:
        a = np.ascontiguousarray(children, np.uint32)
        assert a.size == 8
        idx = self.L.ort_tree_register_node(self.h, _p(a))
        if idx == 0:
            raise OrtError(4, "node table too full (the reference prints and exits here, och_h_octree.h:112-116)")
        return idx

    def remove_node(self, idx: int):
        self.L.ort_tree_remove_node(self.h, idx)

    def set(self, x: int, y: int, z: int, v: int):
        self.L.ort_tree_set(self.h, x & 0xFFFF, y & 0xFFFF, z & 0xFFFF, v)
        if self.L.ort_tree_table_full(self.h):
            raise OrtError(4, "node table too full")

    def set_many(self, xyzv):
        a = np.ascontiguousarray(xyzv, np.uint32).reshape(-1, 4)
        self.L.ort_tree_set_many(self.h, _p(a), a.shape[0])
        if self.L.ort_tree_table_full(self.h):
            raise OrtError(4, "node table too full")

    def set_box(self, cx: int, cy: int, cz: int, ext: int, v: int):
        """The T / Z edit: an ext^3 block of set() calls centred on (cx,cy,cz) (test_och_h_octree.cpp:408-413)."""
        self.L.ort_tree_set_box(self.h, cx & 0xFFFF, cy & 0xFFFF, cz & 0xFFFF, ext, v)
        if self.L.ort_tree_table_full(self.h):
            raise OrtError(4, "node table too full")

    def fill_box(self, lo, hi, v: int):
        """Bulk edit: voxels of [lo, hi) become v (same result as the set() loop, one pass; see ort_tree_fill_box)."""
        self.L.ort_tree_fill_box(self.h, int(lo[0]), int(lo[1]), int(lo[2]), int(hi[0]), int(hi[1]), int(hi[2]), v)
        if self.L.ort_tree_table_full(self.h):
            raise OrtError(4, "node table too full")

    def save(self, path: str):
        """Dump the table (occupied slots, tags, reference counts, root, counters) to a file."""
        check(self.L.ort_tree_save(self.h, os.fsencode(path)))

    def load(self, path: str):
        """Restore a dump made by save(); the device mirror is re-uploaded at the next sync."""
        check(self.L.ort_tree_load(self.h, os.fsencode(path)))

    def at(self, x: int, y: int, z: int) -> int:
        return self.L.ort_tree_at(self.h, x, y, z)

    def set_root(self, idx: int):
        self.L.ort_tree_set_root(self.h, idx)

    def get_root(self) -> int:
        return self.L.ort_tree_get_root(self.h)

    def get_fillcnt(self) -> int:
        return self.L.ort_tree_get_fillcnt(self.h)

    def get_nodecnt(self) -> int:
        return self.L.ort_tree_get_nodecnt(self.h)

    def get_max_refcnt(self) -> int:
        return self.L.ort_tree_get_max_refcnt(self.h)

    def clear(self):
        self.L.ort_tree_clear(self.h)

    # ---- table views -----------------------------------------------------------------------------
    def nodes(self):
        return np.ctypeslib.as_array(self.L.ort_tree_nodes(self.h), shape=(self.table_capacity, 8))

    def cashes(self):
        return np.ctypeslib.as_array(self.L.ort_tree_cashes(self.h), shape=(self.table_capacity,))

    def refcounts(self):
        return np.ctypeslib.as_array(self.L.ort_tree_refcounts(self.h), shape=(self.table_capacity,))

    def flatten(self):
        """(nodes8 copy [n,8], root, level_offsets[depth+1]) in compact level-ordered numbering."""
        p = C.POINTER(C.c_uint32)()
        root = C.c_uint32(0)
        lo = np.zeros(self.depth + 1, np.uint32)
        n = self.L.ort_tree_flatten(self.h, C.byref(p), C.byref(root), _p(lo))
        arr = np.ctypeslib.as_array(p, shape=(n, 8)).copy() if n else np.zeros((0, 8), np.uint32)
        return arr, root.value, lo

    def import_dag(self, nodes8, root: int):
        """Register a compact level-ordered DAG (as flatten() / TraceContext.read_nodes give it) in this EMPTY table;
        reference counts become instance counts, so set / fill_box / sync continue from it (ort_tree_import)."""
        if hasattr(nodes8, "data_ptr"):
            if nodes8.element_size() != 4 or not nodes8.is_contiguous():
                raise ValueError("import_dag: a contiguous 32-bit tensor of n x 8 node words is required")
            if nodes8.is_cuda and self.ctx is None:
                raise ValueError("import_dag: a CUDA tensor needs an attached device context (the copy runs on its stream)")
            if nodes8.is_cuda:
                import torch
                torch.cuda.current_stream(nodes8.device).synchronize()
            n = nodes8.numel() // 8
        else:
            nodes8 = np.ascontiguousarray(nodes8, np.uint32).reshape(-1, 8)
            n = nodes8.shape[0]
        check(self.L.ort_tree_import(self.h, _p(nodes8), n, root))

    def load_voxels(self, grid):
        """Build a dense voxel grid's DAG on the attached context's GPU (TraceContext.upload_voxels), import it into
        this empty table and sync.  Returns (n_nodes, level_offsets)."""
        if self.ctx is None:
            raise OrtError(6, "load_voxels: no device context attached (the builder runs on the GPU)")
        if self.get_root() or self.get_fillcnt():
            raise OrtError(1, f"load_voxels: the table is not empty (root {self.get_root()}, {self.get_fillcnt()} live nodes)")
        n, lo = self.ctx.upload_voxels(grid)
        try:
            self.import_dag(self.ctx.read_nodes(1, n), self.ctx.root)
            self.sync()
        except BaseException:
            # the context now holds the grid, not this table: the next sync must be a full upload of the table
            self.attach(self.ctx)
            raise
        return n, lo

    def take_delta(self):
        """(ids or None, nodes8, root, is_full): the pending device update, consumed."""
        pi = C.POINTER(C.c_uint32)()
        pn = C.POINTER(C.c_uint32)()
        root = C.c_uint32(0)
        full = C.c_int(0)
        n = self.L.ort_tree_take_delta(self.h, C.byref(pi), C.byref(pn), C.byref(root), C.byref(full))
        nodes8 = np.ctypeslib.as_array(pn, shape=(n, 8)).copy() if n else np.zeros((0, 8), np.uint32)
        ids = None if full.value else (np.ctypeslib.as_array(pi, shape=(n,)).copy() if n else np.zeros(0, np.uint32))
        return ids, nodes8, root.value, bool(full.value)

    # ---- tracing (GPU only) ----------------------------------------------------------------------
    def sync(self):
        if self.ctx is None:
            raise OrtError(6, "no device context attached: tracing needs a GPU (there is no CPU path)")
        check(self.L.ort_tree_sync(self.h), self.ctx.h)
        n = C.c_uint64(0)
        full = C.c_int(0)
        self.L.ort_tree_sync_stats(self.h, C.byref(n), C.byref(full))
        return n.value, bool(full.value)

    def sse_trace(self, o, d):
        """One ray -> (Direction, hit_voxel, hit_time), as och_h_octree.h:292 / :449."""
        vox, face, t = self.trace_rays(np.asarray(o, np.float32).reshape(3), np.asarray(d, np.float32).reshape(1, 3))
        return Direction(int(face[0])), int(vox[0]), float(t[0])

    def trace_rays(self, o, d, **kw):
        self.sync()
        return self.ctx.trace_rays(o, d, **kw)

    def trace_frame(self, pos, yaw, pitch, W, H, **kw):
        """tree_camera::update_position + update_image for a camera at pos looking (yaw, pitch)."""
        self.sync()
        rot, fov = camera_coeffs(yaw, pitch)
        return self.ctx.trace_frame(pos, rot, fov, W, H, **kw)


class Octree:
    """och::octree(depth, table_capacity) (och_octree.h:10-69): plain pointer octree over a node pool, GPU tracer.
    Members as in the reference: set, unset, at, get_node_cnt, sse_trace; plus the batched forms."""

    def __init__(self, depth: int, table_capacity: int, device: int | None = 0):
        self.L = lib()
        h = _vp()
        check(self.L.ort_octree_create(C.byref(h), depth, table_capacity))
        self.h = h
        self.depth = depth
        self.dim = 1 << depth
        self.table_capacity = table_capacity
        self.ctx = None
        if device is not None:
            self.attach(TraceContext(depth, device, max(64, min(table_capacity, 1 << 16))))

    def attach(self, ctx: TraceContext):
        self.ctx = ctx
        check(self.L.ort_octree_attach(self.h, ctx.h))

    def __del__(self):
        try:
            if self.h:
                self.L.ort_octree_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def _ck_pool(self):
        if self.L.ort_octree_failed(self.h):
            raise OrtError(4, "Too many allocations (the reference prints this and exits, och_octree.cpp:50-54)")

    def set(self, x: int, y: int, z: int, vx: int):
        self.L.ort_octree_set(self.h, x, y, z, vx)
        self._ck_pool()

    def unset(self, x: int, y: int, z: int):
        self.L.ort_octree_unset(self.h, x, y, z)

    def at(self, x: int, y: int, z: int) -> int:
        return self.L.ort_octree_at(self.h, x, y, z)

    def get_node_cnt(self) -> int:
        return self.L.ort_octree_get_node_cnt(self.h)

    def apply(self, ops):
        """ops: n x (x, y, z, v, kind), kind 0 = set, 1 = unset, applied in order."""
        a = np.ascontiguousarray(ops, np.int32).reshape(-1, 5)
        self.L.ort_octree_apply(self.h, _p(a), a.shape[0])
        self._ck_pool()

    def nodes(self):
        return np.ctypeslib.as_array(self.L.ort_octree_nodes(self.h), shape=(self.table_capacity, 8))

    def sync(self):
        if self.ctx is None:
            raise OrtError(6, "no device context attached: tracing needs a GPU (there is no CPU path)")
        check(self.L.ort_octree_sync(self.h), self.ctx.h)
        n = C.c_uint64(0)
        full = C.c_int(0)
        self.L.ort_octree_sync_stats(self.h, C.byref(n), C.byref(full))
        return n.value, bool(full.value)

    def sse_trace(self, o, d):
        """One ray -> (Direction, hit_voxel, hit_time) as och_octree.cpp:167; a MISS reports hit_time 0.0."""
        vox, face, t = self.trace_rays(np.asarray(o, np.float32).reshape(3), np.asarray(d, np.float32).reshape(1, 3))
        return Direction(int(face[0])), int(vox[0]), float(t[0])

    def trace_rays(self, o, d, **kw):
        self.sync()
        return self.ctx.trace_rays(o, d, **kw)

    def trace_frame(self, pos, yaw, pitch, W, H, **kw):
        self.sync()
        rot, fov = camera_coeffs(yaw, pitch)
        return self.ctx.trace_frame(pos, rot, fov, W, H, **kw)
