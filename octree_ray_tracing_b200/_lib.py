"""ctypes loader for libort_b200.so -- the C ABI declared in include/ort_b200.h.

There is no fallback: if the library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# ORT_B200_EXPERIMENTS=1 selects the measurement build (the same sources with -DORT_EXPERIMENTS: additionally carries the
# kernels that were measured and not adopted, see csrc/ort_experiments.cuh); the default is the product library.
EXPERIMENTS = os.environ.get("ORT_B200_EXPERIMENTS", "") == "1"
LIB_PATH = os.path.join(HERE, "libort_b200_exp.so" if EXPERIMENTS else "libort_b200.so")

_vp = C.c_void_p
_u32p = C.POINTER(C.c_uint32)

ORT_OK, ORT_ERR_INVALID, ORT_ERR_CUDA, ORT_ERR_NO_DEVICE, ORT_ERR_TABLE_FULL, ORT_ERR_CAPACITY, ORT_ERR_NOT_ATTACHED = range(7)


class OrtError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"ort error {code}: {msg}")
        self.code = code


_SIGS = {
    "ort_version": (C.c_char_p, []),
    "ort_last_error": (C.c_char_p, [_vp]),
    "ort_create": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_int, C.c_uint32]),
    "ort_destroy": (C.c_int, [_vp]),
    "ort_set_rcp_table": (C.c_int, [_vp, _vp, C.c_int]),
    "ort_host_rcp_table": (C.c_long, [_vp, C.c_int]),
    "ort_host_rcp_matches": (C.c_int, [_vp, C.c_int]),
    "ort_rcp_host_status": (C.c_int, [_vp]),
    "ort_upload_full": (C.c_int, [_vp, _vp, C.c_size_t, C.c_uint32]),
    "ort_upload_delta": (C.c_int, [_vp, _vp, _vp, C.c_size_t, C.c_uint32]),
    "ort_upload_pool": (C.c_int, [_vp, _vp, C.c_size_t]),
    "ort_build_voxels": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t), _vp]),
    "ort_read_nodes": (C.c_int, [_vp, C.c_uint32, C.c_size_t, _vp]),
    "ort_build_bytes": (C.c_uint64, [_vp]),
    "ort_trace_rays": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_size_t, _vp, _vp, _vp, _vp]),
    "ort_trace_frame": (C.c_int, [_vp, _vp, _vp, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _vp]),
    "ort_trace_frame_async": (C.c_int, [_vp, _vp, _vp, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _vp]),
    "ort_trace_frames_async": (C.c_int, [_vp, _vp, C.c_int]),
    "ort_trace_rays_async": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_size_t, _vp, _vp, _vp, _vp]),
    "ort_set_palette": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32]),
    "ort_parse_voxels": (C.c_int, [C.c_char_p, C.c_size_t, _vp, _vp, C.c_int]),
    "ort_trace_frame_rgba": (C.c_int, [_vp, _vp, _vp, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
    "ort_sync": (C.c_int, [_vp]),
    "ort_stream": (_vp, [_vp]),
    "ort_set_stream": (C.c_int, [_vp, _vp]),
    "ort_device": (C.c_int, [_vp]),
    "ort_node_count": (C.c_uint32, [_vp]),
    "ort_root": (C.c_uint32, [_vp]),
    "ort_launch_count": (C.c_uint64, [_vp]),
    "ort_set_option": (C.c_int, [_vp, C.c_char_p, C.c_int]),
    "ort_measure_gather_peak": (C.c_int, [_vp, C.c_size_t, C.POINTER(C.c_double)]),
    "ort_beam_level": (C.c_int, [_vp, _vp, _vp, C.c_float, C.c_int, C.c_int]),
    "ort_beam_grid": (C.c_int, [_vp, C.c_int, _vp]),
    "ort_beam_builds": (C.c_uint64, [_vp]),
    "ort_band_schedules": (C.c_uint64, [_vp]),
    "ort_host_alloc": (C.c_int, [C.POINTER(_vp), C.c_size_t]),
    "ort_host_free": (C.c_int, [_vp]),
    "ort_camera_coeffs": (None, [C.c_float, C.c_float, _vp, C.POINTER(C.c_float)]),
    "ort_tree_create": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_int]),
    "ort_tree_destroy": (None, [_vp]),
    "ort_tree_register_node": (C.c_uint32, [_vp, _vp]),
    "ort_tree_remove_node": (None, [_vp, C.c_uint32]),
    "ort_tree_set": (None, [_vp, C.c_uint16, C.c_uint16, C.c_uint16, C.c_uint32]),
    "ort_tree_set_many": (None, [_vp, _vp, C.c_size_t]),
    "ort_tree_set_box": (None, [_vp, C.c_uint16, C.c_uint16, C.c_uint16, C.c_int, C.c_uint32]),
    "ort_tree_fill_box": (None, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32]),
    "ort_tree_save": (C.c_int, [_vp, C.c_char_p]),
    "ort_tree_load": (C.c_int, [_vp, C.c_char_p]),
    "ort_tree_at": (C.c_uint32, [_vp, C.c_int, C.c_int, C.c_int]),
    "ort_tree_set_root": (None, [_vp, C.c_uint32]),
    "ort_tree_get_root": (C.c_uint32, [_vp]),
    "ort_tree_get_fillcnt": (C.c_uint32, [_vp]),
    "ort_tree_get_nodecnt": (C.c_uint32, [_vp]),
    "ort_tree_get_max_refcnt": (C.c_uint32, [_vp]),
    "ort_tree_clear": (None, [_vp]),
    "ort_tree_table_full": (C.c_int, [_vp]),
    "ort_tree_depth": (C.c_int, [_vp]),
    "ort_tree_log2_capacity": (C.c_int, [_vp]),
    "ort_tree_nodes": (_u32p, [_vp]),
    "ort_tree_cashes": (C.POINTER(C.c_uint8), [_vp]),
    "ort_tree_refcounts": (_u32p, [_vp]),
    "ort_tree_flatten": (C.c_size_t, [_vp, C.POINTER(_u32p), _u32p, _vp]),
    "ort_tree_import": (C.c_int, [_vp, _vp, C.c_size_t, C.c_uint32]),
    "ort_tree_attach": (C.c_int, [_vp, _vp]),
    "ort_tree_sync": (C.c_int, [_vp]),
    "ort_tree_sync_stats": (None, [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_int)]),
    "ort_tree_take_delta": (C.c_size_t, [_vp, C.POINTER(_u32p), C.POINTER(_u32p), _u32p, C.POINTER(C.c_int)]),
    "ort_octree_create": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_uint32]),
    "ort_octree_destroy": (None, [_vp]),
    "ort_octree_set": (None, [_vp, C.c_int16, C.c_int16, C.c_int16, C.c_uint32]),
    "ort_octree_unset": (None, [_vp, C.c_int16, C.c_int16, C.c_int16]),
    "ort_octree_at": (C.c_uint32, [_vp, C.c_int16, C.c_int16, C.c_int16]),
    "ort_octree_get_node_cnt": (C.c_int, [_vp]),
    "ort_octree_apply": (None, [_vp, _vp, C.c_size_t]),
    "ort_octree_failed": (C.c_int, [_vp]),
    "ort_octree_depth": (C.c_int, [_vp]),
    "ort_octree_table_capacity": (C.c_uint32, [_vp]),
    "ort_octree_nodes": (_u32p, [_vp]),
    "ort_octree_attach": (C.c_int, [_vp, _vp]),
    "ort_octree_sync": (C.c_int, [_vp]),
    "ort_octree_sync_stats": (None, [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_int)]),
    "ort_fixture_heightmap": (None, [C.c_int, _vp, C.c_int]),
    "ort_fixture_heightmap_opensimplex": (None, [C.c_int, C.c_int64, _vp, C.c_int]),
    "ort_opensimplex2": (None, [C.c_int64, _vp, C.c_size_t, _vp]),
    "ort_fixture_build_terrain": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int]),
    "ort_fixture_build_terrain_ex": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    "ort_fixture_heightmap_gpu": (C.c_int, [_vp, C.c_int, _vp]),
    "ort_fixture_carve_gpu": (C.c_int, [_vp, C.c_int, _vp, C.c_int, _vp]),
    "ort_mg_unique_id": (C.c_int, [_vp]),
    "ort_mg_create": (C.c_int, [C.POINTER(_vp), _vp, C.c_int, C.c_int, _vp]),
    "ort_mg_destroy": (C.c_int, [_vp]),
    "ort_mg_rank": (C.c_int, [_vp]),
    "ort_mg_world": (C.c_int, [_vp]),
    "ort_mg_nccl_version": (C.c_int, []),
    "ort_mg_strip_rows": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "ort_mg_broadcast_update": (C.c_int, [_vp, _vp, _vp, C.c_size_t, C.c_uint32, C.c_int, C.c_int]),
    "ort_mg_trace_frame_gather": (C.c_int, [_vp, _vp, _vp, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp]),
    "ort_mg_set_group": (C.c_int, [_vp, C.c_int]),
    "ort_mg_flush": (C.c_int, [_vp]),
    "ort_mg_set_transport": (C.c_int, [_vp, C.c_int]),
    "ort_mg_transport": (C.c_int, [_vp]),
    "ort_mg_set_trace_streams": (C.c_int, [_vp, C.c_int]),
    "ort_mg_wire_ops": (C.c_uint64, [_vp]),
    "ort_mg_trace_frames_gather": (C.c_int, [_vp, _vp, C.c_int]),
    "ort_mg_sync": (C.c_int, [_vp]),
    "ort_mg_stream": (_vp, [_vp]),
    "ort_mg_wire_bytes": (C.c_double, [_vp]),
}

_lib = None


def lib():
    """The loaded library (raises if libort_b200.so has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OSError(f"{LIB_PATH} is missing: run `python -m octree_ray_tracing_b200.build` "
                          "(there is no CPU or PyTorch fallback for the trace path)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def exported_symbols():
    return list(_SIGS)


def check(rc: int, ctx=None):
    if rc != ORT_OK:
        msg = lib().ort_last_error(ctx)
        raise OrtError(rc, msg.decode() if msg else "?")
