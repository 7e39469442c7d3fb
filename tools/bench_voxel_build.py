"""Time ort_build_voxels (the GPU builder of a dense voxel grid's DAG) on the terrain fixture without tunnels.

    python tools/bench_voxel_build.py [--depths 9 10 11] [--reps 5] [--out FILE]

Per depth: the fixture's voxels expanded to a dense uint8 grid on the GPU ([z, y, x], dim^3 bytes), one warm-up build,
then --reps timed builds from that device tensor (host clock around the call, which returns after a device
synchronise).  Reports ms per build, input GB/s, nodes, the device memory the build allocates, the host build_terrain
time of the same scene in the same run, and whether the built DAG equals build_terrain(...).flatten() bitwise.
"build_alloc_gb" is what the builder itself allocated (ort_build_bytes: its peak, as it frees nothing before it ends;
the input tensor is not included).  The HBM floor is one read of the input at the data-sheet 7.7 TB/s; the builder
reads the input at least twice (count, insert), so that floor is not reachable.  Prints one JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import octree_ray_tracing_b200 as ort  # noqa: E402
from octree_ray_tracing_b200 import harness  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], q[1]
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def terrain_grid(heights: np.ndarray, grass: np.ndarray, slab: int = 64) -> torch.Tensor:
    """The tunnel-free terrain's voxels (ort_fixture.cpp, Builder::voxel) as a dense uint8 [z, y, x] grid on cuda:0."""
    dim = heights.shape[0]
    h = torch.from_numpy(heights.astype(np.int32)).cuda()
    g = torch.from_numpy(grass.astype(np.int32)).cuda()
    out = torch.empty((dim, dim, dim), dtype=torch.uint8, device="cuda")
    for z0 in range(0, dim, slab):
        z = torch.arange(z0, min(dim, z0 + slab), device="cuda", dtype=torch.int32).view(-1, 1, 1)
        v = torch.where(z >= h - 2, 4, 1)
        v = torch.where(z == h, 2 + g, v)
        out[z0:z0 + z.shape[0]] = torch.where(z > h, 0, v).to(torch.uint8)
    torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--depths", type=int, nargs="+", default=[9, 10, 11])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_voxel_build: no CUDA device (nothing here runs on the CPU)")
    name, power = card()
    rows = []
    for depth in a.depths:
        dim = 1 << depth
        ctx = ort.TraceContext(depth)
        heights = harness.heightmap_gpu(ctx, depth)
        grass = harness.grass_bits(depth)
        S = ort.HOctree(22 if depth < 11 else 23, depth, device=None)
        t0 = time.perf_counter()
        harness.build_terrain(S, heights, grass, tunnels=False, gpu=False)
        host_ms = (time.perf_counter() - t0) * 1e3
        want, root, lo = S.flatten()
        del S
        grid = terrain_grid(heights, grass)
        ctx.upload_voxels(grid)                                     # warm-up
        times = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            n, blo = ctx.upload_voxels(grid)
            times.append((time.perf_counter() - t0) * 1e3)
        same = bool(n == want.shape[0] and ctx.root == root and np.array_equal(blo, lo) and np.array_equal(ctx.read_nodes(), want))
        nbytes = dim ** 3
        ms = float(np.median(times))
        rows.append(dict(depth=depth, input_bytes=nbytes, nodes=int(n), ms_median=round(ms, 3), ms_min=round(min(times), 3),
                         input_gb_per_s=round(nbytes / ms / 1e6, 1),
                         one_read_floor_ms=round(nbytes / HBM_BYTES_PER_S * 1e3, 3),
                         share_of_one_read_floor=round(nbytes / HBM_BYTES_PER_S * 1e3 / ms, 3),
                         build_alloc_gb=round(ctx.build_bytes / 1e9, 3),
                         host_build_terrain_ms=round(host_ms, 1), bitwise_equal_to_host=same))
        del grid
        ctx.close()
        torch.cuda.empty_cache()
        print(json.dumps(rows[-1]), file=sys.stderr)
    line = json.dumps(dict(tool="bench_voxel_build", gpu=name, power_limit=power, reps=a.reps, input="uint8 CUDA tensor",
                           scene="terrain fixture without tunnels", results=rows))
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not all(r["bitwise_equal_to_host"] for r in rows):
        raise SystemExit("built DAG differs from the host builder's")


if __name__ == "__main__":
    main()
