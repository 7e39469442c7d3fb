"""Time the voxel queries read back from the device DAG: ort_read_voxels and ort_voxels_at.

    python tools/bench_voxel_query.py [--reps 10] [--out FILE]

- read_voxels of the whole cube of the tunnel-free terrain at depths 10 and 11 into a CUDA tensor (4 GB and 34 GB of
  uint32, far beyond L2): GB/s of output and the share of the write floor (output bytes at the data-sheet 7.7 TB/s).
  In the same run, upload_voxels of the grid read back (host clock around the call, which ends in a device
  synchronise) for comparison; the DAG it builds must equal the host's flatten(), which checks the read as well.
- voxels_at on the depth-12 terrain with tunnels, 2^26 random points and 2^26 coherent points (the coordinates of a
  1024 x 256 x 256 box in x order, z 1200-1455: empty air above the terrain, so each walk ends near the root), device
  buffers: lookups per second.  The 44 MiB DAG stays L2-resident.
- read_voxels of a 512^3 box into pageable and pinned host memory: end-to-end GB/s (host clock).
Device calls are timed with CUDA events on the context's stream around the enqueue-only C call, after one warm-up per
shape; medians over --reps.  Prints one JSON line with the card's name and power limit.
"""
from __future__ import annotations

import argparse
import ctypes as C
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


def event_ms(stream, call, reps):
    """median and min ms of call() (an enqueue-only C call on `stream`) over reps, after one warm-up"""
    assert call() == 0, ort.lib().ort_last_error(None)
    stream.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        rc = call()
        b.record(stream)
        b.synchronize()
        assert rc == 0
        times.append(a.elapsed_time(b))
    return float(np.median(times)), float(min(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_voxel_query: no CUDA device (nothing here runs on the CPU)")
    name, power = card()
    L = ort.lib()
    stream = torch.cuda.Stream()
    res = {}

    # ---- whole-cube reads -------------------------------------------------------------------------------------------
    cube = []
    for depth in (10, 11):
        dim = 1 << depth
        T = ort.HOctree(22 if depth < 11 else 23, depth, node_capacity=1 << 20)
        harness.build_terrain(T, tunnels=False)
        T.sync()
        want, root, lo = T.flatten()
        ctx = T.ctx
        ctx.set_stream(stream)
        out = torch.empty((dim, dim, dim), dtype=torch.int32, device="cuda")
        ptr = C.c_void_p(out.data_ptr())
        ms, ms_min = event_ms(stream, lambda: L.ort_read_voxels(ctx.h, 0, 0, 0, dim, dim, dim, ptr), a.reps)
        nbytes = 4 * dim ** 3
        # upload_voxels of what was read, on a second context: the same DAG, and the builder's time on the same grid
        up = ort.TraceContext(depth)
        up.upload_voxels(out)
        up_times = []
        for _ in range(3):
            t0 = time.perf_counter()
            n, blo = up.upload_voxels(out)
            up_times.append((time.perf_counter() - t0) * 1e3)
        same = bool(n == want.shape[0] and up.root == root and np.array_equal(blo, lo) and np.array_equal(up.read_nodes(), want))
        cube.append(dict(depth=depth, output_bytes=nbytes, ms_median=round(ms, 3), ms_min=round(ms_min, 3),
                         output_gb_per_s=round(nbytes / ms / 1e6, 1), write_floor_ms=round(nbytes / HBM_BYTES_PER_S * 1e3, 3),
                         share_of_write_floor=round(nbytes / HBM_BYTES_PER_S * 1e3 / ms, 3),
                         upload_voxels_of_the_read_grid_ms=round(float(np.median(up_times)), 2), round_trip_equal=same))
        print(json.dumps(cube[-1]), file=sys.stderr)
        up.close()
        ctx.set_stream(None)
        del out, T, ctx
        torch.cuda.empty_cache()
    res["read_whole_cube"] = cube

    # ---- points on the depth-12 terrain -----------------------------------------------------------------------------
    T = ort.HOctree(24, 12, node_capacity=1 << 21)
    harness.build_terrain(T, tunnels=True)
    T.sync()
    ctx = T.ctx
    ctx.set_stream(stream)
    n = 1 << 26
    rs = np.random.RandomState(26)
    random_pts = torch.from_numpy(rs.randint(0, 1 << 12, (n, 3)).astype(np.int32)).cuda()
    zz, yy, xx = torch.meshgrid(torch.arange(1200, 1456, device="cuda"), torch.arange(1000, 1256, device="cuda"),
                                torch.arange(1000, 2024, device="cuda"), indexing="ij")
    coherent_pts = torch.stack([xx.reshape(-1), yy.reshape(-1), zz.reshape(-1)], 1).to(torch.int32).contiguous()
    del xx, yy, zz
    out = torch.empty(n, dtype=torch.int32, device="cuda")
    pts_rows = []
    for what, pts in (("random", random_pts), ("coherent", coherent_pts)):
        ms, ms_min = event_ms(stream, lambda: L.ort_voxels_at(ctx.h, C.c_void_p(pts.data_ptr()), n, C.c_void_p(out.data_ptr())), a.reps)
        stream.synchronize()
        sample = rs.randint(0, n, 5000)
        p = pts[torch.from_numpy(sample).cuda()].cpu().numpy()
        got = out.cpu().numpy().view(np.uint32)[sample]
        ok = bool(all(int(g) == T.at(int(x), int(y), int(z)) for g, (x, y, z) in zip(got, p)))
        pts_rows.append(dict(points=what, n=n, ms_median=round(ms, 3), ms_min=round(ms_min, 3),
                             lookups_per_s=float(f"{n / ms * 1e3:.4g}"), nonzero_share=round(float((out != 0).float().mean()), 3),
                             sample_equals_at=ok))
        print(json.dumps(pts_rows[-1]), file=sys.stderr)
    res["voxels_at_depth12"] = pts_rows
    del random_pts, coherent_pts, out
    ctx.set_stream(None)

    # ---- a 512^3 box into host memory -------------------------------------------------------------------------------
    origin, ext = (1000, 1000, 1000), (512, 512, 512)
    nbytes = 4 * 512 ** 3
    host_rows = []
    for what, buf in (("pageable", np.empty((512, 512, 512), np.uint32)), ("pinned", torch.empty((512, 512, 512), dtype=torch.int32).pin_memory())):
        ctx.read_voxels(origin, ext, out=buf)                     # warm-up
        times = []
        for _ in range(max(3, a.reps // 2)):
            t0 = time.perf_counter()
            ctx.read_voxels(origin, ext, out=buf)
            times.append((time.perf_counter() - t0) * 1e3)
        ms = float(np.median(times))
        host_rows.append(dict(output=what, output_bytes=nbytes, ms_median=round(ms, 2), ms_min=round(min(times), 2),
                              end_to_end_gb_per_s=round(nbytes / ms / 1e6, 2)))
        print(json.dumps(host_rows[-1]), file=sys.stderr)
    res["read_box_512_to_host"] = host_rows

    line = json.dumps(dict(tool="bench_voxel_query", gpu=name, power_limit=power, reps=a.reps, **res))
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not all(r["round_trip_equal"] for r in cube) or not all(r["sample_equals_at"] for r in pts_rows):
        raise SystemExit("a query result differs from at() / the host DAG")


if __name__ == "__main__":
    main()
