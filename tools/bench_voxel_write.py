"""Time dense box writes into the device DAG (ort_write_voxels) on the depth-12 terrain with tunnels.

    python tools/bench_voxel_write.py [--reps 10] [--out FILE]

- a 40^3 box (a T / Z-style edit: fill with 3, then erase, alternating, at the surface) written with
  TraceContext.write_voxels from a uint8 CUDA tensor, against today's path for the same edit: HOctree.fill_box on the
  host plus the delta sync (ort_tree_sync);
- a 256^3 box (the terrain's own voxels read back with read_voxels and half of them set to 2) and a whole 2048^3
  brick (read back and written again unchanged) from CUDA tensors;
- the depth-12 terrain assembled into an empty context from its 8 bricks of 2048^3, each read back with read_voxels
  into one CUDA tensor and written: end to end, and checked against the terrain's flatten().
Every time is a host clock around calls that end in a device synchronise (write_voxels returns once the mirror is
installed; the host path's sync waits for its upload), medians over --reps after one warm-up.  ort_build_bytes after
each write.  Prints one JSON line with the card's name and power limit.
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], q[1]
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def host_ms(call, reps):
    """median and min ms of call() (ends in a device synchronise) over reps, after one warm-up"""
    call(0)
    times = []
    for k in range(reps):
        t0 = time.perf_counter()
        call(k + 1)
        times.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(times)), float(min(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    depth = 12
    S = ort.HOctree(24, depth, device=None)
    harness.build_terrain(S, tunnels=True)
    n8, root, lo = S.flatten()
    res = dict(scene=f"depth-12 terrain with tunnels, {n8.shape[0]} nodes")
    column = np.array([S.at(1532, 732, z) for z in range(1 << depth)])
    top = int(np.flatnonzero(column).max())
    origin = (1512, 712, top - 20)

    # 40^3: device write against host fill_box + delta sync
    ctx = ort.TraceContext(depth)
    ctx.upload_full(n8, root)
    boxes = [torch.full((40, 40, 40), v, dtype=torch.uint8, device="cuda") for v in (3, 0)]
    torch.cuda.synchronize()
    res["write_40"] = host_ms(lambda k: ctx.write_voxels(origin, boxes[k & 1]), a.reps)
    res["write_40_build_bytes"] = ctx.build_bytes
    ctx.close()
    T = ort.HOctree(24, depth, node_capacity=n8.shape[0] + (1 << 20))
    T.import_dag(n8, root)
    T.sync()
    hi = tuple(v + 40 for v in origin)

    def host_edit(k):
        T.fill_box(origin, hi, 3 if k % 2 == 0 else 0)
        T.sync()
    res["host_fill_box_sync_40"] = host_ms(host_edit, a.reps)
    del T
    print(json.dumps(res), file=sys.stderr)

    # 256^3 and a whole 2048^3 brick
    ctx = ort.TraceContext(depth)
    ctx.upload_full(n8, root)
    o256 = (1400, 600, top - 128)
    b256 = torch.empty((256, 256, 256), dtype=torch.uint32, device="cuda")
    ctx.read_voxels(o256, (256, 256, 256), out=b256)
    e256 = [b256.clone(), b256.clone()]
    e256[1][::2] = 2
    torch.cuda.synchronize()
    res["write_256"] = host_ms(lambda k: ctx.write_voxels(o256, e256[k & 1]), a.reps)
    res["write_256_build_bytes"] = ctx.build_bytes
    del b256, e256
    brick = torch.empty((2048, 2048, 2048), dtype=torch.uint32, device="cuda")
    ctx.read_voxels((0, 0, 0), (2048, 2048, 2048), out=brick)
    torch.cuda.synchronize()
    res["write_2048_brick"] = host_ms(lambda k: ctx.write_voxels((0, 0, 0), brick), max(3, a.reps // 3))
    res["write_2048_brick_build_bytes"] = ctx.build_bytes
    got = ctx.read_nodes()
    assert ctx.root == root and np.array_equal(got, n8), "brick write changed the scene"
    print(json.dumps(res), file=sys.stderr)

    # brick assembly into an empty context, end to end (read back + write, 8 bricks)
    def assemble(_k):
        dst = ort.TraceContext(depth)
        for k in range(8):
            o = (2048 * (k & 1), 2048 * ((k >> 1) & 1), 2048 * (k >> 2))
            ctx.read_voxels(o, (2048, 2048, 2048), out=brick)
            dst.write_voxels(o, brick)
        assemble.peak = max(getattr(assemble, "peak", 0), dst.build_bytes)
        assemble.rows = (dst.read_nodes(), dst.root)
        dst.close()
    res["assembly_8_bricks"] = host_ms(assemble, max(2, a.reps // 5))
    res["assembly_last_write_build_bytes"] = assemble.peak
    assert assemble.rows[1] == root and np.array_equal(assemble.rows[0], n8), "assembly differs from flatten()"
    del brick
    ctx.close()

    line = json.dumps(dict(tool="bench_voxel_write", gpu=name, power_limit=power, reps=a.reps,
                           note="[median ms, min ms]; host clock around calls that end in a device synchronise", **res))
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
