"""Time the beam start's march launch (beam_start_kernel) and the frame launch after it, per bench pose (depth-12 terrain,
3840x2160, the bench's device-buffer frames), with torch.profiler in a run of its own; also the grid build of a DAG
version and the rounds per ray the frame launches run.  Prints one JSON line.

python tools/bench_beam_march.py [--root TREE] [--reps N]   (TREE: the checkout whose package is timed, default this one)"""
import argparse
import json
import os
import sys
import time

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--reps", type=int, default=20)
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))

import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

import octree_ray_tracing_b200 as ort
from octree_ray_tracing_b200 import harness

W, H, DEPTH = 3840, 2160, 12
ctx = ort.TraceContext(DEPTH, device=0, node_capacity=1 << 21)
tree = ort.HOctree(24, DEPTH, device=None)
harness.build_terrain(tree)
ids, nodes8, root, _ = tree.take_delta()
ctx.upload_full(nodes8, root)
ctx.sync()
cams = {p: (np.array(harness.POSES[p][0], np.float32),) + ort.camera_coeffs(*harness.POSES[p][1:]) for p in "ABC"}
n = W * H
out = (torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.float32, device="cuda"))
own = torch.cuda.ExternalStream(ctx.stream, device=0)


def frame(cam):
    ctx.trace_frame_async(cam[0], cam[1], cam[2], W, H, 0, H, 1, 1, out[0], out[1], out[2], None)


ctx.set_option("beam_after", 0)
torch.cuda.synchronize()
t0 = time.perf_counter()
frame(cams["A"])                     # the first frame of the DAG version builds its grids
own.synchronize()
first_ms = (time.perf_counter() - t0) * 1e3
for cam in cams.values():
    frame(cam)
own.synchronize()

res = {"gpu": torch.cuda.get_device_name(0), "first_frame_ms_with_grid_build": round(first_ms, 3), "grid_builds": ctx.beam_builds, "poses": {}}
for name, cam in cams.items():
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.reps):
            frame(cam)
        own.synchronize()
    per = {}
    for e in prof.key_averages():
        if "beam_start_kernel" in e.key or "trace_frame_kernel" in e.key:
            kind = "march_ms" if "beam_start" in e.key else "frame_ms"
            per[kind] = round(e.device_time_total / 1e3 / e.count, 4) if hasattr(e, "device_time_total") else round(e.cuda_time_total / 1e3 / e.count, 4)
    res["poses"][name] = per
# rounds per ray the frame launches run: counted with option count_beam 2 (the counting launch refines like the frame
# launches; a build without the refinement treats 2 like 1)
dn = torch.empty(n, dtype=torch.int16, device="cuda")
ctx.set_option("count_beam", 2)
rounds = 0
for cam in cams.values():
    ctx.trace_frame_async(cam[0], cam[1], cam[2], W, H, 0, H, 1, 1, out[0], out[1], out[2], dn)
    own.synchronize()
    rounds += int((dn.to(torch.int32) & 0xFFFF).sum().item())
ctx.set_option("count_beam", 0)
res["rounds_run_per_ray"] = round(rounds / (len(cams) * n), 3)
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    ctx.set_option("beam_after", 0)
    tree.set(5, 5, 4000, 1)          # a new DAG version: the next frame builds its grids again
    nodes8, root, _ = tree.flatten()
    ctx.upload_full(nodes8, root)
    frame(cams["B"])
    own.synchronize()
build = {}
for e in prof.key_averages():
    if any(k in e.key for k in ("beam_occupancy", "beam_dilate", "beam_reduce", "beam_skip")):
        t = getattr(e, "device_time_total", None) or e.cuda_time_total
        build[e.key.split("(")[0].replace("void ort::", "")] = round(t / 1e3, 4)      # summed over levels
res["grid_build_kernels_ms"] = build
res["grid_build_ms"] = round(sum(build.values()), 4)
print(json.dumps(res))
ctx.close()
