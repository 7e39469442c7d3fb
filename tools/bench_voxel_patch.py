"""Time in-place box patches of the device DAG (ort_patch_voxels) on the depth-12 terrain with tunnels.

    python tools/bench_voxel_patch.py [--reps 20] [--session 1000] [--out FILE]

- a 40^3 box (a T / Z-style edit: fill with 3, then erase, alternating, at one surface spot) by patch_voxels, by
  write_voxels and by HOctree.fill_box on the host plus the delta sync, interleaved in one loop from the same uint8
  CUDA tensors;
- the first patch after an upload_full, which builds the patch index, on its own;
- a 256^3 and a 512^3 box (the terrain's own voxels read back with read_voxels, half of the z slices set to 2, and
  back, alternating) from uint32 CUDA tensors;
- a session of --session 40^3 fills and erasures at 50 surface spots, visited in turn: the time of each patch and the
  rows it appends ([median, max, mean]; after the first visit to a spot its contents are in the patch index); then a
  3840 x 2160 frame's trace time after the session against after compact(), which must trace the same voxels.
Every time is a host clock around calls that end in a device synchronise (a patch returns after its readback; frames
are synchronised), medians and minima over --reps after one warm-up.  Prints one JSON line with the card's name and
power limit.
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


def clock(call):
    t0 = time.perf_counter()
    r = call()
    return (time.perf_counter() - t0) * 1e3, r


def stats(times):
    return [float(np.median(times)), float(min(times))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--session", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    depth = 12
    S = ort.HOctree(24, depth, device=None)
    harness.build_terrain(S, tunnels=True)
    n8, root, _ = S.flatten()
    res = dict(scene=f"depth-12 terrain with tunnels, {n8.shape[0]} nodes")
    column = np.array([S.at(1532, 732, z) for z in range(1 << depth)])
    top = int(np.flatnonzero(column).max())
    origin = (1512, 712, top - 20)
    hi = tuple(v + 40 for v in origin)
    boxes = [torch.full((40, 40, 40), v, dtype=torch.uint8, device="cuda") for v in (3, 0)]
    torch.cuda.synchronize()

    # 40^3 at one spot: patch, write and host edit interleaved
    P, W = ort.TraceContext(depth), ort.TraceContext(depth)
    P.upload_full(n8, root)
    W.upload_full(n8, root)
    T = ort.HOctree(24, depth, node_capacity=n8.shape[0] + (1 << 20))
    T.import_dag(n8, root)
    T.sync()

    def host_edit(k):
        T.fill_box(origin, hi, 3 if k % 2 == 0 else 0)
        T.sync()
    tp, tw, th, launches = [], [], [], []
    for k in range(2 * a.reps + 2):
        l0 = P.launch_count
        t, _ = clock(lambda: P.patch_voxels(origin, boxes[k & 1]))
        launches.append(P.launch_count - l0)
        tp.append(t)
        tw.append(clock(lambda: W.write_voxels(origin, boxes[k & 1]))[0])
        th.append(clock(lambda: host_edit(k))[0])
    res["patch_40_one_spot"] = stats(tp[2:])
    res["write_40_one_spot"] = stats(tw[2:])
    res["host_fill_box_sync_40"] = stats(th[2:])
    res["patch_40_launches"] = int(np.median(launches[2:]))
    res["write_over_patch_median"] = res["write_40_one_spot"][0] / res["patch_40_one_spot"][0]
    W.close()
    del T
    print(json.dumps(res), file=sys.stderr)

    # the first patch after an upload: the index build
    tf = []
    for k in range(a.reps + 1):
        P.upload_full(n8, root)
        tf.append(clock(lambda: P.patch_voxels(origin, boxes[k & 1]))[0])
    res["first_patch_after_upload_40"] = stats(tf[1:])
    print(json.dumps(res), file=sys.stderr)

    # 256^3 and 512^3 boxes
    for s in (256, 512):
        P.upload_full(n8, root)
        o = (1400, 600, top - s // 2)
        b = torch.empty((s, s, s), dtype=torch.uint32, device="cuda")
        P.read_voxels(o, (s, s, s), out=b)
        e = [b.clone(), b]
        e[0][::2] = 2
        torch.cuda.synchronize()
        P.patch_voxels(o, e[1])                      # (builds the index)
        ts, added = [], []
        for k in range(a.reps + 1):
            t, n = clock(lambda: P.patch_voxels(o, e[k & 1]))
            ts.append(t)
            added.append(n)
        res[f"patch_{s}"] = stats(ts[1:])
        res[f"patch_{s}_rows_appended_first_two"] = added[:2]
        got = torch.empty_like(b)
        P.read_voxels(o, (s, s, s), out=got)
        assert torch.equal(got, e[a.reps & 1]), f"{s}^3 patch reads back wrong"
        del b, e, got
        torch.cuda.empty_cache()
        print(json.dumps(res), file=sys.stderr)

    # a session of edits at 50 surface spots, then a 4K frame before and after compact()
    P.upload_full(n8, root)
    rs = np.random.RandomState(1)
    spots = []
    for x, y in rs.randint(0, 4096 - 40, (50, 2)):
        col = P.read_voxels((int(x) + 20, int(y) + 20, 0), (1, 1, 4096)).ravel()
        z = int(np.flatnonzero(col).max()) - 20 if col.any() else 0
        spots.append((int(x), int(y), int(np.clip(z, 0, 4096 - 40))))
    ts, added = [], []
    for k in range(a.session):
        o = spots[(k // 2) % len(spots)]
        t, n = clock(lambda: P.patch_voxels(o, boxes[k & 1]))
        ts.append(t)
        added.append(n)
    res["session_patches"] = a.session
    res["session_patch_40"] = stats(ts[1:])
    res["session_rows_appended_per_40"] = [float(np.median(added)), int(max(added)), float(np.mean(added))]
    res["session_node_count"] = P.node_count

    pos, yaw, pitch = (1.5, 1.5, 1.5), 0.7, -0.6
    rot, fov = ort.camera_coeffs(yaw, pitch)
    Wd, Hd = 3840, 2160
    outs = (torch.empty(Wd * Hd, dtype=torch.int32, device="cuda"), torch.empty(Wd * Hd, dtype=torch.uint8, device="cuda"),
            torch.empty(Wd * Hd, dtype=torch.float32, device="cuda"))

    def frame_ms():
        def one():
            P.trace_frame_async(pos, rot, fov, Wd, Hd, 0, Hd, 1, 1, *outs)
            P.sync()
        for _ in range(3):
            one()
        return stats([clock(one)[0] for _ in range(a.reps)])
    torch.cuda.synchronize()
    res["frame_4k_after_session"] = frame_ms()
    vox_session = outs[0].clone()
    n_compact, _ = P.compact()
    res["compact_node_count"] = n_compact
    res["frame_4k_after_compact"] = frame_ms()
    assert torch.equal(vox_session, outs[0]), "frames after the session and after compact() differ"
    P.close()

    line = json.dumps(dict(tool="bench_voxel_patch", gpu=name, power_limit=power, reps=a.reps,
                           note="[median ms, min ms]; host clock around calls that end in a device synchronise", **res))
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
