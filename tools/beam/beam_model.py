"""Offline model of a conservative beam start (CPU only, statistics): for the bench frames (depth 12, 4K, poses A/B/C),
how many PUSH rounds of the reference walk lie before a tile-wide conservative start time t0 obtained from a dilated
level-k occupancy grid, and at which level the walk would be re-entered.  python tools/beam/beam_model.py [k] [tile_w tile_h]"""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import octree_ray_tracing_b200 as ort
from octree_ray_tracing_b200 import harness
from oracle import oracle as oc

K = int(sys.argv[1]) if len(sys.argv) > 1 else 6
TW, TH = (int(sys.argv[2]), int(sys.argv[3])) if len(sys.argv) > 3 else (8, 4)
FINE = int(sys.argv[4]) if len(sys.argv) > 4 else 0
DEPTH, W, H = 12, 3840, 2160
so = "/tmp/libbeam_model.so"
subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-ffp-contract=off", "-o", so, os.path.join(ROOT, "tools/beam/beam_model.c"), "-lm"])
L = C.CDLL(so)
p = lambda a: a.ctypes.data_as(C.c_void_p)

tree = ort.HOctree(24, DEPTH, device=None)
harness.build_terrain(tree)
nodes8, root, _ = tree.flatten()
nodes8 = np.ascontiguousarray(nodes8, np.uint32)


def dilated_grid(k):
    """occupancy of level k (ids[z, y, x] of the level-l cells, expanded level by level), dilated by one cell"""
    ids = np.array([[[root]]], np.uint32)
    for l in range(k):
        n = ids.shape[0]
        nxt = np.zeros((2 * n, 2 * n, 2 * n), np.uint32)
        ch = np.where(ids[..., None] != 0, nodes8[np.maximum(ids, 1) - 1], 0)          # (n, n, n, 8)
        for s in range(8):
            nxt[(s >> 2 & 1)::2, (s >> 1 & 1)::2, (s & 1)::2] = ch[..., s]
        ids = nxt
    occ = ids != 0
    N = 1 << k
    print(f"level {k}: {occ.sum()} of {N**3} cells occupied")
    dil = np.zeros_like(occ)
    pad = np.pad(occ, 1)
    for dz in range(3):
        for dy in range(3):
            for dx in range(3):
                dil |= pad[dz:dz + N, dy:dy + N, dx:dx + N]
    print(f"dilated: {dil.sum()} cells")
    return np.ascontiguousarray(dil, np.uint8)


def rcp_eps():
    """largest relative error of the library's reciprocal table (ort::rcp_table_rel_error)"""
    txt = open(os.path.join(ROOT, "octree_ray_tracing_b200", "csrc", "ort_rcp_table.h")).read()
    tab = np.array([int(x, 16) for x in re.findall(r"0x([0-9a-f]{8})u", txt)], np.uint32).view(np.float32).astype(np.float64)
    n = len(tab)
    lo, hi = 1.0 + np.arange(n) / n, 1.0 + np.arange(1, n + 1) / n
    return float(np.maximum(np.abs(tab * lo - 1.0), np.abs(tab * hi - 1.0)).max())


dil8 = dilated_grid(K)
N = 1 << K
fine = dilated_grid(FINE) if FINE else None
EPS = rcp_eps()

step = 4       # every step-th tile in x and y
for name in "ABC":
    pos, yaw, pitch = harness.POSES[name]
    o = np.array(pos, np.float32)
    rot, fov = oc.camera_coeffs(yaw, pitch)
    tot_r = tot_after = tot_skip = tot_n = 0
    miss_free = 0
    worst = 0.0
    lv_hist = np.zeros(16, np.int64)
    refined = tiles = 0
    # the library's tile radius R (ort::beam_tile_radius): 3.5 x 1.5 pixels from the tile's centre, the table's error
    du, dv = 3.5 * (W / H) * (2.0 / W), 1.5 * (2.0 / H)
    R = 1.01 * np.hypot(du, dv) / fov + EPS + 1e-6
    for ty in range(0, H // TH, step):
        rows = oc.gen_rays(rot, fov, W, H, ty * TH, ty * TH + TH).reshape(TH, W, 3)
        txs = np.arange(0, W // TW, step)
        d = np.stack([rows[:, tx * TW:(tx + 1) * TW, :].reshape(-1, 3) for tx in txs])     # (tiles, TW*TH, 3)
        dc = d.astype(np.float64).mean(axis=1)
        dc /= np.linalg.norm(dc, axis=1, keepdims=True)
        dev = np.linalg.norm(d.astype(np.float64) / np.linalg.norm(d.astype(np.float64), axis=2, keepdims=True) - dc[:, None, :], axis=2).max(axis=1)
        te = np.zeros(len(txs), np.float64)
        dc = np.ascontiguousarray(dc)
        L.beam_dda(p(dil8), K, p(o), p(dc), None, C.c_size_t(len(txs)), p(te), None)
        fin = np.isfinite(te)
        tiles += len(txs)
        if FINE:
            tf = np.zeros(len(txs), np.float64)
            tx_ = np.zeros(len(txs), np.float64)
            L.beam_dda(p(fine), FINE, p(o), p(dc), p(np.ascontiguousarray(np.where(fin, te, 0.0))), C.c_size_t(len(txs)), p(tf), p(tx_))
            stop = np.where(np.isfinite(tf), tf, tx_)
            ok = fin & (R * stop + 3e-5 <= 0.7 * 2.0 ** -FINE)
            te = np.where(ok, tf, te)
            refined += int(ok.sum())
        fin = np.isfinite(te)
        worst = max(worst, float((np.where(fin, te, 1.8) * (dev + 4e-4)).max() * N))       # beam radius at t0 in level-k cells (must stay < 1)
        t0 = np.repeat((te * (1 - 1e-3)).astype(np.float32), TW * TH)
        dd = np.ascontiguousarray(d.reshape(-1, 3), np.float32)
        n = len(dd)
        rounds = np.zeros(n, np.int32); at_r = np.zeros(n, np.int32); at_l = np.zeros(n, np.int32); th = np.zeros(n, np.float32)
        L.beam_walk(p(nodes8), C.c_uint32(root), DEPTH, p(o), p(dd), p(t0), C.c_size_t(n), p(rounds), p(at_r), p(at_l), p(th))
        assert not (np.isfinite(th) & (th < t0)).any(), "t0 not conservative"
        found = at_r >= 0
        # rays whose tile start lies beyond their walk: a MISS without any round
        new = np.where(found, at_l + (rounds - at_r - 1), 0)
        new = np.where(~found & np.isfinite(th), rounds, new)      # (hit before any exit time >= t0 cannot happen when conservative)
        miss_free += int((~found & ~np.isfinite(th)).sum())
        tot_r += int(rounds.sum()); tot_after += int(new.sum()); tot_n += n
        np.add.at(lv_hist, at_l[found], 1)
    print(f"pose {name}: rounds/ray {tot_r / tot_n:.2f} -> {tot_after / tot_n:.2f} ({tot_after / tot_r:.3f}); rays that become a MISS without a round: {miss_free / tot_n:.3f}; "
          f"beam radius at t0 <= {worst:.2f} level-{K} cells; re-entry level histogram {lv_hist[1:13].tolist()}"
          + (f"; tiles refined on level {FINE}: {refined / tiles:.3f} (R = {R:.3g}, up to t = {(0.7 * 2.0 ** -FINE - 3e-5) / R:.3f})" if FINE else ""))
