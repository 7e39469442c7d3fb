"""Mint tests/golden/*.npz from the REAL reference (oracle/_ref/libochref.so, built in place from
/root/reference by oracle/Makefile).  Run in the authoring container only:

    python tests/golden/make_golden.py

Each file holds inputs (a DAG as the reference's own table produced it, camera poses) and the outputs of the
reference's own och::h_octree::sse_trace (och_h_octree.h:292-447) on this (Intel) host.  Nothing of
ours is on the producing path except the fixture recursion in ref_wrap.cpp, which drives the
reference's own register_node/set/simplex_n.  The incoherent and edge-case rays are not stored: golden_rays()
draws them again from their seed, and the file keeps their sha256 so that a different draw is caught.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as oc  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
POSES = {"A": ((1.5, 1.5, 1.5), 0.0, 0.0), "B": ((1.5, 1.5, 1.5), 0.7, -0.6), "C": ((1.1, 1.1, 1.4), 0.785, -0.3)}


def compact_of(ref_tree):
    """Compact (level-ordered) copy of a reference table: plain BFS in numpy/python, ids 1..n."""
    nodes = ref_tree.nodes()
    depth = ref_tree.depth
    root = ref_tree.root
    ids = [dict() for _ in range(depth + 2)]
    out = []
    cur = [root]
    ids[1][root] = 1
    nxt_id = 2
    for level in range(1, depth + 1):
        nxt = []
        for slot1 in cur:
            row = nodes[slot1 - 1].copy()
            if level < depth:
                for c in range(8):
                    ch = int(row[c])
                    if ch:
                        m = ids[level + 1]
                        if ch not in m:
                            m[ch] = nxt_id
                            nxt_id += 1
                            nxt.append(ch)
                        row[c] = m[ch]
            out.append(row)
        cur = nxt
    return np.array(out, np.uint32), 1


def edge_rays(rs, n_each=2000):
    """Rays that exercise the corners the reference's arithmetic has: axis-parallel directions
    (coef = -inf, NaN t), origins exactly on cell planes, negative zero, tiny components."""
    o, d = [], []
    # axis parallel, all 6 directions, random origins
    for ax in range(3):
        for s in (1.0, -1.0):
            oo = rs.uniform(1.01, 1.99, (n_each, 3))
            dd = np.zeros((n_each, 3))
            dd[:, ax] = s
            o.append(oo); d.append(dd)
    # two zero components replaced by -0.0
    oo = rs.uniform(1.01, 1.99, (n_each, 3)); dd = np.full((n_each, 3), -0.0); dd[:, 2] = -1.0
    o.append(oo); d.append(dd)
    # one zero component
    oo = rs.uniform(1.01, 1.99, (n_each, 3)); dd = rs.normal(size=(n_each, 3)); dd[:, rs.randint(0, 3, n_each)] *= 1.0
    dd[np.arange(n_each), rs.randint(0, 3, n_each)] = 0.0
    o.append(oo); d.append(dd)
    # origins on cell planes (multiples of 1/256, 1/16, 1/2)
    for q in (256, 16, 2):
        oo = 1.0 + rs.randint(1, q, (n_each, 3)) / q
        dd = rs.normal(size=(n_each, 3))
        o.append(oo); d.append(dd)
    # tiny / huge component magnitudes
    oo = rs.uniform(1.01, 1.99, (n_each, 3)); dd = rs.normal(size=(n_each, 3)) * np.array([1e-30, 1.0, 1e-12])
    o.append(oo); d.append(dd)
    oo = rs.uniform(1.01, 1.99, (n_each, 3)); dd = rs.normal(size=(n_each, 3)) * np.array([1e30, 1e-5, 1.0])
    o.append(oo); d.append(dd)
    # origins inside solid ground (face 7 "inside")
    oo = rs.uniform(1.01, 1.99, (n_each, 3)); oo[:, 2] = rs.uniform(1.01, 1.15, n_each); dd = rs.normal(size=(n_each, 3))
    o.append(oo); d.append(dd)
    return np.concatenate(o).astype(np.float32), np.concatenate(d).astype(np.float32)


RAY_SETS = ("d6_tunnels", "d8_tunnels")         # drawn in this order from one RandomState(12345)
RAY_KEYS = ("rand_o", "rand_d", "edge_o", "edge_d")


def golden_rays(name):
    """The incoherent ("rand") and edge-case ("edge") rays of golden file `name`, drawn again from their seed."""
    rs = np.random.RandomState(12345)
    for set_name in RAY_SETS:
        n = 40000
        o = np.stack([rs.uniform(1.05, 1.95, n), rs.uniform(1.05, 1.95, n), rs.uniform(1.35, 1.95, n)], 1).astype(np.float32)
        d = rs.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True); d = d.astype(np.float32)
        eo, ed = edge_rays(rs)
        if set_name == name:
            return dict(rand_o=o, rand_d=d, edge_o=eo, edge_d=ed)
    raise KeyError(name)


def rays_sha256(rays):
    h = hashlib.sha256()
    for k in RAY_KEYS:
        h.update(np.ascontiguousarray(rays[k]).tobytes())
    return h.hexdigest()


def digest(vox, face, t):
    """FNV-1a-64 over (voxel u32, face u8, t bits u32) per ray, in ray order."""
    rec = np.zeros(vox.size, dtype=[("v", "<u4"), ("f", "u1"), ("t", "<u4")])
    rec["v"], rec["f"], rec["t"] = vox, face, t.view(np.uint32)
    h = 0xCBF29CE484222325
    for b in rec.tobytes():
        h = ((h ^ b) * 0x100000001B3) & 0xFFFFFFFFFFFFFFFF
    return h


def main():
    assert oc.have_ref(), "oracle/_ref/libochref.so missing: run make -C oracle in the authoring container"

    for name, (L, D, tunnels, W, H) in {"d6_tunnels": (16, 6, True, 160, 90), "d8_tunnels": (19, 8, True, 320, 180)}.items():
        hmap = oc.ref_heightmap(D)
        grass = oc.grass_bits(D)
        T = oc.RefTree(L, D)
        T.initialize_terrain(hmap, grass, tunnels)
        nodes8, root = compact_of(T)
        C = oc.RefTree(L, D)
        C.import_compact(nodes8, root)
        data = dict(depth=D, log2cap=L, nodes8=nodes8, root=root, heights=hmap, grass=np.packbits(grass),
                    fillcnt=T.fillcnt, nodecnt=T.nodecnt, W=W, H=H)
        for pn, (pos, yaw, pitch) in POSES.items():
            rot, fov = oc.camera_coeffs(yaw, pitch)
            d = oc.gen_rays(rot, fov, W, H)
            o = np.array(pos, np.float32)
            v1, f1, t1 = T.trace(o, d)          # on the reference's own hashed table
            v2, f2, t2 = C.trace(o, d)          # on the compact copy: must be the same
            assert np.array_equal(v1, v2) and np.array_equal(f1, f2) and np.array_equal(t1.view(np.uint32), t2.view(np.uint32))
            data[f"pose{pn}_rot"] = rot
            data[f"pose{pn}_fov"] = np.float32(fov)
            data[f"pose{pn}_pos"] = o
            data[f"pose{pn}_vox"] = v1.astype(np.uint8)
            data[f"pose{pn}_face"] = f1
            data[f"pose{pn}_t"] = t1
        # incoherent rays and edge cases
        rays = golden_rays(name)
        data["rays_sha256"] = rays_sha256(rays)
        for k in ("rand", "edge"):
            v, f, t = T.trace(rays[f"{k}_o"], rays[f"{k}_d"])
            data.update({f"{k}_vox": v.astype(np.uint8), f"{k}_face": f, f"{k}_t": t})
        np.savez_compressed(os.path.join(OUT, f"{name}.npz"), **data)
        print(name, "nodes", nodes8.shape[0], "fill", T.fillcnt, {k: int((data[f'pose{k}_vox'] != 0).sum()) for k in POSES},
              "rand hits", int((data['rand_vox'] != 0).sum()), "edge faces", np.bincount(f, minlength=9).tolist())

    # full-size digests of the depth-8 default tree (the reference's h_octree<19,8>) at 1280x720
    D, L = 8, 19
    T = oc.RefTree(L, D)
    T.initialize_terrain(oc.ref_heightmap(D), oc.grass_bits(D), True)
    dig = {}
    for pn, (pos, yaw, pitch) in POSES.items():
        rot, fov = oc.camera_coeffs(yaw, pitch)
        d = oc.gen_rays(rot, fov, 1280, 720)
        v, f, t = T.trace(np.array(pos, np.float32), d)
        dig[pn] = f"{digest(v, f, t):016x}"
        dig[pn + "_hits"] = int((v != 0).sum())
    import json
    with open(os.path.join(OUT, "digests.json"), "w") as fp:
        json.dump({"d8_tunnels_1280x720": dig}, fp, indent=1)
    print(dig)


if __name__ == "__main__":
    main()
