"""Dense voxel grids into the library: the GPU builder (ort_build_voxels) against the host table's flatten(), and
ort_tree_import, which hands a compact DAG back to the host table so that edits continue from it.

The CPU tests cover ort_tree_import; the tests marked gpu cover the builder and need a B200."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_same_hits

POSES = {"A": ((1.5, 1.5, 1.5), 0.0, 0.0), "B": ((1.5, 1.5, 1.5), 0.7, -0.6), "C": ((1.1, 1.1, 1.4), 0.785, -0.3)}


# ---- helpers ---------------------------------------------------------------------------------------------------------

def dense_of(nodes8, root, depth):
    """The dense voxel grid [z, y, x] of a compact DAG: numpy for numpy input, torch (on the tensor's device) for a
    tensor.  Child c of a node covers the octant bit 0 = x, bit 1 = y, bit 2 = z."""
    if hasattr(nodes8, "index_select"):
        import torch
        tab = torch.cat([torch.zeros((1, 8), dtype=torch.int64, device=nodes8.device), nodes8.reshape(-1, 8).to(torch.int64)])
        ids = torch.full((1, 1, 1), int(root), dtype=torch.int64, device=nodes8.device)
        for _ in range(depth):
            s = ids.shape[0]
            rows = tab.index_select(0, ids.reshape(-1)).reshape(s, s, s, 2, 2, 2)
            ids = rows.permute(0, 3, 1, 4, 2, 5).reshape(2 * s, 2 * s, 2 * s)
        return ids
    tab = np.concatenate([np.zeros((1, 8), np.uint32), np.asarray(nodes8, np.uint32).reshape(-1, 8)])
    ids = np.full((1, 1, 1), int(root), np.int64)
    for _ in range(depth):
        s = ids.shape[0]
        ids = tab[ids].reshape(s, s, s, 2, 2, 2).transpose(0, 3, 1, 4, 2, 5).reshape(2 * s, 2 * s, 2 * s).astype(np.int64)
    return ids.astype(np.uint32)


def xyzv_of(grid):
    """set_many operations for the non-zero voxels of a [z, y, x] grid"""
    z, y, x = np.nonzero(grid)
    return np.stack([x, y, z, grid[z, y, x]], 1).astype(np.uint32)


def live_mask(tags):
    return (tags != 0) & (tags != 0xFF)


def assert_import_round_trip(ort, A, nodes8, root, lo, depth, log2cap, seed=0):
    """import_dag of (nodes8, root) into an empty table: flatten() gives the input back, at() and the counters equal
    the oracle table A holding the same voxels."""
    T = ort.HOctree(log2cap, depth, device=None)
    T.import_dag(nodes8, root)
    n2, r2, lo2 = T.flatten()
    assert r2 == root and np.array_equal(n2, nodes8) and np.array_equal(lo2, lo)
    assert (T.get_fillcnt(), T.get_nodecnt()) == (A.fillcnt, A.nodecnt)
    assert np.array_equal(np.sort(T.refcounts()[live_mask(T.cashes())]), np.sort(A.refcounts()[live_mask(A.cashes())]))
    rs = np.random.RandomState(seed)
    for q in rs.randint(0, 1 << depth, (3000, 3)):
        assert T.at(*q) == A.at(*q)
    return T


# ---- CPU: ort_tree_import ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("depth,log2cap", [(6, 16), (7, 18), (8, 19)])
def test_import_terrain_with_tunnels(ort, oc, depth, log2cap):
    h, g = oc.heightmap(depth), oc.grass_bits(depth)
    A = oc.OracleTree(log2cap, depth)
    A.initialize_terrain(h, g, True)
    S = ort.HOctree(log2cap, depth, device=None)
    ort.harness.build_terrain(S, h, g, tunnels=True)
    nodes8, root, lo = S.flatten()
    assert_import_round_trip(ort, A, nodes8, root, lo, depth, log2cap, seed=depth)


def test_import_random_set_many_content(ort, oc):
    depth, log2cap = 7, 18
    rs = np.random.RandomState(21)
    ops = np.concatenate([rs.randint(0, 1 << depth, (20000, 3)), rs.randint(1, 6, (20000, 1))], 1).astype(np.uint32)
    A, S = oc.OracleTree(log2cap, depth), ort.HOctree(log2cap, depth, device=None)
    A.set_many(ops)
    S.set_many(ops)
    nodes8, root, lo = S.flatten()
    T = assert_import_round_trip(ort, A, nodes8, root, lo, depth, log2cap)
    # edits continue from the imported table exactly as from the original
    more = np.concatenate([rs.randint(0, 1 << depth, (3000, 3)), rs.randint(0, 4, (3000, 1))], 1).astype(np.uint32)
    A.set_many(more)
    T.set_many(more)
    assert (T.get_fillcnt(), T.get_nodecnt()) == (A.fillcnt, A.nodecnt)
    assert np.array_equal(np.sort(T.refcounts()[live_mask(T.cashes())]), np.sort(A.refcounts()[live_mask(A.cashes())]))


def test_import_golden_reference_dag(ort, oc, golden):
    g = golden("d8_tunnels")
    depth, log2cap = int(g["depth"]), int(g["log2cap"])
    dim = 1 << depth
    grass = np.unpackbits(g["grass"])[: dim * dim].reshape(dim, dim)
    A = oc.OracleTree(log2cap, depth)
    A.initialize_terrain(g["heights"], grass, True)
    assert (A.fillcnt, A.nodecnt) == (int(g["fillcnt"]), int(g["nodecnt"]))
    # the expected level offsets come from the fixture builder's table of the same scene, which must also give the
    # golden rows themselves
    S = ort.HOctree(log2cap, depth, device=None)
    ort.harness.build_terrain(S, g["heights"], grass, tunnels=True, gpu=False)
    nodes8, root, lo = S.flatten()
    assert root == int(g["root"]) and np.array_equal(nodes8, g["nodes8"])
    assert_import_round_trip(ort, A, g["nodes8"], int(g["root"]), lo, depth, log2cap)


def test_import_slot_serving_on_two_levels(ort, oc):
    """Content addressing across levels (the case of test_host_tree's shared-slot test): a row of the last level and an
    interior row with the same bytes are one slot of the table and two rows of the compact DAG."""
    depth, log2cap = 16, 18
    rs = np.random.RandomState(116)
    n = 4000
    pts = rs.randint(0, 1 << depth, (n, 3))
    pts[: n // 2] = 32768 + rs.randint(-40, 40, (n // 2, 3))
    ops = np.concatenate([pts, rs.randint(1, 5, (n, 1))], 1).astype(np.uint32)
    A, S = oc.OracleTree(log2cap, depth), ort.HOctree(log2cap, depth, device=None)
    A.set_many(ops)
    S.set_many(ops)
    nodes8, root, lo = S.flatten()
    assert nodes8.shape[0] > S.get_fillcnt()
    assert_import_round_trip(ort, A, nodes8, root, lo, depth, log2cap)


def test_import_refusals_leave_the_table_untouched(ort, oc):
    depth, log2cap = 6, 16
    h, g = oc.heightmap(depth), oc.grass_bits(depth)
    S = ort.HOctree(log2cap, depth, device=None)
    ort.harness.build_terrain(S, h, g, tunnels=True)
    good, root, lo = S.flatten()
    n = good.shape[0]

    def refused(T, nodes8, r):
        state = (T.get_root(), T.get_fillcnt(), T.get_nodecnt(), T.cashes().copy(), T.refcounts().copy())
        with pytest.raises(ort.OrtError) as e:
            T.import_dag(nodes8, r)
        assert e.value.code == 1, str(e.value)
        assert (T.get_root(), T.get_fillcnt(), T.get_nodecnt()) == state[:3]
        assert np.array_equal(T.cashes(), state[3]) and np.array_equal(T.refcounts(), state[4])

    refused(S, good, root)                                          # a table that is not empty
    E = ort.HOctree(log2cap, depth, device=None)
    bad = good.copy(); bad[lo[1] - 1][np.flatnonzero(bad[lo[1] - 1])[0]] = n + 1
    refused(E, bad, root)                                           # child id out of range
    refused(E, good, n + 1)                                         # root out of range
    bad = good.copy(); bad[lo[2] - 1][np.flatnonzero(bad[lo[2] - 1])[0]] = 1
    refused(E, bad, root)                                           # interior child pointing upward (to the root)
    bad = good.copy(); row = lo[2] - 1; bad[row][np.flatnonzero(bad[row])[0]] = lo[2]
    refused(E, bad, root)                                           # interior child on its own level
    bad = good.copy(); bad[lo[depth - 1] - 1] = 0
    refused(E, bad, root)                                           # a reachable all-zero row (leaf level)
    bad = good.copy(); bad[lo[3] - 1] = 0
    refused(E, bad, root)                                           # a reachable all-zero interior row
    assert E.get_root() == 0 and E.get_fillcnt() == 0
    E.import_dag(good, root)                                        # and the good DAG still goes in
    assert np.array_equal(E.flatten()[0], good)


def test_dense_of_expands_like_at(ort, oc):
    depth = 5
    rs = np.random.RandomState(4)
    ops = np.concatenate([rs.randint(0, 32, (3000, 3)), rs.randint(1, 9, (3000, 1))], 1).astype(np.uint32)
    S = ort.HOctree(16, depth, device=None)
    S.set_many(ops)
    nodes8, root, _ = S.flatten()
    grid = dense_of(nodes8, root, depth)
    for x, y, z in rs.randint(0, 32, (2000, 3)):
        assert grid[z, y, x] == S.at(x, y, z)
    assert np.array_equal(xyzv_of(grid)[:, 3], grid[grid != 0])


# ---- GPU: ort_build_voxels --------------------------------------------------------------------------------------------

def host_flatten(ort, grid, depth, log2cap=22):
    S = ort.HOctree(log2cap, depth, device=None)
    S.set_many(xyzv_of(np.asarray(grid)))
    return S.flatten()


def as_source(grid, kind):
    import torch
    if kind == "host":
        return grid
    t = torch.from_numpy(grid)
    if kind == "pinned":
        return t.pin_memory()
    return t.cuda()


def assert_builds_flatten(ort, ctx, grid, want, what):
    nodes8, root, lo = want
    n, blo = ctx.upload_voxels(grid)
    assert n == nodes8.shape[0] and ctx.node_count == n and ctx.root == root, f"{what}: {n} nodes, root {ctx.root}; want {nodes8.shape[0]}, {root}"
    assert np.array_equal(blo, lo), f"{what}: level offsets {blo} != {lo}"
    got = ctx.read_nodes(1, n)
    assert np.array_equal(got, nodes8), f"{what}: {int((got != nodes8).any(1).sum())} rows differ"


@pytest.mark.gpu
def test_builder_equals_flatten_random_grids(ort):
    """Random grids of densities 0.1 %, 10 % and 90 %, depths 1-8, uint8 / int32 / uint32 (payloads up to 0xFFFFFFFF),
    extents that are not powers of two (nx = 1 among them), from host, CUDA-tensor and pinned memory."""
    rs = np.random.RandomState(2026)
    cases = [  # depth, (nz, ny, nx), density, dtype, largest payload
        (1, (2, 2, 2), 0.5, np.uint8, 3), (1, (1, 2, 1), 0.9, np.uint32, 0xFFFFFFFF), (2, (3, 4, 1), 0.5, np.uint8, 2),
        (3, (8, 8, 8), 0.9, np.uint32, 0xFFFFFFFF), (3, (5, 7, 6), 0.9, np.uint8, 1), (4, (16, 16, 16), 0.1, np.int32, 3),
        (5, (32, 32, 32), 0.9, np.uint8, 2), (5, (31, 17, 1), 0.9, np.uint32, 5), (6, (64, 64, 64), 0.001, np.uint8, 255),
        (6, (50, 1, 64), 0.9, np.uint8, 2), (7, (128, 128, 128), 0.001, np.uint32, 0xFFFFFFFF), (7, (100, 77, 1), 0.9, np.uint8, 3),
        (7, (128, 128, 128), 0.1, np.uint8, 2), (8, (256, 256, 256), 0.001, np.uint8, 200), (8, (200, 130, 90), 0.1, np.uint32, 4),
        (8, (7, 256, 255), 0.9, np.uint8, 2),
    ]
    for k, (depth, shape, dens, dt, vmax) in enumerate(cases):
        vals = rs.randint(1, vmax + 1, size=shape, dtype=np.uint64)
        grid = np.where(rs.random_sample(shape) < dens, vals, 0).astype(dt)
        want = host_flatten(ort, grid, depth)
        ctx = ort.TraceContext(depth)
        for kind in ("host", "cuda", "pinned")[k % 3:] + ("host", "cuda", "pinned")[:k % 3]:
            assert_builds_flatten(ort, ctx, as_source(grid, kind), want, f"case {k} depth {depth} {shape} {dens} {np.dtype(dt).name} {kind}")
        ctx.close()


@pytest.mark.gpu
def test_builder_edge_cases(ort):
    import torch
    for depth in (1, 3, 6):
        dim = 1 << depth
        ctx = ort.TraceContext(depth)
        # all empty: no nodes, root 0, every ray misses
        n, lo = ctx.upload_voxels(np.zeros((dim, dim, dim), np.uint8))
        assert n == 0 and ctx.root == 0 and ctx.node_count == 0 and (lo == 1).all()
        rot, fov = ort.camera_coeffs(0.7, -0.6)
        v, f, t = ctx.trace_frame((1.5, 1.5, 1.5), rot, fov, 64, 36)
        assert (v == 0).all() and (f == 6).all() and np.isinf(t).all()
        # full grid of one value: one node per level
        full = torch.full((dim, dim, dim), 7, dtype=torch.int32, device="cuda")
        n, lo = ctx.upload_voxels(full)
        assert n == depth and ctx.root == 1 and list(lo) == list(range(1, depth + 2))
        assert np.array_equal(ctx.read_nodes(), host_flatten(ort, full.cpu().numpy(), depth)[0])
        # a single voxel at each corner
        for c in range(8):
            g = np.zeros((dim, dim, dim), np.uint8)
            x, y, z = (dim - 1) * (c & 1), (dim - 1) * ((c >> 1) & 1), (dim - 1) * (c >> 2)
            g[z, y, x] = 9
            assert_builds_flatten(ort, ctx, g, host_flatten(ort, g, depth), f"depth {depth} corner {c}")
        ctx.close()


@pytest.mark.gpu
def test_builder_reproduces_the_reference_golden(ort, golden):
    """The golden d8_tunnels DAG expanded to a dense grid and built on the GPU: the same compact DAG, and the golden
    rays and poses A/B/C trace to the reference's stored outputs bit for bit."""
    import torch
    g = golden("d8_tunnels")
    depth = int(g["depth"])
    grid = dense_of(torch.from_numpy(g["nodes8"].astype(np.int32)).cuda(), int(g["root"]), depth).to(torch.int32).contiguous()
    ctx = ort.TraceContext(depth)
    n, _ = ctx.upload_voxels(grid)
    assert n == g["nodes8"].shape[0] and np.array_equal(ctx.read_nodes(), g["nodes8"])
    W, H = int(g["W"]), int(g["H"])
    for p in "ABC":
        got = ctx.trace_frame(g[f"pose{p}_pos"], g[f"pose{p}_rot"], float(g[f"pose{p}_fov"]), W, H)
        assert_same_hits(got, (g[f"pose{p}_vox"], g[f"pose{p}_face"], g[f"pose{p}_t"]), f"built d8 frame {p}")
    for k in ("rand", "edge"):
        assert_same_hits(ctx.trace_rays(g[f"{k}_o"], g[f"{k}_d"]), (g[f"{k}_vox"], g[f"{k}_face"], g[f"{k}_t"]), f"built d8 {k} rays")
    ctx.close()


@pytest.mark.gpu
def test_builder_depth10_terrain_with_tunnels(ort):
    """Scale: a depth-10 terrain with tunnels from a dense grid on the device equals build_terrain's flatten bitwise;
    a 4K frame traces identically with and without the beam start, and the beam grid is built for the new DAG."""
    import torch
    depth = 10
    S = ort.HOctree(22, depth)
    ort.harness.build_terrain(S, tunnels=True)
    nodes8, root, lo = S.flatten()
    grid = dense_of(torch.from_numpy(nodes8.astype(np.int32)).cuda(), root, depth).to(torch.uint8).contiguous()
    ctx = ort.TraceContext(depth)
    n, blo = ctx.upload_voxels(grid)
    del grid
    assert n == nodes8.shape[0] and np.array_equal(blo, lo) and ctx.root == 1
    assert np.array_equal(ctx.read_nodes(), nodes8)
    ctx.set_option("beam_after", 0)
    pos, yaw, pitch = POSES["B"]
    rot, fov = ort.camera_coeffs(yaw, pitch)
    builds = ctx.beam_builds
    with_beam = ctx.trace_frame(pos, rot, fov, 3840, 2160)
    assert ctx.beam_builds > builds
    ctx.set_option("beam", 0)
    assert_same_hits(ctx.trace_frame(pos, rot, fov, 3840, 2160), with_beam, "4K frame, beam 0 vs beam 1")
    assert (with_beam[0] != 0).sum() > 100000
    ctx.close()


@pytest.mark.gpu
def test_load_voxels_then_edits(ort, oc):
    """HOctree.load_voxels, then fill_box and set edits: the syncs after the load are deltas and every frame equals the
    oracle's trace of flatten()."""
    from test_oracle import _builtin_table
    tab = _builtin_table()
    depth = 8
    S = ort.HOctree(19, depth, device=None)
    ort.harness.build_terrain(S, tunnels=True)
    nodes8, root, _ = S.flatten()
    grid = dense_of(nodes8, root, depth).astype(np.uint8)
    T = ort.HOctree(19, depth)
    n, _ = T.load_voxels(grid)
    assert n == nodes8.shape[0] and (T.get_fillcnt(), T.get_nodecnt()) == (S.get_fillcnt(), S.get_nodecnt())
    W, H = 320, 180
    rs = np.random.RandomState(8)
    for step in range(4):
        if step:
            # the same edits on T (loaded from the grid) and on S (the host-built original, never synced: its flatten()
            # is the reference and does not disturb T's mirror bookkeeping)
            lo = rs.randint(0, 200, 3)
            hi, v = lo + rs.randint(4, 50, 3), int(rs.randint(0, 4))
            sets = [(int(x), int(y), int(z), int(rs.randint(0, 5))) for x, y, z in rs.randint(0, 256, (50, 3))]
            for tree in (T, S):
                tree.fill_box(lo, hi, v)
                for q in sets:
                    tree.set(*q)
            up, full = T.sync()
            assert not full and up > 0, f"step {step}: sync uploaded {up} nodes, full={full}"
        f8, r8, _ = S.flatten()
        for p, (pos, yaw, pitch) in POSES.items():
            got = T.trace_frame(pos, yaw, pitch, W, H)
            rot, fov = oc.camera_coeffs(yaw, pitch)
            want = oc.trace_rays(f8, r8, depth, np.array(pos, np.float32), oc.gen_rays(rot, fov, W, H), rcp_tab=tab, nthreads=4)
            assert_same_hits(got, want, f"step {step} pose {p}")
    assert (T.get_fillcnt(), T.get_nodecnt()) == (S.get_fillcnt(), S.get_nodecnt())


@pytest.mark.gpu
def test_failed_builds_leave_the_mirror_intact(ort, golden):
    g = golden("d8_tunnels")
    ctx = ort.TraceContext(8)
    ctx.upload_full(g["nodes8"], int(g["root"]))
    pos, rot, fov = g["poseB_pos"], g["poseB_rot"], float(g["poseB_fov"])
    ref = ctx.trace_frame(pos, rot, fov, 320, 180)
    L = ort.lib()
    grid = np.ones((4, 4, 4), np.uint8)
    p = grid.ctypes.data_as(C.c_void_p)
    n = C.c_size_t(0)
    for what, args in (("elem_bytes 2", (p, 2, 4, 4, 4)), ("elem_bytes 0", (p, 0, 4, 4, 4)), ("nx 0", (p, 1, 0, 4, 4)),
                       ("nz 0", (p, 1, 4, 4, 0)), ("ny 257", (p, 1, 4, 257, 4)), ("null voxels", (None, 1, 4, 4, 4))):
        rc = L.ort_build_voxels(ctx.h, *args, C.byref(n), None)
        assert rc == 1, f"{what}: rc {rc}"
        assert ctx.node_count == g["nodes8"].shape[0] and ctx.root == 1
        assert_same_hits(ctx.trace_frame(pos, rot, fov, 320, 180), ref, f"after the refused build ({what})")
    # a 4-byte device source that is not 4-byte aligned is refused (it would be read with 4-byte loads)
    import torch
    raw = torch.ones(4 * 64 + 4, dtype=torch.uint8, device="cuda")
    rc = L.ort_build_voxels(ctx.h, C.c_void_p(raw.data_ptr() + 1), 4, 4, 4, 4, C.byref(n), None)
    assert rc == 1, f"misaligned device source: rc {rc}"
    assert_same_hits(ctx.trace_frame(pos, rot, fov, 320, 180), ref, "after the refused build (misaligned source)")
    deep = ort.TraceContext(12)
    assert L.ort_build_voxels(deep.h, p, 1, 4, 4, 4, C.byref(n), None) == 1          # depth 12: refused
    deep.close()
    # a pool-layout context returns to the h_octree layout (root 1, MISS at +inf) after a build
    pool = ort.TraceContext(8)
    assert L.ort_upload_pool(pool.h, g["nodes8"].ctypes.data_as(C.c_void_p), g["nodes8"].shape[0]) == 0
    grid = dense_of(g["nodes8"], int(g["root"]), 8).astype(np.uint8)
    pool.upload_voxels(grid)
    assert pool.root == 1
    assert_same_hits(pool.trace_frame(pos, rot, fov, 320, 180), ref, "pool context after a build")
    pool.close()
    ctx.close()


@pytest.mark.gpu
def test_load_voxels_refusals_keep_frames_right(ort, oc, golden):
    """load_voxels on a synced, non-empty tree is refused before anything is built, and the next frame still shows the
    tree.  A refusal after the build (the table fills up during the import) leaves no silent wrong frame behind: the
    tree's next sync reports the full table instead of tracing the grid."""
    from test_oracle import _builtin_table
    tab = _builtin_table()
    g = golden("d8_tunnels")
    depth = 8
    T = ort.HOctree(19, depth)
    ort.harness.build_terrain(T, tunnels=True)
    pos, yaw, pitch = POSES["B"]
    W, H = 320, 180
    before = T.trace_frame(pos, yaw, pitch, W, H)
    n_before = T.ctx.node_count
    grid = dense_of(g["nodes8"], int(g["root"]), depth).astype(np.uint8)
    with pytest.raises(ort.OrtError) as e:
        T.load_voxels(grid)
    assert e.value.code == 1
    assert T.ctx.node_count == n_before
    got = T.trace_frame(pos, yaw, pitch, W, H)
    assert_same_hits(got, before, "frame after the refused load")
    f8, r8, _ = T.flatten()
    rot, fov = oc.camera_coeffs(yaw, pitch)
    want = oc.trace_rays(f8, r8, depth, np.array(pos, np.float32), oc.gen_rays(rot, fov, W, H), rcp_tab=tab, nthreads=4)
    assert_same_hits(got, want, "frame after the refused load vs oracle")

    small = ort.HOctree(10, depth)                          # 1024 slots: the golden DAG does not fit
    small.trace_frame(pos, yaw, pitch, W, H)                # (an empty tree, synced)
    with pytest.raises(ort.OrtError) as e:
        small.load_voxels(grid)
    assert e.value.code == 4
    assert small.get_root() == 0 and small.get_fillcnt() == 0
    with pytest.raises(ort.OrtError) as e:
        small.trace_frame(pos, yaw, pitch, W, H)
    assert e.value.code == 4


@pytest.mark.gpu
def test_import_from_a_cuda_tensor(ort, golden):
    """ort_tree_import reads a device buffer through the tree's context; without a context a CUDA tensor is refused."""
    import torch
    g = golden("d8_tunnels")
    dev = torch.from_numpy(g["nodes8"].astype(np.int32)).cuda()
    T = ort.HOctree(int(g["log2cap"]), int(g["depth"]))
    T.import_dag(dev, int(g["root"]))
    nodes8, root, _ = T.flatten()
    assert root == int(g["root"]) and np.array_equal(nodes8, g["nodes8"])
    assert (T.get_fillcnt(), T.get_nodecnt()) == (int(g["fillcnt"]), int(g["nodecnt"]))
    U = ort.HOctree(int(g["log2cap"]), int(g["depth"]), device=None)
    with pytest.raises(ValueError):
        U.import_dag(dev, int(g["root"]))
    assert U.get_root() == 0 and U.get_fillcnt() == 0
