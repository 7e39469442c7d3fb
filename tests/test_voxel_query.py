"""Voxels read back from the device DAG: ort_voxels_at (n calls of at() in one launch) and ort_read_voxels (a dense box).

The CPU tests run the queries' per-point and per-cell code (csrc/ort_query.cuh) through the host emulation against the
oracle's at() and the host tables' at(), including wrapping coordinates and malformed mirrors; the tests marked gpu run
the kernels and the C entry points on a B200."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from test_voxel_build import dense_of

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emu"))

POSES = {"A": ((1.5, 1.5, 1.5), 0.0, 0.0), "B": ((1.5, 1.5, 1.5), 0.7, -0.6), "C": ((1.1, 1.1, 1.4), 0.785, -0.3)}


@pytest.fixture(scope="module")
def eq():
    import emu_query as m
    m.lib()
    return m


# ---- helpers ---------------------------------------------------------------------------------------------------------

def host_at(at, pts):
    """at() of a host table (or the oracle's) for every row of pts"""
    return np.array([at(int(x), int(y), int(z)) for x, y, z in pts], np.uint32)


def as_int16(pts):
    """coordinates as the int16 arguments of och::octree::at (same low 16 bits)"""
    return (np.asarray(pts, np.int64) + 32768) % 65536 - 32768


def wrap_points(rs, depth, n):
    """points whose coordinates leave the cube: negative, >= dim, >= 65536, and the int32 extremes"""
    dim = 1 << depth
    special = np.array([-1, -dim, dim, dim + 1, 65535, 65536, 65536 + dim - 1, -65536, 2**31 - 1, -2**31, 123456789, -987654], np.int64)
    pts = np.concatenate([rs.randint(-(1 << 20), 1 << 20, (n, 3)), rs.choice(special, (n // 4, 3)),
                          rs.randint(0, dim, (n // 4, 3)) + rs.choice([-65536, 65536, 131072, -dim, dim], (n // 4, 3))])
    return pts.astype(np.int32)


def boxes_for(rs, depth, count):
    """random boxes inside the cube: odd origins and extents, extents of 1, one touching the far corner"""
    dim = 1 << depth
    out = [((dim - 1, dim - 1, dim - 1), (1, 1, 1)), ((0, 0, 0), (min(dim, 9), min(dim, 5), min(dim, 3)))]
    if dim >= 4:
        out.append(((dim - 3, dim - 2, dim - 3), (3, 2, 3)))
    for _ in range(count):
        ext = [int(rs.randint(1, min(dim, 13) + 1)) for _ in range(3)]
        org = [int(rs.randint(0, dim - e + 1)) for e in ext]
        out.append((tuple(org), tuple(ext)))
    return out


def at_box(at, origin, extent):
    x0, y0, z0 = origin
    nx, ny, nz = extent
    zz, yy, xx = np.meshgrid(np.arange(z0, z0 + nz), np.arange(y0, y0 + ny), np.arange(x0, x0 + nx), indexing="ij")
    return host_at(at, np.stack([xx.ravel(), yy.ravel(), zz.ravel()], 1)).reshape(nz, ny, nx)


def box_points(origin, extent):
    """the box's voxels as (n, 3) int32 points in its output order (x fastest)"""
    x0, y0, z0 = origin
    nx, ny, nz = extent
    zz, yy, xx = np.meshgrid(np.arange(z0, z0 + nz), np.arange(y0, y0 + ny), np.arange(x0, x0 + nx), indexing="ij")
    return np.stack([xx.ravel(), yy.ravel(), zz.ravel()], 1).astype(np.int32)


def check_emulation(eq, nodes8, root, depth, at_fns, pts, boxes, pool=False, dense=None):
    """the emulated queries equal every at() in at_fns, out-of-bounds loads 0; boxes at both output alignments"""
    got, oob = eq.voxels_at(nodes8, root, depth, pts, pool=pool)
    assert oob == 0
    q = as_int16(pts) if pool else pts
    for name, at in at_fns.items():
        want = host_at(at, q)
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, f"{name}: {bad.size} of {len(pts)} points differ, first {pts[bad[0]]}: {got[bad[0]]} != {want[bad[0]]}"
    for origin, extent in boxes:
        first = None
        for offset in (0, 1):
            box, oob = eq.read_voxels(nodes8, root, depth, origin, extent, pool=pool, offset=offset)
            assert oob == 0
            if first is None:
                first = box
                x0, y0, z0 = origin
                nx, ny, nz = extent
                want = dense[z0:z0 + nz, y0:y0 + ny, x0:x0 + nx] if dense is not None else at_box(next(iter(at_fns.values())), origin, extent)
                assert np.array_equal(box, want), f"box {origin} {extent}"
            else:
                assert np.array_equal(box, first), f"box {origin} {extent}, unaligned output"


def ref_walk(nodes8, root, depth, pts, pool=False):
    """at() of a mirror of nodes8 with the library's bounds rule: an interior child past the rows reads as empty"""
    n = nodes8.shape[0]
    base = 0 if pool else 1
    out = np.zeros(len(pts), np.uint32)
    for i, (x, y, z) in enumerate(np.asarray(pts, np.int64)):
        node = 0 if pool else int(root)
        if not pool and (node == 0 or node > n):
            continue
        for lvl in range(depth - 1, 0, -1):
            slot = ((x >> lvl) & 1) | (((y >> lvl) & 1) << 1) | (((z >> lvl) & 1) << 2)
            node = int(nodes8[node - base][slot])
            if node == 0 or node - base >= n:
                break
        else:
            out[i] = nodes8[node - base][(x & 1) | ((y & 1) << 1) | ((z & 1) << 2)]
    return out


# ---- CPU: the per-point and per-cell code through the host emulation --------------------------------------------------

@pytest.mark.parametrize("depth,log2cap", [(6, 16), (7, 18), (8, 19)])
def test_emulated_queries_terrain_with_tunnels(ort, oc, eq, depth, log2cap):
    h, g = oc.heightmap(depth), oc.grass_bits(depth)
    A = oc.OracleTree(log2cap, depth)
    A.initialize_terrain(h, g, True)
    S = ort.HOctree(log2cap, depth, device=None)
    ort.harness.build_terrain(S, h, g, tunnels=True)
    nodes8, root, _ = S.flatten()
    rs = np.random.RandomState(depth)
    dim = 1 << depth
    pts = np.concatenate([rs.randint(0, dim, (6000, 3)), wrap_points(rs, depth, 2000)]).astype(np.int32)
    boxes = boxes_for(rs, depth, 12) + [((0, 0, 0), (dim, dim, dim)), ((1, 3, dim // 4 + 1), (dim - 1, dim // 2 - 1, dim // 2 + 3))]
    check_emulation(eq, nodes8, root, depth, {"oracle": A.at, "host": S.at}, pts, boxes, dense=dense_of(nodes8, root, depth))


@pytest.mark.parametrize("depth", list(range(1, 17)))
def test_emulated_queries_random_content(ort, oc, eq, depth):
    """random set_many content at every depth; at depth 16 half the voxels sit around the centre, so that one table slot
    serves two levels (as in test_voxel_build's import test)"""
    dim = 1 << depth
    log2cap = 18
    rs = np.random.RandomState(100 + depth)
    n = min(4000, dim ** 3 // 2 + 1)
    pts = rs.randint(0, dim, (n, 3))
    if depth == 16:
        pts[: n // 2] = 32768 + rs.randint(-40, 40, (n // 2, 3))
    ops = np.concatenate([pts, rs.randint(1, 6, (n, 1))], 1).astype(np.uint32)
    ops[rs.random_sample(n) < 0.1, 3] = 0xFFFFFFFF
    A, S = oc.OracleTree(log2cap, depth), ort.HOctree(log2cap, depth, device=None)
    A.set_many(ops)
    S.set_many(ops)
    nodes8, root, _ = S.flatten()
    if depth == 16:
        assert nodes8.shape[0] > S.get_fillcnt()
    q = np.concatenate([ops[:1500, :3].astype(np.int64), rs.randint(0, dim, (1500, 3)), wrap_points(rs, depth, 800)]).astype(np.int32)
    boxes = boxes_for(rs, depth, 8)
    if depth >= 12:
        boxes.append(((32768 - 8, 32768 - 5, 32768 - 7), (15, 11, 13)) if depth == 16 else ((3, 5, 7), (11, 9, 6)))
    dense = dense_of(nodes8, root, depth) if depth <= 8 else None
    check_emulation(eq, nodes8, root, depth, {"oracle": A.at, "host": S.at}, q, boxes, dense=dense)


def test_emulated_queries_pool_layout(ort, oc, eq):
    """an och::octree pool after random set and unset operations, walked from row 0"""
    for depth in (1, 3, 6, 9):
        dim = 1 << depth
        rs = np.random.RandomState(7 + depth)
        n = 3000
        ops = np.zeros((n, 5), np.int32)
        ops[:, :3] = rs.randint(0, dim, (n, 3))
        ops[:, 3] = rs.randint(1, 9, n)
        ops[:, 4] = rs.random_sample(n) < 0.35
        cap = 1 << 16
        A, T = oc.OracleOctree(depth, cap), ort.Octree(depth, cap, device=None)
        A.apply(ops)
        T.apply(ops)
        pool = T.nodes().copy()
        q = np.concatenate([ops[:800, :3], rs.randint(0, dim, (800, 3)), wrap_points(rs, depth, 400)]).astype(np.int32)
        check_emulation(eq, pool, 0, depth, {"oracle": A.at, "host": T.at}, q, boxes_for(rs, depth, 6), pool=True)


def test_emulated_queries_never_leave_the_mirror(ort, eq):
    """Malformed mirrors: interior children past the last row (a corrupted row, or a mirror cut short), in both layouts.
    The walk reads 0 where it would leave the rows, equals the bounds-checked reference walk everywhere, and the
    emulation's __ldg never loads outside the rows."""
    depth = 7
    dim = 1 << depth
    rs = np.random.RandomState(77)
    ops = np.concatenate([rs.randint(0, dim, (3000, 3)), rs.randint(1, 6, (3000, 1))], 1).astype(np.uint32)
    S = ort.HOctree(18, depth, device=None)
    S.set_many(ops)
    nodes8, root, lo = S.flatten()
    n = nodes8.shape[0]
    pts = np.concatenate([ops[:, :3].astype(np.int64), rs.randint(0, dim, (2000, 3))]).astype(np.int32)
    full = ref_walk(nodes8, root, depth, pts)
    assert np.array_equal(full, host_at(S.at, pts)), "the reference walk is at() on a well-formed mirror"
    cases = []
    bad = nodes8.copy()
    for row in rs.choice(np.arange(lo[1] - 1, lo[depth - 1] - 1), 12, replace=False):      # interior rows (levels above the leaves)
        slots = np.flatnonzero(bad[row])
        bad[row][slots[: max(1, len(slots) // 2)]] = rs.choice([n + 1, n + 1000, 0x1FFFFFFF, 0xFFFFFFFF])
    cases.append(("corrupted rows", bad, root))
    cases.append(("cut short", nodes8[: int(lo[depth - 2])], root))                      # the leaf level missing
    cases.append(("root past the rows", nodes8[:5], 9))
    for what, rows, r in cases:
        got, oob = eq.voxels_at(rows, r, depth, pts)
        assert oob == 0, what
        assert np.array_equal(got, ref_walk(rows, r, depth, pts)), what
        assert (got[full == 0] == 0).all() and (got != full).any(), what
        box, oob = eq.read_voxels(rows, r, depth, (1, 2, 3), (dim - 1, dim - 3, dim - 5))
        assert oob == 0, what
        assert np.array_equal(box.ravel(), ref_walk(rows, r, depth, box_points((1, 2, 3), (dim - 1, dim - 3, dim - 5)))), what

    # pool layout: a child row past the pool's used rows
    T = ort.Octree(depth, 1 << 14, device=None)
    T.apply(np.concatenate([ops[:, :4].astype(np.int32), np.zeros((len(ops), 1), np.int32)], 1))
    used = int(np.flatnonzero(T.nodes().any(1)).max()) + 1
    pool = T.nodes()[:used].copy()
    inner = [r for r in range(used) if pool[r].any() and pool[r].max() < used][:10]
    for r in inner:
        pool[r][np.flatnonzero(pool[r])[:2]] = used + 3
    got, oob = eq.voxels_at(pool, 0, depth, pts, pool=True)
    assert oob == 0 and np.array_equal(got, ref_walk(pool, 0, depth, pts, pool=True))
    box, oob = eq.read_voxels(pool, 0, depth, (0, 1, 0), (dim, dim - 1, 5), pool=True)
    assert oob == 0 and np.array_equal(box.ravel(), ref_walk(pool, 0, depth, box_points((0, 1, 0), (dim, dim - 1, 5)), pool=True))


def test_emulated_queries_empty_mirror(eq):
    rows = np.arange(16, dtype=np.uint32).reshape(2, 8) + 1
    pts = np.array([[0, 0, 0], [1, 1, 1], [-1, 5, 2]], np.int32)
    got, oob = eq.voxels_at(rows, 0, 3, pts)                  # h_octree layout, root 0: no tree
    assert oob == 0 and (got == 0).all()
    box, oob = eq.read_voxels(rows, 0, 3, (0, 0, 0), (8, 8, 8))
    assert oob == 0 and (box == 0).all()


# ---- GPU: the kernels and the C entry points --------------------------------------------------------------------------

def _torch():
    import torch
    return torch


def _u32(t):
    """a torch.uint32 / int32 tensor as a numpy uint32 array"""
    return t.cpu().view(_torch().int32).numpy().view(np.uint32)


@pytest.fixture(scope="module")
def terrain12(ort):
    T = ort.HOctree(24, 12, node_capacity=1 << 21)
    ort.harness.build_terrain(T, tunnels=True)
    T.sync()
    return T


@pytest.mark.gpu
def test_gpu_queries_terrain12(ort, terrain12):
    """depth-12 terrain with tunnels: 2^20 random points and every voxel of three 64^3 boxes (sky, surface, tunnels)
    equal HOctree.at point for point; read_voxels of the boxes equals the same values"""
    torch = _torch()
    T = terrain12
    rs = np.random.RandomState(12)
    pts = rs.randint(0, 1 << 12, (1 << 20, 3)).astype(np.int32)
    got = T.voxels_at(pts)
    assert got.dtype == np.uint32
    assert np.array_equal(got, host_at(T.at, pts))
    launches = T.ctx.launch_count
    column = host_at(T.at, [(1532, 732, z) for z in range(1 << 12)])
    top = int(np.flatnonzero(column).max())                       # the surface above (1532, 732)
    boxes = {"sky": (1000, 2000, 3600), "surface": (1500, 700, top - 32), "tunnels": (2048, 2048, top // 2)}
    for what, origin in boxes.items():
        ext = (64, 64, 64)
        pb = box_points(origin, ext)
        want = host_at(T.at, pb).reshape(64, 64, 64)
        assert np.array_equal(T.voxels_at(pb).reshape(64, 64, 64), want), what
        assert np.array_equal(T.read_voxels(origin, ext), want), what
        assert (want == 0).all() if what == "sky" else (want != 0).any(), what
        dev = T.ctx.voxels_at(torch.from_numpy(pb).cuda())
        assert dev.dtype == torch.uint32 and dev.is_cuda and np.array_equal(_u32(dev).reshape(64, 64, 64), want)
    assert T.ctx.launch_count > launches


@pytest.mark.gpu
def test_gpu_queries_random_dags(ort, oc):
    """random DAGs at depths 1-16 (h_octree layout): points including wrapping ones equal at(); boxes equal dense_of
    (depth <= 8) or at() (above)"""
    for depth in range(1, 17):
        dim = 1 << depth
        rs = np.random.RandomState(300 + depth)
        n = min(5000, dim ** 3 // 2 + 1)
        pts = rs.randint(0, dim, (n, 3))
        if depth == 16:
            pts[: n // 2] = 32768 + rs.randint(-40, 40, (n // 2, 3))
        ops = np.concatenate([pts, rs.randint(1, 6, (n, 1))], 1).astype(np.uint32)
        T = ort.HOctree(18, depth)
        T.set_many(ops)
        q = np.concatenate([ops[:2000, :3].astype(np.int64), rs.randint(0, dim, (2000, 3)), wrap_points(rs, depth, 1000)]).astype(np.int32)
        assert np.array_equal(T.voxels_at(q), host_at(T.at, q)), f"depth {depth}"
        nodes8, root, _ = T.flatten()
        dense = dense_of(nodes8, root, depth) if depth <= 8 else None
        boxes = boxes_for(rs, depth, 8)
        if depth == 16:
            boxes.append(((32768 - 9, 32768 - 6, 32768 - 7), (17, 12, 13)))
        for origin, ext in boxes:
            x0, y0, z0 = origin
            nx, ny, nz = ext
            want = dense[z0:z0 + nz, y0:y0 + ny, x0:x0 + nx] if dense is not None else at_box(T.at, origin, ext)
            assert np.array_equal(T.read_voxels(origin, ext), want), f"depth {depth} box {origin} {ext}"
        if depth <= 7:
            assert np.array_equal(T.read_voxels((0, 0, 0), (dim, dim, dim)), dense), f"depth {depth} whole cube"


@pytest.mark.gpu
def test_gpu_queries_pool_layout(ort, oc):
    for depth in (1, 4, 8):
        dim = 1 << depth
        rs = np.random.RandomState(40 + depth)
        n = 4000
        ops = np.zeros((n, 5), np.int32)
        ops[:, :3] = rs.randint(0, dim, (n, 3))
        ops[:, 3] = rs.randint(1, 9, n)
        ops[:, 4] = rs.random_sample(n) < 0.35
        T = ort.Octree(depth, 1 << 16)
        A = oc.OracleOctree(depth, 1 << 16)
        T.apply(ops)
        A.apply(ops)
        q = np.concatenate([ops[:1000, :3], rs.randint(0, dim, (1000, 3)), wrap_points(rs, depth, 500)]).astype(np.int32)
        got = T.voxels_at(q)
        assert np.array_equal(got, host_at(T.at, as_int16(q))) and np.array_equal(got, host_at(A.at, as_int16(q))), f"depth {depth}"
        for origin, ext in boxes_for(rs, depth, 6) + [((0, 0, 0), (dim, dim, dim))]:
            assert np.array_equal(T.read_voxels(origin, ext), at_box(T.at, origin, ext)), f"depth {depth} box {origin} {ext}"
        # more edits, synced as deltas, read again
        T.apply(np.concatenate([ops[:500, :3], ops[:500, 3:4], np.ones((500, 1), np.int32)], 1))
        assert np.array_equal(T.voxels_at(q), host_at(T.at, as_int16(q)))


@pytest.mark.gpu
def test_gpu_queries_after_deltas(ort):
    """four rounds of fill_box / set_box edits, each synced as a delta: voxels_at and read_voxels equal at() after each"""
    depth = 8
    dim = 1 << depth
    T = ort.HOctree(20, depth)
    ort.harness.build_terrain(T, tunnels=True)
    T.sync()
    rs = np.random.RandomState(5)
    q = rs.randint(0, dim, (20000, 3)).astype(np.int32)
    for step in range(4):
        lo = rs.randint(0, 200, 3)
        T.fill_box(lo, lo + rs.randint(4, 50, 3), int(rs.randint(0, 4)))
        T.set_box(int(rs.randint(0, dim)), int(rs.randint(0, dim)), int(rs.randint(0, dim)), int(rs.randint(1, 12)), int(rs.randint(0, 5)))
        up, full = T.sync()
        assert not full
        edited = np.concatenate([q, box_points(tuple(int(v) for v in lo), (40, 40, 40)) % dim]).astype(np.int32)
        assert np.array_equal(T.voxels_at(edited), host_at(T.at, edited)), f"step {step}"
        nodes8, root, _ = T.flatten()
        assert np.array_equal(T.read_voxels((0, 0, 0), (dim, dim, dim)), dense_of(nodes8, root, depth)), f"step {step}"


@pytest.mark.gpu
def test_gpu_read_voxels_round_trip(ort):
    """upload_voxels then read_voxels: the grid comes back as uint32, cells of the cube outside it read 0"""
    torch = _torch()
    rs = np.random.RandomState(2026)
    cases = [(1, (2, 2, 2), 0.5, np.uint8, 3), (1, (1, 2, 1), 0.9, np.uint32, 0xFFFFFFFF), (2, (3, 4, 1), 0.5, np.uint8, 2),
             (3, (5, 7, 6), 0.9, np.uint8, 1), (4, (16, 16, 16), 0.1, np.int32, 3), (5, (31, 17, 1), 0.9, np.uint32, 5),
             (6, (50, 1, 64), 0.9, np.uint8, 2), (7, (100, 77, 1), 0.9, np.uint8, 3), (7, (128, 128, 128), 0.1, np.uint8, 2),
             (8, (200, 130, 90), 0.1, np.uint32, 4), (8, (7, 256, 255), 0.9, np.uint8, 2)]
    for depth, shape, dens, dt, vmax in cases:
        dim = 1 << depth
        vals = rs.randint(1, vmax + 1, size=shape, dtype=np.uint64)
        grid = np.where(rs.random_sample(shape) < dens, vals, 0).astype(dt)
        ctx = ort.TraceContext(depth)
        ctx.upload_voxels(grid)
        nz, ny, nx = shape
        back = ctx.read_voxels((0, 0, 0), (nx, ny, nz))
        assert back.dtype == np.uint32 and np.array_equal(back, grid.astype(np.uint32)), f"{depth} {shape}"
        cube = ctx.read_voxels((0, 0, 0), (dim, dim, dim))
        assert np.array_equal(cube[:nz, :ny, :nx], back)
        cube[:nz, :ny, :nx] = 0
        assert not cube.any()
        ctx.upload_voxels(back)                                   # the read-back grid goes straight back in
        assert np.array_equal(ctx.read_voxels((0, 0, 0), (nx, ny, nz)), back)
        ctx.close()
    # depth-10 terrain into a CUDA tensor, compared on the device
    depth, dim = 10, 1 << 10
    S = ort.HOctree(22, depth, device=None)
    ort.harness.build_terrain(S, tunnels=True)
    nodes8, root, _ = S.flatten()
    src = dense_of(torch.from_numpy(nodes8.astype(np.int32)).cuda(), root, depth).to(torch.uint8).contiguous()
    ctx = ort.TraceContext(depth)
    ctx.upload_voxels(src)
    out = torch.empty((dim, dim, dim), dtype=torch.int32, device="cuda")
    assert ctx.read_voxels((0, 0, 0), (dim, dim, dim), out=out) is out
    assert torch.equal(out, src.to(torch.int32))
    ctx.close()


@pytest.mark.gpu
def test_gpu_queries_memory_kinds(ort, terrain12):
    torch = _torch()
    T = terrain12
    ctx = T.ctx
    rs = np.random.RandomState(9)
    pts = rs.randint(-100, (1 << 12) + 100, (300001, 3)).astype(np.int32)
    want = host_at(T.at, pts)
    kinds = {"pageable": lambda a: torch.from_numpy(a.copy()), "pinned": lambda a: torch.from_numpy(a.copy()).pin_memory(),
             "cuda": lambda a: torch.from_numpy(a.copy()).cuda()}
    for ki, mk_in in kinds.items():
        for ko, mk_out in kinds.items():
            out = mk_out(np.zeros(len(pts), np.uint32).view(np.int32))
            r = ctx.voxels_at(mk_in(pts), out=out)
            assert r is out and np.array_equal(_u32(out), want), f"xyz {ki}, out {ko}"
    assert np.array_equal(ctx.voxels_at(pts.astype(np.int64)), want)             # numpy of another integer dtype
    # a host-output box of about 300^3 (more than one 64 MiB staging chunk), unaligned dimensions
    origin, ext = (1301, 999, 2401), (301, 299, 297)
    box = T.read_voxels(origin, ext)
    sub = rs.randint(0, 297 * 299 * 301, 200000)
    bp = np.stack([origin[0] + sub % 301, origin[1] + sub // 301 % 299, origin[2] + sub // (301 * 299)], 1)
    assert np.array_equal(box.ravel()[sub], host_at(T.at, bp))
    dbox = torch.empty(ext[::-1], dtype=torch.uint32, device="cuda")
    ctx.read_voxels(origin, ext, out=dbox)
    assert np.array_equal(_u32(dbox), box)
    pinned = torch.empty(ext[::-1], dtype=torch.int32).pin_memory()
    ctx.read_voxels(origin, ext, out=pinned)
    assert np.array_equal(pinned.numpy().view(np.uint32), box)
    # a device-only C call is only enqueued; ctx.sync() completes it
    d_xyz = torch.from_numpy(pts).cuda()
    d_out = torch.zeros(len(pts), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    assert ort.lib().ort_voxels_at(ctx.h, C.c_void_p(d_xyz.data_ptr()), len(pts), C.c_void_p(d_out.data_ptr())) == 0
    ctx.sync()
    assert np.array_equal(_u32(d_out), want)
    d_box = torch.zeros(ext[::-1], dtype=torch.int32, device="cuda")
    assert ort.lib().ort_read_voxels(ctx.h, *origin, *ext, C.c_void_p(d_box.data_ptr())) == 0
    ctx.sync()
    assert np.array_equal(_u32(d_box), box)
    # on a stream handed over with set_stream
    s = torch.cuda.Stream()
    ctx.set_stream(s)
    try:
        assert np.array_equal(ctx.voxels_at(pts), want)
        with torch.cuda.stream(s):
            o2 = torch.zeros(ext[::-1], dtype=torch.int32, device="cuda")
        s.synchronize()
        ctx.read_voxels(origin, ext, out=o2)
        assert np.array_equal(_u32(o2), box)
    finally:
        ctx.set_stream(None)


@pytest.mark.gpu
def test_gpu_queries_with_a_deferred_frame_in_flight(ort, terrain12):
    """a defer_sync host frame in flight, then read_voxels to host, then sync(): the frame equals an undeferred one and
    the box is right"""
    T = terrain12
    ctx = T.ctx
    pos, yaw, pitch = POSES["B"]
    rot, fov = ort.camera_coeffs(yaw, pitch)
    W, H = 1920, 1080
    ref = ctx.trace_frame(pos, rot, fov, W, H)
    boxes = [((1500, 700, 900), (64, 64, 64)), ((1501, 699, 901), (300, 300, 200))]   # within the frame's staging, and beyond it
    want = [T.read_voxels(o, e) for o, e in boxes]
    for (origin, ext), w in zip(boxes, want):
        out = tuple(np.zeros(W * H, dt) for dt in (np.uint32, np.uint8, np.float32)) + (None,)
        ctx.set_option("defer_sync", 1)
        try:
            ctx.trace_frame(pos, rot, fov, W, H, out=out)
            box = ctx.read_voxels(origin, ext)
            ctx.sync()
        finally:
            ctx.set_option("defer_sync", 0)
        for a, b in zip(out[:3], ref):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), ext
        assert np.array_equal(box, w), ext


@pytest.mark.gpu
def test_gpu_queries_empty_and_refused(ort, terrain12):
    torch = _torch()
    L = ort.lib()
    # a context never uploaded to, and an h_octree mirror with root 0: zeros
    ctx = ort.TraceContext(6)
    pts = np.random.RandomState(1).randint(-70, 70, (1000, 3)).astype(np.int32)
    assert (ctx.voxels_at(pts) == 0).all() and (ctx.read_voxels((0, 0, 0), (64, 64, 64)) == 0).all()
    ctx.upload_full(np.ones((3, 8), np.uint32), 0)
    assert (ctx.voxels_at(pts) == 0).all() and (ctx.read_voxels((3, 0, 1), (61, 64, 63)) == 0).all()
    ctx.close()

    T = terrain12
    ctx = T.ctx
    pos, yaw, pitch = POSES["A"]
    rot, fov = ort.camera_coeffs(yaw, pitch)
    before = ctx.trace_frame(pos, rot, fov, 640, 360)
    dim = 1 << 12
    host = np.full(64, 0xABCD, np.uint32)
    dev = torch.full((65,), 7, dtype=torch.int32, device="cuda")
    xyz_dev = torch.zeros((9, 3), dtype=torch.int32, device="cuda")
    pv = lambda a: C.c_void_p(a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr())
    refused = [
        lambda: L.ort_read_voxels(ctx.h, -1, 0, 0, 4, 4, 4, pv(host)),
        lambda: L.ort_read_voxels(ctx.h, 0, 0, 0, 0, 4, 4, pv(host)),
        lambda: L.ort_read_voxels(ctx.h, dim - 3, 0, 0, 4, 1, 1, pv(host)),
        lambda: L.ort_read_voxels(ctx.h, 0, 0, dim, 1, 1, 1, pv(host)),
        lambda: L.ort_read_voxels(ctx.h, 0, 0, 0, 1, 1, -2, pv(host)),
        lambda: L.ort_read_voxels(ctx.h, 0, 0, 0, 4, 4, 4, None),
        lambda: L.ort_read_voxels(None, 0, 0, 0, 4, 4, 4, pv(host)),
        lambda: L.ort_read_voxels(ctx.h, 0, 0, 0, 4, 4, 4, C.c_void_p(dev.data_ptr() + 2)),
        lambda: L.ort_voxels_at(ctx.h, None, 4, pv(host)),
        lambda: L.ort_voxels_at(ctx.h, pv(xyz_dev), 4, None),
        lambda: L.ort_voxels_at(None, pv(xyz_dev), 4, pv(host)),
        lambda: L.ort_voxels_at(ctx.h, C.c_void_p(xyz_dev.data_ptr() + 2), 4, pv(host)),
        lambda: L.ort_voxels_at(ctx.h, pv(xyz_dev), 4, C.c_void_p(dev.data_ptr() + 1)),
    ]
    for k, call in enumerate(refused):
        torch.cuda.synchronize()
        assert call() == 1, f"call {k} not refused"
        ctx.sync()
        assert (host == 0xABCD).all() and (dev.cpu() == 7).all(), f"call {k} wrote"
    assert L.ort_voxels_at(ctx.h, None, 0, None) == 0                           # n == 0: nothing to do
    with pytest.raises(ort.OrtError):
        ctx.read_voxels((0, 0, 0), (dim + 1, 1, 1))
    with pytest.raises(TypeError):
        ctx.voxels_at(torch.zeros((4, 3), dtype=torch.int64))
    with pytest.raises(ValueError):
        ctx.voxels_at(torch.zeros((3, 4), dtype=torch.int32))
    with pytest.raises(ValueError):
        ctx.voxels_at(torch.zeros((4, 3), dtype=torch.int32).t().contiguous().t())
    with pytest.raises(TypeError):
        ctx.voxels_at(np.zeros((4, 3), np.float32))
    after = ctx.trace_frame(pos, rot, fov, 640, 360)
    for a, b in zip(before, after):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    builds = ctx.beam_builds
    ctx.voxels_at(pts)
    ctx.read_voxels((0, 0, 0), (64, 64, 64))
    assert ctx.beam_builds == builds
