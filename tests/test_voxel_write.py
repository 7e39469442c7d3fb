"""A dense box of voxels written into the device DAG (ort_write_voxels, TraceContext.write_voxels) against two
references: canonical_dag of the old dense grid with the box replaced, and a host table holding the old rows
(import_dag) edited with set_many / fill_box, then flatten().

The CPU tests check the two references against each other; the tests marked gpu check the write and need a B200."""
import ctypes as C

import numpy as np
import pytest

from conftest import PRODUCT_VARIANTS, assert_same_hits
from test_voxel_build import dense_of, xyzv_of
from test_voxel_build_scale import canonical_dag, cuda_free_bytes, release_cuda

POSES = {"A": ((1.5, 1.5, 1.5), 0.0, 0.0), "B": ((1.5, 1.5, 1.5), 0.7, -0.6), "C": ((1.1, 1.1, 1.4), 0.785, -0.3)}
GIB = 1 << 30


# ---- references --------------------------------------------------------------------------------------------------------

def replaced(dense, origin, box):
    """the dense grid [z, y, x] with the box at origin (x0, y0, z0) replaced"""
    out = np.array(dense, np.uint32, copy=True)
    x0, y0, z0 = origin
    nz, ny, nx = box.shape
    out[z0:z0 + nz, y0:y0 + ny, x0:x0 + nx] = np.asarray(box).astype(np.uint32)
    return out


def box_ops(origin, box):
    """set_many operations writing every voxel of the box, zeros included"""
    x0, y0, z0 = origin
    z, y, x = np.indices(box.shape).reshape(3, -1)
    return np.stack([x + x0, y + y0, z + z0, np.asarray(box).astype(np.uint32).ravel()], 1).astype(np.uint32)


def host_write(ort, nodes8, root, depth, origin, box, log2cap=20):
    """flatten() of a host table holding (nodes8, root) after set_many of every voxel of the box"""
    T = ort.HOctree(log2cap, depth, device=None)
    if root:
        T.import_dag(nodes8, root)
    T.set_many(box_ops(origin, box))
    return T.flatten()


def random_grid(rs, depth, density, vmax=4):
    dim = 1 << depth
    vals = rs.randint(1, vmax + 1, (dim, dim, dim)).astype(np.uint32)
    return np.where(rs.random_sample((dim, dim, dim)) < density, vals, 0).astype(np.uint32)


def random_box(rs, depth, kind):
    """(origin, extent) of a box of the given kind inside the cube of depth `depth`"""
    dim = 1 << depth
    if kind == "voxel":
        return tuple(int(v) for v in rs.randint(0, dim, 3)), (1, 1, 1)
    if kind == "cube":
        return (0, 0, 0), (dim, dim, dim)
    if kind == "aligned":
        s = 1 << int(rs.randint(0, depth))
        return tuple(int(s * rs.randint(0, dim // s)) for _ in range(3)), (s, s, s)
    if kind == "face":                              # touches the low face on some axes and the high face on the others
        ext = tuple(int(rs.randint(1, dim + 1)) for _ in range(3))
        return tuple(0 if rs.randint(2) else dim - e for e in ext), ext
    ext = tuple(int(rs.randint(1, dim + 1)) for _ in range(3))
    return tuple(int(rs.randint(0, dim - e + 1)) for e in ext), ext


def random_box_content(rs, ext, density, vmax=4):
    nx, ny, nz = ext
    vals = rs.randint(1, vmax + 1, (nz, ny, nx)).astype(np.uint32)
    return np.where(rs.random_sample((nz, ny, nx)) < density, vals, 0).astype(np.uint32)


BOX_KINDS = ("voxel", "aligned", "unaligned", "face", "cube")


def assert_rows(got, want, what):
    n8, root, lo = want
    g8, groot, glo = got
    assert groot == root, f"{what}: root {groot} != {root}"
    assert g8.shape == n8.shape, f"{what}: {g8.shape[0]} rows != {n8.shape[0]}"
    assert np.array_equal(g8, n8), f"{what}: rows differ"
    assert np.array_equal(np.asarray(glo, np.uint32), np.asarray(lo, np.uint32)), f"{what}: level offsets {glo} != {lo}"


# ---- CPU: the two references agree --------------------------------------------------------------------------------------

@pytest.mark.parametrize("depth", list(range(1, 9)))
def test_references_agree_on_random_scenes(ort, depth):
    """canonical_dag of the replaced dense grid == a host table importing the old rows, edited with set_many"""
    rs = np.random.RandomState(700 + depth)
    grid = random_grid(rs, depth, 0.3 if depth <= 5 else 0.01)
    old = canonical_dag(grid, depth)
    assert np.array_equal(dense_of(old[0], old[1], depth), grid)
    for kind in BOX_KINDS:
        if depth == 8 and kind in ("cube", "face"):
            continue                                # (a 256^3 set_many is slow on the host; the GPU tests cover them)
        origin, ext = random_box(rs, depth, kind)
        box = random_box_content(rs, ext, float(rs.choice([0.0, 0.5, 1.0])))
        want = canonical_dag(replaced(grid, origin, box), depth)
        assert_rows(host_write(ort, old[0], old[1], depth, origin, box), want, f"depth {depth} {kind} box {origin} {ext}")


def test_references_agree_when_the_scene_becomes_empty(ort):
    depth = 5
    rs = np.random.RandomState(5)
    grid = np.zeros((32, 32, 32), np.uint32)
    grid[3:9, 10:12, 20:31] = rs.randint(1, 3, (6, 2, 11))
    old = canonical_dag(grid, depth)
    box = np.zeros((6, 2, 11), np.uint32)
    want = canonical_dag(replaced(grid, (20, 10, 3), box), depth)
    assert want[1] == 0 and want[0].shape[0] == 0
    assert_rows(host_write(ort, old[0], old[1], depth, (20, 10, 3), box), want, "emptied")


# ---- GPU ----------------------------------------------------------------------------------------------------------------

def _torch():
    import torch
    return torch


def mirror_of(ctx, ret):
    """(rows, root, level_offsets) of the context's mirror; checks the write's return value against it"""
    n, lo = ret
    assert ctx.node_count == n
    return ctx.read_nodes(1, n), ctx.root, lo


def write_and_check(ctx, dense, origin, box, depth, what, src=None):
    """ctx.write_voxels(origin, src or box); the mirror equals canonical_dag of the replaced grid.  Returns the new grid."""
    new = replaced(dense, origin, box)
    got = mirror_of(ctx, ctx.write_voxels(origin, box if src is None else src))
    assert_rows(got, canonical_dag(new, depth), what)
    return new


@pytest.mark.gpu
@pytest.mark.parametrize("depth", list(range(1, 9)))
def test_gpu_write_random_scenes(ort, depth):
    """random scenes built by upload_voxels, then a chain of writes of every box kind: rows, root, n and level offsets
    equal canonical_dag of the grid each write leaves"""
    rs = np.random.RandomState(800 + depth)
    dense = random_grid(rs, depth, 0.3 if depth <= 5 else 0.02)
    ctx = ort.TraceContext(depth)
    ctx.upload_voxels(dense)
    rounds = 3 if depth <= 6 else 1
    for r in range(rounds):
        for kind in BOX_KINDS:
            origin, ext = random_box(rs, depth, kind)
            box = random_box_content(rs, ext, float(rs.choice([0.0, 0.02, 0.5, 1.0])))
            dense = write_and_check(ctx, dense, origin, box, depth, f"depth {depth} round {r} {kind} {origin} {ext}")
        assert np.array_equal(ctx.read_voxels((0, 0, 0), (1 << depth,) * 3), dense)
    ctx.close()


@pytest.mark.gpu
def test_gpu_write_dtypes_and_memory_kinds(ort):
    """uint8 / int32 / uint32 sources as numpy, CPU, pinned and CUDA tensors; read_voxels output taken as it is"""
    torch = _torch()
    depth = 6
    rs = np.random.RandomState(61)
    dense = random_grid(rs, depth, 0.2)
    ctx = ort.TraceContext(depth)
    ctx.upload_voxels(dense)
    tdt = {np.uint8: torch.uint8, np.int32: torch.int32, np.uint32: torch.uint32}
    kinds = {"numpy": lambda a, dt: a.astype(dt),
             "cpu": lambda a, dt: torch.from_numpy(a.astype(np.int64)).to(tdt[dt]),
             "pinned": lambda a, dt: torch.from_numpy(a.astype(np.int64)).to(tdt[dt]).pin_memory(),
             "cuda": lambda a, dt: torch.from_numpy(a.astype(np.int64)).to(tdt[dt]).cuda()}
    for dt in (np.uint8, np.int32, np.uint32):
        for kn, mk in kinds.items():
            origin, ext = random_box(rs, depth, "unaligned")
            box = random_box_content(rs, ext, 0.5, vmax=255 if dt == np.uint8 else 1 << 20)
            dense = write_and_check(ctx, dense, origin, box, depth, f"{dt.__name__} {kn}", src=mk(box, dt))
    # 32-bit values above 2^31 through int32 and uint32
    box = np.full((3, 4, 5), 0xFFFFFFF0, np.uint32)
    dense = write_and_check(ctx, dense, (7, 8, 9), box, depth, "int32 high bit", src=box.view(np.int32))
    # read_voxels' output, numpy and a CUDA tensor, written elsewhere
    back = ctx.read_voxels((10, 20, 30), (17, 9, 11))
    dense = write_and_check(ctx, dense, (40, 1, 2), back, depth, "read_voxels numpy")
    dback = torch.empty((11, 9, 17), dtype=torch.uint32, device="cuda")
    ctx.read_voxels((1, 2, 3), (17, 9, 11), out=dback)
    dense = write_and_check(ctx, dense, (0, 50, 40), dback.cpu().view(torch.int32).numpy().view(np.uint32), depth, "read_voxels cuda", src=dback)
    ctx.close()


@pytest.mark.gpu
def test_gpu_write_erasing(ort):
    """an erasing write that empties the scene (rays miss, node_count 0), writes into a context never uploaded to"""
    depth = 5
    rs = np.random.RandomState(51)
    dense = np.zeros((32, 32, 32), np.uint32)
    dense[4:20, 6:9, 10:30] = rs.randint(1, 4, (16, 3, 20))
    ctx = ort.TraceContext(depth)
    ctx.upload_voxels(dense)
    n, lo = ctx.write_voxels((10, 6, 4), np.zeros((16, 3, 20), np.uint8))
    assert n == 0 and ctx.node_count == 0 and ctx.root == 0 and (lo == 1).all()
    vox, face, t = ctx.trace_rays(np.array([[1.5, 1.5, 1.5]], np.float32), np.array([[0.3, -0.5, 0.8]], np.float32))[:3]
    assert vox[0] == 0 and np.isinf(t[0])
    assert (ctx.read_voxels((0, 0, 0), (32, 32, 32)) == 0).all()
    dense[:] = 0
    dense = write_and_check(ctx, dense, (1, 2, 3), random_box_content(rs, (7, 8, 9), 0.5), depth, "after empty")
    ctx.close()
    for d in (1, 3, 8):
        ctx = ort.TraceContext(d)
        dense = np.zeros((1 << d,) * 3, np.uint32)
        dense = write_and_check(ctx, dense, (0, 0, 0), np.zeros((1, 1, 1), np.uint32), d, f"never uploaded, zero, depth {d}")
        origin, ext = random_box(rs, d, "unaligned")
        dense = write_and_check(ctx, dense, origin, random_box_content(rs, ext, 0.4), d, f"never uploaded, depth {d}")
        ctx.close()


@pytest.mark.gpu
def test_gpu_write_over_mirrors_that_are_not_compact(ort, oc):
    """a host table synced through several deltas (unreachable rows left in the mirror), and a full upload of a hashed
    table in which one slot serves two levels"""
    depth = 7
    ctx = ort.TraceContext(depth)
    T = ort.HOctree(18, depth)
    T.attach(ctx)
    ort.harness.build_terrain(T, tunnels=True)
    T.sync()
    rs = np.random.RandomState(77)
    for _ in range(4):
        lo = rs.randint(0, 100, 3)
        T.fill_box(lo, lo + rs.randint(4, 28, 3), int(rs.randint(0, 4)))
        up, full = T.sync()
        assert not full
    n8, root, _ = T.flatten()
    assert not np.array_equal(ctx.read_nodes(), n8)          # the deltas left the mirror out of flatten()'s order
    dense = dense_of(n8, root, depth)
    for kind in BOX_KINDS:
        origin, ext = random_box(rs, depth, kind)
        dense = write_and_check(ctx, dense, origin, random_box_content(rs, ext, 0.3), depth, f"after deltas {kind}")
    ctx.close()

    # one table slot serving a leaf row and an interior row (test_voxel_build_scale), uploaded as the raw table
    depth = 5
    grid = np.zeros((32, 32, 32), np.uint32)
    pts = rs.randint(0, 32, (300, 3))
    grid[pts[:, 2], pts[:, 1], pts[:, 0]] = rs.randint(1, 3, 300)
    S = ort.HOctree(12, depth, device=None)
    S.set_many(xyzv_of(grid))
    child = int(S.nodes()[S.get_root() - 1][0])
    cell = np.array(S.nodes()[child - 1], np.uint32)
    for c in range(8):
        S.set(30 + (c & 1), 30 + ((c >> 1) & 1), 30 + (c >> 2), int(cell[c]))
    n8, root, _ = S.flatten()
    assert n8.shape[0] > S.get_fillcnt()
    dense = dense_of(n8, root, depth)
    ctx = ort.TraceContext(depth)
    for origin, ext in [((0, 0, 0), (1, 1, 1)), ((5, 7, 9), (3, 3, 3)), ((16, 0, 0), (16, 16, 16)), ((29, 29, 29), (3, 3, 3))]:
        ctx.upload_full(np.array(S.nodes()), S.get_root())
        box = random_box_content(rs, ext, 0.5)
        write_and_check(ctx, dense, origin, box, depth, f"two-level slot, box {origin} {ext}")
    ctx.close()


@pytest.fixture(scope="module")
def terrain12_rows(ort):
    S = ort.HOctree(24, 12, device=None)
    ort.harness.build_terrain(S, tunnels=True)
    return S


def frames_equal(ort, ctx, ref, what, W=640, H=360):
    for variant in PRODUCT_VARIANTS:
        ctx.set_option("variant", variant)
        ref.set_option("variant", variant)
        for name, (pos, yaw, pitch) in POSES.items():
            rot, fov = ort.camera_coeffs(yaw, pitch)
            assert_same_hits(ctx.trace_frame(pos, rot, fov, W, H), ref.trace_frame(pos, rot, fov, W, H), f"{what} variant {variant} pose {name}")
    ctx.set_option("variant", 13)
    ref.set_option("variant", 13)


@pytest.mark.gpu
def test_gpu_write_terrain12_edits(ort, terrain12_rows):
    """T / Z-style 40^3 fills and erasures on the depth-12 terrain with tunnels: rows equal the host table's fill_box +
    flatten(); frames after each write equal a context loaded from the reference rows (beam start on, grids built at
    once, so a stale grid would show)"""
    S = terrain12_rows
    n8, root, _ = S.flatten()
    T = ort.HOctree(24, 12, device=None)
    T.import_dag(n8, root)
    ctx, ref = ort.TraceContext(12), ort.TraceContext(12)
    for c in (ctx, ref):
        c.set_option("beam_after", 0)
    ctx.upload_full(n8, root)
    ref.upload_full(n8, root)
    frames_equal(ort, ctx, ref, "before")
    column = np.array([T.at(1532, 732, z) for z in range(1 << 12)])
    top = int(np.flatnonzero(column).max())
    edits = [((1512, 712, top - 20), 0), ((1512, 712, top - 20), 3), ((2048, 2048, top // 2), 0), ((1300, 700, top + 5), 2),
             ((4056, 0, 0), 1), ((0, 4056, 4056), 0)]
    for k, (lo, v) in enumerate(edits):
        box = np.full((40, 40, 40), v, np.uint8)
        got = mirror_of(ctx, ctx.write_voxels(lo, box))
        T.fill_box(lo, tuple(a + 40 for a in lo), v)
        want = T.flatten()
        assert_rows(got, want, f"edit {k} at {lo} value {v}")
        ref.upload_full(want[0], want[1])
        frames_equal(ort, ctx, ref, f"after edit {k}")
    ctx.close()
    ref.close()


@pytest.mark.gpu
def test_gpu_write_brick_assembly_depth12(ort, terrain12_rows):
    """the depth-12 terrain rebuilt brick by brick: its 8 bricks of 2048^3, read back with read_voxels into a CUDA
    tensor, written into an empty context, give the terrain's flatten()"""
    torch = _torch()
    need = 2048 ** 3 * 4 + 40 * GIB
    if cuda_free_bytes() < need:
        pytest.skip(f"needs about {need / GIB:.0f} GiB of free device memory, {cuda_free_bytes() / GIB:.0f} GiB free")
    n8, root, lo = terrain12_rows.flatten()
    src = ort.TraceContext(12)
    src.upload_full(n8, root)
    dst = ort.TraceContext(12)
    brick = torch.empty((2048, 2048, 2048), dtype=torch.uint32, device="cuda")
    for k in range(8):
        origin = (2048 * (k & 1), 2048 * ((k >> 1) & 1), 2048 * (k >> 2))
        src.read_voxels(origin, (2048, 2048, 2048), out=brick)
        ret = dst.write_voxels(origin, brick)
    assert_rows(mirror_of(dst, ret), (n8, root, lo), "brick assembly")
    del brick
    src.close()
    dst.close()
    release_cuda()


@pytest.mark.gpu
def test_gpu_write_depth16(ort):
    """small boxes near both ends of the depth-16 cube, against a host table importing the old rows + set_many"""
    depth, dim = 16, 1 << 16
    rs = np.random.RandomState(16)
    n = 3000
    pts = np.concatenate([rs.randint(0, 40, (n // 2, 3)), dim - 1 - rs.randint(0, 40, (n // 2, 3))])
    S = ort.HOctree(18, depth, device=None)
    S.set_many(np.concatenate([pts, rs.randint(1, 5, (n, 1))], 1).astype(np.uint32))
    n8, root, _ = S.flatten()
    ctx = ort.TraceContext(depth)
    ctx.upload_full(n8, root)
    boxes = [((0, 0, 0), (13, 9, 17)), ((dim - 21, dim - 8, dim - 30), (21, 8, 30)), ((dim - 1, dim - 1, dim - 1), (1, 1, 1)),
             ((5, dim - 12, 3), (20, 12, 31)), ((32760, 32761, 32759), (9, 9, 9))]
    for origin, ext in boxes:
        box = random_box_content(rs, ext, 0.5)
        want = host_write(ort, n8, root, depth, origin, box)
        got = mirror_of(ctx, ctx.write_voxels(origin, box))
        assert_rows(got, want, f"depth 16 box {origin} {ext}")
        n8, root = want[0], want[1]
    ctx.close()


@pytest.mark.gpu
def test_gpu_write_refusals_leave_everything_unchanged(ort, oc):
    torch = _torch()
    L = ort.lib()
    depth = 12
    S = ort.HOctree(20, 8, device=None)
    ort.harness.build_terrain(S, tunnels=True)
    n8, root, _ = S.flatten()
    ctx = ort.TraceContext(depth)
    # the depth-8 terrain in the corner of a depth-12 cube: the write's ids stay small, its frames are cheap
    ctx.write_voxels((0, 0, 0), dense_of(n8, root, 8))
    pos, yaw, pitch = (1.03, 1.03, 1.06), 0.785, -0.3
    rot, fov = ort.camera_coeffs(yaw, pitch)
    before = (ctx.read_nodes(), ctx.root, ctx.trace_frame(pos, rot, fov, 320, 200))
    dim = 1 << depth
    host = np.ones(64, np.uint32)
    dev = torch.ones(65, dtype=torch.int32, device="cuda")
    pv = lambda a: C.c_void_p(a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr())
    n = C.c_size_t(0)
    lo = np.zeros(depth + 1, np.uint32)
    w = lambda x0, y0, z0, p, eb, nx, ny, nz: L.ort_write_voxels(ctx.h, x0, y0, z0, p, eb, nx, ny, nz, C.byref(n), pv(lo))
    refused = [
        (1, lambda: w(-1, 0, 0, pv(host), 4, 4, 4, 4)),
        (1, lambda: w(0, 0, 0, pv(host), 4, 0, 4, 4)),
        (1, lambda: w(dim - 3, 0, 0, pv(host), 4, 4, 1, 1)),
        (1, lambda: w(0, 0, dim, pv(host), 4, 1, 1, 1)),
        (1, lambda: w(0, 0, 0, pv(host), 4, 1, 1, -2)),
        (1, lambda: w(0, 0, 0, pv(host), 4, 2049, 1, 1)),
        (1, lambda: w(0, 0, 0, pv(host), 2, 4, 4, 4)),
        (1, lambda: w(0, 0, 0, None, 4, 4, 4, 4)),
        (1, lambda: L.ort_write_voxels(None, 0, 0, 0, pv(host), 4, 4, 4, 4, C.byref(n), pv(lo))),
        (1, lambda: w(0, 0, 0, C.c_void_p(dev.data_ptr() + 2), 4, 4, 4, 4)),
    ]
    if torch.cuda.device_count() > 1:
        other = torch.ones(64, dtype=torch.int32, device="cuda:1")
        refused.append((1, lambda: w(0, 0, 0, pv(other), 4, 4, 4, 4)))
    for k, (code, call) in enumerate(refused):
        torch.cuda.synchronize()
        assert call() == code, f"call {k} not refused"
    with pytest.raises(ort.OrtError):
        ctx.write_voxels((dim - 1, 0, 0), np.ones((1, 1, 2), np.uint8))
    with pytest.raises(TypeError):
        ctx.write_voxels((0, 0, 0), np.ones((2, 2, 2), np.int64))
    with pytest.raises(ValueError):
        ctx.write_voxels((0, 0, 0), np.ones((2, 2), np.uint8))
    # more than 2^29 - 1 ids: 2^30 distinct leaf cells in a 2048^3 box
    if cuda_free_bytes() >= 2048 ** 3 * 4 + 48 * GIB:
        big = torch.zeros((2048, 2048, 2048), dtype=torch.int32, device="cuda")
        big[::2, ::2, ::2] = torch.arange(1, (1 << 30) + 1, dtype=torch.int32, device="cuda").reshape(1024, 1024, 1024)
        with pytest.raises(ort.OrtError) as e:
            ctx.write_voxels((0, 0, 0), big)
        assert e.value.code == 5, e.value
        del big
        release_cuda()
    after = (ctx.read_nodes(), ctx.root, ctx.trace_frame(pos, rot, fov, 320, 200))
    assert np.array_equal(after[0], before[0]) and after[1] == before[1]
    assert_same_hits(after[2], before[2], "after refusals")
    ctx.close()
    # the och::octree pool layout is not a DAG
    P = ort.Octree(4, 1 << 10)
    P.apply(np.array([[1, 2, 3, 5, 0]], np.int32))
    P.sync()
    pctx = P.ctx
    rows = pctx.read_nodes()
    with pytest.raises(ort.OrtError) as e:
        pctx.write_voxels((0, 0, 0), np.ones((2, 2, 2), np.uint8))
    assert e.value.code == 1
    assert np.array_equal(pctx.read_nodes(), rows)
    assert P.voxels_at(np.array([[1, 2, 3]]))[0] == 5


@pytest.mark.gpu
def test_gpu_write_with_work_in_flight(ort, terrain12_rows):
    """a write while a defer_sync host frame is still in flight, and while work is queued on a caller's stream: the
    outgoing frame equals one traced before the write, the mirror is the reference"""
    torch = _torch()
    n8, root, _ = terrain12_rows.flatten()
    ctx = ort.TraceContext(12)
    ctx.upload_full(n8, root)
    pos, yaw, pitch = POSES["B"]
    rot, fov = ort.camera_coeffs(yaw, pitch)
    W, H = 1920, 1080
    before = ctx.trace_frame(pos, rot, fov, W, H)
    T = ort.HOctree(24, 12, device=None)
    T.import_dag(n8, root)
    lo = (1500, 700, 1000)
    T.fill_box(lo, tuple(a + 40 for a in lo), 0)
    want = T.flatten()
    out = tuple(np.zeros(W * H, dt) for dt in (np.uint32, np.uint8, np.float32)) + (None,)
    ctx.set_option("defer_sync", 1)
    try:
        ctx.trace_frame(pos, rot, fov, W, H, out=out)
        got = mirror_of(ctx, ctx.write_voxels(lo, np.zeros((40, 40, 40), np.uint8)))
        ctx.sync()
    finally:
        ctx.set_option("defer_sync", 0)
    assert_same_hits(out, before, "deferred frame")
    assert_rows(got, want, "deferred")

    # work queued on a caller's stream handed over with set_stream: a frame into CUDA tensors behind a long kernel
    ctx.upload_full(n8, root)
    s = torch.cuda.Stream()
    ctx.set_stream(s)
    try:
        with torch.cuda.stream(s):
            a = torch.randn(4096, 4096, device="cuda")
            for _ in range(20):
                a = a @ a
                a = a / a.norm()
            vox = torch.empty(W * H, dtype=torch.int32, device="cuda")
            face = torch.empty(W * H, dtype=torch.uint8, device="cuda")
            t = torch.empty(W * H, dtype=torch.float32, device="cuda")
        ctx.trace_frame_async(pos, rot, fov, W, H, 0, H, 1, 1, vox, face, t)
        got = mirror_of(ctx, ctx.write_voxels(lo, np.zeros((40, 40, 40), np.uint8)))
        s.synchronize()
    finally:
        ctx.set_stream(None)
    assert_same_hits((vox.cpu().numpy().view(np.uint32), face.cpu().numpy(), t.cpu().numpy()), before, "frame on the caller's stream")
    assert_rows(got, want, "caller's stream")
    ctx.close()
