"""A dense box of voxels patched into the device DAG in place (ort_patch_voxels, TraceContext.patch_voxels) against
host_patch, a plain restatement of the mirror contract: rows 1 .. n_old untouched, new contents appended level by level
from the leaf level up, in the raster order of their first cell, unless the patch index already holds them.

The CPU tests check host_patch against the references of test_voxel_write.py; the tests marked gpu check the patch and
need a B200."""
import ctypes as C

import numpy as np
import pytest

from conftest import PRODUCT_VARIANTS, assert_same_hits
from test_voxel_build import dense_of, xyzv_of
from test_voxel_build_scale import canonical_dag, cuda_free_bytes, release_cuda
from test_voxel_write import (BOX_KINDS, POSES, assert_rows, frames_equal, host_write, random_box, random_box_content,
                              random_grid, replaced)

ID_MASK = (1 << 29) - 1
GIB = 1 << 30


# ---- reference -----------------------------------------------------------------------------------------------------------

def reachable(rows, root, depth):
    """the ids reachable at each level 1 .. depth (sorted; index 0 unused); a child at or past the rows reads as empty"""
    n = rows.shape[0]
    lv = [None] * (depth + 1)
    cur = np.array([root] if 0 < root <= n else [], np.int64)
    for l in range(1, depth + 1):
        lv[l] = np.unique(cur)
        if l < depth:
            ch = rows[lv[l] - 1].ravel().astype(np.int64)
            cur = ch[(ch > 0) & (ch <= n)]
    return lv


def build_index(rows, root, depth):
    """the patch index of a mirror: per level, content -> smallest id among the reachable rows holding it"""
    index = [dict() for _ in range(depth + 1)]
    for l, ids in enumerate(reachable(rows, root, depth)):
        if l:
            for i in ids:
                index[l].setdefault(rows[i - 1].tobytes(), int(i))
    return index


def _cells(lo, ext):
    """absolute (x, y, z) of the cells of a box of cells, raster order (x fastest)"""
    z, y, x = np.indices((ext[2], ext[1], ext[0])).reshape(3, -1).astype(np.int64)
    return x + lo[0], y + lo[1], z + lo[2]


def host_patch(rows, root, depth, index, origin, box):
    """(rows, root, index, n_added) after patching box (a [z, y, x] grid) at origin into the mirror (rows, root);
    index: the patch index carried from the previous patch, or None for a fresh one (the first patch after an upload)"""
    rows = np.asarray(rows, np.uint32).reshape(-1, 8)
    box = np.asarray(box).astype(np.uint32)
    n_old = rows.shape[0]
    if index is None:
        index = build_index(rows, root, depth)
    old_root = root if 0 < root <= n_old else 0
    b0 = np.array(origin, np.int64)
    b1 = b0 + np.array(box.shape[::-1], np.int64) - 1
    ro = {l: b0 >> (depth - l + 1) for l in range(1, depth + 1)}
    re = {l: (b1 >> (depth - l + 1)) - ro[l] + 1 for l in range(1, depth + 1)}

    tab = np.concatenate([np.zeros((1, 8), np.uint32), rows])     # row of id i at tab[i]; tab[0]: no old node

    def child(p, c):                                # interior child c of old nodes p, 0 where it is at or past the rows
        w = tab[p, c].astype(np.int64)
        return np.where(w <= n_old, w, 0)

    old_at = {1: np.array([old_root], np.int64)}
    for l in range(2, depth + 1):
        x, y, z = _cells(ro[l], re[l])
        P = ((((z >> 1) - ro[l - 1][2]) * re[l - 1][1] + ((y >> 1) - ro[l - 1][1])) * re[l - 1][0] + ((x >> 1) - ro[l - 1][0]))
        old_at[l] = child(old_at[l - 1][P], (x & 1) | ((y & 1) << 1) | ((z & 1) << 2))
    appended, entered, next_id, final = [], [], n_old + 1, {}
    for l in range(depth, 0, -1):
        x, y, z = _cells(ro[l], re[l])
        p = old_at[l]
        content = np.zeros((x.size, 8), np.uint32)
        for c in range(8):
            cx, cy, cz = 2 * x + (c & 1), 2 * y + ((c >> 1) & 1), 2 * z + (c >> 2)
            if l == depth:
                inside = (cx >= b0[0]) & (cx <= b1[0]) & (cy >= b0[1]) & (cy <= b1[1]) & (cz >= b0[2]) & (cz <= b1[2])
                old = tab[p, c]
                vals = box[np.clip(cz - b0[2], 0, box.shape[0] - 1), np.clip(cy - b0[1], 0, box.shape[1] - 1), np.clip(cx - b0[0], 0, box.shape[2] - 1)]
                content[:, c] = np.where(inside, vals, old)
            else:
                q, e = ro[l + 1], re[l + 1]
                inside = (cx - q[0] >= 0) & (cx - q[0] < e[0]) & (cy - q[1] >= 0) & (cy - q[1] < e[1]) & (cz - q[2] >= 0) & (cz - q[2] < e[2])
                k = ((cz - q[2]) * e[1] + (cy - q[1])) * e[0] + (cx - q[0])
                content[:, c] = np.where(inside, final[l + 1][np.where(inside, k, 0)], child(p, c))
        uniq, first, inv = np.unique(content, axis=0, return_index=True, return_inverse=True)
        uid = np.zeros(uniq.shape[0], np.int64)
        for k in np.argsort(first):                 # new contents in the raster order of their first cell
            if not uniq[k].any():
                continue
            key = uniq[k].tobytes()
            h = index[l].get(key)
            if h is None:
                h = next_id
                next_id += 1
                appended.append(uniq[k])
                entered.append((l, key, h))
            uid[k] = h
        final[l] = uid[inv.reshape(-1)]
    assert next_id - 1 <= ID_MASK
    for l, key, h in entered:
        index[l][key] = h
    new_rows = np.concatenate([rows, np.array(appended, np.uint32).reshape(-1, 8)])
    return new_rows, int(final[1][0]), index, len(appended)


def reachable_dag(rows, root, depth):
    """(reachable node count, True when no two reachable rows of a level are equal)"""
    lv = reachable(rows, root, depth)
    count, distinct = 0, True
    for l in range(1, depth + 1):
        count += lv[l].size
        if lv[l].size:
            distinct &= np.unique(rows[lv[l] - 1], axis=0).shape[0] == lv[l].size
    return count, distinct


def check_patch_result(ort, before, after, depth, dense, what):
    """the contract on one host_patch step: old rows untouched, voxels replaced, reachable DAG == flatten()'s"""
    rows0, rows1, root1 = before, after[0], after[1]
    assert np.array_equal(rows1[:rows0.shape[0]], rows0), f"{what}: old rows changed"
    assert np.array_equal(dense_of(rows1, root1, depth), dense), f"{what}: voxels"
    count, distinct = reachable_dag(rows1, root1, depth)
    want = canonical_dag(dense, depth)
    assert distinct and count == want[0].shape[0], f"{what}: {count} reachable rows, flatten() has {want[0].shape[0]}"


# ---- CPU ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("depth", list(range(1, 9)))
def test_host_patch_on_random_scenes(ort, depth):
    """host_patch on random scenes, every box kind: voxels replaced, old rows kept, the reachable DAG is host_write's
    flatten() renumbered (canonical_dag of its voxels, same node count, no duplicate)"""
    rs = np.random.RandomState(900 + depth)
    grid = random_grid(rs, depth, 0.3 if depth <= 5 else 0.01)
    rows, root, _ = canonical_dag(grid, depth)
    for kind in BOX_KINDS:
        if depth == 8 and kind in ("cube", "face"):
            continue                                # (slow on the host; the GPU tests cover them)
        origin, ext = random_box(rs, depth, kind)
        box = random_box_content(rs, ext, float(rs.choice([0.0, 0.5, 1.0])))
        new = replaced(grid, origin, box)
        got = host_patch(rows, root, depth, None, origin, box)
        check_patch_result(ort, rows, got, depth, new, f"depth {depth} {kind} {origin} {ext}")
        hw = host_write(ort, rows, root, depth, origin, box)
        assert np.array_equal(dense_of(hw[0], hw[1], depth), new)
        assert reachable_dag(got[0], got[1], depth)[0] == hw[0].shape[0]
        assert got[3] == got[0].shape[0] - rows.shape[0]


@pytest.mark.parametrize("depth", [3, 5, 7])
def test_host_patch_chains(ort, depth):
    """chains of 20 patches with the index carried along: after each, the contract holds against the dense grid"""
    rs = np.random.RandomState(950 + depth)
    grid = random_grid(rs, depth, 0.2 if depth <= 5 else 0.02)
    rows, root, _ = canonical_dag(grid, depth)
    index = None
    for k in range(20):
        kind = BOX_KINDS[k % 4]                     # (no whole-cube box: it leaves nothing of the old scene)
        origin, ext = random_box(rs, depth, kind)
        if depth == 7:
            ext = tuple(min(e, 24) for e in ext)
        box = random_box_content(rs, ext, float(rs.choice([0.0, 0.1, 1.0])))
        grid = replaced(grid, origin, box)
        got = host_patch(rows, root, depth, index, origin, box)
        check_patch_result(ort, rows, got, depth, grid, f"depth {depth} patch {k}")
        rows, root, index = got[0], got[1], got[2]


def test_host_patch_numbering_rule():
    """a hand-checked case: depth 2, one voxel into an empty scene, then the same voxel again, then an erase"""
    rows = np.zeros((0, 8), np.uint32)
    r = host_patch(rows, 0, 2, None, (3, 0, 0), np.full((1, 1, 1), 7, np.uint32))
    # leaf cell (1, 0, 0) holds voxel (3, 0, 0) at child 1; the root holds that leaf at child 1
    assert r[3] == 2 and r[1] == 2
    assert r[0][0].tolist() == [0, 7, 0, 0, 0, 0, 0, 0] and r[0][1].tolist() == [0, 1, 0, 0, 0, 0, 0, 0]
    r2 = host_patch(r[0], r[1], 2, r[2], (3, 0, 0), np.full((1, 1, 1), 7, np.uint32))
    assert r2[3] == 0 and r2[1] == 2
    r3 = host_patch(r2[0], r2[1], 2, r2[2], (3, 0, 0), np.zeros((1, 1, 1), np.uint32))
    assert r3[3] == 0 and r3[1] == 0 and r3[0].shape[0] == 2


# ---- GPU ---------------------------------------------------------------------------------------------------------------

def _torch():
    import torch
    return torch


class Chain:
    """a context and host_patch's mirror, patched side by side; every patch checks the mirror bit for bit.  dense: the
    scene's voxels, kept up to date for check_all (None: not kept)"""

    def __init__(self, ort, ctx, depth, dense=None):
        self.ort, self.ctx, self.depth = ort, ctx, depth
        self.dense = None if dense is None else np.array(dense, np.uint32)
        self.rows = ctx.read_nodes()
        self.root = ctx.root
        self.index = None

    def patch(self, origin, box, what, src=None):
        n_old = self.ctx.node_count
        added = self.ctx.patch_voxels(origin, box if src is None else src)
        rows, root, self.index, n_added = host_patch(self.rows, self.root, self.depth, self.index, origin, box)
        assert added == n_added, f"{what}: n_added {added} != {n_added}"
        assert self.ctx.node_count == n_old + added and self.ctx.root == root, f"{what}: root {self.ctx.root} != {root}"
        assert np.array_equal(self.ctx.read_nodes(n_old + 1, added), rows[n_old:]), f"{what}: appended rows differ"
        self.rows, self.root = rows, root
        if self.dense is not None:
            self.dense = replaced(self.dense, origin, box)
        return added

    def check_all(self, what):
        assert np.array_equal(self.ctx.read_nodes(), self.rows), f"{what}: mirror differs"
        assert np.array_equal(self.ctx.read_voxels((0, 0, 0), (1 << self.depth,) * 3), self.dense), f"{what}: voxels"


@pytest.mark.gpu
@pytest.mark.parametrize("depth", list(range(1, 9)))
def test_gpu_patch_random_scenes(ort, depth):
    """random scenes built by upload_voxels, then chains of patches of every box kind: the mirror equals host_patch's
    bit for bit, n_added and root included, with the index carried from patch to patch"""
    rs = np.random.RandomState(1000 + depth)
    dense = random_grid(rs, depth, 0.3 if depth <= 5 else 0.02)
    ctx = ort.TraceContext(depth)
    ctx.upload_voxels(dense)
    ch = Chain(ort, ctx, depth, dense)
    for r in range(3 if depth <= 6 else 2):
        for kind in BOX_KINDS:
            origin, ext = random_box(rs, depth, kind)
            box = random_box_content(rs, ext, float(rs.choice([0.0, 0.02, 0.5, 1.0])))
            ch.patch(origin, box, f"depth {depth} round {r} {kind} {origin} {ext}")
        ch.check_all(f"depth {depth} round {r}")
    count, distinct = reachable_dag(ch.rows, ch.root, depth)
    assert distinct and count == canonical_dag(ch.dense, depth)[0].shape[0]
    ctx.close()


@pytest.mark.gpu
def test_gpu_patch_512_limit(ort):
    """boxes 512 wide on two axes at depth 10, unaligned, across the middle of the cube, chained, against host_patch;
    a whole depth-9 cube (512^3) replaced by a patch reads back as its source"""
    rs = np.random.RandomState(512)
    depth, dim = 10, 1 << 10
    S = ort.HOctree(20, depth, device=None)
    pts = rs.randint(0, dim, (20000, 3))
    S.set_many(np.concatenate([pts, rs.randint(1, 5, (20000, 1))], 1).astype(np.uint32))
    n8, root, _ = S.flatten()
    ctx = ort.TraceContext(depth)
    ctx.upload_full(n8, root)
    ch = Chain(ort, ctx, depth)
    for origin, shape in (((257, 300, 129), (9, 512, 512)), ((511, 3, 100), (512, 13, 512)), ((0, 512, 512), (512, 512, 5))):
        box = np.zeros(shape, np.uint8)
        box[shape[0] // 4:, : shape[1] // 2, 7:] = 3
        box[::7, ::5, ::3] = rs.randint(0, 9, box[::7, ::5, ::3].shape)
        n_old = ctx.node_count
        added = ctx.patch_voxels(origin, box)
        rows, root2, ch.index, n_added = host_patch(ch.rows, ch.root, depth, ch.index, origin, box)
        assert added == n_added and ctx.root == root2, f"box {origin} {shape}"
        assert np.array_equal(ctx.read_nodes(n_old + 1, added), rows[n_old:])
        ch.rows, ch.root = rows, root2
    ctx.close()
    ctx = ort.TraceContext(9)
    ctx.upload_voxels(random_grid(rs, 9, 0.001))
    box = random_box_content(rs, (512, 512, 512), 0.01)
    ctx.patch_voxels((0, 0, 0), box)
    assert np.array_equal(ctx.read_voxels((0, 0, 0), (512, 512, 512)), box)
    ctx.close()


@pytest.mark.gpu
def test_gpu_patch_dtypes_and_memory_kinds(ort):
    """uint8 / int32 / uint32 sources as numpy, CPU, pinned and CUDA tensors; read_voxels output taken as it is"""
    torch = _torch()
    depth = 6
    rs = np.random.RandomState(66)
    dense = random_grid(rs, depth, 0.2)
    ctx = ort.TraceContext(depth)
    ctx.upload_voxels(dense)
    ch = Chain(ort, ctx, depth, dense)
    tdt = {np.uint8: torch.uint8, np.int32: torch.int32, np.uint32: torch.uint32}
    kinds = {"numpy": lambda a, dt: a.astype(dt),
             "cpu": lambda a, dt: torch.from_numpy(a.astype(np.int64)).to(tdt[dt]),
             "pinned": lambda a, dt: torch.from_numpy(a.astype(np.int64)).to(tdt[dt]).pin_memory(),
             "cuda": lambda a, dt: torch.from_numpy(a.astype(np.int64)).to(tdt[dt]).cuda()}
    for dt in (np.uint8, np.int32, np.uint32):
        for kn, mk in kinds.items():
            origin, ext = random_box(rs, depth, "unaligned")
            box = random_box_content(rs, ext, 0.5, vmax=255 if dt == np.uint8 else 1 << 20)
            ch.patch(origin, box, f"{dt.__name__} {kn}", src=mk(box, dt))
    box = np.full((3, 4, 5), 0xFFFFFFF0, np.uint32)
    ch.patch((7, 8, 9), box, "int32 high bit", src=box.view(np.int32))
    back = ctx.read_voxels((10, 20, 30), (17, 9, 11))
    ch.patch((40, 1, 2), back, "read_voxels numpy")
    dback = torch.empty((11, 9, 17), dtype=torch.uint32, device="cuda")
    ctx.read_voxels((1, 2, 3), (17, 9, 11), out=dback)
    ch.patch((0, 50, 40), dback.cpu().view(torch.int32).numpy().view(np.uint32), "read_voxels cuda", src=dback)
    ch.check_all("dtypes")
    ctx.close()


@pytest.mark.gpu
def test_gpu_patch_erasing_and_never_uploaded(ort):
    """a patch that empties the scene (root 0, rows stay, rays miss), patches after it, and patches into contexts never
    uploaded to"""
    depth = 5
    rs = np.random.RandomState(55)
    dense = np.zeros((32, 32, 32), np.uint32)
    dense[4:20, 6:9, 10:30] = rs.randint(1, 4, (16, 3, 20))
    ctx = ort.TraceContext(depth)
    ctx.upload_voxels(dense)
    ch = Chain(ort, ctx, depth, dense)
    n0 = ctx.node_count
    assert ch.patch((10, 6, 4), np.zeros((16, 3, 20), np.uint8), "erase") == 0
    assert ctx.root == 0 and ctx.node_count == n0
    vox, face, t = ctx.trace_rays(np.array([[1.5, 1.5, 1.5]], np.float32), np.array([[0.3, -0.5, 0.8]], np.float32))[:3]
    assert vox[0] == 0 and np.isinf(t[0])
    assert (ctx.read_voxels((0, 0, 0), (32, 32, 32)) == 0).all()
    ch.patch((1, 2, 3), random_box_content(rs, (7, 8, 9), 0.5), "after empty")
    ch.check_all("after empty")
    ctx.close()
    for d in (1, 3, 8):
        ctx = ort.TraceContext(d)
        ch = Chain(ort, ctx, d, np.zeros((1 << d,) * 3, np.uint32))
        assert ch.patch((0, 0, 0), np.zeros((1, 1, 1), np.uint32), f"never uploaded, zero, depth {d}") == 0
        for k in range(3):
            origin, ext = random_box(rs, d, "unaligned")
            ch.patch(origin, random_box_content(rs, ext, 0.4), f"never uploaded, depth {d}, patch {k}")
        ch.check_all(f"never uploaded, depth {d}")
        ctx.close()


@pytest.mark.gpu
def test_gpu_patch_after_other_routes(ort):
    """the index is rebuilt after every other route that changes the rows: a raw hashed table with a slot serving two
    levels (upload_full), delta syncs, upload_voxels and write_voxels; each time the patch equals host_patch from a
    fresh index"""
    rs = np.random.RandomState(88)
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
    raw = np.array(S.nodes())
    assert S.flatten()[0].shape[0] > S.get_fillcnt()
    ctx = ort.TraceContext(depth)
    ctx.upload_full(raw, S.get_root())
    ch = Chain(ort, ctx, depth, dense_of(raw, S.get_root(), depth))
    for k in range(4):
        origin, ext = random_box(rs, depth, "unaligned")
        ch.patch(origin, random_box_content(rs, ext, 0.3), f"raw table patch {k}")
    ch.check_all("raw table")

    # upload_voxels, then write_voxels, each followed by patches (a fresh index each time)
    n, _ = ctx.upload_voxels(ch.dense)
    ch = Chain(ort, ctx, depth, ch.dense)
    for k in range(3):
        origin, ext = random_box(rs, depth, BOX_KINDS[k])
        ch.patch(origin, random_box_content(rs, ext, 0.3), f"after upload_voxels {k}")
    ctx.write_voxels((3, 4, 5), random_box_content(rs, (6, 7, 8), 0.5))
    ch = Chain(ort, ctx, depth, ctx.read_voxels((0, 0, 0), (32, 32, 32)))
    for k in range(3):
        origin, ext = random_box(rs, depth, BOX_KINDS[k + 1])
        ch.patch(origin, random_box_content(rs, ext, 0.3), f"after write_voxels {k}")
    ch.check_all("after write_voxels")
    ctx.close()

    # a host table synced through deltas, patched in between
    depth = 7
    ctx = ort.TraceContext(depth)
    T = ort.HOctree(18, depth)
    T.attach(ctx)
    ort.harness.build_terrain(T, tunnels=True)
    T.sync()
    for k in range(3):
        lo = rs.randint(0, 100, 3)
        T.fill_box(lo, lo + rs.randint(4, 28, 3), int(rs.randint(0, 4)))
        up, full = T.sync()
        assert not full
        n8, root, _ = T.flatten()
        ch = Chain(ort, ctx, depth, dense_of(n8, root, depth))
        for j in range(2):
            origin, ext = random_box(rs, depth, "unaligned")
            ch.patch(origin, random_box_content(rs, ext, 0.3), f"after delta {k} patch {j}")
        ch.check_all(f"after delta {k}")
        T.attach(ctx)                               # the patches replaced what the table mirrored: a full sync follows
        T.sync()
    ctx.close()


@pytest.fixture(scope="module")
def terrain12_rows(ort):
    S = ort.HOctree(24, 12, device=None)
    ort.harness.build_terrain(S, tunnels=True)
    return S


def reachable_count_gpu(ctx, depth):
    """reachable node count of a context's mirror, walked on the GPU"""
    torch = _torch()
    n = ctx.node_count
    rows = torch.empty((max(n, 1), 8), dtype=torch.int32, device="cuda")
    assert ctx.L.ort_read_nodes(ctx.h, 1, n, C.c_void_p(rows.data_ptr())) == 0
    rows = rows.to(torch.int64)
    cur = torch.tensor([ctx.root] if ctx.root else [], dtype=torch.int64, device="cuda")
    count = 0
    for l in range(1, depth + 1):
        cur = torch.unique(cur)
        count += int(cur.numel())
        if l < depth:
            ch = rows[cur - 1].reshape(-1)
            cur = ch[(ch > 0) & (ch <= n)]
    return count


@pytest.mark.gpu
def test_gpu_patch_terrain12_edit_chain(ort, terrain12_rows):
    """T / Z-style 40^3 fills and erasures at varied surface positions of the depth-12 terrain with tunnels, 120 patches:
    after each, the box and its shell read as the host table's voxels and the reachable node count is flatten()'s n;
    at several points frames over every product variant (beam start on) equal those of the flatten() mirror; at the
    end compact() gives flatten() bit for bit"""
    S = terrain12_rows
    n8, root, _ = S.flatten()
    T = ort.HOctree(24, 12, device=None)
    T.import_dag(n8, root)
    ctx, ref = ort.TraceContext(12), ort.TraceContext(12)
    for c in (ctx, ref):
        c.set_option("beam_after", 0)
    ctx.upload_full(n8, root)
    rs = np.random.RandomState(12)
    heights = {}
    added = []
    for k in range(120):
        x, y = (int(v) for v in rs.randint(0, 4096 - 40, 2))
        if (x, y) not in heights:
            column = ctx.read_voxels((x + 20, y + 20, 0), (1, 1, 4096)).ravel()
            heights[(x, y)] = int(np.flatnonzero(column).max()) if column.any() else 0
        z = int(np.clip(heights[(x, y)] - 20 + rs.randint(-10, 11), 0, 4096 - 40))
        v = 0 if k % 2 == 0 else int(rs.randint(1, 4))
        lo = (x, y, z)
        added.append(ctx.patch_voxels(lo, np.full((40, 40, 40), v, np.uint8)))
        T.fill_box(lo, tuple(a + 40 for a in lo), v)
        want = T.flatten()
        ref.upload_full(want[0], want[1])
        shell_lo = tuple(max(a - 1, 0) for a in lo)
        shell_ext = tuple(min(a + 41, 4096) - b for a, b in zip(lo, shell_lo))
        assert np.array_equal(ctx.read_voxels(shell_lo, shell_ext), ref.read_voxels(shell_lo, shell_ext)), f"patch {k} at {lo}"
        assert reachable_count_gpu(ctx, 12) == want[0].shape[0], f"patch {k}: reachable count"
        if k in (0, 1, 59, 119):
            frames_equal(ort, ctx, ref, f"after patch {k}")
    assert max(added) < 20000
    n, lo = ctx.compact()
    assert_rows((ctx.read_nodes(1, n), ctx.root, lo), T.flatten(), "compact")
    ctx.close()
    ref.close()


@pytest.mark.gpu
def test_gpu_patch_depth16(ort):
    """small boxes near both ends of the depth-16 cube, against host_patch"""
    depth, dim = 16, 1 << 16
    rs = np.random.RandomState(160)
    n = 3000
    pts = np.concatenate([rs.randint(0, 40, (n // 2, 3)), dim - 1 - rs.randint(0, 40, (n // 2, 3))])
    S = ort.HOctree(18, depth, device=None)
    S.set_many(np.concatenate([pts, rs.randint(1, 5, (n, 1))], 1).astype(np.uint32))
    n8, root, _ = S.flatten()
    ctx = ort.TraceContext(depth)
    ctx.upload_full(n8, root)
    ch = Chain(ort, ctx, depth)
    boxes = [((0, 0, 0), (13, 9, 17)), ((dim - 21, dim - 8, dim - 30), (21, 8, 30)), ((dim - 1, dim - 1, dim - 1), (1, 1, 1)),
             ((5, dim - 12, 3), (20, 12, 31)), ((32760, 32761, 32759), (9, 9, 9))]
    for origin, ext in boxes:
        box = random_box_content(rs, ext, 0.5)
        added = ctx.patch_voxels(origin, box)
        rows, root2, ch.index, n_added = host_patch(ch.rows, ch.root, depth, ch.index, origin, box)
        assert added == n_added and ctx.root == root2
        ch.rows, ch.root = rows, root2
        assert np.array_equal(ctx.read_nodes(), rows)
        back = ctx.read_voxels(origin, ext)
        assert np.array_equal(back, box)
    ctx.close()


@pytest.mark.gpu
def test_gpu_patch_replicas_stay_identical(ort, terrain12_rows):
    """two contexts fed the same chain of patches end byte-identical"""
    n8, root, _ = terrain12_rows.flatten()
    a, b = ort.TraceContext(12), ort.TraceContext(12)
    a.upload_full(n8, root)
    b.upload_full(n8, root)
    rs = np.random.RandomState(2)
    for k in range(30):
        lo = tuple(int(v) for v in rs.randint(0, 4096 - 64, 3))
        box = random_box_content(rs, tuple(int(v) for v in rs.randint(1, 64, 3)), float(rs.choice([0.0, 0.3, 1.0])))
        assert a.patch_voxels(lo, box) == b.patch_voxels(lo, box)
    assert a.root == b.root and a.node_count == b.node_count
    assert np.array_equal(a.read_nodes(n8.shape[0] + 1), b.read_nodes(n8.shape[0] + 1))
    a.close()
    b.close()


@pytest.mark.gpu
def test_gpu_patch_with_frames_in_flight(ort, terrain12_rows):
    """an async frame and a defer_sync host frame queued before a patch give the old scene; frames queued after it
    give the new one"""
    torch = _torch()
    n8, root, _ = terrain12_rows.flatten()
    ctx = ort.TraceContext(12)
    ctx.upload_full(n8, root)
    T = ort.HOctree(24, 12, device=None)
    T.import_dag(n8, root)
    lo = (1500, 700, 1000)
    T.fill_box(lo, tuple(a + 40 for a in lo), 0)
    ref = ort.TraceContext(12)
    ref.upload_full(*T.flatten()[:2])
    pos, yaw, pitch = POSES["B"]
    rot, fov = ort.camera_coeffs(yaw, pitch)
    W, H = 1920, 1080
    old = ctx.trace_frame(pos, rot, fov, W, H)
    new = ref.trace_frame(pos, rot, fov, W, H)

    def bufs():
        return (torch.empty(W * H, dtype=torch.int32, device="cuda"), torch.empty(W * H, dtype=torch.uint8, device="cuda"),
                torch.empty(W * H, dtype=torch.float32, device="cuda"))

    def host(b):
        return b[0].cpu().numpy().view(np.uint32), b[1].cpu().numpy(), b[2].cpu().numpy()

    before, after = bufs(), bufs()
    out_old = tuple(np.zeros(W * H, dt) for dt in (np.uint32, np.uint8, np.float32)) + (None,)
    out_new = tuple(np.zeros(W * H, dt) for dt in (np.uint32, np.uint8, np.float32)) + (None,)
    torch.cuda.synchronize()
    ctx.set_option("defer_sync", 1)
    try:
        ctx.trace_frame_async(pos, rot, fov, W, H, 0, H, 1, 1, *before)
        ctx.trace_frame(pos, rot, fov, W, H, out=out_old)
        ctx.patch_voxels(lo, np.zeros((40, 40, 40), np.uint8))
        ctx.trace_frame_async(pos, rot, fov, W, H, 0, H, 1, 1, *after)
        ctx.trace_frame(pos, rot, fov, W, H, out=out_new)
        ctx.sync()
    finally:
        ctx.set_option("defer_sync", 0)
    assert_same_hits(host(before), old, "async frame queued before the patch")
    assert_same_hits(out_old, old, "deferred host frame queued before the patch")
    assert_same_hits(host(after), new, "async frame queued after the patch")
    assert_same_hits(out_new, new, "deferred host frame queued after the patch")
    ctx.close()
    ref.close()


@pytest.mark.gpu
def test_gpu_patch_refusals_leave_everything_unchanged(ort):
    torch = _torch()
    L = ort.lib()
    depth = 12
    S = ort.HOctree(20, 8, device=None)
    ort.harness.build_terrain(S, tunnels=True)
    n8, root, _ = S.flatten()
    ctx = ort.TraceContext(depth)
    ctx.write_voxels((0, 0, 0), dense_of(n8, root, 8))
    ch = Chain(ort, ctx, depth)
    ch.patch((10, 20, 30), random_box_content(np.random.RandomState(1), (9, 8, 7), 0.5), "before")
    pos, yaw, pitch = (1.03, 1.03, 1.06), 0.785, -0.3
    rot, fov = ort.camera_coeffs(yaw, pitch)

    def state():
        return ctx.read_nodes(), ctx.root, ctx.node_count, ctx.trace_frame(pos, rot, fov, 320, 200)

    before = state()
    dim = 1 << depth
    host = np.ones(64, np.uint32)
    dev = torch.ones(65, dtype=torch.int32, device="cuda")
    pv = lambda a: C.c_void_p(a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr())
    n = C.c_size_t(0)
    p = lambda x0, y0, z0, q, eb, nx, ny, nz: L.ort_patch_voxels(ctx.h, x0, y0, z0, q, eb, nx, ny, nz, C.byref(n))
    refused = [
        lambda: p(-1, 0, 0, pv(host), 4, 4, 4, 4),
        lambda: p(0, 0, 0, pv(host), 4, 0, 4, 4),
        lambda: p(dim - 3, 0, 0, pv(host), 4, 4, 1, 1),
        lambda: p(0, 0, dim, pv(host), 4, 1, 1, 1),
        lambda: p(0, 0, 0, pv(host), 4, 1, 1, -2),
        lambda: p(0, 0, 0, pv(host), 4, 513, 1, 1),
        lambda: p(0, 0, 0, pv(host), 4, 1, 513, 1),
        lambda: p(0, 0, 0, pv(host), 2, 4, 4, 4),
        lambda: p(0, 0, 0, None, 4, 4, 4, 4),
        lambda: L.ort_patch_voxels(None, 0, 0, 0, pv(host), 4, 4, 4, 4, C.byref(n)),
        lambda: p(0, 0, 0, C.c_void_p(dev.data_ptr() + 2), 4, 4, 4, 4),
    ]
    if torch.cuda.device_count() > 1:
        other = torch.ones(64, dtype=torch.int32, device="cuda:1")
        refused.append(lambda: p(0, 0, 0, pv(other), 4, 4, 4, 4))
    for k, call in enumerate(refused):
        torch.cuda.synchronize()
        assert call() == 1, f"call {k} not refused"
    with pytest.raises(ort.OrtError):
        ctx.patch_voxels((dim - 1, 0, 0), np.ones((1, 1, 2), np.uint8))
    with pytest.raises(TypeError):
        ctx.patch_voxels((0, 0, 0), np.ones((2, 2, 2), np.int64))
    after = state()
    assert np.array_equal(after[0], before[0]) and after[1:3] == before[1:3]
    assert_same_hits(after[3], before[3], "after refusals")
    ch.patch((100, 50, 20), random_box_content(np.random.RandomState(2), (30, 20, 10), 0.5), "after refusals")
    ctx.close()
    # the och::octree pool layout is not a DAG
    P = ort.Octree(4, 1 << 10)
    P.apply(np.array([[1, 2, 3, 5, 0]], np.int32))
    P.sync()
    rows = P.ctx.read_nodes()
    with pytest.raises(ort.OrtError) as e:
        P.ctx.patch_voxels((0, 0, 0), np.ones((2, 2, 2), np.uint8))
    assert e.value.code == 1
    assert np.array_equal(P.ctx.read_nodes(), rows)


@pytest.mark.gpu
def test_gpu_patch_id_limit(ort):
    """a mirror of kIdMask - 40 rows (unreachable filler, then a small DAG): a patch that would append past the id limit
    is refused with ORT_ERR_CAPACITY and changes nothing; a patch that fits still equals host_patch"""
    torch = _torch()
    need = 2 * ID_MASK * 32 + 6 * GIB
    if cuda_free_bytes() < need:
        pytest.skip(f"needs about {need / GIB:.0f} GiB of free device memory, {cuda_free_bytes() / GIB:.0f} GiB free")
    depth = 6
    rs = np.random.RandomState(29)
    grid = random_grid(rs, depth, 0.05)
    small, sroot, _ = canonical_dag(grid, depth)
    n_fill = ID_MASK - 40 - small.shape[0]
    rows = torch.zeros((ID_MASK - 40, 8), dtype=torch.int32, device="cuda")
    rows[:n_fill, 0] = 1                                # filler: unreachable leaf rows
    # the small DAG behind the filler: its interior ids shifted (leaf words are voxels, kept)
    lv = reachable(small, sroot, depth)
    leaf = np.zeros(small.shape[0] + 1, bool)
    leaf[lv[depth]] = True
    shifted = np.where(leaf[1:, None] | (small == 0), small.astype(np.int64), small.astype(np.int64) + n_fill)
    tail = torch.from_numpy(shifted).to(torch.int32).cuda()
    rows[n_fill:] = tail
    ctx = ort.TraceContext(depth)
    assert L_upload(ort, ctx, rows, sroot + n_fill) == 0
    del rows, tail
    release_cuda()
    n0, r0 = ctx.node_count, ctx.root
    tail_rows = ctx.read_nodes(n_fill + 1)
    dense = ctx.read_voxels((0, 0, 0), (64, 64, 64))
    assert np.array_equal(dense, grid)
    with pytest.raises(ort.OrtError) as e:
        ctx.patch_voxels((0, 0, 0), random_box_content(rs, (64, 64, 64), 0.5))
    assert e.value.code == 5, e.value
    assert ctx.node_count == n0 and ctx.root == r0
    assert np.array_equal(ctx.read_nodes(n_fill + 1, n0 - n_fill), tail_rows)
    assert np.array_equal(ctx.read_voxels((0, 0, 0), (64, 64, 64)), grid)
    # a patch that fits: one voxel of a new value, one new row per level.  host_patch of the small DAG alone, its
    # interior ids (old and new) shifted by the filler, is the expectation
    box = np.full((1, 1, 1), 9, np.uint32)
    added = ctx.patch_voxels((5, 6, 7), box)
    want = host_patch(small, sroot, depth, None, (5, 6, 7), box)
    assert added == want[3] == depth and ctx.node_count == n0 + added and ctx.root == want[1] + n_fill
    new = want[0][small.shape[0]:].astype(np.int64)
    new[1:] = np.where(new[1:] > 0, new[1:] + n_fill, 0)
    assert np.array_equal(ctx.read_nodes(n0 + 1, added), new.astype(np.uint32))
    ctx.close()
    release_cuda()


def L_upload(ort, ctx, rows, root):
    """ort_upload_full of a CUDA tensor of rows"""
    return ctx.L.ort_upload_full(ctx.h, C.c_void_p(rows.data_ptr()), rows.shape[0], root)
