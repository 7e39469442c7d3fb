"""The GPU builder of a dense voxel grid (ort_build_voxels) over its whole documented range: depth 11 and DAGs of up to
kIdMask = 2^29 - 1 compact ids, against references written from the contract alone.

The contract: per level, the distinct node contents, numbered breadth-first by first occurrence, root = id 1.
- canonical_dag() computes that with NumPy and nothing else; the CPU tests hold it to HOctree.flatten().
- morton_grid() fills the first M leaf cells in Morton order with distinct contents.  Its DAG is known in closed form
  (morton_rows()), so grids far too large for any host reference (depth 11, 2^29 - 1 ids) are checked row by row on the
  device.  The CPU tests hold the formula to canonical_dag() and flatten().
- The hash mirror (build_hash_np) equals the device's build_hash, compiled for the host; the adversarial grids (all
  contents on one table slot) are made with it.

The tests marked gpu need a B200.  The one at the id limit needs about 46 GiB of free device memory and 22 GiB of
available host memory, the others at most 18 GiB of device memory; each skips with the reason when that is not free."""
import ctypes as C
import os
import sys
import time

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emu"))

from conftest import PRODUCT_VARIANTS, assert_same_hits
from test_voxel_build import as_source, dense_of, host_flatten

KID_MASK = (1 << 29) - 1                   # the largest compact id (ort_trace.cuh kIdMask)
SCAN_TILE = 1024                           # ort_build.cuh kScanTile
GIB = 1 << 30


# ---- references --------------------------------------------------------------------------------------------------------

def _cells(a, s):
    """(2s, 2s, 2s) [z, y, x] -> (s, s, s, 8): the 8 words of each 2x2x2 cell, child c = x | y << 1 | z << 2"""
    return a.reshape(s, 2, s, 2, s, 2).transpose(0, 2, 4, 1, 3, 5).reshape(s, s, s, 8)


def canonical_dag(grid, depth):
    """(nodes8, root, level_offsets) of a [z, y, x] grid, from the contract alone: pad to 2^depth, deduplicate each level
    bottom-up, then number top-down by the first occurrence among the frontier's 8 n child slots."""
    grid = np.asarray(grid)
    if grid.dtype == np.int32:
        grid = grid.view(np.uint32)
    dim = 1 << depth
    a = np.zeros((dim, dim, dim), np.uint32)
    a[: grid.shape[0], : grid.shape[1], : grid.shape[2]] = grid
    uniq = [None] * (depth + 1)                 # uniq[l]: distinct contents of level l (children as level-(l+1) indices + 1)
    for l in range(depth, 0, -1):
        s = a.shape[0] // 2
        rows = _cells(a, s).reshape(-1, 8)
        ne = rows.any(1)
        uniq[l], inv = np.unique(rows[ne], axis=0, return_inverse=True)
        ids = np.zeros(rows.shape[0], np.uint32)
        ids[ne] = inv.reshape(-1) + 1
        a = ids.reshape(s, s, s)
    if a[0, 0, 0] == 0:
        return np.zeros((0, 8), np.uint32), 0, np.ones(depth + 1, np.uint32)
    frontier, base, out = a.reshape(1), [0, 1], []
    for l in range(1, depth + 1):
        rows = uniq[l][frontier - 1]
        if l == depth:
            out.append(rows)
            break
        flat = rows.reshape(-1)
        nz = np.flatnonzero(flat)
        _, first = np.unique(flat[nz], return_index=True)
        nxt = flat[nz[np.sort(first)]]
        assert len(nxt) == len(uniq[l + 1])     # every distinct content of a level is some node's child
        base.append(base[l] + len(frontier))
        remap = np.zeros(len(nxt) + 1, np.uint32)
        remap[nxt] = base[l + 1] + np.arange(len(nxt))
        out.append(remap[rows])
        frontier = nxt
    nodes8 = np.concatenate(out).astype(np.uint32)
    return nodes8, 1, np.array(base[1:] + [nodes8.shape[0] + 1], np.uint32)


def morton_counts(depth, M):
    """n[l] nodes and first id base[l] of level l = 1 .. depth of morton_grid(depth, M); base[depth + 1] = total + 1"""
    n = [0] + [-(-M // 8 ** (depth - l)) for l in range(1, depth + 1)]
    base = [0, 1]
    for l in range(1, depth + 1):
        base.append(base[l] + n[l])
    return n, base


def morton_total(depth, M):
    return morton_counts(depth, M)[1][depth + 1] - 1


def morton_cell_xyz(i, depth):
    """leaf-cell coordinates (cx, cy, cz) of Morton indices i (numpy or torch int64): bit 3b = x, 3b + 1 = y, 3b + 2 = z"""
    cx, cy, cz = i & 0, i & 0, i & 0
    for b in range(depth - 1):
        cx = cx | (((i >> (3 * b)) & 1) << b)
        cy = cy | (((i >> (3 * b + 1)) & 1) << b)
        cz = cz | (((i >> (3 * b + 2)) & 1) << b)
    return cx, cy, cz


def morton_voxels(i, c):
    """voxel c (0..7) of leaf cell i in morton_grid: byte c of i + 1 for c < 4, else 0"""
    return ((i + 1) >> (8 * c)) & 255 if c < 4 else i & 0


def morton_grid(depth, M, dtype=np.uint8, device=None, chunk=1 << 25):
    """The [z, y, x] grid whose first M leaf cells in Morton order hold voxels 0-3 = the 4 bytes of i + 1: numpy, or a
    torch tensor on `device` (built chunk by chunk)."""
    dim = 1 << depth
    assert 0 <= M <= 8 ** (depth - 1)
    if device is None:
        g = np.zeros(dim ** 3, dtype)
        i = np.arange(M, dtype=np.int64)
        cx, cy, cz = morton_cell_xyz(i, depth)
        for c in range(4):
            g[((2 * cz) * dim + 2 * cy + (c >> 1)) * dim + 2 * cx + (c & 1)] = morton_voxels(i, c)
        return g.reshape(dim, dim, dim)
    import torch
    tdt = {np.uint8: torch.uint8, np.uint32: torch.int32}[dtype]
    g = torch.zeros(dim ** 3, dtype=tdt, device=device)
    for k0 in range(0, M, chunk):
        i = torch.arange(k0, min(M, k0 + chunk), dtype=torch.int64, device=device)
        cx, cy, cz = morton_cell_xyz(i, depth)
        at = ((2 * cz) * dim + 2 * cy) * dim + 2 * cx
        del cx, cy, cz
        for c in range(4):
            g[at + ((c >> 1) * dim + (c & 1))] = morton_voxels(i, c).to(tdt)
        del i, at
    return g.reshape(dim, dim, dim)


def morton_rows(depth, M, level, k0, k1, device=None):
    """Rows of nodes k0 .. k1 - 1 of level `level` (1 = root, depth = leaf rows) of morton_grid(depth, M)'s DAG: int64,
    numpy or a torch tensor on `device`.  Node k of an interior level has children base[l+1] + 8k + c where 8k + c is
    below the next level's count, 0 elsewhere; leaf node k holds leaf cell k's voxels."""
    n, base = morton_counts(depth, M)
    assert 0 <= k0 <= k1 <= n[level]
    if device is None:
        xp, k, c = np, np.arange(k0, k1, dtype=np.int64), np.arange(8, dtype=np.int64)
    else:
        import torch
        xp = torch
        k, c = torch.arange(k0, k1, dtype=torch.int64, device=device), torch.arange(8, dtype=torch.int64, device=device)
    if level == depth:
        return xp.stack([morton_voxels(k, j) for j in range(8)], 1)
    child = 8 * k[:, None] + c[None, :]
    return xp.where(child < n[level + 1], base[level + 1] + child, child & 0)


def morton_dag(depth, M):
    """every row of morton_grid(depth, M)'s DAG (numpy uint32), from morton_rows"""
    n, base = morton_counts(depth, M)
    rows = [morton_rows(depth, M, l, 0, n[l]) for l in range(1, depth + 1)]
    return np.concatenate(rows).astype(np.uint32), 1, np.array(base[1:], np.uint32)


def build_hash_np(w8):
    """NumPy mirror of ort_build.cuh's build_hash over the rows of an (n, 8) uint32 array"""
    w8 = np.asarray(w8, np.uint32).reshape(-1, 8).astype(np.uint64)
    h = np.full(w8.shape[0], 0x9E3779B97F4A7C15, np.uint64)
    for i in range(8):
        h ^= w8[:, i]
        h *= np.uint64(0xFF51AFD7ED558CCD)
        h ^= h >> np.uint64(29)
    return ((h ^ (h >> np.uint64(32))) & np.uint64(0xFFFFFFFF)).astype(np.uint32)


def table_cap(n_nonempty):
    """ort_device.cu's leaf table size for n non-empty leaf cells: pow2_at_least(2 n), at least 64"""
    p = 64
    while p < 2 * n_nonempty:
        p <<= 1
    return p


def scan_scratch_words(n):
    words, m = 0, n
    while m > 1:
        m = -(-m // SCAN_TILE)
        words += m
    return words + 1


def morton_build_bytes(depth, M, cap_nodes):
    """What build_voxels allocates for morton_grid(depth, M) read from device memory into a context whose mirror holds
    cap_nodes rows (ort_build_bytes): per-level ids and tables, counters, frontiers, the top-down scratch, and the new
    mirror (or a temporary copy of the rows when the old one is big enough).  Every non-empty cell of a Morton grid has
    distinct content, so a level's non-empty count is its node count."""
    n, _ = morton_counts(depth, M)
    total = sum(n)
    cells = {l: 8 ** (l - 1) for l in range(1, depth + 1)}
    cap = {l: table_cap(min(M if l == depth else n[l + 1], cells[l])) for l in range(1, depth + 1)}
    b = sum(4 * cells[l] for l in cells) + 16 * (depth + 1) + sum(4 * cap[l] for l in cap)
    b += 32 * min(total + total // 4 + 4096, KID_MASK) if total > cap_nodes else 32 * total
    b += sum(4 * n[l] for l in range(1, depth + 1))
    max_slots = max(8 * n[l] for l in range(1, depth))
    b += 4 * (2 * max_slots + max(cap[l] for l in range(2, depth + 1)) + scan_scratch_words(max_slots))
    return b


def id_limit_M(depth=11):
    """the largest M whose Morton DAG fits the 2^29 - 1 compact ids, and whether some M fills them exactly"""
    lo, hi = 1, 8 ** (depth - 1)
    while lo < hi:
        mid = (lo + hi + 1) // 2
        if morton_total(depth, mid) <= KID_MASK:
            lo = mid
        else:
            hi = mid - 1
    return lo, morton_total(depth, lo) == KID_MASK


# ---- CPU: the references against each other and against flatten() ---------------------------------------------------------

def assert_dag_equal(got, want, what):
    g8, gr, glo = got
    w8, wr, wlo = want
    assert gr == wr, f"{what}: root {gr} != {wr}"
    assert np.array_equal(np.asarray(glo, np.int64), np.asarray(wlo, np.int64)), f"{what}: level offsets {glo} != {wlo}"
    assert g8.shape == w8.shape, f"{what}: {g8.shape[0]} rows, want {w8.shape[0]}"
    bad = np.flatnonzero((np.asarray(g8, np.int64) != np.asarray(w8, np.int64)).any(1))
    assert bad.size == 0, f"{what}: {bad.size} rows differ, first ids {bad[:5] + 1}"


def test_canonical_dag_equals_flatten_random_grids(ort):
    rs = np.random.RandomState(29)
    cases = [  # depth, (nz, ny, nx), density, dtype, largest payload
        (1, (2, 2, 2), 0.5, np.uint8, 2), (1, (1, 1, 1), 1.0, np.uint32, 0xFFFFFFFF), (2, (4, 3, 1), 0.7, np.uint8, 3),
        (3, (8, 8, 8), 0.9, np.uint32, 0xFFFFFFFF), (3, (5, 8, 7), 0.3, np.int32, 3), (4, (16, 16, 16), 0.05, np.uint8, 255),
        (4, (16, 9, 13), 0.95, np.uint8, 2), (5, (32, 32, 32), 0.5, np.uint8, 2), (5, (17, 32, 1), 0.9, np.uint32, 7),
        (6, (64, 64, 64), 0.01, np.uint32, 0xFFFFFFFF), (6, (64, 50, 64), 0.9, np.uint8, 1), (7, (128, 128, 128), 0.002, np.uint8, 200),
        (7, (99, 128, 70), 0.3, np.uint8, 2), (8, (256, 256, 256), 0.0005, np.uint32, 9), (8, (256, 255, 3), 0.5, np.uint8, 3),
    ]
    for k, (depth, shape, dens, dt, vmax) in enumerate(cases):
        vals = rs.randint(1, vmax + 1, size=shape, dtype=np.uint64)
        grid = np.where(rs.random_sample(shape) < dens, vals, 0).astype(dt)
        assert_dag_equal(canonical_dag(grid, depth), host_flatten(ort, grid, depth), f"case {k} depth {depth} {shape}")


@pytest.mark.parametrize("depth,log2cap", [(6, 16), (7, 18), (8, 19)])
def test_canonical_dag_equals_flatten_terrain_with_tunnels(ort, oc, depth, log2cap):
    S = ort.HOctree(log2cap, depth, device=None)
    ort.harness.build_terrain(S, oc.heightmap(depth), oc.grass_bits(depth), tunnels=True)
    want = S.flatten()
    assert_dag_equal(canonical_dag(dense_of(want[0], want[1], depth), depth), want, f"terrain depth {depth}")


def test_canonical_dag_with_content_on_two_levels(ort):
    """A table slot that serves a leaf row and an interior row (the same 8 words) is two rows of the compact DAG in both."""
    depth = 5
    rs = np.random.RandomState(3)
    grid = np.zeros((32, 32, 32), np.uint32)
    pts = rs.randint(0, 32, (300, 3))
    grid[pts[:, 2], pts[:, 1], pts[:, 0]] = rs.randint(1, 3, 300)
    S = ort.HOctree(16, depth, device=None)
    from test_voxel_build import xyzv_of
    S.set_many(xyzv_of(grid))
    # a leaf cell (in the root's octant 7) whose 8 voxels are the 8 table slots of an interior node the edit leaves
    # alone (the root's child in octant 0): one slot then serves both levels
    child = int(S.nodes()[S.get_root() - 1][0])          # (table rows: id - 1)
    assert child
    cell = np.array(S.nodes()[child - 1], np.uint32)
    for c in range(8):
        S.set(30 + (c & 1), 30 + ((c >> 1) & 1), 30 + (c >> 2), int(cell[c]))
    nodes8, root, lo = S.flatten()
    assert nodes8.shape[0] > S.get_fillcnt()          # the shared slot really is one table entry and two rows
    assert_dag_equal(canonical_dag(dense_of(nodes8, root, depth), depth), (nodes8, root, lo), "content on two levels")


def test_morton_rows_equal_canonical_and_flatten(ort):
    """morton_rows is the closed form of morton_grid's DAG: every M at depths 3 and 4, the 8^j boundaries at 5 and 6."""
    cases = [(3, M) for M in range(0, 65)] + [(4, M) for M in range(0, 513)]
    for depth in (5, 6):
        cases += [(depth, M) for M in sorted({1, 2, 7, 8, 9, 63, 64, 65, 511, 512, 513, 4095, 4096, 4097, 8 ** (depth - 1) - 1, 8 ** (depth - 1)})
                  if M <= 8 ** (depth - 1)]
    for depth, M in cases:
        grid = morton_grid(depth, M)
        want = canonical_dag(grid, depth)
        if M == 0:
            assert want[0].shape[0] == 0
            continue
        assert_dag_equal(morton_dag(depth, M), want, f"depth {depth} M {M}")
        if depth >= 5 or M % 37 == 0:
            assert_dag_equal(want, host_flatten(ort, grid, depth), f"depth {depth} M {M} flatten")
        assert morton_total(depth, M) == want[0].shape[0]


def test_morton_grid_on_torch_equals_numpy():
    torch = pytest.importorskip("torch")
    for depth, M in ((4, 300), (5, 4096), (6, 20001)):
        for dt in (np.uint8, np.uint32):
            t = morton_grid(depth, M, dt, device="cpu", chunk=1000)
            assert np.array_equal(t.numpy().view(dt), morton_grid(depth, M, dt)), f"depth {depth} M {M} {np.dtype(dt).name}"
        for level in range(1, depth + 1):
            n = morton_counts(depth, M)[0][level]
            assert np.array_equal(morton_rows(depth, M, level, 0, n, device="cpu").numpy(), morton_rows(depth, M, level, 0, n))


def test_hash_mirror_equals_build_hash():
    import emu_build
    rs = np.random.RandomState(11)
    w = rs.randint(0, 1 << 32, (100000, 8), dtype=np.uint64).astype(np.uint32)
    w[:1000] = rs.choice(np.array([0, 1, 2, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFE, 0xFFFFFFFF], np.uint32), (1000, 8))
    w[1000:2000] = rs.randint(0, 256, (1000, 8))
    assert np.array_equal(build_hash_np(w), emu_build.build_hash(w))


def test_id_limit_constants():
    M, exact = id_limit_M(11)
    assert morton_total(11, M) <= KID_MASK < morton_total(11, M + 1)
    assert morton_total(11, M) >= KID_MASK - 7             # one more leaf adds at most 11 nodes
    # some M fills the ids exactly, so the test at the id limit builds a DAG whose highest id is 2^29 - 1 itself
    assert exact and M == 469762046 and morton_total(11, M) == KID_MASK


# ---- GPU helpers ---------------------------------------------------------------------------------------------------------

def probe_chain_contents(n_want, n_copies, dtype, seed):
    """n_want distinct leaf contents whose build_hash all falls on slot cap - 1 of the leaf table that n_want * n_copies
    non-empty leaf cells get"""
    cap = table_cap(n_want * n_copies)
    rs = np.random.RandomState(seed)
    top = 256 if dtype == np.uint8 else 1 << 32
    found = []
    while sum(len(f) for f in found) < n_want:
        w = rs.randint(0, top, (1 << 21, 8), dtype=np.uint64).astype(np.uint32)
        w = w[w.any(1)]
        found.append(w[(build_hash_np(w) & (cap - 1)) == cap - 1])
    w = np.unique(np.concatenate(found), axis=0)[:n_want]
    assert w.shape[0] == n_want
    return w[rs.permutation(n_want)], cap


def grid_of_leaf_contents(depth, cells, contents):
    """a grid whose leaf cells `cells` (flat indices into the (2^(depth-1))^3 leaf cell grid, [z, y, x]) hold `contents`"""
    s = 1 << (depth - 1)
    rows = np.zeros((s ** 3, 8), contents.dtype)
    rows[cells] = contents
    return rows.reshape(s, s, s, 2, 2, 2).transpose(0, 3, 1, 4, 2, 5).reshape(2 * s, 2 * s, 2 * s).copy()


def assert_builds(ctx, grid, want, what):
    nodes8, root, lo = want
    n, blo = ctx.upload_voxels(grid)
    assert n == nodes8.shape[0] and ctx.node_count == n and ctx.root == root, f"{what}: {n} nodes, root {ctx.root}; want {nodes8.shape[0]}, {root}"
    assert np.array_equal(blo, lo), f"{what}: level offsets {blo} != {lo}"
    if n:
        got = ctx.read_nodes(1, n)
        bad = np.flatnonzero((got != nodes8).any(1))
        assert bad.size == 0, f"{what}: {bad.size} rows differ, first ids {bad[:5] + 1}"


def read_rows_cuda(ctx, first, n):
    """rows first .. first + n - 1 of the mirror into a CUDA tensor (ort_read_nodes copies to any pointer)"""
    import torch
    out = torch.empty((n, 8), dtype=torch.int32, device=f"cuda:{ctx.device}")
    torch.cuda.current_stream(ctx.device).synchronize()
    ctx._ck(ctx.L.ort_read_nodes(ctx.h, first, n, C.c_void_p(out.data_ptr())))
    return out


def assert_morton_rows_on_device(ctx, depth, M, chunk=1 << 23):
    """every row of the mirror against morton_rows, chunk by chunk on the device"""
    import torch
    n, base = morton_counts(depth, M)
    for l in range(1, depth + 1):
        for k0 in range(0, n[l], chunk):
            k1 = min(n[l], k0 + chunk)
            got = read_rows_cuda(ctx, base[l] + k0, k1 - k0).to(torch.int64) & 0xFFFFFFFF
            bad = (got != morton_rows(depth, M, l, k0, k1, device=got.device)).any(1)
            if bool(bad.any()):
                first = int(torch.nonzero(bad)[0, 0])
                raise AssertionError(f"depth {depth} M {M}: level {l}: {int(bad.sum())} rows differ in ids {base[l] + k0} .. {base[l] + k1 - 1}, "
                                     f"first id {base[l] + k0 + first}: {got[first].tolist()}")
            del got, bad


def cuda_free_bytes():
    import torch
    return torch.cuda.mem_get_info()[0]


def host_available_bytes():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


def release_cuda():
    import gc

    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


# ---- GPU: adversarial content at depths 6-9 ----------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("dtype,kind", [(np.uint32, "host"), (np.uint8, "pinned"), (np.uint32, "cuda"), (np.uint8, "cuda")])
def test_probe_chains_that_wrap(ort, dtype, kind):
    """1500 distinct leaf contents, twice each, that all hash to the last slot of the 8192-entry leaf table: one probe
    chain of 1500 entries that wraps from slot cap - 1 to slot 0, walked by 3000 racing threads."""
    depth = 7
    contents, cap = probe_chain_contents(1500, 2, dtype, seed=7 if dtype == np.uint8 else 8)
    assert (build_hash_np(contents) & (cap - 1) == cap - 1).all() and cap == 8192
    contents = contents.astype(dtype)
    rs = np.random.RandomState(70)
    cells = rs.choice(8 ** (depth - 1), 3000, replace=False)
    grid = grid_of_leaf_contents(depth, cells, np.concatenate([contents, contents[rs.permutation(1500)]]))
    ctx = ort.TraceContext(depth)
    assert_builds(ctx, as_source(grid, kind), canonical_dag(grid, depth), f"probe chain {np.dtype(dtype).name} {kind}")
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["host", "cuda"])
def test_dedup_under_contention(ort, kind):
    """Five contents, each in ~350 000 leaf cells spread over a depth-8 grid (one of them all 0xFFFFFFFF, the table's
    free marker), then every cell the same 0xFFFFFFFF content: hundreds of thousands of threads insert the same
    content at once."""
    depth = 8
    rs = np.random.RandomState(81)
    palette = np.array([[0] * 8, [0xFFFFFFFF] * 8, [1, 0, 0, 0, 0, 0, 0, 0], [0, 0, 0, 0, 0, 0, 0, 0xFFFFFFFF],
                        [7, 7, 7, 7, 7, 7, 7, 7], [0xFFFFFFFF, 1, 0xFFFFFFFF, 2, 0xFFFFFFFF, 3, 0xFFFFFFFF, 4]], np.uint32)
    pick = rs.randint(0, 6, 8 ** (depth - 1))
    assert (np.bincount(pick, minlength=6) > 100000).all()
    grid = grid_of_leaf_contents(depth, np.arange(8 ** (depth - 1)), palette[pick])
    ctx = ort.TraceContext(depth)
    assert_builds(ctx, as_source(grid, kind), canonical_dag(grid, depth), f"five contents {kind}")
    full = np.full((256, 256, 256), 0xFFFFFFFF, np.uint32)
    want = canonical_dag(full, depth)
    assert want[0].shape[0] == depth
    assert_builds(ctx, as_source(full, kind), want, f"all 0xFFFFFFFF {kind}")
    ctx.close()


@pytest.mark.gpu
def test_all_distinct_leaves(ort):
    """Every leaf cell distinct (no deduplication: the leaf table at its largest load, 1/2), from random uint32 content
    and from the full Morton grid, whose interior levels are all distinct too."""
    depth = 7
    rs = np.random.RandomState(77)
    n = 8 ** (depth - 1)
    rows = rs.randint(1, 1 << 32, (n, 8), dtype=np.uint64).astype(np.uint32)
    assert np.unique(rows, axis=0).shape[0] == n and table_cap(n) == 2 * n
    grid = grid_of_leaf_contents(depth, np.arange(n), rows)
    ctx = ort.TraceContext(depth)
    assert_builds(ctx, as_source(grid, "cuda"), canonical_dag(grid, depth), "random distinct leaves")
    grid = morton_grid(depth, n)
    want = canonical_dag(grid, depth)
    assert_dag_equal(want, morton_dag(depth, n), "full Morton grid")
    assert_builds(ctx, as_source(grid, "pinned"), want, "full Morton grid")
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("depth,M,slots", [(8, 1013, 1016), (8, 1021, 1024), (8, 1027, 1032),
                                           (9, (1 << 20) - 3, 1 << 20), (9, (1 << 20) + 5, (1 << 20) + 8)])
def test_scan_tile_boundaries(ort, depth, M, slots):
    """The leaf level's parents give the widest top-down pass: 8 ceil(M / 8) child slots = one scan tile less a row,
    exactly one, one and a row; 2^20 (1024 tiles: two scan levels) and 2^20 + 8 (three scan levels)."""
    n, _ = morton_counts(depth, M)
    assert 8 * n[depth - 1] == slots
    grid = morton_grid(depth, M)
    want = morton_dag(depth, M)
    assert_dag_equal(canonical_dag(grid, depth), want, f"depth {depth} M {M} reference")
    ctx = ort.TraceContext(depth)
    assert_builds(ctx, as_source(grid, "cuda"), want, f"depth {depth} M {M}")
    ctx.close()


@pytest.mark.gpu
def test_extents_that_are_not_powers_of_two(ort):
    """Clipped grids from every memory kind, 1- and 4-byte elements: Morton content and random content."""
    rs = np.random.RandomState(90)
    ctx = ort.TraceContext(9)
    cases = [(morton_grid(9, 300000)[:301, :512, :257], "host"), (morton_grid(9, 300000, np.uint32)[:512, :77, :300], "pinned"),
             (morton_grid(9, 4 ** 9)[:129, :1, :511], "cuda")]
    for shape, dt in (((333, 170, 1), np.uint32), ((1, 400, 300), np.uint8), ((511, 3, 257), np.uint8)):
        cases.append((np.where(rs.random_sample(shape) < 0.4, rs.randint(1, 4, shape), 0).astype(dt), ("host", "pinned", "cuda")[len(cases) % 3]))
    for k, (grid, kind) in enumerate(cases):
        grid = np.ascontiguousarray(grid)
        assert_builds(ctx, as_source(grid, kind), canonical_dag(grid, 9), f"case {k} {grid.shape} {grid.dtype} {kind}")
    ctx.close()


# ---- GPU: depth 11 -------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_depth11_terrain_with_tunnels(ort):
    """The depth-11 terrain with tunnels, read back into an 8 GiB uint8 grid with read_voxels and built again: the
    same rows and level offsets as flatten()."""
    import torch
    need = 8 * GIB + 14 * GIB
    if cuda_free_bytes() < need:
        pytest.skip(f"needs {need / GIB:.0f} GiB of free device memory, {cuda_free_bytes() / GIB:.1f} GiB free")
    depth, dim, slab = 11, 2048, 64
    T = ort.HOctree(24, depth, node_capacity=1 << 21)
    ort.harness.build_terrain(T, tunnels=True)
    nodes8, root, lo = T.flatten()
    grid = torch.empty((dim, dim, dim), dtype=torch.uint8, device="cuda")
    buf = torch.empty((slab, dim, dim), dtype=torch.int32, device="cuda")
    for z0 in range(0, dim, slab):
        T.read_voxels((0, 0, z0), (dim, dim, slab), out=buf)
        assert int(buf.max()) < 256
        grid[z0:z0 + slab] = buf.to(torch.uint8)
    del buf
    ctx = ort.TraceContext(depth)
    t0 = time.perf_counter()
    assert_builds(ctx, grid, (nodes8, root, lo), "depth-11 terrain")
    print(f"depth-11 terrain: {nodes8.shape[0]} nodes, build {time.perf_counter() - t0:.2f} s with the read-back, build_bytes {ctx.build_bytes / GIB:.2f} GiB")
    ctx.close()
    del grid, T
    release_cuda()


# ---- GPU: the id limit ---------------------------------------------------------------------------------------------------

LEAN_MAX_NODES = 0x16000000               # ort_device.cu lean_capable: LeanWalker and the beam start take mirrors below it


@pytest.mark.gpu
@pytest.mark.parametrize("n_rows", [LEAN_MAX_NODES - 1, KID_MASK])
def test_interior_ids_up_to_2pow29_minus_1(ort, golden, n_rows):
    """The builder numbers the leaf level last, so at depth 11 its interior ids stay below 2^28, and only a walker's
    parent stack holds interior ids.  Here the golden depth-8 DAG is moved to the top of a mirror of n_rows rows (the
    rows below are empty and never referenced): every interior id has bit 28 set, the root is the highest interior id.
    n_rows = LEAN_MAX_NODES - 1 is the largest mirror LeanWalker and the beam start take; at 2^29 - 1 the frames run on
    FastWalker without the beam start.  Frames of every product variant, with the beam option on and off, and the
    golden rays trace to the reference's outputs; voxel queries read the golden grid."""
    import torch
    need = 32 * n_rows + 2 * GIB
    if cuda_free_bytes() < need:
        pytest.skip(f"needs {need / GIB:.0f} GiB of free device memory, {cuda_free_bytes() / GIB:.1f} GiB free")
    g = golden("d8_tunnels")
    depth, root = int(g["depth"]), int(g["root"])
    nodes8 = g["nodes8"].astype(np.uint32)
    N = nodes8.shape[0]
    interior = np.zeros(N + 1, bool)
    lvl = np.array([root])
    for _ in range(depth - 1):
        interior[lvl] = True
        ch = nodes8[lvl - 1].reshape(-1)
        lvl = np.unique(ch[ch != 0])
    off = n_rows - N
    rows = nodes8.copy()
    rows[interior[1:]] = np.where(rows[interior[1:]] != 0, rows[interior[1:]] + off, 0)
    big = np.zeros((n_rows, 8), np.uint32)                # (untouched pages: no host memory behind the empty rows)
    big[off:] = rows
    assert off + root >= 1 << 28 and (rows[interior[1:]] >= 1 << 28).sum() > 0
    ctx = ort.TraceContext(depth)
    ctx.upload_full(big, off + root)
    del big
    assert ctx.node_count == n_rows and ctx.root == off + root
    W, H = int(g["W"]), int(g["H"])
    ctx.set_option("beam_after", 0)
    for variant in PRODUCT_VARIANTS:
        ctx.set_option("variant", variant)
        for beam in (1, 0):
            ctx.set_option("beam", beam)
            for p in "ABC":
                got = ctx.trace_frame(g[f"pose{p}_pos"], g[f"pose{p}_rot"], float(g[f"pose{p}_fov"]), W, H)
                assert_same_hits(got, (g[f"pose{p}_vox"], g[f"pose{p}_face"], g[f"pose{p}_t"]), f"pose {p} variant {variant} beam {beam}")
    # a 4K frame with the beam option on (the grid of this DAG built and used where the lean tier takes the mirror)
    # against the same frame without it
    ctx.set_option("variant", PRODUCT_VARIANTS[-1])
    ctx.set_option("beam", 1)
    pos, rot, fov = g["poseB_pos"], g["poseB_rot"], float(g["poseB_fov"])
    lean = n_rows < LEAN_MAX_NODES
    assert (ctx.beam_level(pos, rot, fov, 3840, 2160) > 0) == lean
    builds = ctx.beam_builds
    with_beam = ctx.trace_frame(pos, rot, fov, 3840, 2160)
    assert (ctx.beam_builds > builds) == lean and (with_beam[0] != 0).sum() > 100000
    ctx.set_option("beam", 0)
    assert_same_hits(ctx.trace_frame(pos, rot, fov, 3840, 2160), with_beam, "4K frame, beam 0 vs beam 1")
    for k in ("rand", "edge"):
        assert_same_hits(ctx.trace_rays(g[f"{k}_o"], g[f"{k}_d"]), (g[f"{k}_vox"], g[f"{k}_face"], g[f"{k}_t"]), f"{k} rays")
    dense = dense_of(nodes8, root, depth)
    xyz = np.random.RandomState(12).randint(0, 1 << depth, (100000, 3))
    assert np.array_equal(ctx.voxels_at(xyz), dense[xyz[:, 2], xyz[:, 1], xyz[:, 0]])
    assert np.array_equal(ctx.read_voxels((0, 0, 0), (256, 256, 256)), dense)
    ctx.close()
    release_cuda()


def tail_rays(depth, M, n, seed):
    """Rays from the empty voxel layer just above the last n filled leaf cells, straight down (but for a tilt of 1e-4)
    onto a non-zero voxel of that cell: each hits the cell, so the rays reach the highest leaf ids, up to the last.
    Returns (origins, directions, the voxel each ray hits)."""
    dim = 1 << depth
    rs = np.random.RandomState(seed)
    i = np.arange(M - n, M, dtype=np.int64)
    vals = np.stack([morton_voxels(i, c) for c in range(4)], 1)
    c = np.array([rs.choice(np.flatnonzero(v)) for v in vals])
    cx, cy, cz = morton_cell_xyz(i, depth)
    p = np.stack([2 * cx + (c & 1) + 0.5, 2 * cy + (c >> 1) + 0.5, 2 * cz + 1.25 + 0.5 * rs.random_sample(n)], 1)
    o = (1.0 + p / dim).astype(np.float32)
    d = np.stack([rs.uniform(-1e-4, 1e-4, n), rs.uniform(-1e-4, 1e-4, n), -np.ones(n)], 1).astype(np.float32)
    return o, d, vals[np.arange(n), c].astype(np.uint32)


@pytest.mark.gpu
def test_id_limit_2pow29_minus_1(ort, oc):
    """morton_grid(11, M*), M* the largest M whose DAG fits the 2^29 - 1 compact ids: every row, level offset, voxel
    query, box read-back and traced ray (every product frame variant, beam option on and off) is right up to the
    highest id.  One more leaf cell is refused with ORT_ERR_CAPACITY and leaves the mirror as it was."""
    import torch
    from test_oracle import _builtin_table
    depth = 11
    dim = 1 << depth
    M, exact = id_limit_M(depth)
    total = morton_total(depth, M)
    n_lvl, base = morton_counts(depth, M)
    est = morton_build_bytes(depth, M, 1 << 16)
    need_dev, need_host = 8 * GIB + est + 2 * GIB, 32 * (total + 1) + 6 * GIB
    if cuda_free_bytes() < need_dev:
        pytest.skip(f"needs {need_dev / GIB:.1f} GiB of free device memory, {cuda_free_bytes() / GIB:.1f} GiB free")
    if host_available_bytes() < need_host:
        pytest.skip(f"needs {need_host / GIB:.1f} GiB of available host memory for the oracle's copy of the rows, {host_available_bytes() / GIB:.1f} GiB available")

    grid = morton_grid(depth, M, device="cuda")
    ctx = ort.TraceContext(depth)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n, lo = ctx.upload_voxels(grid)
    dt = time.perf_counter() - t0
    print(f"id limit: M* = {M}, {n} nodes (highest id {n}; 2^29 - 1 = {KID_MASK}; exactly reachable: {exact}), "
          f"build {dt:.2f} s, build_bytes {ctx.build_bytes / GIB:.2f} GiB (estimate {est / GIB:.2f} GiB), "
          f"device free after {cuda_free_bytes() / GIB:.1f} GiB")
    assert n == total and ctx.node_count == total and ctx.root == 1
    assert n >= KID_MASK - 7 and (n == KID_MASK or not exact)     # (M* fills them exactly: test_id_limit_constants)
    assert list(lo) == base[1:], f"level offsets {list(lo)} != {base[1:]}"
    assert ctx.build_bytes == est, f"build_bytes {ctx.build_bytes} != {est}"
    assert_morton_rows_on_device(ctx, depth, M)

    # voxel queries at the first and last filled cells, past them, and spread over the cube
    rs = np.random.RandomState(29)
    cells = np.concatenate([np.arange(0, 64), np.arange(M - 64, M + 64), rs.randint(0, 8 ** (depth - 1), 4096)]).astype(np.int64)
    cx, cy, cz = morton_cell_xyz(cells, depth)
    xyz, want = [], []
    for c in range(8):
        xyz.append(np.stack([2 * cx + (c & 1), 2 * cy + ((c >> 1) & 1), 2 * cz + (c >> 2)], 1))
        want.append(np.where(cells < M, morton_voxels(cells, c), 0))
    xyz, want = np.concatenate(xyz), np.concatenate(want).astype(np.uint32)
    assert np.array_equal(ctx.voxels_at(xyz), want)
    got = ctx.voxels_at(torch.from_numpy(xyz.astype(np.int32)).cuda())
    assert np.array_equal(got.cpu().numpy().view(np.uint32), want)
    # a box around the last filled cell, against the grid itself
    tx, ty, tz = (int(v[0]) for v in morton_cell_xyz(np.array([M - 1], np.int64), depth))
    org = [min(max(2 * v - 40, 0), dim - 96) for v in (tx, ty, tz)]
    box = ctx.read_voxels(org, (96, 96, 96), out=torch.empty((96, 96, 96), dtype=torch.int32, device="cuda"))
    ref = grid[org[2]:org[2] + 96, org[1]:org[1] + 96, org[0]:org[0] + 96].to(torch.int32)
    assert torch.equal(box, ref) and int((ref != 0).sum()) > 1000 and int((ref == 0).sum()) > 1000

    # tracing: explicit rays and frames from above the tail, against the oracle on a host copy of the rows
    tab = _builtin_table()
    nodes8 = ctx.read_nodes(1, n)
    o, d, want_vox = tail_rays(depth, M, 4096, seed=5)
    want_rays = oc.trace_rays(nodes8, 1, depth, o, d, rcp_tab=tab, nthreads=8)
    assert np.array_equal(want_rays[0], want_vox)                   # the oracle too sees the analytic voxels
    assert_same_hits(ctx.trace_rays(o, d), want_rays, "rays onto the last leaf cells")
    rot, fov = oc.camera_coeffs(np.pi + 0.3, 0.25)                  # looking down (-z), slightly tilted
    pos = ((np.array([tx, ty, tz], np.float64) * 2 + [1.0, 1.0, 5.5]) / dim + 1.0).astype(np.float32)
    W, H = 320, 180
    want_frame = oc.trace_rays(nodes8, 1, depth, pos, oc.gen_rays(rot, fov, W, H), rcp_tab=tab, nthreads=8)
    assert (want_frame[0] != 0).mean() > 0.3
    del nodes8
    ctx.set_option("beam_after", 0)
    for variant in PRODUCT_VARIANTS:
        ctx.set_option("variant", variant)
        for beam in (1, 0):
            ctx.set_option("beam", beam)
            assert_same_hits(ctx.trace_frame(pos, rot, fov, W, H), want_frame, f"frame variant {variant} beam {beam}")
    ctx.set_option("variant", PRODUCT_VARIANTS[-1])
    # a 4K frame from the centre, looking down into the filled part, with the beam option on and off.  A mirror this
    # large is past the lean tier (LEAN_MAX_NODES): the frames run on FastWalker and no beam grid is built
    ctx.set_option("beam", 1)
    rot4, fov4 = oc.camera_coeffs(np.pi + 0.7, -0.6)
    pos4 = np.full(3, 1.5, np.float32)
    assert n > LEAN_MAX_NODES and ctx.beam_level(pos4, rot4, fov4, 3840, 2160) == 0
    builds = ctx.beam_builds
    with_beam = ctx.trace_frame(pos4, rot4, fov4, 3840, 2160)
    assert ctx.beam_builds == builds and (with_beam[0] != 0).sum() > 100000
    ctx.set_option("beam", 0)
    assert_same_hits(ctx.trace_frame(pos4, rot4, fov4, 3840, 2160), with_beam, "4K frame, beam 0 vs beam 1")
    ctx.set_option("beam", 1)

    # one more leaf cell: refused, and the mirror stays as it was
    i = torch.tensor([M], dtype=torch.int64, device="cuda")
    cx, cy, cz = morton_cell_xyz(i, depth)
    for c in range(4):
        grid[2 * cz, 2 * cy + (c >> 1), 2 * cx + (c & 1)] = morton_voxels(i, c).to(torch.uint8)
    assert morton_total(depth, M + 1) > KID_MASK
    torch.cuda.synchronize()
    before = ctx.trace_frame(pos, rot, fov, W, H)
    nn = C.c_size_t(0)
    rc = ctx.L.ort_build_voxels(ctx.h, C.c_void_p(grid.data_ptr()), 1, dim, dim, dim, C.byref(nn), None)
    assert rc == 5, f"rc {rc}"
    assert ctx.node_count == total and ctx.root == 1
    assert_same_hits(ctx.trace_frame(pos, rot, fov, W, H), before, "after the refused build")
    assert_same_hits(before, want_frame, "before the refused build")
    ctx.close()
    del grid
    release_cuda()
