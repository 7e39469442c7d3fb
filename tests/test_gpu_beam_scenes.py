"""Beam start of camera frames on the GPU (csrc/ort_beam.cuh, csrc/ort_device.cu) against the oracle on the scenes where a
wrong bound would show: random DAGs seen from random cameras, needles / a one-voxel sheet / a rod at depths 12 and 16,
voxels on the cube's faces, edges and corners seen by grazing cameras, foreign reciprocal tables, every frame entry
point, batched launches that mix grid levels or split into several launches, and DAGs built, written and patched on
the device.

Every frame is held to the oracle run with the reciprocal table the context uses, bit for bit on every ray traced.  Two
more checks tie the device to the host emulation (tests/host_emu), whose tile starts tests/test_beam.py and
tests/test_beam_refine.py hold to the bound on the CPU:
  - ctx.beam_level equals the emulation's level for the same camera and table (the host-side plumbing);
  - with option count_beam = 2 the per-ray PUSH counts of the device equal the emulation's on the same rows: equal rounds
    per ray means the device started every tile where the emulation did.
Each test asserts its own coverage (grid levels, refining frames, certified tiles).

The scenes the emulation had not seen before (the depth-16 thin scene, the face and corner voxels, the 2^16-entry and
the 8-bit tables) also run through the emulation alone, without the gpu mark."""
import os
import sys

import numpy as np
import pytest

from conftest import assert_same_hits

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emu"))

NCPU = max(1, min(32, os.cpu_count() or 1))
EXIT, INSIDE = 0xFFFEBF00, 0xFF07193F


@pytest.fixture(scope="module")
def emu():
    import emu as m
    m.lib()
    return m


@pytest.fixture(scope="module")
def refine():
    import emu_refine as m
    m.lib()
    return m


# ---- reciprocal tables ---------------------------------------------------------------------------------------------

def table_24bit(log2n=11):
    """Correctly rounded reciprocals of the bin centres (24 significant bits)."""
    n = 1 << log2n
    return (np.float32(1.0) / (np.float32(1.0) + (np.arange(n, dtype=np.float32) + np.float32(0.5)) / np.float32(n))).astype(np.float32).view(np.uint32)


def table_rounded_up(log2n, bits):
    """Reciprocals of the bin centres rounded up to `bits` significant bits: every entry stays in (0.5, 1]."""
    n = 1 << log2n
    x = 1.0 / (1.0 + (np.arange(n) + 0.5) / n)
    s = 2.0 ** (bits - 1 - np.floor(np.log2(x)))
    return (np.ceil(x * s) / s).astype(np.float32).view(np.uint32)


def foreign_tables():
    return {"24-bit 2^11": table_24bit(11), "12-bit 2^16": table_rounded_up(16, 12), "8-bit 2^11": table_rounded_up(11, 8)}


# ---- one frame: oracle, emulation, device ----------------------------------------------------------------------------

def on_grid(pos, depth):
    return any(float(np.float32(c)) * (1 << depth) == int(float(np.float32(c)) * (1 << depth)) for c in pos)


class Scene:
    """A DAG (compact layout) with its emulation grids, built on first use."""

    def __init__(self, emu, nodes8, root, depth, name):
        self.emu, self.nodes8, self.root, self.depth, self.name = emu, nodes8, root, depth, name
        self.grids = {}

    def grid(self, k):
        if k not in self.grids:
            self.grids[k] = self.emu.beam_grid(self.nodes8, self.root, k)
        return self.grids[k]


class Coverage:
    def __init__(self):
        self.frames = self.refining = self.certified = self.zero_round_misses = 0
        self.levels = set()

    def add(self, r):
        self.frames += 1
        self.levels.add(r["k"])
        self.refining += r["fine_t"] > 0
        self.certified += r["stats"]["beam_tile_misses"]
        self.zero_round_misses += r["zero_round_misses"]


def frame_rows(y0, rows, tr, ts):
    return [y0 + (r // tr) * tr * ts + r % tr for r in range(rows)] if ts > 1 else list(range(y0, y0 + rows))


def frame_dirs(oc, rot, fov, W, H, y0, rows, tr=1, ts=1):
    if ts == 1:
        return oc.gen_rays(rot, fov, W, H, y0, y0 + rows)
    return np.concatenate([oc.gen_rays(rot, fov, W, H, y, y + 1) for y in frame_rows(y0, rows, tr, ts)])


def check_frame(emu, refine, oc, sc, pos, rot, fov, W, H, y0=0, rows=None, tr=1, ts=1, tab=None, ctx=None, what="", lean_only=True):
    """The rows (y0, rows, tr, ts) of a W x H frame: the oracle, the emulation of the library's beam start with the level
    and refinement the library picks for this camera and table (equal to the oracle; the tile starts bound the hit times,
    the guard never fires, no tile is certified wrongly) and, with ctx, the device: ctx.beam_level is the emulation's,
    the frame equals the oracle and its per-ray PUSH counts under count_beam = 2 are the emulation's.
    lean_only: every ray is a lean-tier ray, so every hit time bounds its tile's start."""
    tab = emu.default_rcp_table() if tab is None else tab
    rows = H - y0 if rows is None else rows
    pos = np.asarray(pos, np.float32)
    what = f"{sc.name}: {what} camera {pos.tolist()}, {W}x{H} rows {y0}+{rows} tiles {tr}/{ts}"
    k = emu.beam_level(pos, rot, fov, W, H, sc.depth, rcp_tab=tab)
    assert k > 0, f"{what}: the camera should have a beam level"
    fine_t = refine.beam_fine_t(pos, rot, fov, W, H, sc.depth, rcp_tab=tab)
    want = oc.trace_rays(sc.nodes8, sc.root, sc.depth, pos, frame_dirs(oc, rot, fov, W, H, y0, rows, tr, ts), rcp_tab=tab, nthreads=NCPU)
    e = refine.trace_frame(sc.nodes8, sc.root, sc.depth, pos, rot, fov, W, H, sc.grid(k), sc.grid(8) if fine_t > 0 else None,
                           y0=y0, rows=rows, tile_rows=tr, tile_step=ts, rcp_tab=tab, want_npush=True, nthreads=NCPU)
    what += f", level {k}" + (f" refined to t {fine_t:.3f}" if fine_t > 0 else "")
    assert_same_hits(e, want, f"{what}: emulation")
    st, tau = e[4], e[5]
    assert st["beam_guard"] == 0 and st["beam_cert_wrong"] == 0, what
    hit = (want[0] != 0) & lean_only
    assert (tau[hit] <= want[2][hit]).all(), f"{what}: a tile start later than a hit time of the tile"
    if ctx is not None:
        assert ctx.beam_level(pos, rot, fov, W, H) == k, f"{what}: device level {ctx.beam_level(pos, rot, fov, W, H)}"
        got = ctx.trace_frame(pos, rot, fov, W, H, y0=y0, rows=rows, tile_rows=tr, tile_step=ts)
        assert_same_hits(got, want, f"{what}: device")
        cnt = ctx.trace_frame(pos, rot, fov, W, H, y0=y0, rows=rows, tile_rows=tr, tile_step=ts, want_npush=True)
        assert_same_hits(cnt, want, f"{what}: device, counting launch")
        bad = np.flatnonzero(cnt[3] != e[3])
        assert bad.size == 0, (f"{what}: {bad.size} rays with other PUSH counts than the emulation's, first at ray {bad[:3]} "
                               f"(device {cnt[3][bad[:3]]}, emulation {e[3][bad[:3]]}): a tile started elsewhere")
    return {"k": k, "fine_t": fine_t, "stats": st, "want": want, "zero_round_misses": int(((e[3] == 0) & (e[1] == 6)).sum())}


def device_ctx(ort, depth, nodes8=None, root=0):
    ctx = ort.TraceContext(depth)
    ctx.set_option("beam_after", 0)
    ctx.set_option("count_beam", 2)
    if nodes8 is not None:
        ctx.upload_full(nodes8, root)
    return ctx


# ---- scenes ----------------------------------------------------------------------------------------------------------

def thin_scene(ort, emu, depth):
    """test_beam.py's needles, one-voxel sheet and rod at depth 12, scaled to `depth` (the objects stay one voxel thin)."""
    s = 1 << (depth - 12)
    T = ort.HOctree(18, depth, device=None)
    rs = np.random.RandomState(9)
    for i in range(40):
        x, y, z = 2100 + 37 * i, 2048 + int(rs.randint(-300, 300)), 2048 + int(rs.randint(-200, 200))
        T.set(x * s, y * s, z * s, 1 + (x % 5))
    T.fill_box((3500 * s, 1000 * s, 1000 * s), (3500 * s + 1, 3000 * s, 3000 * s), 3)
    T.fill_box((2300 * s, 2047 * s, 1500 * s), (3400 * s, 2047 * s + 1, 1500 * s + 1), 4)
    nodes8, root, _ = T.flatten()
    return Scene(emu, nodes8, root, depth, f"thin scene, depth {depth}")


THIN_VIEWS = [(0.0, 0.0), (0.03, -0.12), (-0.05, 0.04)]
THIN_ROWS = [(758, 641), (2157 - 643, 643)]          # middle rows, and the last rows of the frame (partial tiles)


def face_scene(ort, emu, depth=12):
    """Voxels on the cube's faces (value 1), edges (2) and corners (3): single voxels, and a one-voxel line on face x = max."""
    dim = 1 << depth
    m = dim - 1
    T = ort.HOctree(18, depth, device=None)
    rs = np.random.RandomState(21)
    for _ in range(400):
        a, b = (int(v) for v in rs.randint(0, dim, 2))
        for v in ((m, a, b), (0, a, b), (a, m, b), (a, 0, b), (a, b, m), (a, b, 0)):
            T.set(*v, 1)
    for _ in range(100):
        a = int(rs.randint(0, dim))
        for v in ((m, m, a), (m, 0, a), (0, m, a), (m, a, m), (m, a, 0), (a, m, m), (a, 0, m)):
            T.set(*v, 2)
    for x in (0, m):
        for y in (0, m):
            for z in (0, m):
                T.set(x, y, z, 3)
    T.fill_box((m, dim // 4, dim // 2), (dim, 3 * dim // 4, dim // 2 + 1), 1)
    nodes8, root, _ = T.flatten()
    return Scene(emu, nodes8, root, depth, "face, edge and corner voxels")


# grazing cameras next to a face (most of the face is seen at a shallow angle, tiles leave the cube through it), and one
# looking at a corner
FACE_VIEWS = [((1.985, 1.5, 1.5), 1.5708, 0.0), ((1.97, 1.03, 1.5), 1.2, 0.1), ((1.5, 1.5, 1.992), 0.4, -0.05), ((1.02, 1.97, 1.03), -0.78, 0.35),
              ((1.97, 1.03, 1.03), -0.7854, -0.6155)]


def terrain_scene(ort, emu, depth, tunnels=True, ctx_device=False):
    T = ort.HOctree(14 + depth, depth, device=0 if ctx_device else None)
    ort.harness.build_terrain(T, tunnels=tunnels)
    nodes8, root, _ = T.flatten()
    return T, Scene(emu, nodes8, root, depth, f"terrain, depth {depth}")


TABLE_ORIGINS = [(1.5, 1.5, 1.5), (1.0 + 77 / 256.0, 1.5, 1.75), (1.3, 1.6, 1.9)]
TABLE_FRAMES = [(3840, 2160, 1000, 64), (1920, 1080, 448, 128)]


# ---- the emulation alone on the new scenes (CPU) -------------------------------------------------------------------

def test_thin_scene_at_depth_16_in_the_emulation(emu, refine, ort, oc):
    sc = thin_scene(ort, emu, 16)
    cov = Coverage()
    for yaw, pitch in THIN_VIEWS:
        rot, fov = oc.camera_coeffs(yaw, pitch)
        r = check_frame(emu, refine, oc, sc, (1.5, 1.5, 1.5), rot, fov, 3838, 2157, 758, 641, what=f"yaw {yaw} pitch {pitch}")
        hit = r["want"][0] != 0
        assert hit.sum() > 100 and len(np.unique(r["want"][0][hit])) >= 2, "the sheet and needles (sub-pixel at depth 16) in sight"
        cov.add(r)
    assert cov.levels == {7} and cov.refining == len(THIN_VIEWS) and cov.certified > 0


def test_face_edge_and_corner_voxels_in_the_emulation(emu, refine, ort, oc):
    sc = face_scene(ort, emu)
    cov = Coverage()
    kinds = set()
    for pos, yaw, pitch in FACE_VIEWS:
        rot, fov = oc.camera_coeffs(yaw, pitch)
        r = check_frame(emu, refine, oc, sc, pos, rot, fov, 3838, 2157, 758, 641, what=f"yaw {yaw} pitch {pitch}")
        kinds |= set(np.unique(r["want"][0]).tolist())
        cov.add(r)
    assert {1, 2, 3} <= kinds, f"faces, edges and corners should be in sight ({kinds})"
    assert cov.refining >= 2 and cov.certified > 0, (cov.refining, cov.certified)


def test_foreign_tables_in_the_emulation(emu, refine, ort, oc):
    """The 2^16-entry and the 8-bit table on the terrain: frames equal the oracle run with the same table; the coarse
    table's larger error widens the beam, so its 1080p launches take a coarser level."""
    _, sc = terrain_scene(ort, emu, 8)
    tabs = foreign_tables()
    rot, fov = oc.camera_coeffs(0.7, -0.6)
    for pos in TABLE_ORIGINS:
        assert emu.beam_level(pos, rot, fov, 1920, 1080, 8, rcp_tab=tabs["8-bit 2^11"]) < emu.beam_level(pos, rot, fov, 1920, 1080, 8)
    for name in ("12-bit 2^16", "8-bit 2^11"):
        cov = Coverage()
        for pos in TABLE_ORIGINS:
            for W, H, y0, rows in TABLE_FRAMES:
                cov.add(check_frame(emu, refine, oc, sc, pos, rot, fov, W, H, y0, rows, tab=tabs[name], what=f"{name} table,"))
        assert cov.certified > 0, name
        assert (cov.refining > 0) == (name == "12-bit 2^16"), (name, cov.refining)


# ---- the device --------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_random_dags_and_cameras(emu, refine, ort, oc):
    """test_fuzz_random_dags' scenes at depths 3-10 from three cameras each (one on a level's grid), 64-row strips of
    frames from 256 x 144 to 4K; the device's grids equal the emulation's for every level used, and for level 8."""
    from test_fuzz_random_dags import random_scene
    cov = Coverage()
    ctxs = {}
    for seed in range(120):
        depth, nodes8, root, _, _ = random_scene(ort, 5000 + seed, depth=3 + seed % 8)
        if root == 0:
            continue
        sc = Scene(emu, nodes8, root, depth, f"seed {seed} (kind {(5000 + seed) % 4}, depth {depth})")
        ctx = ctxs.get(depth) or ctxs.setdefault(depth, device_ctx(ort, depth))
        ctx.upload_full(nodes8, root)
        rs = np.random.RandomState(seed)
        sizes = [(1920, 1080), (2560, 1440), (3840, 2160)] if depth >= 8 else [(256, 144), (640, 360), (1280, 720), (1920, 1080), (3840, 2160)]
        used = set()
        for cam in range(3):
            pos = rs.uniform(1.02, 1.98, 3).astype(np.float32)
            if cam == 1:
                q = 1 << int(rs.randint(1, depth + 1))
                pos = (np.floor((pos - 1.0) * q) / q + 1.0 + (1.0 / q if rs.rand() < 0.5 else 0.0)).astype(np.float32)      # on some level's grid
                pos = np.clip(pos, np.float32(1.0) + np.float32(1.0 / q), np.float32(2.0) - np.float32(1.0 / q))
            rot, fov = oc.camera_coeffs(float(rs.uniform(-3.1, 3.1)), float(rs.uniform(-1.5, 1.5)))
            W, H = sizes[(seed + cam) % len(sizes)]
            rows = min(H, 64)
            y0 = int(rs.randint(0, H - rows + 1)) & ~3
            if emu.beam_level(pos, rot, fov, W, H, depth) == 0:
                assert ctx.beam_level(pos, rot, fov, W, H) == 0, sc.name
                continue
            r = check_frame(emu, refine, oc, sc, pos, rot, fov, W, H, y0, rows, ctx=ctx, what=f"camera {cam}")
            used.add(r["k"])
            if r["fine_t"] > 0:
                used.add(8)
            cov.add(r)
        for k in sorted(used | ({8} if depth >= 8 else set())):
            assert np.array_equal(ctx.beam_grid(k), sc.grid(k)), f"{sc.name}: level-{k} grid"
    for ctx in ctxs.values():
        ctx.close()
    assert cov.frames >= 150 and len(cov.levels) >= 3 and cov.refining >= 50, (cov.frames, cov.levels, cov.refining)
    assert cov.certified > 0 and cov.zero_round_misses > 0


@pytest.mark.gpu
def test_thin_geometry_at_depths_12_and_16(emu, refine, ort, oc):
    """Needles, a one-voxel sheet and a rod at depths 12 and 16, and voxels on the cube's faces, edges and corners seen by
    grazing cameras, in 3838 x 2157 frames (partial tiles on the right and at the bottom), refined."""
    cov = Coverage()
    for sc, views in [(thin_scene(ort, emu, 12), [((1.5, 1.5, 1.5), y, p) for y, p in THIN_VIEWS]),
                      (thin_scene(ort, emu, 16), [((1.5, 1.5, 1.5), y, p) for y, p in THIN_VIEWS]),
                      (face_scene(ort, emu), FACE_VIEWS)]:
        ctx = device_ctx(ort, sc.depth, sc.nodes8, sc.root)
        for i, (pos, yaw, pitch) in enumerate(views):
            rot, fov = oc.camera_coeffs(yaw, pitch)
            y0, rows = THIN_ROWS[i % 2]
            r = check_frame(emu, refine, oc, sc, pos, rot, fov, 3838, 2157, y0, rows, ctx=ctx, what=f"yaw {yaw} pitch {pitch}")
            assert (r["want"][0] != 0).sum() > 50, f"{sc.name}: yaw {yaw} pitch {pitch} should see something"
            cov.add(r)
        for k in (7, 8):
            assert np.array_equal(ctx.beam_grid(k), sc.grid(k)), f"{sc.name}: level-{k} grid"
        ctx.close()
    assert cov.levels == {7} and cov.refining >= 8 and cov.certified > 0, (cov.levels, cov.refining, cov.certified)


@pytest.mark.gpu
def test_foreign_reciprocal_tables(emu, refine, ort, oc):
    """ctx.set_rcp_table with the 24-bit, the 2^16-entry and the 8-bit table, switched on the same DAG version without a
    re-upload: levels follow the table, frames equal the oracle run with the table in use, an on-grid origin with the
    24-bit table certifies no tile and an off-grid one does; the default table restores the default frames."""
    tabs = foreign_tables()
    default = emu.default_rcp_table()
    rot, fov = oc.camera_coeffs(0.7, -0.6)
    for depth in (8, 12):
        T, sc = terrain_scene(ort, emu, depth, ctx_device=True)
        T.sync()
        ctx = T.ctx
        ctx.set_option("beam_after", 0)
        ctx.set_option("count_beam", 2)
        first = {}
        used = set()
        for name, tab in [("default", default)] + list(tabs.items()) + [("default again", default)]:
            if name != "default":
                ctx.set_rcp_table(tab)
            levels = set()
            for pos in TABLE_ORIGINS:
                for W, H, y0, rows in TABLE_FRAMES:
                    r = check_frame(emu, refine, oc, sc, pos, rot, fov, W, H, y0, rows, tab=tab, ctx=ctx, what=f"{name} table,",
                                    lean_only=not name.startswith("24"))
                    levels.add(r["k"])
                    used |= {r["k"]} | ({8} if r["fine_t"] > 0 else set())
                    if name.startswith("24"):
                        if on_grid(pos, depth):
                            assert r["stats"]["beam_tile_misses"] == 0, f"{name}, origin {pos}: an on-grid origin with inexact products certified a tile"
                        else:
                            assert r["stats"]["beam_tile_misses"] > 0, f"{name}, origin {pos}: off the grid, tiles that see nothing should be certified"
                    key = (pos, W)
                    if name == "default":
                        first[key] = r["want"]
                    elif name == "default again":
                        assert_same_hits(r["want"], first[key], f"depth {depth}, origin {pos}, {W}: the default table's frame again")
            if name.startswith("8-bit"):
                assert min(levels) < 6, f"depth {depth}: the coarse table should coarsen the level ({levels})"
        for k in sorted(used):
            assert np.array_equal(ctx.beam_grid(k), sc.grid(k)), f"depth {depth}: level-{k} grid after the table switches"
        ctx.close()


@pytest.mark.gpu
def test_every_frame_entry_point_on_a_refining_scene(emu, refine, ort, oc):
    """Terrain at depth 10 with needles floating above it, one camera whose 1080p launches run at level 7 and refine:
    host-buffer frames in 1, 3 and 8 chunks and deferred, device buffers, shaded frames to the host and to the device,
    cyclic strips, repeated views (band schedules applied) -- and the pool layout at depth 8 and 4K."""
    import torch
    depth = 10
    T = ort.HOctree(24, depth, device=0)
    ort.harness.build_terrain(T, tunnels=True)
    rs = np.random.RandomState(4)
    for i in range(60):
        T.set(512 + 7 * i, 512 + int(rs.randint(-200, 200)), 600 + int(rs.randint(-60, 60)), 1 + i % 4)
    T.sync()
    ctx = T.ctx
    ctx.set_option("beam_after", 0)
    ctx.set_option("count_beam", 2)
    cols, _ = ort.harness.parse_voxels(ort.harness.DEMO_VOXELS)
    ctx.set_palette(cols, EXIT, INSIDE)
    nodes8, root, _ = T.flatten()
    sc = Scene(emu, nodes8, root, depth, "terrain + needles, depth 10")
    pos = np.array([1.5, 1.5, 1.5], np.float32)
    rot, fov = oc.camera_coeffs(0.2, -0.35)
    W, H = 1920, 1080
    r = check_frame(emu, refine, oc, sc, pos, rot, fov, W, H, ctx=ctx, what="whole frame")
    want = r["want"]
    assert r["k"] == 7 and r["fine_t"] > 0 and r["stats"]["beam_tile_misses"] > 0 and r["zero_round_misses"] > 0
    assert (want[0] != 0).sum() > 10_000 and np.isin(np.arange(1, 5), want[0]).all()
    for chunks in (1, 3, 8):
        ctx.set_option("frame_chunks", chunks)
        assert_same_hits(ctx.trace_frame(pos, rot, fov, W, H), want, f"{chunks} chunks")
    ctx.set_option("frame_chunks", 0)
    ctx.set_option("defer_sync", 1)
    outs = [ctx.trace_frame(pos, rot, fov, W, H) for _ in range(2)]
    ctx.sync()
    ctx.set_option("defer_sync", 0)
    for o in outs:
        assert_same_hits(o, want, "deferred host-buffer frame")
    n = W * H
    dv = torch.empty(n, dtype=torch.int32, device="cuda"); df = torch.empty(n, dtype=torch.uint8, device="cuda"); dt = torch.empty(n, dtype=torch.float32, device="cuda")
    s0 = ctx.band_schedules
    for rep in range(4):
        ctx.trace_frame_async(pos, rot, fov, W, H, 0, H, 1, 1, dv, df, dt)
        ctx.sync()
        assert_same_hits((dv.cpu().numpy().view(np.uint32), df.cpu().numpy(), dt.cpu().numpy()), want, f"device buffers, repetition {rep}")
    assert ctx.band_schedules > s0, "a repeated view should have had its band schedule applied"
    colour = np.where(want[1] == 6, np.uint32(EXIT), np.where(want[1] == 7, np.uint32(INSIDE),
                      cols.ravel()[np.minimum(6 * (want[0].astype(np.int64) - 1) + want[1], cols.size - 1).clip(0)])).astype(np.uint32)
    assert np.array_equal(ctx.trace_frame_rgba(pos, rot, fov, W, H), colour), "shaded frame to the host"
    d = torch.empty(n, dtype=torch.int32, device="cuda")
    ctx.trace_frame_rgba(pos, rot, fov, W, H, out=d)
    ctx.sync()
    assert np.array_equal(d.cpu().numpy().view(np.uint32), colour), "shaded frame to the device"
    strips = [(8, 4, 2, 200), (4, 8, 3, 216), (12, 12, 4, 180), (20, 16, 5, 160), (16, 16, 2, 256)]
    for y0, tr, ts, rows in strips:
        r = check_frame(emu, refine, oc, sc, pos, rot, fov, W, H, y0, rows, tr, ts, ctx=ctx, what="cyclic strip,")
        sel = np.concatenate([np.arange(y * W, (y + 1) * W) for y in frame_rows(y0, rows, tr, ts)])
        assert np.array_equal(ctx.trace_frame_rgba(pos, rot, fov, W, H, y0=y0, rows=rows, tile_rows=tr, tile_step=ts), colour[sel]), f"shaded strip {tr}/{ts}"
    ctx.close()

    # the pool layout (och::octree rows, root = row 0, MISS time 0.0F) at depth 8, refined 4K rows
    from test_oracle import _builtin_table
    depth, cap = 8, 1 << 18
    P = ort.Octree(depth, cap)
    ops = [(int(x), int(y), int(z), 1 + int(x) % 4, 0) for x, y, z in np.random.RandomState(12).randint(0, 256, (3000, 3)) if z < 160]
    ops += [(x, y, z, 2, 0) for x in range(0, 256, 3) for y in range(0, 256, 5) for z in range(0, 24)]
    P.apply(np.array(ops, np.int32))
    P.sync()
    P.ctx.set_option("beam_after", 0)
    tab = _builtin_table()
    assert np.array_equal(tab, emu.default_rcp_table())
    pool = P.nodes().copy()
    rot, fov = oc.camera_coeffs(0.9, -0.4)
    pos = np.array([1.4, 1.45, 1.85], np.float32)
    W, H, y0, rows = 3840, 2160, 900, 320
    k = emu.beam_level(pos, rot, fov, W, H, depth)
    assert k == 7 and P.ctx.beam_level(pos, rot, fov, W, H) == 7 and refine.beam_fine_t(pos, rot, fov, W, H, depth) > 0
    got = P.ctx.trace_frame(pos, rot, fov, W, H, y0=y0, rows=rows)
    want = oc.octree_trace_rays(pool, depth, pos, frame_dirs(oc, rot, fov, W, H, y0, rows), rcp_tab=tab, nthreads=NCPU)
    assert_same_hits(got, want, "pool layout, 4K rows")
    assert (want[0] != 0).sum() > 1000 and (want[1] == 6).sum() > 1000
    for k in (7, 8):
        assert np.array_equal(P.ctx.beam_grid(k), emu.beam_grid(pool, 0, k, pool=True)), f"pool layout: level-{k} grid"
    P.ctx.close()


@pytest.mark.gpu
def test_batched_launches(emu, refine, ort, oc):
    """Batch A: one launch of jobs whose levels differ (a refining 4K job at level 7, 1080p and 640 x 360 jobs, origins on
    and off the grid), then the same jobs as a counting launch (one job with PUSH counts) under count_beam = 2.  Batch B:
    40 jobs, two launches; an origin outside the cube in the second runs that launch without the beam, the first keeps it."""
    import torch
    depth = 9
    T = ort.HOctree(22, depth, device=0)
    ort.harness.build_terrain(T, tunnels=True)
    for i in range(30):
        T.set(300 + 5 * i, 250 + (37 * i) % 40, 400, 3)
    T.sync()
    ctx = T.ctx
    ctx.set_option("beam_after", 0)
    nodes8, root, _ = T.flatten()
    sc = Scene(emu, nodes8, root, depth, "terrain, depth 9")
    tab = emu.default_rcp_table()

    def run(jobs, npush_job=None):
        outs, arg = [], []
        for i, (pos, rot, fov, W, H, y0, rows, tr, ts) in enumerate(jobs):
            m = rows * W
            o = [torch.empty(m, dtype=torch.int32, device="cuda"), torch.empty(m, dtype=torch.uint8, device="cuda"), torch.empty(m, dtype=torch.float32, device="cuda")]
            if i == npush_job:
                o.append(torch.empty(m, dtype=torch.int16, device="cuda"))
            outs.append(o)
            arg.append((pos, rot, fov, W, H, y0, rows, tr, ts, *o))
        torch.cuda.synchronize()
        ctx.trace_frames_async(arg)
        ctx.sync()
        return [tuple(a.cpu().numpy() for a in o) for o in outs]

    def oracle(job):
        pos, rot, fov, W, H, y0, rows, tr, ts = job
        return oc.trace_rays(nodes8, root, depth, pos, frame_dirs(oc, rot, fov, W, H, y0, rows, tr, ts), rcp_tab=tab, nthreads=NCPU)

    def check(jobs, outs, wants, what):
        for i, (o, w) in enumerate(zip(outs, wants)):
            assert_same_hits((o[0].view(np.uint32), o[1], o[2]), w, f"{what}, job {i}")

    cam = lambda p, yaw, pitch: (np.array(p, np.float32),) + tuple(oc.camera_coeffs(yaw, pitch))
    jobs_a = [cam((1.5, 1.5, 1.5), 0.7, -0.6) + (3840, 2160, 1000, 96, 1, 1),
              cam((1.3, 1.6, 1.9), 0.3, -0.8) + (1920, 1080, 16, 192, 8, 2),
              cam((1.0 + 77 / 256.0, 1.25, 1.75), 2.0, -0.5) + (640, 360, 0, 360, 1, 1),
              cam((1.1, 1.8, 1.6), -2.2, -0.3) + (3838, 2157, 2157 - 99, 99, 1, 1)]
    levels = [emu.beam_level(j[0], j[1], j[2], j[3], j[4], depth) for j in jobs_a]
    fine = [refine.beam_fine_t(j[0], j[1], j[2], j[3], j[4], depth) for j in jobs_a]
    assert levels[0] == 7 and fine[0] > 0 and len(set(levels)) >= 3 and min(levels) > 0, levels
    for j, k in zip(jobs_a, levels):
        assert ctx.beam_level(j[0], j[1], j[2], j[3], j[4]) == k
    wants = [oracle(j) for j in jobs_a]
    l0 = ctx.launch_count
    check(jobs_a, run(jobs_a), wants, "batch A")
    assert ctx.launch_count - l0 >= 2, "batch A: a march and a trace launch"
    ctx.set_option("count_beam", 2)
    for counted in (0, 2):
        outs = run(jobs_a, npush_job=counted)
        check(jobs_a, outs, wants, f"batch A, counting job {counted}")
        pos, rot, fov, W, H, y0, rows, tr, ts = jobs_a[counted]
        e = refine.trace_frame(nodes8, root, depth, pos, rot, fov, W, H, sc.grid(levels[counted]), sc.grid(8) if fine[counted] > 0 else None,
                               y0=y0, rows=rows, tile_rows=tr, tile_step=ts, want_npush=True, nthreads=NCPU)
        assert_same_hits(e, wants[counted], f"batch A, job {counted}: emulation")
        got_n = outs[counted][3].view(np.uint16)
        bad = np.flatnonzero(got_n != e[3])
        assert bad.size == 0, f"batch A, job {counted}: {bad.size} rays with other PUSH counts than the emulation's, first at {bad[:3]}"
        assert ((e[3] == 0) & (e[1] == 6)).any() and e[4]["beam_tile_misses"] > 0
    ctx.set_option("count_beam", 0)

    # batch B: 40 jobs -> launches of 32 and 8; job 35's origin is outside the cube
    rs = np.random.RandomState(8)
    jobs_b = []
    for i in range(40):
        W, H = [(640, 360), (1280, 720), (1920, 1080)][i % 3]
        p = (2.4, 1.5, 1.6) if i == 35 else tuple(rs.uniform(1.1, 1.9, 3))
        yaw = 3.1416 if i == 35 else float(rs.uniform(-3.1, 3.1))
        rows = 32
        jobs_b.append(cam(p, yaw, float(rs.uniform(-0.9, 0.1))) + (W, H, int(rs.randint(0, H - rows)) & ~3, rows, 1, 1))
    lv = [emu.beam_level(j[0], j[1], j[2], j[3], j[4], depth) for j in jobs_b]
    assert lv[35] == 0 and all(k > 0 for i, k in enumerate(lv) if i != 35) and len(set(lv[:32])) >= 2, lv
    wants = [oracle(j) for j in jobs_b]
    check(jobs_b, run(jobs_b), wants, "batch B")
    l0, b0 = ctx.launch_count, ctx.beam_builds
    check(jobs_b, run(jobs_b), wants, "batch B again")
    assert ctx.beam_builds == b0 and ctx.launch_count - l0 == 3, "the first launch of 32 jobs with its march, the second without"
    assert (wants[35][0] != 0).any()
    ctx.close()


def _sky_scene(dim):
    """A slab and two blocks (z < 64) -- and what goes into the sky above: isolated voxels and a one-voxel sheet."""
    base = np.zeros((dim, dim, dim), np.uint8)
    base[:48] = 1
    base[48:64, 40:90, 30:120] = 2
    base[48:60, 150:200, 100:220] = 4
    sky = []
    rs = np.random.RandomState(6)
    for i in range(40):
        sky.append((170 + 2 * i, 96 + int(rs.randint(0, 64)), 112 + int(rs.randint(0, 60)), 1 + i % 4))
    return base, sky


@pytest.mark.gpu
def test_dags_made_on_the_device(emu, refine, ort, oc):
    """Voxels put into sky that was free at levels 1-3 by upload_voxels, write_voxels and patch_voxels, then erased again:
    every version's frames equal the oracle of a host table with the same voxels, its grids of levels 3-8 equal the
    emulation's (a patched mirror, with its appended rows, gives the same bytes), each traced version builds its grids
    once, and a patch that empties the scene gives an all-MISS frame without a grid build."""
    depth = 8
    dim = 1 << depth
    base, sky = _sky_scene(dim)
    full = base.copy()
    for x, y, z, v in sky:
        full[z, y, x] = v
    full[112:172, 80:176, 240] = 3                                   # the sheet, one voxel thick
    box_o, box_n = (160, 64, 96), (96, 128, 96)                      # the sky part that changes: [x0, x0 + nx) ...
    sl = (slice(box_o[2], box_o[2] + box_n[2]), slice(box_o[1], box_o[1] + box_n[1]), slice(box_o[0], box_o[0] + box_n[0]))
    changed = full != base
    assert not base[sl].any() and changed[sl].sum() == changed.sum() > 0

    def host_scene(grid, name):
        T = ort.HOctree(20, depth, device=None)
        T.fill_box((0, 0, 0), (dim, dim, 48), 1)
        T.fill_box((30, 40, 48), (120, 90, 64), 2)
        T.fill_box((100, 150, 48), (220, 200, 60), 4)
        if grid is full:
            for x, y, z, v in sky:
                T.set(x, y, z, v)
            T.fill_box((240, 80, 112), (241, 176, 172), 3)
        nodes8, root, _ = T.flatten()
        return Scene(emu, nodes8, root, depth, name)

    sc_base, sc_full = host_scene(base, "slab"), host_scene(full, "slab + sky voxels")
    # the changed voxels sit in cells that were free at levels 1-3 of the level-3 grid, and are marked now
    g3b, g3f = sc_base.grid(3), sc_full.grid(3)
    cells = {(z >> 5, y >> 5, x >> 5) for x, y, z, _ in sky}
    assert all(1 <= g3b[c] <= 3 for c in cells) and all(g3f[c] == 0 for c in cells)
    views = [((1.5, 1.5, 1.55), 0.05, -0.1, 3840, 2160, 920, 160), ((1.5, 1.5, 1.55), -0.1, -0.05, 640, 360, 0, 360)]

    def frames(ctx, sc, what):
        b0 = ctx.beam_builds
        levels = set()
        for pos, yaw, pitch, W, H, y0, rows in views:
            rot, fov = oc.camera_coeffs(yaw, pitch)
            r = check_frame(emu, refine, oc, sc, pos, rot, fov, W, H, y0, rows, ctx=ctx, what=f"{what},")
            levels.add(r["k"])
            if sc is sc_full and W == 3840:
                assert r["fine_t"] > 0 and np.isin([1, 2, 3, 4], r["want"][0]).all(), "the sky voxels and the sheet in sight, refined"
        # one build per launch level of the DAG version (the refinement's level-8 grid is built with the level-7 one)
        assert len(levels) == 2 and ctx.beam_builds == b0 + len(levels), f"{what}: one grid build per level used ({levels})"
        for k in range(3, 9):
            assert np.array_equal(ctx.beam_grid(k), sc.grid(k)), f"{what}: level-{k} grid"

    for method in ("upload_voxels", "write_voxels", "patch_voxels"):
        ctx = device_ctx(ort, depth)
        ctx.upload_voxels(base)
        frames(ctx, sc_base, f"{method}: the slab")
        if method == "upload_voxels":
            ctx.upload_voxels(full)
        else:
            getattr(ctx, method)(box_o, np.ascontiguousarray(full[sl]))
        frames(ctx, sc_full, f"{method}: sky voxels put in")
        if method == "upload_voxels":
            ctx.upload_voxels(base)
        else:
            getattr(ctx, method)(box_o, np.zeros_like(full[sl]))
        frames(ctx, sc_base, f"{method}: sky voxels erased")
        if method == "patch_voxels":
            ctx.patch_voxels((0, 0, 0), np.zeros((dim, dim, dim), np.uint8))
            b0 = ctx.beam_builds
            pos, yaw, pitch, W, H, y0, rows = views[0]
            rot, fov = oc.camera_coeffs(yaw, pitch)
            v, f, t = ctx.trace_frame(pos, rot, fov, W, H, y0=y0, rows=rows)
            assert (v == 0).all() and (f == 6).all() and np.isinf(t).all(), "an empty scene: every ray a MISS"
            assert ctx.beam_builds == b0, "an empty scene builds no grid"
        ctx.close()
