"""Refinement of the beam start on the level-8 grid (csrc/ort_beam.cuh, item 2: a tile marches on from its level-k stop on
the level-8 grid and keeps that stop where its own beam still fits a level-8 cell there), on the CPU through the host
emulation -- everywhere tests/test_beam.py holds the one-level march: terrain from nine cameras at three frame sizes, the
24-bit reciprocal table with on-grid origins, random DAGs, needles / a one-voxel sheet / a rod at depth 12 and 4K.

For each: frames with the refinement equal the oracle bit for bit, no tile start exceeds a hit time of its tile, the guard
never fires, no tile is certified wrongly, and a refined start is never earlier than the one-level start."""
import os
import sys

import numpy as np
import pytest

from conftest import assert_same_hits

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emu"))

POSES = {"A": ((1.5, 1.5, 1.5), 0.0, 0.0), "B": ((1.5, 1.5, 1.5), 0.7, -0.6), "C": ((1.1, 1.1, 1.4), 0.785, -0.3)}
NCPU = max(1, min(16, os.cpu_count() or 1))


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


def check_frame(emu, refine, oc, nodes8, root, depth, pos, rot, fov, W, H, grid, fine, what, y0=0, rows=None, tr=1, ts=1, tab=None, counts=False, lean_only=True):
    """One frame with and without the refinement against the oracle; returns (stats, tiles refined, rounds without, rounds with).
    lean_only: every ray is a lean-tier ray, so every hit time bounds its tile's start (with the 24-bit table some rays of an
    on-grid origin take other tiers, which ignore the start and measure hit times on another clock)."""
    tab = emu.default_rcp_table() if tab is None else tab
    rows = H - y0 if rows is None else rows
    frame_rows = [y0 + (r // tr) * tr * ts + r % tr for r in range(rows)] if ts > 1 else list(range(y0, y0 + rows))
    d = np.concatenate([oc.gen_rays(rot, fov, W, H, y, y + 1) for y in frame_rows])
    want = oc.trace_rays(nodes8, root, depth, np.array(pos, np.float32), d, rcp_tab=tab, nthreads=NCPU)
    kw = dict(y0=y0, rows=rows, tile_rows=tr, tile_step=ts, rcp_tab=tab, want_npush=counts)
    base = refine.trace_frame(nodes8, root, depth, pos, rot, fov, W, H, grid, None, **kw)
    got = refine.trace_frame(nodes8, root, depth, pos, rot, fov, W, H, grid, fine, **kw)
    # without the refinement the frame is the one emu.py traces with the same grid
    one = emu.trace_frame(nodes8, root, depth, pos, rot, fov, W, H, walker=13, beam=grid, want_tau=True, **kw)
    assert all(np.array_equal(a, b) for a, b in zip(one[:3 + counts], base[:3 + counts])) and np.array_equal(one[-1], base[-1]), what
    assert_same_hits(got, want, what)
    st, tau, tau0 = got[-2], got[-1], base[-1]
    assert st["beam_guard"] == 0, what
    assert st["beam_cert_wrong"] == 0, f"{what}: a tile was ended as a whole although some of its rays are not lean-tier rays"
    hit = (want[0] != 0) & lean_only
    assert (tau[hit] <= want[2][hit]).all(), f"{what}: a tile start later than a hit time of the tile"
    assert (tau >= tau0).all(), f"{what}: a refined start earlier than the one-level start"
    refined = int((tau > tau0).sum())
    n0 = int(base[3].astype(np.int64).sum()) if counts else 0
    n1 = int(got[3].astype(np.int64).sum()) if counts else 0
    return st, refined, n0, n1


@pytest.mark.parametrize("depth,tunnels", [(8, True), (10, False)])
def test_refined_frames_on_terrain_equal_the_oracle(emu, refine, ort, oc, depth, tunnels):
    """The cameras of test_beam.py's terrain test (the bench poses, corners of the cube, next to the terrain and inside
    tunnels) at three frame sizes: rows of 4K frames and cyclic 4K strips, where launches run at level 7 and refine, and
    whole 640 x 360 frames, where they do not."""
    T = ort.HOctree(14 + depth, depth, device=None)
    ort.harness.build_terrain(T, tunnels=tunnels)
    nodes8, root, _ = T.flatten()
    cams = [POSES["A"], POSES["B"], POSES["C"],
            ((1.02, 1.03, 1.9), 0.785, -0.9), ((1.97, 1.96, 1.95), 3.9, -0.5), ((1.5, 1.5, 1.999), 0.3, -1.5),
            ((1.25, 1.75, 1.0 + 5.0 / 16.0 + 0.02), 1.1, -0.05), ((1.5, 1.5, 1.2), 2.0, 0.4), ((1.0625, 1.5, 1.5), 0.0, 0.0)]
    grids = {}
    fine = emu.beam_grid(nodes8, root, 8)
    refined = n_base = n_fine = frames = 0
    for ci, (pos, yaw, pitch) in enumerate(cams):
        rot, fov = oc.camera_coeffs(yaw, pitch)
        for (W, H, y0, rows, tr, ts) in [(3840, 2160, 1000, 48, 1, 1), (3840, 2160, 512, 48, 8, 2), (640, 360, 0, 360, 1, 1)][: 3 if ci < 4 else 1]:
            k = emu.beam_level(pos, rot, fov, W, H, depth)
            if k == 0:
                continue
            if k not in grids:
                grids[k] = emu.beam_grid(nodes8, root, k)
            what = f"depth {depth}, camera {ci}, {W}x{H} rows {y0}+{rows} tiles {tr}/{ts}, level {k} + 8"
            _, r, a, b = check_frame(emu, refine, oc, nodes8, root, depth, pos, rot, fov, W, H, grids[k], fine, what, y0, rows, tr, ts, counts=True)
            assert b <= a, what
            refined += r; n_base += a; n_fine += b; frames += 1
    assert frames >= 10 and refined > 10_000, (frames, refined)
    assert n_fine < n_base, "the refinement should save rounds"


def test_refined_frames_with_a_full_precision_reciprocal_table(emu, refine, ort, oc):
    """On-grid and off-grid origins with a table of correctly rounded reciprocals (test_beam.py's on-grid test), on the
    middle rows of 4K frames."""
    depth = 8
    T = ort.HOctree(20, depth, device=None)
    ort.harness.build_terrain(T, tunnels=True)
    nodes8, root, _ = T.flatten()
    n = 1 << 11
    tab = (np.float32(1.0) / (np.float32(1.0) + (np.arange(n, dtype=np.float32) + np.float32(0.5)) / np.float32(n))).astype(np.float32).view(np.uint32)
    fine = emu.beam_grid(nodes8, root, 8)
    W, H = 3840, 2160                   # (launches at level 7 refine: not at 640 x 360)
    refined = 0
    for pos in [(1.5, 1.5, 1.5), (1.0 + 77 / 256.0, 1.5, 1.75), (1.3, 1.6, 1.9)]:
        rot, fov = oc.camera_coeffs(0.7, -0.6)
        k = emu.beam_level(pos, rot, fov, W, H, depth, rcp_tab=tab)
        assert k > 0 and refine.beam_fine_t(pos, rot, fov, W, H, depth, rcp_tab=tab) > 0
        st, r, _, _ = check_frame(emu, refine, oc, nodes8, root, depth, pos, rot, fov, W, H, emu.beam_grid(nodes8, root, k), fine, f"origin {pos}, 24-bit table", y0=1000, rows=100, tab=tab, lean_only=False)
        on_grid = any(float(c) * 256 == int(float(c) * 256) for c in pos)
        if on_grid:
            assert st["beam_tile_misses"] == 0, "an on-grid origin with inexact products must not certify tiles"
        refined += r
    assert refined > 0


def test_refined_frames_on_random_dags(emu, refine, ort, oc):
    """The 120 scenes of test_fuzz_random_dags.py (isolated voxels, boxes, dense noise, a solid cube with holes) at depths
    8-10, where a level-8 grid exists, from random cameras, on-grid origins included, at frame sizes from 1600 x 900
    to 4K."""
    from test_fuzz_random_dags import random_scene
    frames = refined = refining_frames = 0
    for seed in range(120):
        depth, nodes8, root, _, _ = random_scene(ort, 5000 + seed, depth=8 + seed % 3)
        if root == 0:
            continue
        rs = np.random.RandomState(seed)
        grids = {}
        fine = None
        for cam in range(3):
            pos = rs.uniform(1.02, 1.98, 3).astype(np.float32)
            if cam == 1:
                q = 1 << int(rs.randint(1, depth + 1))
                pos = (np.floor((pos - 1.0) * q) / q + 1.0 + (1.0 / q if rs.rand() < 0.5 else 0.0)).astype(np.float32)      # on some level's grid
                pos = np.clip(pos, np.float32(1.0) + np.float32(1.0 / q), np.float32(2.0) - np.float32(1.0 / q))
            rot, fov = oc.camera_coeffs(float(rs.uniform(-3.1, 3.1)), float(rs.uniform(-1.5, 1.5)))
            W, H = [(1600, 900), (2560, 1440), (3840, 2160)][(seed + cam) % 3]
            rows = min(H, 64)
            y0 = int(rs.randint(0, H - rows + 1)) & ~3
            k = emu.beam_level(pos, rot, fov, W, H, depth)
            if k == 0:
                continue
            if k not in grids:
                grids[k] = emu.beam_grid(nodes8, root, k)
            if fine is None:
                fine = emu.beam_grid(nodes8, root, 8)
            what = f"seed {seed} (kind {(5000 + seed) % 4}, depth {depth}), camera {cam} at {pos.tolist()}, {W}x{H}, level {k} + 8"
            _, r, _, _ = check_frame(emu, refine, oc, nodes8, root, depth, pos, rot, fov, W, H, grids[k], fine, what, y0, rows)
            frames += 1; refined += r; refining_frames += refine.beam_fine_t(pos, rot, fov, W, H, depth) > 0
    assert frames > 150 and refining_frames > 50 and refined > 0, (frames, refining_frames, refined)


def test_refined_needles_and_sheets_are_not_flown_past(emu, refine, ort, oc):
    """test_beam.py's thin geometry at depth 12 and 4K: single voxels at several distances, a one-voxel sheet far away and
    a one-voxel rod along x; with the level-8 refinement the tiles start up to 16 voxels from what they see."""
    depth = 12
    T = ort.HOctree(16, depth, device=None)
    rs = np.random.RandomState(9)
    needles = [(2100 + 37 * i, 2048 + int(rs.randint(-300, 300)), 2048 + int(rs.randint(-200, 200))) for i in range(40)]
    for x, y, z in needles:
        T.set(x, y, z, 1 + (x % 5))
    T.fill_box((3500, 1000, 1000), (3501, 3000, 3000), 3)
    T.fill_box((2300, 2047, 1500), (3400, 2048, 1501), 4)
    nodes8, root, _ = T.flatten()
    W, H = 3840, 2160
    pos = np.array([1.5, 1.5, 1.5], np.float32)
    grid, fine = emu.beam_grid(nodes8, root, 7), emu.beam_grid(nodes8, root, 8)
    refined = 0
    for yaw, pitch in [(0.0, 0.0), (0.03, -0.12), (-0.05, 0.04)]:
        rot, fov = oc.camera_coeffs(yaw, pitch)
        assert emu.beam_level(pos, rot, fov, W, H, depth) == 7 and refine.beam_fine_t(pos, rot, fov, W, H, depth) > 0.5
        st, r, _, _ = check_frame(emu, refine, oc, nodes8, root, depth, pos, rot, fov, W, H, grid, fine, f"needles, yaw {yaw} pitch {pitch}", 760, 640)
        assert st["beam_tile_misses"] > 0
        refined += r
    assert refined > 0


def test_refinement_limit(emu, refine, oc):
    """The host's choice: refinement needs a level-8 DAG and a launch at level 7; the limit shrinks with the pixel size."""
    rot, fov = oc.camera_coeffs(0.7, -0.6)
    c = (1.5, 1.5, 1.5)
    t4k, t1080 = refine.beam_fine_t(c, rot, fov, 3840, 2160, 12), refine.beam_fine_t(c, rot, fov, 1920, 1080, 12)
    assert 0.5 < t4k and 0 < t1080 < t4k
    assert emu.beam_level(c, rot, fov, 640, 360, 12) < 7 and refine.beam_fine_t(c, rot, fov, 640, 360, 12) == 0.0
    assert refine.beam_fine_t(c, rot, fov, 3840, 2160, 7) == 0.0
    assert refine.beam_fine_t(c, rot, fov, 3840, 2160, 8) == t4k
    assert refine.beam_fine_t(c, rot, fov, 8, 4, 12) == 0.0
    assert refine.beam_fine_t(c, rot * 1.01, fov, 3840, 2160, 12) == 0.0
