"""Refinement of the beam start on the level-8 grid (csrc/ort_beam.cuh, item 2) on the GPU: the level-8 grid's bytes equal
the host rebuild, and frames with the refinement equal frames without it (option "beam_level" forces the launch's level
and turns the refinement off) bit for bit, with fewer rounds, for host-buffer, shaded and batched launches.  Launches
that return PUSH counts refine only with option count_beam = 2."""
import os
import sys

import numpy as np
import pytest

from conftest import assert_same_hits

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emu"))

pytestmark = pytest.mark.gpu

POSES = {"A": ((1.5, 1.5, 1.5), 0.0, 0.0), "B": ((1.5, 1.5, 1.5), 0.7, -0.6), "C": ((1.1, 1.1, 1.4), 0.785, -0.3)}


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


def test_gpu_level8_grid_equals_host_grid_and_follows_edits(ort, emu):
    depth = 9
    T = ort.HOctree(21, depth, device=0)
    ort.harness.build_terrain(T, tunnels=True)
    T.sync()
    nodes8, root, _ = T.flatten()
    assert np.array_equal(T.ctx.beam_grid(8), emu.beam_grid(nodes8, root, 8))
    T.set_box(300, 300, 470, 12, 3)
    T.sync()
    nodes8, root, _ = T.flatten()
    g = T.ctx.beam_grid(8)
    assert np.array_equal(g, emu.beam_grid(nodes8, root, 8)), "after the edit"
    assert g[(470 * 256) >> depth, (300 * 256) >> depth, (300 * 256) >> depth] == 0
    T.ctx.close()


def test_bench_frames_refined_equal_unrefined(ort, oc, emu, refine):
    """Depth 12, 3840x2160, poses A/B/C: every ray with the refinement == every ray with level 7 alone; rounds counted on
    the device with the refinement (count_beam = 2) == the host emulation's and fewer than without (count_beam = 1, or a
    forced level); one grid build for both levels."""
    import torch
    depth = 12
    T = ort.HOctree(24, depth, device=0)
    ort.harness.build_terrain(T)
    T.sync()
    ctx = T.ctx
    ctx.set_option("beam_after", 0)
    nodes8, root, _ = T.flatten()
    W, H = 3840, 2160
    fine_host = None
    tot_on = tot_off = 0
    for name, (pos, yaw, pitch) in POSES.items():
        rot, fov = oc.camera_coeffs(yaw, pitch)
        assert ctx.beam_level(pos, rot, fov, W, H) == 7
        ctx.set_option("beam_level", 7)
        off = ctx.trace_frame(pos, rot, fov, W, H)
        ctx.set_option("count_beam", 2)
        n_off = ctx.trace_frame(pos, rot, fov, W, H, want_npush=True)[3]
        ctx.set_option("beam_level", 0)
        ctx.set_option("count_beam", 1)
        assert np.array_equal(ctx.trace_frame(pos, rot, fov, W, H, want_npush=True)[3], n_off), "count_beam 1 counts the level-7 start alone"
        ctx.set_option("count_beam", 2)
        b0 = ctx.beam_builds
        n_on = ctx.trace_frame(pos, rot, fov, W, H, want_npush=True)[3]
        assert ctx.beam_builds - b0 <= 1, "the level-8 grid is built with the launch's grid, as one build"
        ctx.set_option("count_beam", 0)
        on = ctx.trace_frame(pos, rot, fov, W, H)
        assert_same_hits(on, off, f"pose {name}: refined vs level 7 alone")
        tot_on += int(n_on.astype(np.int64).sum()); tot_off += int(n_off.astype(np.int64).sum())
        a, b = ctx.trace_frame_rgba(pos, rot, fov, W, H), None
        ctx.set_option("beam_level", 7)
        b = ctx.trace_frame_rgba(pos, rot, fov, W, H)
        ctx.set_option("beam_level", 0)
        assert np.array_equal(a, b), f"pose {name}: shaded frame"
        if name == "C":
            fine_host = emu.beam_grid(nodes8, root, 8)
            e = refine.trace_frame(nodes8, root, depth, pos, rot, fov, W, H, emu.beam_grid(nodes8, root, 7), fine_host, y0=1024, rows=64, want_npush=True)
            assert np.array_equal(e[3], n_on[1024 * W:(1024 + 64) * W]), "per-ray rounds with the refinement differ from the host emulation's"
    assert tot_on < 0.97 * tot_off, (tot_on, tot_off)

    # batched launch on device buffers: strips of all poses in one launch, refined and not
    def batched():
        outs, jobs = [], []
        for k, (pos, yaw, pitch) in enumerate(POSES.values()):
            rot, fov = oc.camera_coeffs(yaw, pitch)
            rows = 8 * (((H // 8) - k % 2 + 1) // 2)
            n = rows * W
            o = (torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.float32, device="cuda"))
            outs.append(o)
            jobs.append((np.array(pos, np.float32), rot, fov, W, H, 8 * (k % 2), rows, 8, 2, o[0], o[1], o[2]))
        ctx.trace_frames_async(jobs)
        ctx.sync()
        return [(o[0].cpu().numpy().view(np.uint32), o[1].cpu().numpy(), o[2].cpu().numpy()) for o in outs]
    ctx.set_option("beam_level", 7)
    a = batched()
    ctx.set_option("beam_level", 0)
    b = batched()
    for k in range(len(a)):
        assert_same_hits(b[k], a[k], f"batched job {k}")
    ctx.close()
