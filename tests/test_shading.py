"""Shading epilogue (SURVEY 8f-4): voxels.txt parsing and the fused colour lookup of trace_pixel."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, ROOT


def test_parse_voxels_format_and_errors(ort):
    h = ort.harness
    cols, names = h.parse_voxels(h.DEMO_VOXELS)
    assert names == ["Stone", "Grass", "Dark Grass", "Dirt"] and cols.shape == (4, 6)
    assert cols[0, 0] == 0xFF5D4444          # "44445D" -> r=0x44 g=0x44 b=0x5D, alpha 0xFF, packed like olc::Pixel::n
    # the reference's palette (voxels.txt): stored under tests/golden, and live where oracle/_ref is built from its sources
    pal = json.load(open(os.path.join(GOLDEN, "voxels_palette.json")))
    rgb = np.array([[int(c, 16) for c in row] for row in pal["faces_rrggbb"]], np.uint32)
    want = 0xFF000000 | (rgb & 0xFF) << 16 | (rgb & 0xFF00) | (rgb >> 16)       # RRGGBB -> r | g<<8 | b<<16 | a<<24
    assert names == pal["names"] and np.array_equal(cols, want)
    ref_file = os.path.join(ROOT, "oracle", "_ref", "voxels.txt")
    if os.path.exists(ref_file):
        c2, n2 = h.parse_voxels(open(ref_file).read())
        assert n2 == names and np.array_equal(c2, cols)
    for bad in ("Stone: 44445D 4E4E5B", "X: 12345G 000000 000000 000000 000000 000000", ": 000000 000000 000000 000000 000000 000000",
                "ANameThatIsFarTooLongForIt: 000000 000000 000000 000000 000000 000000"):
        with pytest.raises(ValueError):
            h.parse_voxels(bad)
    assert h.parse_voxels("  \n")[0].shape == (0, 6)


@pytest.mark.gpu
def test_rgba_frame_equals_colour_lookup_of_the_hits(ort, golden):
    import torch
    g = golden("d8_tunnels")
    ctx = ort.TraceContext(8)
    ctx.upload_full(g["nodes8"], int(g["root"]))
    cols, _ = ort.harness.parse_voxels(ort.harness.DEMO_VOXELS)
    EXIT, INSIDE = 0xFFFEBF00, 0xFF07193F      # olc::Pixel{0x00,0xBF,0xFE}, {0x3F,0x19,0x07} (test_och_h_octree.cpp:76-77)
    ctx.set_palette(cols, EXIT, INSIDE)
    W, H = 640, 360
    for p in "ABC":
        pos, rot, fov = g[f"pose{p}_pos"], g[f"pose{p}_rot"], float(g[f"pose{p}_fov"])
        v, f, t = ctx.trace_frame(pos, rot, fov, W, H)
        want = np.where(f == 6, np.uint32(EXIT), np.where(f == 7, np.uint32(INSIDE),
                        cols.ravel()[np.minimum(6 * (v.astype(np.int64) - 1) + f, cols.size - 1).clip(0)])).astype(np.uint32)
        got = ctx.trace_frame_rgba(pos, rot, fov, W, H)
        assert np.array_equal(got, want), f"pose {p}"
        part = ctx.trace_frame_rgba(pos, rot, fov, W, H, y0=16, rows=80, tile_rows=8, tile_step=4)
        rows = np.concatenate([np.arange(16 + 32 * k, 24 + 32 * k) for k in range(10)])
        assert np.array_equal(part, want.reshape(H, W)[rows].ravel())
        d = torch.empty(W * H, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        ctx.trace_frame_rgba(pos, rot, fov, W, H, out=d)
        ctx.sync()
        assert np.array_equal(d.cpu().numpy().view(np.uint32), want)
    # inside a solid voxel -> the "inside" colour everywhere; empty tree -> sky everywhere
    got = ctx.trace_frame_rgba(np.array([1.5, 1.5, 1.05], np.float32), g["poseA_rot"], float(g["poseA_fov"]), 64, 36)
    assert (got == INSIDE).all()
    ctx.upload_full(np.zeros((0, 8), np.uint32), 0)
    assert (ctx.trace_frame_rgba(g["poseA_pos"], g["poseA_rot"], float(g["poseA_fov"]), 64, 36) == EXIT).all()


def test_save_png_round_trip(ort, tmp_path):
    """harness.save_png: a valid RGBA PNG whose decoded scanlines are the pixels that went in."""
    import struct
    import zlib
    W, H = 37, 21
    rs = np.random.RandomState(0)
    px = rs.randint(0, 2**32, W * H, dtype=np.uint64).astype(np.uint32)
    path = tmp_path / "f.png"
    ort.harness.save_png(str(path), px, W, H)
    raw = path.read_bytes()
    assert raw[:8] == b"\x89PNG\r\n\x1a\n"
    pos, chunks = 8, {}
    while pos < len(raw):
        n, tag = struct.unpack(">I4s", raw[pos:pos + 8])
        data = raw[pos + 8:pos + 8 + n]
        assert struct.unpack(">I", raw[pos + 8 + n:pos + 12 + n])[0] == zlib.crc32(tag + data) & 0xFFFFFFFF
        chunks[tag] = data
        pos += 12 + n
    assert struct.unpack(">IIBBBBB", chunks[b"IHDR"]) == (W, H, 8, 6, 0, 0, 0)
    rows = np.frombuffer(zlib.decompress(chunks[b"IDAT"]), np.uint8).reshape(H, 1 + 4 * W)
    assert (rows[:, 0] == 0).all()
    assert np.array_equal(rows[:, 1:].reshape(-1).view(np.uint32), px)
