"""bench.py's output contract, checked on the arm that needs no GPU (--impl reference): exactly one JSON line on
stdout with the keys the driver reads; everything else goes to stderr.  --dump-outputs on both arms (the product's on a GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

DUMP_NAMES = sorted(f"frame{k}_pose{p}_{o}.npy" for k, p in enumerate("ABC") for o in ("voxel", "face", "t"))


def bench(*args, timeout=600):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return out


def check_dump(dump):
    """--dump-outputs: voxel / face / t of the same sampled rays of every pose's frame, float64 / float32, 64 MB at most;
    t of the rays that leave the volume (face 6) written as -1."""
    assert sorted(p.name for p in dump.iterdir()) == DUMP_NAMES
    assert sum(p.stat().st_size for p in dump.iterdir()) <= 64 << 20
    for k, p in enumerate("ABC"):
        v, f, t = (np.load(dump / f"frame{k}_pose{p}_{o}.npy") for o in ("voxel", "face", "t"))
        assert (v.dtype, f.dtype, t.dtype) == (np.float64, np.float32, np.float32) and v.shape == f.shape == t.shape
        assert v.size > 1_000_000 and (v == np.round(v)).all() and set(np.unique(f)) <= set(range(8)) and (v != 0).any()
        assert np.isfinite(t).all() and (f == 6).any() and (t[f == 6] == -1.0).all() and (t[f != 6] >= 0.0).all()


def test_reference_arm_prints_one_json_line(tmp_path):
    dump = tmp_path / "dump"
    out = bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(dump))
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["gpu_launches"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]
    check_dump(dump)


@pytest.mark.gpu
def test_product_arm_dumps_what_the_cpu_trace_computes(tmp_path):
    """The product's timed frames through --dump-outputs, on both launch modes, equal the reference arm's dump of the same
    rays file for file, bit for bit."""
    bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path / "cpu"))
    for launch in ("streams", "batch"):
        out = bench("--quick", "--no-cpu", "--steps", "1", "--launch", launch, "--dump-outputs", str(tmp_path / launch))
        assert json.loads(out.stdout)["quick"] is True
        check_dump(tmp_path / launch)
        for name in DUMP_NAMES:
            assert (tmp_path / launch / name).read_bytes() == (tmp_path / "cpu" / name).read_bytes(), f"{launch}: {name}"


def test_product_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "no CUDA device" in (out.stderr + out.stdout)
    assert not [l for l in out.stdout.splitlines() if l.strip().startswith("{")]
