#!/usr/bin/env bash
# Host-side memory safety check (CPU only): builds a copy of the library with the host code under
# AddressSanitizer + UndefinedBehaviorSanitizer (nvcc -Xcompiler -fsanitize=address,undefined) in a scratch
# directory and runs the CPU test-suite's host legs against it -- the node table, the pool octree, the fixture
# builder, the delta stream, the voxels.txt parser, the fuzz scenes and the world-size-2 gloo test.  The device code
# cannot be sanitised here (no GPU; compute-sanitizer is closed on the GPU pool): its per-ray walk is covered by the
# host emulation instead (tests/host_emu), which checks every global load itself and is built with ASan + UBSan here so
# that the walkers' local arrays (parent stacks) are checked as well.
# Usage: tools/sanitize_host.sh [scratch-dir]      exit code 0 = no finding
set -euo pipefail
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
SCRATCH="${1:-/tmp/ort_sanitize}"
rm -rf "$SCRATCH" && mkdir -p "$SCRATCH"
tar -C "$ROOT" --exclude=.git --exclude=gpurun_out --exclude='libort_b200.so' --exclude='__pycache__' --exclude='.pytest_cache' -cf - . | tar -C "$SCRATCH" -xf -
python - "$SCRATCH" <<'PY'
import sys
p = sys.argv[1] + "/octree_ray_tracing_b200/build.py"
s = open(p).read()
old = '"-Xcompiler", "-fPIC,-O2,-ffp-contract=off,-Wall",'
assert old in s
s = s.replace(old, '"-Xcompiler", "-fPIC,-O1,-g,-ffp-contract=off,-Wall,-fsanitize=address,-fsanitize=undefined,-fno-omit-frame-pointer", "-Xlinker", "-lasan", "-Xlinker", "-lubsan",')
open(p, "w").write(s)
PY
cd "$SCRATCH"
python -c "from octree_ray_tracing_b200 import build as b; b.build(force=True)"
# (grep -c, not -q: with pipefail an early exit of grep would make nm's SIGPIPE look like a failure)
[ "$(nm -D octree_ray_tracing_b200/libort_b200.so | grep -c __asan_)" -gt 0 ] || { echo "library is not instrumented"; exit 2; }
export LD_PRELOAD="$(gcc -print-file-name=libasan.so) $(gcc -print-file-name=libubsan.so)"
export ASAN_OPTIONS=detect_leaks=0:halt_on_error=1 UBSAN_OPTIONS=print_stacktrace=1:halt_on_error=0
export ORT_EMU_SANITIZE=1      # the host emulation of the device walkers too: their parent stacks are plain local arrays
python -m pytest tests/test_host_tree.py tests/test_octree.py tests/test_shading.py tests/test_capi_symbols.py \
       tests/test_fuzz_random_dags.py tests/test_multi_gpu_cpu.py tests/test_host_emu.py tests/test_beam.py tests/test_voxel_query.py -q -s -m "not gpu" 2>&1 | tee sanitize.log | tail -3
if grep -q "runtime error\|AddressSanitizer" sanitize.log; then
	grep "runtime error\|AddressSanitizer" sanitize.log | sort | uniq -c | sort -rn | head -20
	exit 1
fi
grep -q " passed" sanitize.log && ! grep -q " failed" sanitize.log
echo "host code: no ASan / UBSan finding"
