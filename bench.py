#!/usr/bin/env python
"""bench.py -- headline benchmark of the h_octree trace path on B200.

Metric (BASELINE.json): Mrays/s on the depth-12 (4096^3) synthetic terrain DAG, 3840x2160 primary rays.
A *step* = one pass over the camera poses A, B, C (SURVEY.md section 6) = 3 frames = 24 883 200 rays per
GPU.  At N GPUs every step holds 3*N frames; each frame is cut into cyclic 8-row tile strips, rank r
tracing tiles r, r+N, ... of every frame with its own replica of the DAG (weak scaling: per-GPU work is
fixed, no data-path collective).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # product (CUDA, libort_b200.so)
    python bench.py --impl reference [...]                         # the reference's own CPU sse_trace
    python bench.py [...] --dump-outputs DIR                       # also write the last timed step's outputs (sampled)

One JSON line on stdout (rank 0).  `value`: device-resident throughput (outputs stay in HBM; L2 is
flushed before every step).  `parity`: the timed frames against the CPU checker, in the same run.
`e2e`: the same frames through the public host-buffer entry point (ort_trace_frame: camera in, voxel/face/t out to
pinned host memory, copies inside the timed region), next to what the host can ingest from all ranks at once.
`roofline`: the bound that binds -- warp-instruction issue -- with the instruction count from the committed ncu
capture (used only if it was taken from the kernel sources this run uses), the SIMT picture measured in-run, and the
memory-side figures (SURVEY.md 8d's byte model as a rate, compulsory and measured HBM / L2 traffic as fractions).
`with_gather` (N > 1): frames assembled on their consumer by the library's NCCL gather.  `cpu_baseline`: the
reference's CPU trace (oracle/_ref when present, else the oracle port) on the host cores, all rays of a step.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DEPTH, LOG2CAP = 12, 24
W, H = 3840, 2160
TILE_ROWS = 8
POSE_NAMES = ("A", "B", "C")
METRIC = "Mrays/s, depth-12 terrain DAG, 3840x2160 primary rays"
WORKLOAD = "h_octree<24,12> simplex terrain (no tunnels), 3840x2160, poses A/B/C per step"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_capture():
    """The committed `ncu --set full` capture of the step's three frame launches (profiles/traffic.json, written by
    tools/ncu_summary.py --traffic) -- but only if it was taken from the kernel sources this run uses: the file carries
    the hash of those sources, and on a mismatch every number that would come from it is reported as null."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        cap = json.load(open(p))
    except Exception:
        return None, "profiles/traffic.json missing"
    from octree_ray_tracing_b200.build import kernel_source_hash
    have, want = cap.get("kernel_source_sha16"), kernel_source_hash()
    if have != want:
        return None, f"profiles/traffic.json is a capture of other kernel sources (sha16 {have}, running {want}): not used"
    if len(cap.get("warp_instructions_per_launch", [])) != len(POSE_NAMES):
        return None, "profiles/traffic.json does not hold the three frame launches of a step"
    return cap, f"profiles/traffic.json (ncu --set full, kernel sources sha16 {want})"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()
        self.active = False

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
            }
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
            while not self._halt.is_set():
                if self.active:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    r = get_reasons(h)
                    for bit, nm in names.items():
                        if r & bit:
                            self.reasons.add(nm)
                time.sleep(0.002)
        except Exception as e:  # NVML missing: report nothing rather than fail the bench
            self.error = repr(e)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ------------------------------------------------------------------------------------------------
# product arm
# ------------------------------------------------------------------------------------------------

def run_product(args):
    import torch
    import torch.distributed as dist
    import octree_ray_tracing_b200 as ort
    from octree_ray_tracing_b200 import harness, multi_gpu

    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if world != args.gpus:
        log(f"note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference for the CPU trace)")
    torch.cuda.set_device(local_rank)
    numa_bound = False
    if world > 1 and not args.no_numa:
        numa_bound = multi_gpu.bind_to_gpu_numa(physical_gpu_index(local_rank))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    # rank 0 owns the host table: it builds the DAG; the library's communicator (ort_mg_*, NCCL inside libort_b200.so)
    # broadcasts the flattened nodes and every rank uploads its replica from the received device buffer.
    t0 = time.time()
    ctx = ort.TraceContext(DEPTH, device=local_rank, node_capacity=1 << 21)
    mg = multi_gpu.MultiGpu(ctx, rank, world) if world > 1 else None
    tree = None
    if rank == 0:
        tree = ort.HOctree(LOG2CAP, DEPTH, device=None)
        harness.build_terrain(tree)
    if mg is not None:
        n_up = mg.broadcast_update(tree.take_delta() if rank == 0 else None)
    else:
        ids, nodes8_up, root_up, _full = tree.take_delta()
        ctx.upload_full(nodes8_up, root_up)
        n_up = ctx.node_count
    ctx.sync()
    if args.variant is not None:
        ctx.set_option("variant", args.variant)
    for kv in args.opt:
        k, v = kv.split("=")
        ctx.set_option(k, int(v))
    log(f"[rank {rank}] DAG built + broadcast + uploaded in {time.time() - t0:.1f}s: {n_up} nodes ({n_up * 32 / 2**20:.1f} MiB)")

    poses = [harness.POSES[p] for p in POSE_NAMES]
    cams = [(np.array(p[0], np.float32),) + ort.camera_coeffs(p[1], p[2]) for p in poses]

    # every rank must hold the same DAG: each traces the same small frames and the digests are compared across ranks
    replica_check = None
    if world > 1:
        dig = []
        for cam in cams:
            v, f, t = ctx.trace_frame(cam[0], cam[1], cam[2], 480, 270)
            dig += [int(v.astype(np.uint64).sum()), int(f.astype(np.uint64).sum()), int(t.view(np.uint32).astype(np.uint64).sum() & 0x7FFFFFFFFFFFFFFF), int((v != 0).sum())]
        mine = torch.tensor(dig, dtype=torch.int64, device="cuda")
        lo, hi = mine.clone(), mine.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        if not torch.equal(lo, hi) or dig[3] < 1000:
            raise SystemExit(f"[rank {rank}] replica check FAILED: the ranks do not trace the same DAG (digests {dig[:4]} vs min {lo[:4].tolist()} max {hi[:4].tolist()})")
        replica_check = f"ok: {len(dig)} digests of 3 traced 480x270 frames equal on all {world} ranks"
    # partition rank / world: the process's own, or (--as-rank r/n, a one-GPU measurement aid for --quick) the share
    # rank r of an n-GPU job would trace -- same strips, same frames per step, same number of streams
    prank, pworld = rank, world
    if args.as_rank:
        if world != 1 or not args.quick:
            raise SystemExit("bench.py: --as-rank is a single-GPU measurement aid and needs --quick")
        prank, pworld = (int(x) for x in args.as_rank.split("/"))
    y0, rows, frame_rows = multi_gpu.strip_rows(prank, pworld, H, TILE_ROWS)
    n_local = rows * W
    frames_per_step = len(cams) * pworld
    rays_per_step_total = frames_per_step * W * H          # all ranks together
    rays_per_step_local = frames_per_step * n_local

    own = torch.cuda.ExternalStream(ctx.stream, device=local_rank)
    # frames in flight: small strips need more of them to hide launch tails, but too many concurrent launches dilute
    # the L1 locality of each (measured in round 1: 2 GPUs 3/4/6 streams -> 28.2/28.2/26.5, 4 GPUs 4/6/8 -> 54.0/52.1/53.2, 8 GPUs 5/8/12 -> 101.8/104.5/102.3 Grays/s)
    NS = args.streams or (3 if pworld == 1 else (4 if pworld <= 4 else 8))
    streams = [torch.cuda.Stream(device=local_rank) for _ in range(NS)]
    outs = [(torch.empty(n_local, dtype=torch.int32, device="cuda"), torch.empty(n_local, dtype=torch.uint8, device="cuda"),
             torch.empty(n_local, dtype=torch.float32, device="cuda")) for _ in range(NS)]
    dv, df, dt = outs[0]
    dn = torch.empty(n_local, dtype=torch.int16, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def frame(cam, out=outs[0], npush=None):
        ctx.trace_frame_async(cam[0], cam[1], cam[2], W, H, y0, rows, TILE_ROWS, pworld, out[0], out[1], out[2], npush)

    # a DAG version gets its beam grid at the third frame call that meets it (ort_set_option "beam_after"): three throw-away
    # frames, so that the counting passes below see the kernels the timed loop runs
    with torch.cuda.stream(own):
        for cam in cams:
            frame(cam)
        own.synchronize()

    # algorithmic bytes: PUSH counts from an (untimed) counting pass -- identical to the oracle's counts (tests).  The same
    # pass yields the SIMT picture of the round loop: a warp (8 x 4 pixel tile) runs as many rounds as its longest ray.
    pushes = 0
    hits = 0
    warp_rounds = 0
    with torch.cuda.stream(own):
        for cam in cams:
            frame(cam, outs[0], dn)
            own.synchronize()
            cnt = (dn.to(torch.int32) & 0xFFFF).view(rows, W)
            pushes += int(cnt.sum().item())
            hits += int((dv != 0).sum().item())
            if rows % 4 == 0 and W % 8 == 0:
                warp_rounds += int(cnt.view(rows // 4, 4, W // 8, 8).amax(dim=(1, 3)).sum().item())
    # the rounds the timed kernels actually run: with the beam start (csrc/ort_beam.cuh) most rays re-enter their walk at the
    # tile's lower bound, or end as a MISS at once -- counted by the same kind of pass with option count_beam
    pushes_run, warp_rounds_run = pushes, warp_rounds
    beam_levels = [ctx.beam_level(cam[0], cam[1], cam[2], W, H) for cam in cams]
    if any(beam_levels):
        ctx.set_option("count_beam", 1)
        pushes_run = warp_rounds_run = 0
        with torch.cuda.stream(own):
            for cam in cams:
                frame(cam, outs[0], dn)
                own.synchronize()
                cnt = (dn.to(torch.int32) & 0xFFFF).view(rows, W)
                pushes_run += int(cnt.sum().item())
                if rows % 4 == 0 and W % 8 == 0:
                    warp_rounds_run += int(cnt.view(rows // 4, 4, W // 8, 8).amax(dim=(1, 3)).sum().item())
        ctx.set_option("count_beam", 0)
    pushes_per_step_local = pushes * pworld
    bytes_per_step_local = 32 * pushes_per_step_local + 9 * rays_per_step_local
    step_cams = [cam for _rep in range(pworld) for cam in cams]

    if args.launch == "auto":
        args.launch = "streams"       # measured: 1 GPU 14.8 (streams) vs 14.6 (batch); 8 GPUs 105 vs 92 Grays/s (DESIGN.md section 9)
    # one output set per frame of the step for the batched launch (ort_trace_frames_async: the whole step in one launch)
    batch_outs = [(torch.empty(n_local, dtype=torch.int32, device="cuda"), torch.empty(n_local, dtype=torch.uint8, device="cuda"),
                   torch.empty(n_local, dtype=torch.float32, device="cuda")) for _ in range(frames_per_step)] if args.launch == "batch" else []
    batch_jobs = [(cam[0], cam[1], cam[2], W, H, y0, rows, TILE_ROWS, pworld, o[0], o[1], o[2]) for cam, o in zip(step_cams, batch_outs)]

    def timed_steps_batched(steps, do_flush):
        """One timed interval per STEP, the step's frames in one batched launch on one stream."""
        evs = []
        s0 = streams[0]
        ctx.set_stream(s0)
        for _ in range(steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(s0):
                if do_flush:
                    flush.zero_()
                a.record(s0)
            ctx.trace_frames_async(batch_jobs)
            b.record(s0)
            evs.append((a, b))
        ctx.set_stream(None)
        return evs

    def timed_steps(steps, do_flush):
        if args.launch == "batch":
            return timed_steps_batched(steps, do_flush)
        return timed_steps_streams(steps, do_flush)

    def timed_steps_streams(steps, do_flush):
        """One timed interval per STEP: L2 flushed before it (outside the interval), then the step's frames are
        queued round-robin on NS streams so that the latency tail of one launch overlaps the next launch."""
        evs = []
        s0 = streams[0]
        for _ in range(steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(s0):
                if do_flush:
                    flush.zero_()
                a.record(s0)
            for st in streams[1:]:
                st.wait_event(a)
            for k, cam in enumerate(step_cams):
                ctx.set_stream(streams[k % NS])
                frame(cam, outs[k % NS])
            for st in streams[1:]:
                e = torch.cuda.Event()
                e.record(st)
                s0.wait_event(e)
            b.record(s0)
            evs.append((a, b))
        ctx.set_stream(None)
        return evs

    def serial_launches(steps, do_flush):
        """Reference measurement: one stream, one timed interval per LAUNCH (no overlap between launches)."""
        evs = []
        with torch.cuda.stream(own):
            for _ in range(steps):
                for cam in step_cams:
                    if do_flush:
                        flush.zero_()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(own)
                    frame(cam)
                    b.record(own)
                    evs.append((a, b))
        return evs

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure_gather():
        # Frames assembled on their consumer (ort_mg_trace_frame_gather: strips traced into a ring of slots, ONE NCCL message
        # per rank and frame on the communicator's stream, unpacked at their final rows on the consumer).  Two consumer
        # layouts: round robin (frame k of the step is consumed on rank k mod N -- the weak-scaling shape: N times the frames,
        # N consumers) and everything on rank 0 (one consumer for N times the frames: bound by one GPU's NVLink ingest).
        gather = {}
        if mg is not None:
            fv = torch.empty(W * H, dtype=torch.int32, device="cuda")
            ff = torch.empty(W * H, dtype=torch.uint8, device="cuda")
            ft = torch.empty(W * H, dtype=torch.float32, device="cuda")

            def jobs_of(mode):
                js = []
                for k, cam in enumerate(step_cams):
                    dst = k % world if mode == "round_robin" else 0
                    mine = dst == rank
                    js.append((cam[0], cam[1], cam[2], W, H, TILE_ROWS, dst, fv if mine else None, ff if mine else None, ft if mine else None))
                return mg.make_jobs(js)
            step_jobs = {mode: jobs_of(mode) for mode in ("round_robin", "rank0")}

            def gather_step(mode):
                mg.trace_frames_gather(step_jobs[mode])         # the step's frames in one call (ort_mg_trace_frames_gather)

            g_steps = max(1, min(args.steps, 10))
            # (consumers, frames per wire operation): per-frame messages, and the whole step's strips as one NCCL group
            # frames per wire operation of the headline leg: a whole step up to 12 frames, half-steps of 12 beyond (8 GPUs, 24 frames
            # per step: one operation per step 122, per 12 frames 139, per 8 frames 121 Grays/s; profiles/r2_n8_gather_legs.json)
            G = min(len(step_cams), 12)
            for mode, grp, tr in (("round_robin", 1, 1), ("round_robin", G, 1), ("rank0", G, 1), ("round_robin", G, 0), ("round_robin", len(step_cams), 1)):
                mg.set_transport(tr)
                mg.set_group(grp)
                gather_step(mode)
                mg.sync()
                barrier()
                w0 = mg.wire_bytes
                g0 = time.perf_counter()
                for _ in range(g_steps):
                    gather_step(mode)
                mg.sync()
                barrier()
                if tr == 1:
                    gather["transport"] = mg.transport
                gather[(mode, grp) if tr == 1 else (mode + "_nccl_sendrecv", grp)] = ((time.perf_counter() - g0) / g_steps, (mg.wire_bytes - w0) / g_steps)
            # measurement aid: extra legs "mode:group:transport:trace_streams,..." from ORT_BENCH_GATHER_LEGS (quick mode prints them)
            for leg in filter(None, os.environ.get("ORT_BENCH_GATHER_LEGS", "").split(",")):
                mode, grp, tr, ts = leg.split(":")
                mg.set_transport(int(tr)); mg.set_group(int(grp)); mg.set_trace_streams(int(ts))
                gather_step(mode); mg.sync(); barrier()
                g0 = time.perf_counter()
                for _ in range(g_steps):
                    gather_step(mode)
                mg.sync(); barrier()
                gather[(f"extra_{mode}_t{tr}_s{ts}", int(grp))] = ((time.perf_counter() - g0) / g_steps, 0.0)
            if os.environ.get("ORT_BENCH_GATHER_LEGS"):
                mg.set_trace_streams(8 if world > 4 else 4)
            mg.set_transport(1)
            mg.set_group(1)
            # one frame at a time, nothing in flight: the latency of "trace my strips + gather" for a single frame
            lat = []
            for cam in cams[:1]:                    # (untimed: the settings above rebuild the rings at the next frame)
                mg.trace_frame_gather(cam[0], cam[1], cam[2], W, H, tile_rows=TILE_ROWS, dst=0, d_vox=fv if rank == 0 else None, d_face=ff if rank == 0 else None, d_t=ft if rank == 0 else None)
                mg.sync()
            for cam in cams:
                barrier()
                g0 = time.perf_counter()
                mg.trace_frame_gather(cam[0], cam[1], cam[2], W, H, tile_rows=TILE_ROWS, dst=0, d_vox=fv if rank == 0 else None, d_face=ff if rank == 0 else None, d_t=ft if rank == 0 else None)
                mg.sync()
                barrier()
                lat.append(time.perf_counter() - g0)
            gather["latency"] = lat
            # the last assembled frame (pose C, consumer rank 0) against the single-GPU trace of the same frame on rank 0
            if rank == 0:
                full = (torch.empty(W * H, dtype=torch.int32, device="cuda"), torch.empty(W * H, dtype=torch.uint8, device="cuda"), torch.empty(W * H, dtype=torch.float32, device="cuda"))
                cam = cams[-1]
                ctx.trace_frame_async(cam[0], cam[1], cam[2], W, H, 0, H, 1, 1, full[0], full[1], full[2], None)
                ctx.sync()
                gather["assembled_equals_single_gpu"] = bool(torch.equal(full[0], fv) and torch.equal(full[1], ff) and torch.equal(full[2].view(torch.int32), ft.view(torch.int32)))

        return gather

    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()

    sampler.active = True          # warm-up, timed loops and e2e are all load
    timed_steps(args.warmup, True)
    barrier()
    launches0 = ctx.launch_count
    wall0 = time.perf_counter()
    evs = timed_steps(args.steps, True)
    host_enqueue_s = time.perf_counter() - wall0          # the host's share: queueing the steps' launches, nothing waited for
    barrier()
    wall = time.perf_counter() - wall0
    launches = ctx.launch_count - launches0
    kernel_ms = sum(a.elapsed_time(b) for a, b in evs)

    # Parity of the TIMED frames: the output buffers still hold the last frames the timed loop wrote -- buffer j the frame
    # k = the largest index with k % NS == j, i.e. pose k % 3 of the step.  Every 8th row of each (this rank's strip rows)
    # goes to the CPU checker: the reference's own sse_trace (oracle/_ref) where it travelled, else the oracle port.
    parity = None
    if args.launch == "streams" and not args.no_cpu:
        parity = parity_of_timed_frames(ort, tree, n_up, ctx, mg, world, rank, outs, NS, len(step_cams), cams, frame_rows, torch, dist)
    if args.dump_outputs and rank == 0:
        # the timed loop's output buffers still hold the last step: every frame with the batched launch, else frame k of the
        # step in buffer k % NS for the last k of each residue (with N > 1, this rank's strip rows of those frames)
        n_step = len(step_cams)
        held = list(enumerate(batch_outs)) if args.launch == "batch" else \
            [(max(k for k in range(n_step) if k % NS == j), outs[j]) for j in range(min(NS, n_step))]

        def take(buf):
            def rows(idx):
                sel = torch.from_numpy(idx).cuda()
                return buf[0][sel].cpu().numpy().view(np.uint32), buf[1][sel].cpu().numpy(), buf[2][sel].cpu().numpy()
            return rows
        dump_outputs(args.dump_outputs, [(f"frame{k}_pose{POSE_NAMES[k % len(cams)]}", take(buf)) for k, buf in held], n_local)

    # per-launch view of the same work: serialised launches, each timed alone
    serial_launches(1, True)
    barrier()
    evs_s = serial_launches(args.steps, True)
    barrier()
    serial_per_launch = [a.elapsed_time(b) for a, b in evs_s]
    serial_ms = sum(serial_per_launch)

    if args.quick:
        sampler.stop()
        ms = kernel_ms / args.steps
        gq = None
        if world > 1:
            g = measure_gather()
            keys = sorted(k for k in g if isinstance(k, tuple))
            tq = torch.tensor([ms, serial_ms] + [g[k][0] for k in keys] + [max(g["latency"])], dtype=torch.float64, device="cuda")
            dist.all_reduce(tq, op=dist.ReduceOp.MAX)
            ms, serial_ms = float(tq[0]), float(tq[1])
            gq = {f"{k[0]}_group{k[1]}_Mrays/s": round(rays_per_step_total / float(tq[2 + i]) / 1e6, 1) for i, k in enumerate(keys)}
            gq["single_frame_latency_ms"] = round(float(tq[-1]) * 1e3, 3)
            gq["assembled_equals_single_gpu"] = g.get("assembled_equals_single_gpu")
            mg.close()
            dist.barrier()
            dist.destroy_process_group()
        if rank != 0:
            return None
        emit({"quick": True, "value": round(rays_per_step_total / (ms * 1e-3) / 1e6, 2), "unit": "Mrays/s", "ms_per_step": round(ms, 4),
                          "serial_value": round(rays_per_step_total / (serial_ms / args.steps * 1e-3) / 1e6, 2),
                          "pushes_per_ray": round(pushes_per_step_local / rays_per_step_local, 3),
                          "rounds_run_per_ray": round(pushes_run / (len(cams) * n_local), 3), "beam_levels": beam_levels, "launches": launches,
                          "host_enqueue_ms_per_step": round(host_enqueue_s / args.steps * 1e3, 4), "band_schedules": ctx.band_schedules,
                          "per_frame_ms_serial": [round(x, 4) for x in serial_per_launch[-len(step_cams):]],
                          "tile_rows": TILE_ROWS, "streams": NS, "parity": parity, "gather": gq,
                          "as_rank": (f"{prank}/{pworld}: value = what {pworld} GPUs would total if every rank ran like this one" if args.as_rank else None)})
        return None

    # same loop without the flush (steady state of a real frame loop: DAG stays L2-resident)
    timed_steps(1, False)
    barrier()
    evs_w = timed_steps(args.steps, False)
    barrier()
    warm_ms = sum(a.elapsed_time(b) for a, b in evs_w)

    # end to end through the host-buffer entry point: pinned outputs, D2H inside the timed region.  One set of host
    # buffers per frame of the step; the calls are enqueued with deferred completion (ort_set_option defer_sync) and
    # the step ends with ort_sync(), so frame k+1 is traced while frame k's 9 B/ray are still crossing PCIe.
    n_host = min(len(step_cams), 3)
    houts = []
    for _ in range(n_host):
        hv = torch.empty(n_local, dtype=torch.int32).pin_memory()
        hf = torch.empty(n_local, dtype=torch.uint8).pin_memory()
        ht = torch.empty(n_local, dtype=torch.float32).pin_memory()
        houts.append((hv.numpy().view(np.uint32), hf.numpy(), ht.numpy(), None))

    def e2e_step():
        ctx.set_option("defer_sync", 1)
        for k, cam in enumerate(step_cams):
            ctx.trace_frame(cam[0], cam[1], cam[2], W, H, y0=y0, rows=rows, tile_rows=TILE_ROWS, tile_step=world, out=houts[k % n_host])
        ctx.sync()
        ctx.set_option("defer_sync", 0)

    for _ in range(max(1, min(args.warmup, 3))):
        e2e_step()
    barrier()
    e0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 10))
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - e0
    e2e_check = int((houts[(len(step_cams) - 1) % n_host][0] != 0).sum())
    # measurement aid: the same with other numbers of launches per host-buffer frame (ORT_BENCH_E2E_CHUNKS="1,2,4")
    e2e_chunk_legs = {}
    for nck in filter(None, os.environ.get("ORT_BENCH_E2E_CHUNKS", "").split(",")):
        ctx.set_option("frame_chunks", int(nck))
        e2e_step()
        barrier()
        c0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        barrier()
        sec = time.perf_counter() - c0
        if world > 1:
            tsec = torch.tensor([sec], dtype=torch.float64, device="cuda")
            dist.all_reduce(tsec, op=dist.ReduceOp.MAX)
            sec = float(tsec.item())
        e2e_chunk_legs[f"frame_chunks={nck}"] = round(rays_per_step_total * e2e_steps / sec / 1e6, 2)
    ctx.set_option("frame_chunks", 0)

    # the same, one synchronous call per frame (each call returns with its results on the host)
    def e2e_sync_step():
        for k, cam in enumerate(step_cams):
            ctx.trace_frame(cam[0], cam[1], cam[2], W, H, y0=y0, rows=rows, tile_rows=TILE_ROWS, tile_step=world, out=houts[k % n_host])
    e2e_sync_step()
    barrier()
    e0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_sync_step()
    barrier()
    e2e_sync_s = time.perf_counter() - e0

    # What the host can take from all GPUs of the box AT ONCE: every rank copies a 256 MiB device buffer to pinned host
    # memory, all ranks together, timed on the device.  The e2e figure cannot exceed (sum over ranks) / 9 B per ray.
    probe_d = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    probe_h = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
    probe_h.copy_(probe_d, non_blocking=True)
    barrier()
    pa, pb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pa.record()
    for _ in range(4):
        probe_h.copy_(probe_d, non_blocking=True)
    pb.record()
    barrier()
    d2h_gbs_local = 4 * (256 << 20) / (pa.elapsed_time(pb) * 1e-3) / 1e9
    del probe_d, probe_h

    gather = measure_gather()

    # shaded frames (the pixels update_image draws): 4 B per ray cross PCIe instead of 9
    cols, _ = harness.parse_voxels(harness.DEMO_VOXELS)
    ctx.set_palette(cols)
    hrgba = [torch.empty(n_local, dtype=torch.int32).pin_memory() for _ in range(n_host)]

    def rgba_step():
        ctx.set_option("defer_sync", 1)
        for k, cam in enumerate(step_cams):
            ctx.trace_frame_rgba(cam[0], cam[1], cam[2], W, H, y0=y0, rows=rows, tile_rows=TILE_ROWS, tile_step=world, out=hrgba[k % n_host])
        ctx.sync()
        ctx.set_option("defer_sync", 0)
    rgba_step()
    barrier()
    r0 = time.perf_counter()
    for _ in range(e2e_steps):
        rgba_step()
    barrier()
    rgba_s = time.perf_counter() - r0

    clocks = sampler.stop()
    # memory-side ceilings measured on this GPU: random 32-B sector gathers over a buffer of the DAG's size (L2-resident)
    # and over 4 GiB (HBM-resident)
    gather_l2 = ctx.measure_gather_peak(int(n_up) * 32) if rank == 0 else 0.0
    gather_hbm = ctx.measure_gather_peak(4 << 30) if rank == 0 else 0.0

    # max over ranks
    n_step_frames = len(step_cams)
    G = min(n_step_frames, 12)
    g_rr, g_r0 = gather.get(("round_robin", G), (0.0, 0.0)), gather.get(("rank0", G), (0.0, 0.0))
    g_rr1 = gather.get(("round_robin", 1), (0.0, 0.0))
    g_rrn = gather.get(("round_robin_nccl_sendrecv", G), (0.0, 0.0))
    g_rrw = gather.get(("round_robin", n_step_frames), (0.0, 0.0))
    g_lat = max(gather.get("latency", [0.0]))
    d2h_sum = d2h_gbs_local
    if world > 1:
        tt = torch.tensor([kernel_ms, warm_ms, e2e_s, wall, g_rr[0], g_r0[0], g_lat, rgba_s, e2e_sync_s, serial_ms, g_rr1[0], g_rrn[0], g_rrw[0]], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        kernel_ms, warm_ms, e2e_s, wall, g_rr_s, g_r0_s, g_lat, rgba_s, e2e_sync_s, serial_ms, g_rr1_s, g_rrn_s, g_rrw_s = (float(x) for x in tt.tolist())
        cnt = torch.tensor([launches, bytes_per_step_local, pushes_per_step_local, d2h_gbs_local, g_rr[1], g_r0[1]], dtype=torch.float64, device="cuda")
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        launches_all = int(cnt[0].item())
        pushes_per_ray_all = float(cnt[2].item()) / rays_per_step_total
        d2h_sum = float(cnt[3].item())
        wire_rr, wire_r0 = float(cnt[4].item()) / 2, float(cnt[5].item()) / 2           # every message is counted by its sender and its receiver
        wmax = torch.tensor([g_r0[1]], dtype=torch.float64, device="cuda")
        dist.all_reduce(wmax, op=dist.ReduceOp.MAX)
        ingest_r0 = float(wmax.item())                                                  # the consumer's share (rank 0 receives everything)
    else:
        launches_all = launches
        pushes_per_ray_all = pushes_per_step_local / rays_per_step_local
        g_rr_s = g_r0_s = g_rr1_s = g_rrn_s = g_rrw_s = 0.0
        wire_rr = wire_r0 = ingest_r0 = 0.0

    result = None
    if rank == 0:
        peak, peak_src = measured_peak()
        ms_per_step = kernel_ms / args.steps
        value_trace = rays_per_step_total / (ms_per_step * 1e-3) / 1e6
        n_launch_local = args.steps * frames_per_step
        avg_launch_s = kernel_ms * 1e-3 / n_launch_local      # effective: launches of a step overlap
        algorithmic_rate = (bytes_per_step_local / frames_per_step) / avg_launch_s / 1e9
        e2e_val = rays_per_step_total * e2e_steps / e2e_s / 1e6
        cap, cap_src = ncu_capture()
        sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
        mhz = (clocks or {}).get("sm_mhz")
        issue_peak = sms * 4 * mhz * 1e6 if mhz else None
        inst_per_step = int(sum(cap["warp_instructions_per_launch"]) + sum(cap.get("march_warp_instructions_per_launch", []))) if cap else None   # one GPU's share of a step = 3 full frames' worth (+ their marches)
        issue_achieved = inst_per_step / (ms_per_step * 1e-3) if inst_per_step else None
        # compulsory HBM traffic of a launch: every output byte once + the DAG once (it does not fit L1, it does fit L2)
        compulsory = 9 * n_local + int(n_up) * 32
        roofline = {
            "bound": "issue",
            "achieved": round(issue_achieved / 1e9, 1) if issue_achieved else None,
            "peak": round(issue_peak / 1e9, 1) if issue_peak else None,
            "unit": "G warp-instr/s",
            "frac": round(issue_achieved / issue_peak, 4) if issue_achieved and issue_peak else None,
            "traffic": cap["dram_bytes_per_launch"] if cap else None,
            "kernel": ("ort::trace_frame_kernel<13,false,true> (LeanWalker tiers, beam start) + ort::beam_start_kernel" if any(beam_levels) else
                       "ort::trace_frame_kernel<13,false,false> (LeanWalker tiers)") if args.variant in (None, 13) else f"variant {args.variant}",
            "peak_source": f"{sms} SMs x 4 schedulers x {mhz} MHz (SM clock sampled through NVML during the timed region)",
            "warp_instructions_per_step_per_gpu": inst_per_step,
            "counters_source": cap_src,
            "avg_launch_ms": round(avg_launch_s * 1e3, 4),
            "why_issue": "the DAG is cache resident (ncu: L1 hit ~90 %, DRAM traffic ~1 % of the algorithmic bytes, DRAM and L2 throughput a few % of peak) and every scheduler has ~6 eligible "
                         "warps per cycle: the kernel is bound by warp-instruction issue, so that is the roofline it is held against; the memory-side figures are listed under `memory`",
            "simt": {"lane_rounds_per_ray": round(pushes_run / (len(cams) * n_local), 3),
                     "warp_rounds_per_warp": round(warp_rounds_run / (len(cams) * n_local / 32), 3) if warp_rounds_run else None,
                     "lanes_busy_per_warp_round": round(pushes_run / warp_rounds_run, 2) if warp_rounds_run else None,
                     "reference_walk": {"lane_rounds_per_ray": round(pushes / (len(cams) * n_local), 3),
                                        "warp_rounds_per_warp": round(warp_rounds / (len(cams) * n_local / 32), 3) if warp_rounds else None},
                     "active_threads_per_warp_instruction_ncu": cap.get("active_threads_per_warp_instruction") if cap else None,
                     "note": "measured in this run from per-ray round counts (untimed counting passes, with and without the beam start): a warp = an 8x4 pixel tile runs as many rounds as its longest ray"},
            "memory": {
                "algorithmic_bytes_per_launch": int(bytes_per_step_local / frames_per_step),
                "algorithmic_rate_gbs": round(algorithmic_rate, 1),
                "algorithmic_note": "SURVEY 8d's byte model: 32 B per child-slot load (PUSH) + 9 B of output per ray, over the measured launch time.  ~90 % of those loads are L1 hits, "
                                    "so this rate is NOT bytes that left the SM and is not a fraction of anything",
                "hbm_peak_gbs": peak, "hbm_peak_source": peak_src,
                "compulsory_bytes_per_launch": compulsory,
                "compulsory_hbm_frac": round(compulsory / avg_launch_s / 1e9 / peak, 4),
                "dram_bytes_per_launch_ncu": cap["dram_bytes_per_launch"] if cap else None,
                "dram_hbm_frac_ncu": round(cap["dram_bytes_per_launch"] / avg_launch_s / 1e9 / peak, 4) if cap else None,
                "l2_bytes_per_launch_ncu": int(np.mean(cap["l2_sectors_per_launch"]) * 32) if cap and cap.get("l2_sectors_per_launch") else None,
                "l2_sector_gather_peak_gbs": round(gather_l2, 1), "hbm_sector_gather_peak_gbs": round(gather_hbm, 1),
                "l2_gather_frac_ncu": round(float(np.mean(cap["l2_sectors_per_launch"])) * 32 / avg_launch_s / 1e9 / gather_l2, 4) if cap and cap.get("l2_sectors_per_launch") and gather_l2 else None,
                "how": "ort_measure_gather_peak: independent random 4-B loads, one 32-B sector each, over a buffer of the DAG's size (L2-resident) / 4 GiB (HBM-resident); "
                       "ncu figures from the capture named in counters_source",
            },
        }
        # N > 1: the headline is the throughput WITH the gather (frames assembled on their consumers inside the library);
        # the trace-only figure stands beside it (no_gather).  N = 1 assembles nothing: the frame is already whole.
        value = rays_per_step_total / g_rr_s / 1e6 if mg is not None else value_trace
        result = {
            "metric": METRIC, "value": round(value, 2), "unit": "Mrays/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round((g_rr_s * 1e3) if mg is not None else ms_per_step, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32+u32", "data": "synthetic",
            "config": {
                "workload": WORKLOAD, "frames_per_step": frames_per_step, "rays_per_step": rays_per_step_total,
                "partition": f"cyclic {TILE_ROWS}-row tile strips over {world} GPU(s), DAG replicated",
                "replica_check": replica_check,
                "host_placement": "rank pinned to its GPU's NUMA node (NVML ideal CPUs)" if numa_bound else "default",
                "l2": "flushed before every step (256 MiB memset outside the timed interval)",
                "in_flight": ("one batched launch per step (ort_trace_frames_async): the frames' blocks stream through the SMs back to back"
                              if args.launch == "batch" else f"{NS} streams: the frames of a step are queued round-robin so launch tails overlap"),
                "dag_nodes": int(n_up), "dag_mib": round(n_up * 32 / 2**20, 1),
                "pushes_per_ray": round(pushes_per_ray_all, 3),
                "beam_start": {"grid_level_per_pose": beam_levels, "rounds_run_per_ray": round(pushes_run / (len(cams) * n_local), 3),
                               "note": "pushes_per_ray counts the reference walk (och_h_octree.h:344 executions, what the byte model of SURVEY 8d is stated in); the kernels "
                                       "start every 8x4 tile at a proven lower bound of its rays' hit times (csrc/ort_beam.cuh) and run rounds_run_per_ray -- same outputs, see parity"},
                "hit_fraction": round(hits / (len(cams) * n_local), 4),
                "timing": ("value: wall clock over whole steps of trace + gather (ort_mg_trace_frames_gather ... ort_mg_sync), barrier + synchronize on both sides, max over ranks; "
                           "no_gather / roofline: sum of CUDA-event intervals around each step, max over ranks" if mg is not None else
                           "sum of CUDA-event intervals around each step (start after the flush, end after all streams joined), max over ranks"),
            },
            "parity": parity,
            "serial": {"value": round(rays_per_step_total / (serial_ms / args.steps * 1e-3) / 1e6, 2), "unit": "Mrays/s",
                       "note": "same frames on ONE stream, one event interval per launch, L2 flushed before every launch",
                       "per_launch_ms": [round(x, 4) for x in serial_per_launch[-len(step_cams):]]},
            "warm_l2": {"value": round(rays_per_step_total / (warm_ms / args.steps * 1e-3) / 1e6, 2), "unit": "Mrays/s",
                        "note": "same loop without the L2 flush (DAG stays L2-resident between steps)"},
            "e2e": {"value": round(e2e_val, 2), "unit": "Mrays/s", "h2d_bytes_per_step": frames_per_step * 52,
                    "d2h_bytes_per_step": frames_per_step * n_local * 9, "steps": e2e_steps,
                    "api": "ort_trace_frame, pinned host outputs (voxel u32 + face u8 + t f32), option defer_sync: the step's frames are "
                           "enqueued back to back and ort_sync() ends the step; chunk kernels on 3 streams, D2H on the copy engine",
                    "per_call_sync": {"value": round(rays_per_step_total * e2e_steps / e2e_sync_s / 1e6, 2), "unit": "Mrays/s",
                                      "note": "same frames, every ort_trace_frame call returns with its results on the host"},
                    "host_ingest_peak_gbs": round(d2h_sum, 1),
                    "host_ingest_note": f"measured in this run: all {world} rank(s) copy 256 MiB device -> pinned host at the same time (sum over ranks); "
                                        f"at 9 B per ray this caps e2e at {d2h_sum / 9 * 1e3:.0f} Mrays/s on this box",
                    "frac_of_host_ingest": round(e2e_val * 9 / 1e3 / d2h_sum, 4) if d2h_sum else None,
                    "hits_last_frame": e2e_check, **({"chunk_legs_Mrays/s": e2e_chunk_legs} if e2e_chunk_legs else {})},
            "e2e_rgba": {"value": round(rays_per_step_total * e2e_steps / rgba_s / 1e6, 2), "unit": "Mrays/s",
                         "d2h_bytes_per_step": frames_per_step * n_local * 4,
                         "api": "ort_trace_frame_rgba: trace_pixel's colour lookup fused into the kernel, one uint32 pixel per ray to pinned host memory"},
            "gpu_launches": launches_all,
            "roofline": roofline,
            "clocks": clocks,
            "wall_s_timed_region": round(wall, 3),
        }
        if mg is not None:
            result["with_gather"] = {
                "value": round(rays_per_step_total / g_rr_s / 1e6, 2), "unit": "Mrays/s",
                "frac_of_no_gather": round(rays_per_step_total / g_rr_s / 1e6 / value_trace, 4),
                "consumers": "round robin: frame k of the step is assembled on rank k mod N (N times the frames, N consumers)",
                "wire": f"ort_mg_set_group({G}): the strips of {G} of a step's {n_step_frames} frames leave in ONE wire operation that overlaps the traces of the next frames",
                "wire_bytes_per_step": int(wire_rr), "wire_gbs_aggregate": round(wire_rr / g_rr_s / 1e9, 1),
                "transport": ("peer copies: every strip block moves with one cudaMemcpyAsync on the copy engines into the consumer's staging area (CUDA IPC mapping), one 4-byte ncclAllReduce per wire operation orders it"
                              if gather.get("transport") == 1 else "NCCL ncclSend / ncclRecv (CUDA IPC not available between the ranks)"),
                "nccl_sendrecv_transport": {"value": round(rays_per_step_total / g_rrn_s / 1e6, 2), "unit": "Mrays/s",
                                            "note": "the same exchange with ort_mg_set_transport(0): NCCL's copy kernels share the SMs with the issue-bound trace kernels"},
                "whole_step_per_operation": {"value": round(rays_per_step_total / g_rrw_s / 1e6, 2), "unit": "Mrays/s",
                                             "note": f"ort_mg_set_group({n_step_frames}): all strips of a step in one wire operation (the same leg as the headline up to 12 frames per step)"},
                "per_frame_messages": {"value": round(rays_per_step_total / g_rr1_s / 1e6, 2), "unit": "Mrays/s",
                                       "note": "ort_mg_set_group(1): every frame's strips leave as soon as they are traced (one wire operation per frame)"},
                "api": "ort_mg_trace_frame_gather (inside libort_b200.so): strips traced into a ring of blocks on 4-8 trace streams, moved on the communicator's "
                       "stream, one unpack kernel per frame writes final rows on the consumer; wall clock over whole steps, max over ranks",
                "rank0_only": {"value": round(rays_per_step_total / g_r0_s / 1e6, 2), "unit": "Mrays/s",
                               "note": "every frame assembled on rank 0: one GPU's NVLink ingest carries (N-1)/N of ALL frames",
                               "rank0_ingest_bytes_per_step": int(ingest_r0), "rank0_ingest_gbs": round(ingest_r0 / g_r0_s / 1e9, 1)},
                "strong_scaling_single_frame": {"latency_ms": round(g_lat * 1e3, 3), "value": round(W * H / g_lat / 1e6, 2), "unit": "Mrays/s",
                                                "note": "ONE 4K frame traced by N GPUs and assembled on rank 0, nothing else in flight (worst pose), wall clock"},
                "assembled_equals_single_gpu": gather.get("assembled_equals_single_gpu"),
            }
            result["no_gather"] = {"value": round(value_trace, 2), "unit": "Mrays/s", "ms_per_step": round(ms_per_step, 4),
                                   "note": "trace only: every rank's strips stay on the GPU that traced them (round 1's headline); L2 flushed before every step, CUDA events"}
        if world == 1 and not args.no_cpu:
            result["cpu_baseline"] = cpu_baseline(tree)
        emit(result)
    if mg is not None:
        mg.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return result


def parity_of_timed_frames(ort, tree, n_nodes, ctx, mg, world, rank, outs, NS, n_frames, cams, frame_rows, torch, dist):
    """Compare what the timed loop left in its output buffers with the CPU checker (every rank its own strip rows; the
    counts are summed over ranks).  The DAG reaches the other ranks' checkers as plain data (torch broadcast)."""
    import numpy as _np
    from oracle import oracle as oc
    if world > 1:
        meta = torch.zeros(1, dtype=torch.int64, device="cuda")
        nodes8 = root = None
        if rank == 0:
            nodes8, root, _ = tree.flatten()
            meta[0] = root
        dist.broadcast(meta, src=0)
        nn = torch.from_numpy(nodes8.view(_np.int32)).cuda() if rank == 0 else torch.empty((int(n_nodes), 8), dtype=torch.int32, device="cuda")
        dist.broadcast(nn, src=0)
        nodes8, root = nn.cpu().numpy().view(_np.uint32), int(meta[0])
        del nn
    else:
        nodes8, root, _ = tree.flatten()
    kind, fn = cpu_tracer(nodes8, root)
    cores = os.cpu_count() or 1
    tot = {"rays": 0, "voxel_mismatch": 0, "face_mismatch": 0, "t_bitwise_mismatch": 0}
    poses_seen = set()
    for j in range(min(NS, n_frames)):
        k = max(kk for kk in range(n_frames) if kk % NS == j)
        cam = cams[k % len(cams)]
        poses_seen.add(POSE_NAMES[k % len(cams)])
        local = _np.arange(3, len(frame_rows), 8)                          # every 8th row of this rank's strip
        sel = torch.from_numpy((local[:, None] * W + _np.arange(W)[None, :]).ravel()).cuda()
        gv = outs[j][0][sel].cpu().numpy().view(_np.uint32)
        gf = outs[j][1][sel].cpu().numpy()
        gt = outs[j][2][sel].cpu().numpy().view(_np.uint32)
        d = _np.concatenate([oc.gen_rays(cam[1], cam[2], W, H, int(frame_rows[r]), int(frame_rows[r]) + 1) for r in local])
        wv, wf, wt = fn(cam[0], d, cores)
        tot["rays"] += int(gv.size)
        tot["voxel_mismatch"] += int((gv != wv).sum())
        tot["face_mismatch"] += int((gf != wf).sum())
        tot["t_bitwise_mismatch"] += int((gt != wt.view(_np.uint32)).sum())
    if world > 1:
        c = torch.tensor([tot[k] for k in ("rays", "voxel_mismatch", "face_mismatch", "t_bitwise_mismatch")], dtype=torch.int64, device="cuda")
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        tot = dict(zip(("rays", "voxel_mismatch", "face_mismatch", "t_bitwise_mismatch"), (int(x) for x in c.tolist())))
    tot["poses"] = sorted(poses_seen)
    tot["checker"] = f"{kind}: " + ("the reference's own sse_trace (oracle/_ref)" if kind == "reference" else "oracle port (oracle/och_oracle.c)")
    tot["what"] = "the frames the TIMED loop left in its output buffers, every 8th row of each rank's strip, bitwise (voxel, face, t)"
    return tot


# ------------------------------------------------------------------------------------------------
# CPU arms (the reference's own sse_trace where oracle/_ref exists, else the oracle port)
# ------------------------------------------------------------------------------------------------

def cpu_tracer(nodes8, root):
    """Returns (kind, fn(o, d, nthreads) -> (vox, face, t))."""
    from oracle import oracle as oc
    if oc.have_ref():
        R = oc.RefTree(LOG2CAP, DEPTH)
        R.import_compact(nodes8, root)
        return "reference", lambda o, d, nt: R.trace(o, d, nthreads=nt)
    return "port", lambda o, d, nt: oc.trace_rays(nodes8, root, DEPTH, o, d, nthreads=nt)


def sample_rays(sample_tiles: int):
    """Every `sample_tiles`-th 8-row tile of each pose's 4K frame: (origin, directions) per pose."""
    from oracle import oracle as oc
    from octree_ray_tracing_b200 import harness
    out = []
    for p in POSE_NAMES:
        pos, yaw, pitch = harness.POSES[p]
        rot, fov = oc.camera_coeffs(yaw, pitch)
        d = np.concatenate([oc.gen_rays(rot, fov, W, H, t * TILE_ROWS, (t + 1) * TILE_ROWS) for t in range(0, H // TILE_ROWS, sample_tiles)])
        out.append((np.array(pos, np.float32), d))
    return out


DUMP_BYTES = 60 << 20          # --dump-outputs writes at most this much: 16 B per sampled ray and frame


def dump_outputs(out_dir, frames, n_rays):
    """--dump-outputs: the outputs a caller of the timed path receives -- voxel id, face, hit time t -- for a fixed, seeded
    sample of the n_rays rays of each frame (the same ray indices in every frame and every run), as
    out_dir/<frame>_{voxel,face,t}.npy: voxel as float64 (exact for any uint32), face and t as float32 (t bit for bit).
    A ray that leaves the volume without a hit (face 6) has t = +inf; the file holds -1 there, never a hit time, so that a
    correct build writes only finite values.  Any other non-finite t is written as it is.
    frames: [(name, take)], take(idx) -> (voxel, face, t) of the rays at the sorted indices idx."""
    n = min(n_rays, DUMP_BYTES // (16 * len(frames)))
    idx = np.sort(np.random.RandomState(0).choice(n_rays, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, take in frames:
        v, f, t = take(idx)
        np.save(os.path.join(out_dir, f"{name}_voxel.npy"), np.asarray(v, np.uint32).astype(np.float64))
        f, t = np.asarray(f, np.uint8), np.asarray(t, np.float32)
        np.save(os.path.join(out_dir, f"{name}_face.npy"), f.astype(np.float32))
        np.save(os.path.join(out_dir, f"{name}_t.npy"), np.where((f == 6) & (t == np.inf), np.float32(-1.0), t))
    log(f"--dump-outputs: {len(frames)} frame(s), {n} of {n_rays} rays each, written to {out_dir}")


CPU_LAYOUT = ("compact level-ordered node array (the product's flatten) imported into the reference's nodes[]: 44 MiB contiguous instead of "
              "1.44 M nodes hashed over a 512 MiB table -- this favours the CPU arm; the traced function is the reference's own sse_trace")


def cpu_baseline(tree):
    """The reference's CPU trace over the WHOLE ray set of a step (3 poses x 3840x2160), all host cores."""
    nodes8, root, _ = tree.flatten()
    kind, fn = cpu_tracer(nodes8, root)
    cores = os.cpu_count() or 1
    rays = sample_rays(1)
    n = sum(d.shape[0] for _, d in rays)
    fn(rays[0][0], rays[0][1][:100000], cores)          # warm-up
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        for o, d in rays:
            fn(o, d, cores)
    dt = (time.perf_counter() - t0) / reps
    t1 = time.perf_counter()
    fn(rays[1][0], rays[1][1][: 1 << 20], 1)
    one = (1 << 20) / (time.perf_counter() - t1) / 1e6
    return {"value": round(n / dt / 1e6, 2), "unit": "Mrays/s", "cores": cores, "kind": kind,
            "sample": f"all rays of a step: the 3 poses' full 4K frames ({n} rays), {reps} passes, {cores} threads",
            "cpu_layout": CPU_LAYOUT, "one_thread_mrays": round(one, 2)}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from octree_ray_tracing_b200 import harness
    import octree_ray_tracing_b200 as ort
    tree = ort.HOctree(LOG2CAP, DEPTH, device=None)        # host table only: this arm never touches the GPU
    harness.build_terrain(tree)
    nodes8, root, _ = tree.flatten()
    kind, fn = cpu_tracer(nodes8, root)
    cores = os.cpu_count() or 1
    rays = sample_rays(1)                                   # every ray of the product arm's step (N = 1 share)
    n = sum(d.shape[0] for _, d in rays)

    def step():
        return [fn(o, d, cores) for o, d in rays]

    for _ in range(max(1, min(args.warmup, 2))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        last = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [(f"frame{k}_pose{p}", lambda idx, r=r: tuple(a[idx] for a in r))
                                         for k, (p, r) in enumerate(zip(POSE_NAMES, last))], last[0][0].size)
    value = n * args.steps / dt / 1e6
    sample = f"all rays of a step: the 3 poses' full 4K frames ({n} rays per step), {cores} threads"
    emit({
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": "Mrays/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", args.gpus)), "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32+u32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step": len(rays), "rays_per_step": n, "sample": sample, "cpu_layout": CPU_LAYOUT},
        "cpu_baseline": {"value": round(value, 3), "unit": "Mrays/s", "cores": cores, "kind": kind, "sample": sample, "cpu_layout": CPU_LAYOUT},
        "e2e": {"value": round(value, 3), "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


_JSON_OUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries write there too (NCCL prints its version banner when
    NCCL_DEBUG is set in the environment), so the real stdout is kept aside for the result line and file descriptor 1
    is pointed at stderr for everybody else."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(obj):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def main():
    global TILE_ROWS
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--launch", default="auto", choices=["auto", "batch", "streams"],
                    help="device-resident loop: the step's frames in one batched launch (ort_trace_frames_async) or one launch per frame on several streams")
    ap.add_argument("--streams", type=int, default=0, help="frames in flight in the device-resident loop (0 = 3 on one GPU, up to 8 on several)")
    ap.add_argument("--no-numa", action="store_true", help="do not pin the rank to its GPU's NUMA node")
    ap.add_argument("--quick", action="store_true", help="profiling aid: only the device-resident timed loop (no warm-L2 loop, no e2e, no CPU leg)")
    ap.add_argument("--tile-rows", type=int, default=TILE_ROWS, help="rows per tile of the cyclic strip partition (a multiple of 8)")
    ap.add_argument("--as-rank", default=None, metavar="R/N", help="with --quick on one GPU: trace the share rank R of an N-GPU job would")
    ap.add_argument("--variant", type=int, default=None, help="kernel variant (ort_set_option 'variant')")
    ap.add_argument("--opt", action="append", default=[], help="key=value passed to ort_set_option")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the last step's outputs (voxel, face, t) of a fixed, seeded sample of each "
                         "frame's rays as DIR/<frame>_<output>.npy, at most 60 MiB in all, so that two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    TILE_ROWS = args.tile_rows
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_product(args)


if __name__ == "__main__":
    main()
