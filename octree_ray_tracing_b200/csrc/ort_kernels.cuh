// ort_kernels.cuh -- the __global__ functions of libort_b200.so (sm_100a): the trace kernels, the delta scatter, the
// strip unpack of the multi-GPU gather, the fixture noise kernels and the roofline diagnostic.  Included by
// ort_device.cu only; the per-ray traversal itself lives in ort_trace.cuh.  Kernels that were measured and not adopted
// live in ort_experiments.cuh and are compiled into libort_b200_exp.so only (-DORT_EXPERIMENTS).
#pragma once

#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "ort_noise.h"
#include "ort_trace.cuh"
#include "ort_beam.cuh"

namespace ort {

// ------------------------------------------------------------------------------------------------
// small kernels
// ------------------------------------------------------------------------------------------------

// delta upload: one thread per 16-byte half node.  The source rows need only 4-byte alignment (a broadcast payload
// [ids | nodes] puts them at any word offset); the destination halves are 16-byte aligned.
__global__ void scatter_nodes_kernel(uint4* __restrict__ nodes, const uint32_t* __restrict__ ids, const uint32_t* __restrict__ src, uint32_t n)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < 2u * n)
	{
		const uint32_t* s = src + 4u * static_cast<size_t>(i);
		nodes[2u * static_cast<size_t>(ids[i >> 1] - 1u) + (i & 1u)] = make_uint4(s[0], s[1], s[2], s[3]);
	}
}

__global__ void fill_miss_kernel(uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* __restrict__ t, uint16_t* __restrict__ npush, float miss_t, size_t n)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i < n)
	{
		voxel[i] = 0;
		face[i] = 6;
		t[i] = miss_t;
		if (npush) npush[i] = 0;
	}
}

__global__ void fill_u32_kernel(uint32_t* __restrict__ dst, uint32_t v, size_t n)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i < n) dst[i] = v;
}

// ------------------------------------------------------------------------------------------------
// the walk of one ray
// ------------------------------------------------------------------------------------------------

// What every trace kernel needs to know about the DAG (one kernel parameter).
struct Dag
{
	const uint32_t*    nodes_m1;     // node id i at nodes_m1[8 * i ..] (h_octree layout: ids 1-based; och::octree pool: raw rows)
	unsigned long long base_biased;  // address of nodes_m1 minus 4 * kMagicBits (LeanWalker's slot words carry the 2^23 magic)
	uint32_t           root;
	int                depth;
	float              leaf_dimf;    // 2^-depth: the size of a voxel = the children's size at the last level
	float              miss_t;       // hit_time of a MISS: INFINITY (och_h_octree.h:429) or 0.0F (och_octree.cpp:302)
	uint32_t           plane_mask;   // (1 << (23 - depth)) - 1: origin mantissa bits below the finest grid (Ray::t0or)
	RcpTable           rt;
};

// walk selection ("variant" option): 0 = traverse(), the reference's state machine in integer ops; 1 = round 1's
// FastWalker (+ traverse() outside its domain); kLean = round 2's tiers: LeanWalker where a negative t can never
// occur, FastWalker for rays with a degenerate axis or an on-grid origin whose t rounds below zero, traverse()
// outside [1,2)^3.
constexpr int kLean = 13;
constexpr int kLeanShift = 13;      // LeanStack column pitch: 23 - log2(256 threads * 4 bytes); lean kernels run 256-thread blocks

// dynamic shared memory of a lean kernel: one column of (depth - 1) parent-stack words per thread
inline size_t lean_smem_bytes(int depth) { return static_cast<size_t>(depth > 1 ? depth - 1 : 1) * 256 * 4; }

__device__ __forceinline__ uint32_t lean_stack_base(const uint32_t* s_stack, int depth)
{
	// the entry of level L sits at exponent field 127 - L; the deepest level pushed is depth - 1
	return static_cast<uint32_t>(__cvta_generic_to_shared(s_stack)) + threadIdx.x * 4u - (static_cast<uint32_t>(128 - depth) << (23 - kLeanShift));
}

// Loop shape of the lean tier ("descend-while"): a lane keeps descending while the slot it lands on holds a child and
// only then takes ONE advance (step / pop) -- measured against the plain "one load, then descend or advance" round and
// the "advance-while" shape on the bench step: 18.57 vs 18.38 vs 18.34 Grays/s (profiles/r2_loop_shapes.json).
// The walk of one ray from its set-up state.  origin_ok: the origin part of fast_path_ok holds (tested per ray for
// explicit rays, known for the whole launch for camera frames).
template<int VARIANT, bool COUNT>
__device__ __forceinline__ Hit walk_ray(const Dag& g, float ox, float oy, float oz, const Ray& ray, bool origin_ok, const uint32_t* s_stack, float tau = 0.0f)
{
	// lean tier: origin inside the cube, no degenerate axis, no negative t possible
	if (VARIANT == kLean && origin_ok && lean_path_ok(ray))
	{
		LeanWalker<COUNT> w;
		const LeanStack<kLeanShift> st{ lean_stack_base(s_stack, g.depth) };
		// tau > 0: the tile's beam start (ort_beam.cuh) -- re-enter the walk there, or end as a MISS right away
		bool beam_used;
		if (lean_start(w, g.root, ray, tau, g.miss_t, beam_used))
			return w.hit;
		for (;;)
		{
			for (;;)
			{
				uint32_t child;
				bool done = false;
				while ((child = w.load_child(g.base_biased)) != 0u)
					if (w.descend(child, g.leaf_dimf, st)) { done = true; break; }
				if (done || w.advance(g.miss_t, st)) break;
			}
			// guard of the beam start: a voxel reached without a single STEP (min_t_idx untouched) means tau was not a
			// lower bound of this ray's hit time -- walk it from the start (an origin inside a solid voxel never gets tau > 0)
			if (!(beam_used && w.mti == 8u)) break;
			beam_used = false;
			w.start(g.root, ray);
		}
		return w.hit;
	}
	return traverse_variant<VARIANT, COUNT>(g.nodes_m1, g.root, g.depth, g.miss_t, ox, oy, oz, ray);
}

// explicit ray: every ray has its own origin, the origin tests run per ray
template<int VARIANT, bool COUNT>
__device__ __forceinline__ Hit trace_ray(const Dag& g, float ox, float oy, float oz, float dx, float dy, float dz, const uint32_t* s_stack)
{
	const Ray ray = ray_setup(g.rt, ox, oy, oz, dx, dy, dz, VARIANT == kLean ? g.plane_mask : 0u);
	return walk_ray<VARIANT, COUNT>(g, ox, oy, oz, ray, VARIANT == kLean && origin_in_cube(ox, oy, oz, ray), s_stack);
}

// camera ray: the origin facts were established once on the host (Camera::origin_flags)
template<int VARIANT, bool COUNT>
__device__ __forceinline__ Hit trace_camera_ray(const Dag& g, const Camera& cam, float dx, float dy, float dz, const uint32_t* s_stack, float tau = 0.0f)
{
	if (VARIANT != kLean)
		return trace_ray<VARIANT, COUNT>(g, cam.ox, cam.oy, cam.oz, dx, dy, dz, s_stack);
	const Ray ray = ray_setup_camera(g.rt, cam.ox, cam.oy, cam.oz, dx, dy, dz, cam.origin_flags);
	return walk_ray<VARIANT, COUNT>(g, cam.ox, cam.oy, cam.oz, ray, (cam.origin_flags & kOriginInCube) != 0u, s_stack, tau);
}

// ------------------------------------------------------------------------------------------------
// trace kernels
// ------------------------------------------------------------------------------------------------

// explicit rays: thread i traces ray i
template<int VARIANT, bool COUNT>
__global__ void __launch_bounds__(256)
trace_rays_kernel(const Dag g, const float* __restrict__ o3, int o_stride, const float* __restrict__ d3, size_t n,
                  uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* __restrict__ t, uint16_t* __restrict__ npush)
{
	extern __shared__ uint32_t s_stack[];
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float* o = o3 + i * static_cast<size_t>(o_stride);
	const float* d = d3 + i * 3;
	const Hit h = trace_ray<VARIANT, COUNT>(g, __ldg(o), __ldg(o + 1), __ldg(o + 2), __ldg(d), __ldg(d + 1), __ldg(d + 2), s_stack);
	voxel[i] = h.voxel;
	face[i] = static_cast<uint8_t>(h.face);
	t[i] = h.t;
	if (COUNT) npush[i] = static_cast<uint16_t>(min(h.npush, 65535u));
}

// FrameRows / frame_row (strip-local row -> frame row) live in ort_trace.cuh, next to the camera

// camera rays: a warp owns an 8 x 4 pixel tile (coherent rays -> shared upper-level nodes), a 256-thread block a
// 16 x 16 pixel tile; block row b of the launch is traced by blockIdx.y = (b - band_rotate) mod (number of bands).
__device__ __forceinline__ bool frame_pixel(const FrameRows& fr, unsigned block_y, unsigned bands, int& x, int& r)
{
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	unsigned by;
	if (fr.band_order)
		by = __ldg(fr.band_order + block_y);
	else
	{
		by = block_y + static_cast<unsigned>(fr.band_rotate);
		if (by >= bands) by -= bands;
	}
	x = blockIdx.x * 16 + (warp & 1) * 8 + (lane & 7);
	r = static_cast<int>(by) * 16 + (warp >> 1) * 4 + (lane >> 3);
	return x < fr.W && r < fr.rows;
}

// Beam start of the thread's 8 x 4 tile: beam_start_kernel left it in the output word of the tile's first pixel (nobody but
// the tile's own warp touches that word, and the warp reads it here before any of its lanes can have stored a result).
// All 32 lanes take part, also those outside the frame.
__device__ __forceinline__ float read_tile_start(const FrameRows& fr, const float* tile_word, int x, int r)
{
	const int x0 = x & ~7, r0 = r & ~3;
	float tau = 0.0f;
	if (x0 < fr.W && r0 < fr.rows)
		tau = tile_word[static_cast<size_t>(r0) * fr.W + x0];
	__syncwarp();
	return tau;
}

// (register budget: 6 resident blocks per SM = 40 registers; the 32-register build reloads the node base pointer from the
// constant bank every round and measures 1-2 % slower, although it fits 8 blocks)
// BEAM: the launch was preceded by beam_start_kernel over the same rows and the same `t` array.
// RECORD: the launch measures what its bands cost (FrameRows::band_cost) -- a separate instantiation, because the clock
// value kept across the walk costs the ordinary kernel four registers and a tenth of its speed.
template<int VARIANT, bool COUNT, bool BEAM = false, bool RECORD = false>
__global__ void __launch_bounds__(256, 6)
trace_frame_kernel(const Dag g, Camera cam, FrameRows fr,
                   uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* t, uint16_t* __restrict__ npush)
{
	extern __shared__ uint32_t s_stack[];
	int x, r;
	const bool inside = frame_pixel(fr, blockIdx.y, gridDim.y, x, r);
	const float tau = BEAM ? read_tile_start(fr, t, x, r) : 0.0f;
	if (!inside) return;
	const size_t i = static_cast<size_t>(r) * fr.W + x;
	if (BEAM && __float_as_uint(tau) == kBeamAllMissBits)
	{
		// nothing in sight for the whole tile and every ray certain to be in the lean tier: 32 MISSes (och_h_octree.h:423-431)
		voxel[i] = 0u;
		face[i] = 6;
		t[i] = g.miss_t;
		if (COUNT) npush[i] = 0;
		return;
	}
	const long long t_start = RECORD ? clock64() : 0ll;
	const int y = frame_row(fr, r);

	float dx, dy, dz;
	camera_ray(cam, x, y, dx, dy, dz);
	const Hit h = trace_camera_ray<VARIANT, COUNT>(g, cam, dx, dy, dz, s_stack, tau);

	voxel[i] = h.voxel;
	face[i] = static_cast<uint8_t>(h.face);
	t[i] = h.t;
	if (COUNT) npush[i] = static_cast<uint16_t>(min(h.npush, 65535u));
	if (RECORD)
	{
		// what this band costs, for the schedule of the next launch of the same view: the longest a warp of the band was busy
		// (a scheduling hint, nothing reads it for results; one atomic per warp where the lanes have reconverged)
		const unsigned m = __activemask();
		const unsigned dur = __reduce_max_sync(m, static_cast<unsigned>((clock64() - t_start) >> 4));
		if ((threadIdx.x & 31u) == static_cast<unsigned>(__ffs(static_cast<int>(m)) - 1))
			atomicMax(fr.band_cost + (r >> 4), dur);
	}
}

// The march of the beam start (ort_beam.cuh), one thread per 8 x 4 pixel tile of the rows a frame launch traces: the tile's
// start time goes into the output word of its first pixel -- `t` for the voxel / face / t kernels, the pixel for the
// shaded kernel -- where the trace kernel picks it up.
// fine / fine_t: the level-8 grid and the time limit of the refinement (fine_t = 0: none).
__global__ void __launch_bounds__(128)
beam_start_kernel(const BeamGrid grid, const BeamGrid fine, float fine_t, Camera cam, FrameRows fr, float min_comp, float* __restrict__ tile_word)
{
	const int tiles_x = (fr.W + 7) >> 3, tiles_y = (fr.rows + 3) >> 2;
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= tiles_x * tiles_y) return;
	const int x0 = (i % tiles_x) * 8, r0 = (i / tiles_x) * 4;
	tile_word[static_cast<size_t>(r0) * fr.W + x0] = beam_tile_start(grid, cam, x0, frame_row(fr, r0), min_comp, nullptr, fine, fine_t);
}

// Several frame jobs in ONE launch (blockIdx.z = job): strips of different frames, or the views of a multi-camera
// rig.  Separate launches each end with the latency tail of their longest rays; here the blocks of all jobs stream
// through the SMs back to back and only the last job's tail is exposed.  The jobs travel in the kernel parameters.
constexpr int kMaxJobs = 32;

struct FrameJob
{
	Camera cam;
	FrameRows fr;
	uint32_t* voxel;
	uint8_t*  face;
	float*    t;
	uint16_t* npush;    // may be null
	int       beam_k;   // level of the beam grid this job's tile starts come from (0: the job runs without)
	float     beam_min_comp;   // beam_certify_min_comp() of the job's camera
	float     beam_fine_t;     // beam_fine_t_limit() of the job's camera: its tiles refine their start on the level-8 grid (0: not)
};

struct FrameJobBatch
{
	FrameJob job[kMaxJobs];
};

template<int VARIANT, bool COUNT, bool BEAM = false>          // COUNT: some job of the batch wants per-ray PUSH counts (jobs without an npush pointer skip the store)
__global__ void __launch_bounds__(256, 6)
trace_frames_kernel(const Dag g, const __grid_constant__ FrameJobBatch batch)
{
	extern __shared__ uint32_t s_stack[];
	const FrameJob& jb = batch.job[blockIdx.z];
	const FrameRows& fr = jb.fr;
	const unsigned bands = static_cast<unsigned>((fr.rows + 15) >> 4);
	if (blockIdx.y >= bands) return;                                    // the grid is sized for the largest job
	int x, r;
	const bool inside = frame_pixel(fr, blockIdx.y, bands, x, r);
	const float tau = BEAM ? read_tile_start(fr, jb.t, x, r) : 0.0f;
	if (!inside) return;
	const size_t i = static_cast<size_t>(r) * fr.W + x;
	if (BEAM && __float_as_uint(tau) == kBeamAllMissBits)
	{
		jb.voxel[i] = 0u;
		jb.face[i] = 6;
		jb.t[i] = g.miss_t;
		if (COUNT && jb.npush) jb.npush[i] = 0;
		return;
	}
	const int y = frame_row(fr, r);

	float dx, dy, dz;
	camera_ray(jb.cam, x, y, dx, dy, dz);
	const Hit h = trace_camera_ray<VARIANT, COUNT>(g, jb.cam, dx, dy, dz, s_stack, tau);

	jb.voxel[i] = h.voxel;
	jb.face[i] = static_cast<uint8_t>(h.face);
	jb.t[i] = h.t;
	if (COUNT && jb.npush) jb.npush[i] = static_cast<uint16_t>(min(h.npush, 65535u));
}

// the march for every job of a batch (blockIdx.y = job); grids[k] = the context's grid of level k (kBeamFineLevel: the
// refinement's, where some job refines)
struct BeamGridSet
{
	const uint8_t* skip[kBeamFineLevel + 1];
};

__global__ void __launch_bounds__(128)
beam_start_batch_kernel(const BeamGridSet grids, const __grid_constant__ FrameJobBatch batch)
{
	const FrameJob& jb = batch.job[blockIdx.y];
	if (!jb.beam_k) return;
	const FrameRows& fr = jb.fr;
	const int tiles_x = (fr.W + 7) >> 3, tiles_y = (fr.rows + 3) >> 2;
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= tiles_x * tiles_y) return;
	const int x0 = (i % tiles_x) * 8, r0 = (i / tiles_x) * 4;
	jb.t[static_cast<size_t>(r0) * fr.W + x0] = beam_tile_start(BeamGrid{ grids.skip[jb.beam_k], jb.beam_k }, jb.cam, x0, frame_row(fr, r0), jb.beam_min_comp, nullptr,
	                                                               BeamGrid{ grids.skip[kBeamFineLevel], kBeamFineLevel }, jb.beam_fine_t);
}

// Shading epilogue (tree_camera::trace_pixel, test_och_h_octree.cpp:76-84) fused into the frame kernel: the hit is
// turned into the pixel the demo would Draw() -- colours[6 * (voxel - 1) + face], the sky colour on exit, the
// "inside" colour when the origin sits in a solid voxel -- and only that uint32 leaves the SM (4 B per pixel
// instead of 9).  Voxel types beyond the palette (the reference reads past its array there) shade as 0.
struct Palette
{
	const uint32_t* colours;
	uint32_t n_voxels;
	uint32_t exit_rgba, inside_rgba;
};

template<int VARIANT, bool BEAM = false>
__global__ void __launch_bounds__(256, 6)
trace_frame_rgba_kernel(const Dag g, Camera cam, FrameRows fr, Palette pal, uint32_t* rgba)
{
	extern __shared__ uint32_t s_stack[];
	int x, r;
	const bool inside = frame_pixel(fr, blockIdx.y, gridDim.y, x, r);
	const float tau = BEAM ? read_tile_start(fr, reinterpret_cast<const float*>(rgba), x, r) : 0.0f;
	if (!inside) return;
	if (BEAM && __float_as_uint(tau) == kBeamAllMissBits)
	{
		rgba[static_cast<size_t>(r) * fr.W + x] = pal.exit_rgba;
		return;
	}
	const int y = frame_row(fr, r);

	float dx, dy, dz;
	camera_ray(cam, x, y, dx, dy, dz);
	const Hit h = trace_camera_ray<VARIANT, false>(g, cam, dx, dy, dz, s_stack, tau);

	uint32_t px;
	if (h.face == 6u) px = pal.exit_rgba;
	else if (h.face == 7u) px = pal.inside_rgba;
	else px = (h.voxel - 1u < pal.n_voxels) ? __ldg(pal.colours + 6u * (h.voxel - 1u) + h.face) : 0u;
	rgba[static_cast<size_t>(r) * fr.W + x] = px;
}

// ------------------------------------------------------------------------------------------------
// Persistent warps with lane refill ("warp-level ray compaction").
//
// A fixed grid (one resident wave) walks the ray list: each warp draws batches of ray indices from a global
// counter and keeps its 32 lanes busy -- when a lane's ray ends, the lane writes its result and goes idle;
// once the number of busy lanes (ballot + popc) falls to `low_water` and rays remain, the idle lanes are
// refilled before traversal continues.  This trades a ballot per traversal round and scattered result
// writes for lanes that no longer wait on the slowest ray of their warp: worth little on coherent camera
// rays, a lot on incoherent rays (BASELINE config 3: 10 PUSHes on average, 600 worst case).
// FRAME = true enumerates the pixels of the strip in 8x4 tile order (index = 32 * tile + lane-in-tile) so
// that consecutive indices stay spatially coherent.
// The resumable walker is LeanWalker (its parent stack is the thread's shared-memory column); a ray outside its
// preconditions is walked to the end right away when it is drawn (FastWalker / traverse()), like any other rare case.
// `counter` is the launch's own work counter (a ring of them lives in the context, so launches on different streams
// never share one).
// ------------------------------------------------------------------------------------------------

constexpr unsigned kBatch = 128;    // ray indices a warp draws per atomicAdd

// MINB = minimum resident blocks per SM the compiler must allow for (register budget)
template<bool COUNT, bool FRAME, int MINB = 1>
__global__ void __launch_bounds__(256, MINB)
trace_persistent_kernel(const Dag g, const float* __restrict__ o3, int o_stride, const float* __restrict__ d3, Camera cam, FrameRows fr,
                        unsigned long long n, unsigned long long* __restrict__ counter, int low_water,
                        uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* __restrict__ t, uint16_t* __restrict__ npush)
{
	extern __shared__ uint32_t s_stack[];
	const unsigned lane = threadIdx.x & 31u;
	const unsigned lt_mask = (1u << lane) - 1u;
	const unsigned tiles_x = FRAME ? (fr.W + 7) / 8 : 1;
	const LeanStack<kLeanShift> st{ lean_stack_base(s_stack, g.depth) };

	LeanWalker<COUNT> w;
	bool active = false;
	size_t out = 0;                              // where this lane's result goes
	unsigned long long next = 0, end = 0;        // the warp's current batch (uniform)
	bool exhausted = false;                      // (uniform)

	auto store = [&](size_t i, const Hit& h) {
		voxel[i] = h.voxel;
		face[i] = static_cast<uint8_t>(h.face);
		t[i] = h.t;
		if (COUNT) npush[i] = static_cast<uint16_t>(min(h.npush, 65535u));
	};

	for (;;)
	{
		// ---- refill idle lanes ---------------------------------------------------------------
		unsigned idle = __ballot_sync(0xFFFFFFFFu, !active);
		while (idle != 0u && !exhausted)
		{
			if (next == end)
			{
				unsigned long long b = 0;
				if (lane == 0) b = atomicAdd(counter, static_cast<unsigned long long>(kBatch));
				b = __shfl_sync(0xFFFFFFFFu, b, 0);
				if (b >= n) { exhausted = true; break; }
				next = b;
				end = b + kBatch < n ? b + kBatch : n;
			}
			const unsigned long long left = end - next;
			const unsigned n_idle = __popc(idle);
			const unsigned avail = left < n_idle ? static_cast<unsigned>(left) : n_idle;
			const unsigned rank = __popc(idle & lt_mask);
			if (!active && rank < avail)
			{
				const unsigned long long i = next + rank;
				float ox, oy, oz, dx, dy, dz;
				bool valid = true;
				if (FRAME)
				{
					const unsigned tile = static_cast<unsigned>(i >> 5), l = static_cast<unsigned>(i) & 31u;
					const int x = static_cast<int>(tile % tiles_x) * 8 + static_cast<int>(l & 7u);
					const int r = static_cast<int>(tile / tiles_x) * 4 + static_cast<int>(l >> 3);
					valid = x < fr.W && r < fr.rows;
					const int y = frame_row(fr, r);
					ox = cam.ox; oy = cam.oy; oz = cam.oz;
					camera_ray(cam, x, y, dx, dy, dz);
					out = static_cast<size_t>(r) * fr.W + x;
				}
				else
				{
					const float* o = o3 + i * static_cast<unsigned long long>(o_stride);
					const float* d = d3 + i * 3ull;
					ox = __ldg(o); oy = __ldg(o + 1); oz = __ldg(o + 2);
					dx = __ldg(d); dy = __ldg(d + 1); dz = __ldg(d + 2);
					out = static_cast<size_t>(i);
				}
				if (valid)
				{
					const Ray ray = ray_setup(g.rt, ox, oy, oz, dx, dy, dz, g.plane_mask);
					if (origin_in_cube(ox, oy, oz, ray) && lean_path_ok(ray))
					{
						w.start(g.root, ray);
						active = true;
					}
					else
						store(out, traverse_variant<1, COUNT>(g.nodes_m1, g.root, g.depth, g.miss_t, ox, oy, oz, ray));   // rare ray: walked to the end right away
				}
			}
			next += avail;
			idle = __ballot_sync(0xFFFFFFFFu, !active);
		}

		if (__ballot_sync(0xFFFFFFFFu, active) == 0u)
			break;

		// ---- traverse until too few lanes are busy ---------------------------------------------
		for (;;)
		{
			if (active && w.round(g.base_biased, g.leaf_dimf, g.miss_t, st))
			{
				store(out, w.hit);
				active = false;
			}
			const unsigned busy = __ballot_sync(0xFFFFFFFFu, active);
			if (busy == 0u || (!exhausted && __popc(busy) <= low_water))
				break;
		}
	}
}

// ------------------------------------------------------------------------------------------------
// multi-GPU strip gather (ort_mg_*): received strips -> their rows of the assembled frame
// ------------------------------------------------------------------------------------------------

// A rank's strip block holds its tiles back to back (tile k of the strip = frame tile rank + k * world, tile_rows rows
// each) in three sections of max_n entries: voxel u32 | t f32 | face u8 (max_n = pixels of the longest strip, a
// multiple of 4 because W is).  The consumer holds one block per rank, `pitch` bytes apart, in rank order.
// One thread moves 4 pixels of all three outputs: grid = (ceil(max_n / 4 / 256), world).
struct StripMap
{
	int W, H, tile_rows, world;
	unsigned long long max_n, pitch;
};

__global__ void __launch_bounds__(256)
unpack_strips_kernel(uint4* __restrict__ voxel, uint4* __restrict__ t, uint32_t* __restrict__ face, const char* __restrict__ blocks, StripMap m)
{
	const int W4 = m.W >> 2;
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;     // 4-pixel group within the strip
	if (i * 4 >= m.max_n) return;
	const int rk = static_cast<int>(blockIdx.y);
	const int r = static_cast<int>(i / W4), x4 = static_cast<int>(i % W4);
	const int tile = r / m.tile_rows, in_tile = r % m.tile_rows;
	const int y = (rk + tile * m.world) * m.tile_rows + in_tile;
	if (y >= m.H) return;                                                            // past the rank's last tile / the frame's last row
	const char* blk = blocks + static_cast<size_t>(rk) * m.pitch;
	const size_t o = static_cast<size_t>(y) * W4 + x4;
	voxel[o] = reinterpret_cast<const uint4*>(blk)[i];
	t[o] = reinterpret_cast<const uint4*>(blk + m.max_n * 4)[i];
	face[o] = reinterpret_cast<const uint32_t*>(blk + m.max_n * 8)[i];
}

// ------------------------------------------------------------------------------------------------
// beam grid (ort_beam.cuh): level-k occupancy of the DAG -> dilation -> empty-cell pyramid -> skip levels
// ------------------------------------------------------------------------------------------------

// one thread per level-k cell (index (z * N + y) * N + x): is anything below it?  Slot bit a = upper half on world axis a.
__global__ void __launch_bounds__(256)
beam_occupancy_kernel(const uint32_t* __restrict__ nodes_m1, uint32_t root, int k, uint8_t* __restrict__ occ)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= (1u << (3 * k))) return;
	const uint32_t m = (1u << k) - 1u, x = i & m, y = (i >> k) & m, z = i >> (2 * k);
	uint32_t node = root, child = 1u;
	for (int l = k - 1; l >= 0 && child; --l)
	{
		const uint32_t slot = ((x >> l) & 1u) | (((y >> l) & 1u) << 1) | (((z >> l) & 1u) << 2);
		child = __ldg(nodes_m1 + (static_cast<size_t>(node) << 3) + slot);
		node = child;
	}
	occ[i] = child != 0u;
}

// dil = 1 where any of the 27 cells around the cell is occupied
__global__ void __launch_bounds__(256)
beam_dilate_kernel(const uint8_t* __restrict__ occ, int k, uint8_t* __restrict__ dil)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= (1u << (3 * k))) return;
	const int N = 1 << k, x = i & (N - 1), y = (i >> k) & (N - 1), z = i >> (2 * k);
	uint32_t any = 0;
	for (int dz = -1; dz <= 1; ++dz)
		for (int dy = -1; dy <= 1; ++dy)
			for (int dx = -1; dx <= 1; ++dx)
			{
				const int xx = x + dx, yy = y + dy, zz = z + dz;
				if (xx >= 0 && xx < N && yy >= 0 && yy < N && zz >= 0 && zz < N)
					any |= occ[(static_cast<size_t>(zz) * N + yy) * N + xx];
			}
	dil[i] = any != 0u;
}

// level j of the pyramid from level j + 1: a cell is marked when any of its 8 children is
__global__ void __launch_bounds__(256)
beam_reduce_kernel(const uint8_t* __restrict__ fine, int j, uint8_t* __restrict__ coarse)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= (1u << (3 * j))) return;
	const int N = 1 << j, F = 2 * N, x = i & (N - 1), y = (i >> j) & (N - 1), z = i >> (2 * j);
	uint32_t any = 0;
	for (int c = 0; c < 8; ++c)
		any |= fine[(static_cast<size_t>(2 * z + (c >> 2)) * F + (2 * y + ((c >> 1) & 1))) * F + (2 * x + (c & 1))];
	coarse[i] = any != 0u;
}

// skip[cell] = 0 where the cell is dilated-occupied, else the coarsest level whose cell around it is unmarked.
// pyr: the levels 1 .. k of the dilation pyramid back to back (level j at offset sum of 8^i for i in 1 .. j - 1)
__global__ void __launch_bounds__(256)
beam_skip_kernel(const uint8_t* __restrict__ pyr, int k, uint8_t* __restrict__ skip)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= (1u << (3 * k))) return;
	const uint32_t m = (1u << k) - 1u, x = i & m, y = (i >> k) & m, z = i >> (2 * k);
	size_t off = 0;
	int s = 0;
	for (int j = 1; j <= k; ++j)
	{
		const int sh = k - j;
		const size_t c = ((((static_cast<size_t>(z >> sh) << j) | (y >> sh)) << j) | (x >> sh));
		if (!pyr[off + c]) { s = j; break; }
		off += static_cast<size_t>(1) << (3 * j);
	}
	skip[i] = static_cast<uint8_t>(s);
}

// Fixture kernels (SURVEY 8f.3): the noise evaluations of the demo's terrain set-up, one thread per column / voxel.
// get_terrain_heigth over the whole map (test_och_h_octree.cpp:561-566, :587-592)
__global__ void __launch_bounds__(256)
fixture_heightmap_kernel(uint16_t* __restrict__ heights, int dim)
{
	const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
	if (x < dim) heights[static_cast<size_t>(y) * dim + x] = ort_noise::terrain_height(x, y, dim);
}

// remove(tree, splatter_noise(-0.5F, .., 1/16))'s dim^3 test (:735-743, :755-763) for the voxels at or below the
// surface: bit (y * dim + x) of slab z = "carved".  A warp covers 32 consecutive x and writes one 32-bit word.
__global__ void __launch_bounds__(256)
fixture_carve_kernel(const uint16_t* __restrict__ heights, int dim, uint32_t* __restrict__ bits, size_t words32_per_slab)
{
	const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, z = blockIdx.z;
	const bool carved = x < dim && z <= static_cast<int>(heights[static_cast<size_t>(y) * dim + x]) && ort_noise::carve_test(x, y, z);
	const unsigned w = __ballot_sync(0xFFFFFFFFu, carved);
	if ((threadIdx.x & 31u) == 0u && x < dim)
		bits[static_cast<size_t>(z) * words32_per_slab + ((static_cast<size_t>(y) * dim + x) >> 5)] = w;
}

// Diagnostic: random 32-byte-sector gather over an L2-resident buffer -- the memory-side ceiling of a
// traversal whose nodes live in L2 (one 4-byte child read moves one sector).  Independent loads, 8 in
// flight per thread, addresses from a counter hash so that L1 cannot help.
__global__ void __launch_bounds__(256)
gather_peak_kernel(const uint32_t* __restrict__ buf, uint32_t n_sectors, uint32_t iters, uint32_t* __restrict__ sink)
{
	uint32_t x = (blockIdx.x * blockDim.x + threadIdx.x) * 2654435761u + 12345u;
	uint32_t acc = 0;
	for (uint32_t i = 0; i < iters; ++i)
	{
		uint32_t v[8];
#pragma unroll
		for (int k = 0; k < 8; ++k)
		{
			x = x * 1664525u + 1013904223u;
			const uint32_t s = __umulhi(x ^ (x >> 15), n_sectors);            // uniform in [0, n_sectors)
			v[k] = __ldg(buf + (static_cast<size_t>(s) << 3) + (x & 7u));
		}
#pragma unroll
		for (int k = 0; k < 8; ++k) acc ^= v[k];
	}
	if (acc == 0x9E3779B9u) *sink = acc;                                      // keep the loads alive
}

}  // namespace ort
