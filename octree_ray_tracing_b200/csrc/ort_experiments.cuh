// ort_experiments.cuh -- kernels that were built to answer a design question, measured, and NOT adopted.  They are
// compiled only with -DORT_EXPERIMENTS (libort_b200_exp.so, built next to the product library by build.py) so that the
// decisions in DESIGN.md section 4 can be re-measured; the product library does not carry them.  Selected through
// ort_set_option("variant", n): 3 shared-memory staging of the top levels, 4 deferred phases, 5 / 6 TightWalker,
// 7 PipeWalker, 8-11 pipe probes, 12 persistent warps over tiles, 14 straight-line (predicated) round, 15 128-bit half-node
// fetches, 16 / 17 while-while loop shapes, 18 local-memory parent stack, 19 a 40-register budget; options "tile_shape" / "block" select other warp tiles and block heights of the round-1 default kernel.
// Included by ort_device.cu after the context definition.
#pragma once

#include "ort_kernels.cuh"
#include "ort_trace_experiments.cuh"

namespace ort {

// round 1's default frame kernel with selectable warp tiles (fr.tile_shape: 0 = 8x4, 1 = 16x2, 2 = 4x8, 3 = 8x4 in a
// 32x8 block) and block heights (blockDim.x / 16 rows); no band rotation
template<bool COUNT>
__global__ void __launch_bounds__(256)
trace_frame_shaped_kernel(const uint32_t* __restrict__ nodes_m1, uint32_t root, int depth, float miss_t, RcpTable rt, Camera cam, FrameRows fr,
                   uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* __restrict__ t, uint16_t* __restrict__ npush)
{
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	int x, r;
	if (fr.tile_shape == 1)      { x = blockIdx.x * 16 + (lane & 15);                   r = blockIdx.y * 16 + warp * 2 + (lane >> 4); }
	else if (fr.tile_shape == 2) { x = blockIdx.x * 16 + (warp & 3) * 4 + (lane & 3);   r = blockIdx.y * 16 + (warp >> 2) * 8 + (lane >> 2); }
	else if (fr.tile_shape == 3) { x = blockIdx.x * 32 + (warp & 3) * 8 + (lane & 7);   r = blockIdx.y * 8 + (warp >> 2) * 4 + (lane >> 3); }   // 32 x 8 block: stays inside one 8-row strip
	else                         { x = blockIdx.x * 16 + (warp & 1) * 8 + (lane & 7);   r = blockIdx.y * static_cast<int>(blockDim.x >> 4) + (warp >> 1) * 4 + (lane >> 3); }
	if (x >= fr.W || r >= fr.rows) return;
	const int y = frame_row(fr, r);

	float dx, dy, dz;
	camera_ray(cam, x, y, dx, dy, dz);
	const Ray ray = ray_setup(rt, cam.ox, cam.oy, cam.oz, dx, dy, dz);
	const Hit h = traverse_variant<1, COUNT>(nodes_m1, root, depth, miss_t, cam.ox, cam.oy, cam.oz, ray);

	const size_t i = static_cast<size_t>(r) * fr.W + x;
	voxel[i] = h.voxel;
	face[i] = static_cast<uint8_t>(h.face);
	t[i] = h.t;
	if (COUNT) npush[i] = static_cast<uint16_t>(min(h.npush, 65535u));
}


// Variants 5 / 6: TightWalker (leaner bookkeeping per round, see ort_trace.cuh).  WW = false keeps the
// "if-if" round of the default kernel (one child load, then descend OR advance); WW = true is the "while-while"
// shape: every lane first advances over empty child slots until it holds a non-empty child (or leaves the tree),
// then the whole warp descends together.
template<bool COUNT, bool WW>
__global__ void __launch_bounds__(256)
trace_frame_tight_kernel(const uint32_t* __restrict__ nodes_m1, uint32_t root, int depth, float miss_t, RcpTable rt, Camera cam, FrameRows fr,
                         uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* __restrict__ t, uint16_t* __restrict__ npush)
{
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int x = blockIdx.x * 16 + (warp & 1) * 8 + (lane & 7);
	const int r = blockIdx.y * 16 + (warp >> 1) * 4 + (lane >> 3);
	if (x >= fr.W || r >= fr.rows) return;
	const int y = frame_row(fr, r);

	float dx, dy, dz;
	camera_ray(cam, x, y, dx, dy, dz);
	const Ray ray = ray_setup(rt, cam.ox, cam.oy, cam.oz, dx, dy, dz);
	uint32_t stack[kMaxDepth];
	Hit h;
	if (fast_path_ok(cam.ox, cam.oy, cam.oz, ray))
	{
		TightWalker<COUNT> w;
		w.start(root, miss_t, ray);
		if (WW)
		{
			for (;;)
			{
				uint32_t child;
				bool done = false;
				while ((child = w.load_child(nodes_m1)) == 0u)
					if (w.advance(stack)) { done = true; break; }
				if (done || w.descend(child, depth, stack))
					break;
			}
		}
		else
		{
			for (;;)
			{
				const uint32_t child = w.load_child(nodes_m1);
				if (child ? w.descend(child, depth, stack) : w.advance(stack))
					break;
			}
		}
		h = w.hit;
	}
	else
		h = traverse(nodes_m1, root, depth, miss_t, ray, stack);

	const size_t i = static_cast<size_t>(r) * fr.W + x;
	voxel[i] = h.voxel;
	face[i] = static_cast<uint8_t>(h.face);
	t[i] = h.t;
	if (COUNT) npush[i] = static_cast<uint16_t>(min(h.npush, 65535u));
}

// Variant 12: persistent warps over tiles.  The default kernel's blocks retire when their slowest warp does, which
// leaves warp slots empty (achieved occupancy 83 %).  Here a resident grid is launched once and every WARP draws its
// next 8 x 4 tile from a global counter as soon as it is done, in the order the default kernel would have used
// (8 consecutive tiles = one 16 x 16 block tile), so slots never wait for a block mate.
template<bool COUNT>
__global__ void __launch_bounds__(256, 8)
trace_frame_tiles_kernel(const uint32_t* __restrict__ nodes_m1, uint32_t root, int depth, float miss_t, RcpTable rt, Camera cam, FrameRows fr,
                         unsigned int n_tiles, unsigned int* __restrict__ counter,
                         uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* __restrict__ t, uint16_t* __restrict__ npush)
{
	const unsigned lane = threadIdx.x & 31u;
	const unsigned blocks_x = (fr.W + 15) / 16;
	for (;;)
	{
		unsigned tile = 0;
		if (lane == 0) tile = atomicAdd(counter, 1u);
		tile = __shfl_sync(0xFFFFFFFFu, tile, 0);
		if (tile >= n_tiles) return;
		const unsigned blk = tile >> 3, sub = tile & 7u;
		const int x = static_cast<int>(blk % blocks_x) * 16 + static_cast<int>(sub & 1u) * 8 + static_cast<int>(lane & 7u);
		const int r = static_cast<int>(blk / blocks_x) * 16 + static_cast<int>(sub >> 1) * 4 + static_cast<int>(lane >> 3);
		if (x >= fr.W || r >= fr.rows) continue;
		const int y = frame_row(fr, r);

		float dx, dy, dz;
		camera_ray(cam, x, y, dx, dy, dz);
		const Ray ray = ray_setup(rt, cam.ox, cam.oy, cam.oz, dx, dy, dz);
		const Hit h = traverse_variant<1, COUNT>(nodes_m1, root, depth, miss_t, cam.ox, cam.oy, cam.oz, ray);

		const size_t i = static_cast<size_t>(r) * fr.W + x;
		voxel[i] = h.voxel;
		face[i] = static_cast<uint8_t>(h.face);
		t[i] = h.t;
		if (COUNT) npush[i] = static_cast<uint16_t>(min(h.npush, 65535u));
	}
}

// Variant 7: PipeWalker (ALU-lean bookkeeping, see ort_trace.cuh).
template<bool COUNT>
__global__ void __launch_bounds__(256)
trace_frame_pipe_kernel(const uint32_t* __restrict__ nodes_m1, unsigned long long base_biased, uint32_t root, int depth, float miss_t, RcpTable rt, Camera cam, FrameRows fr,
                        uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* __restrict__ t, uint16_t* __restrict__ npush)
{
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int x = blockIdx.x * 16 + (warp & 1) * 8 + (lane & 7);
	const int r = blockIdx.y * 16 + (warp >> 1) * 4 + (lane >> 3);
	if (x >= fr.W || r >= fr.rows) return;
	const int y = frame_row(fr, r);

	float dx, dy, dz;
	camera_ray(cam, x, y, dx, dy, dz);
	const Ray ray = ray_setup(rt, cam.ox, cam.oy, cam.oz, dx, dy, dz);
	Hit h;
	if (fast_path_ok(cam.ox, cam.oy, cam.oz, ray))
	{
		uint32_t stack_n[kMaxDepth];
		float stack_f[kMaxDepth];
		PipeWalker<COUNT> w;
		w.start(root, miss_t, ray);
		for (;;)
		{
			const uint32_t child = w.load_child(base_biased);
			if (child ? w.descend(child, depth, stack_n, stack_f) : w.advance(stack_n, stack_f))
				break;
		}
		h = w.hit;
	}
	else
	{
		uint32_t stack[kMaxDepth];
		h = traverse(nodes_m1, root, depth, miss_t, ray, stack);
	}

	const size_t i = static_cast<size_t>(r) * fr.W + x;
	voxel[i] = h.voxel;
	face[i] = static_cast<uint8_t>(h.face);
	t[i] = h.t;
	if (COUNT) npush[i] = static_cast<uint16_t>(min(h.npush, 65535u));
}

// Probe kernels (variants 8 / 9): the default walk plus PROBE_FMA dependent-free FMA-pipe instructions or PROBE_ALU
// ALU-pipe instructions per round, on dummy accumulators that are folded into the result only if they take an
// impossible value.  They answer "which resource binds the loop?": extra work on a unit that has slack is free.
template<int PROBE_FMA, int PROBE_ALU>
__global__ void __launch_bounds__(256)
trace_frame_probe_kernel(const uint32_t* __restrict__ nodes_m1, uint32_t root, int depth, float miss_t, RcpTable rt, Camera cam, FrameRows fr,
                         uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* __restrict__ t)
{
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int x = blockIdx.x * 16 + (warp & 1) * 8 + (lane & 7);
	const int r = blockIdx.y * 16 + (warp >> 1) * 4 + (lane >> 3);
	if (x >= fr.W || r >= fr.rows) return;
	const int y = frame_row(fr, r);

	float dx, dy, dz;
	camera_ray(cam, x, y, dx, dy, dz);
	const Ray ray = ray_setup(rt, cam.ox, cam.oy, cam.oz, dx, dy, dz);
	uint32_t stack[kMaxDepth];
	Hit h;
	float facc[3] = { dx, dy, dz };
	uint32_t iacc[3] = { ray.px, ray.py, ray.pz };
	if (fast_path_ok(cam.ox, cam.oy, cam.oz, ray))
	{
		FastWalker<false> w;
		w.start(root, miss_t, ray);
		for (;;)
		{
			const uint32_t child = w.load_child(nodes_m1);
#pragma unroll
			for (int k = 0; k < PROBE_FMA; ++k)
				asm volatile("fma.rn.f32 %0, %0, %1, %2;" : "+f"(facc[k % 3]) : "f"(w.cx), "f"(w.bx));
#pragma unroll
			for (int k = 0; k < PROBE_ALU; ++k)
				asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(iacc[k % 3]) : "r"(w.idx), "r"(w.inv));
			if (child ? w.descend(child, depth, stack) : w.advance(stack))
				break;
		}
		h = w.hit;
	}
	else
		h = traverse(nodes_m1, root, depth, miss_t, ray, stack);
	if (facc[0] + facc[1] + facc[2] == 1.2345e-30f || (iacc[0] ^ iacc[1] ^ iacc[2]) == 0xDEADBEEFu)
		h.voxel ^= 0x80000000u;                                                  // never true; keeps the probes alive

	const size_t i = static_cast<size_t>(r) * fr.W + x;
	voxel[i] = h.voxel;
	face[i] = static_cast<uint8_t>(h.face);
	t[i] = h.t;
}

// Experiment kernel for the SIMT-efficiency question (variant 4): "deferred phases".  In the default kernel every
// round of the loop runs the descend block for the lanes whose child exists AND the advance block for the lanes
// whose child is empty -- each with about two thirds of the warp.  Here a phase that fewer than `threshold` lanes
// want is postponed (those lanes keep their loaded child and wait) as long as the other phase has enough takers, in
// the hope that the stragglers' phase fills up.  Costs two ballots per round.
template<bool COUNT>
__global__ void __launch_bounds__(256)
trace_frame_deferred_kernel(const uint32_t* __restrict__ nodes_m1, uint32_t root, int depth, float miss_t, RcpTable rt, Camera cam, FrameRows fr,
                            int threshold,
                            uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* __restrict__ t, uint16_t* __restrict__ npush)
{
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int x = blockIdx.x * 16 + (warp & 1) * 8 + (lane & 7);
	const int r = blockIdx.y * 16 + (warp >> 1) * 4 + (lane >> 3);
	const bool valid = x < fr.W && r < fr.rows;
	const int y = frame_row(fr, r);

	float dx, dy, dz;
	camera_ray(cam, x, y, dx, dy, dz);
	const Ray ray = ray_setup(rt, cam.ox, cam.oy, cam.oz, dx, dy, dz);
	uint32_t stack[kMaxDepth];
	FastWalker<COUNT> w;
	w.start(root, miss_t, ray);
	int st = 0;                       // 0 load next child, 1 wants descend (child held), 2 wants advance, 3 finished
	uint32_t child = 0;
	if (!valid)
		st = 3;
	else if (!fast_path_ok(cam.ox, cam.oy, cam.oz, ray))
	{
		w.hit = traverse(nodes_m1, root, depth, miss_t, ray, stack);
		st = 3;
	}

	for (;;)
	{
		if (st == 0)
		{
			child = w.load_child(nodes_m1);
			st = child ? 1 : 2;
		}
		const unsigned md = __ballot_sync(0xFFFFFFFFu, st == 1), ma = __ballot_sync(0xFFFFFFFFu, st == 2);
		if ((md | ma) == 0u)
			break;
		const int nd = __popc(md), na = __popc(ma);
		const bool run_d = nd >= threshold || na < threshold;
		const bool run_a = na >= threshold || nd < threshold;
		if (run_d && st == 1) st = w.descend(child, depth, stack) ? 3 : 0;
		if (run_a && st == 2) st = w.advance(stack) ? 3 : 0;
	}

	if (valid)
	{
		const size_t i = static_cast<size_t>(r) * fr.W + x;
		voxel[i] = w.hit.voxel;
		face[i] = static_cast<uint8_t>(w.hit.face);
		t[i] = w.hit.t;
		if (COUNT) npush[i] = static_cast<uint16_t>(min(w.hit.npush, 65535u));
	}
}

// Experiment kernel for the "upper levels in shared memory" question: 1024-thread blocks (a 32 x 32 pixel tile,
// warps still 8 x 4) copy the first n_staged nodes -- the top levels, a contiguous prefix of the level-ordered
// array -- into shared memory and serve PUSHes on those nodes from there.  Only valid in the h_octree layout.
// Kept selectable (variant 3) so that the decision can be re-measured; see DESIGN.md section 4 for the numbers.
template<bool COUNT>
__global__ void __launch_bounds__(1024)
trace_frame_staged_kernel(const uint32_t* __restrict__ nodes_m1, uint32_t root, int depth, float miss_t, RcpTable rt, Camera cam, FrameRows fr,
                          uint32_t n_staged,
                          uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* __restrict__ t, uint16_t* __restrict__ npush)
{
	extern __shared__ uint4 s_raw[];
	uint32_t* s_nodes = reinterpret_cast<uint32_t*>(s_raw);
	{
		const uint4* src = reinterpret_cast<const uint4*>(nodes_m1 + 8);            // id 1
		for (uint32_t i = threadIdx.x; i < 2u * n_staged; i += blockDim.x) s_raw[i] = __ldg(src + i);
	}
	__syncthreads();
	const uint32_t* s_nodes_m1 = s_nodes - 8;

	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int x = blockIdx.x * 32 + (warp & 3) * 8 + (lane & 7);
	const int r = blockIdx.y * 32 + (warp >> 2) * 4 + (lane >> 3);
	if (x >= fr.W || r >= fr.rows) return;
	const int y = frame_row(fr, r);

	float dx, dy, dz;
	camera_ray(cam, x, y, dx, dy, dz);
	const Ray ray = ray_setup(rt, cam.ox, cam.oy, cam.oz, dx, dy, dz);
	uint32_t stack[kMaxDepth];
	Hit h;
	if (fast_path_ok(cam.ox, cam.oy, cam.oz, ray))
	{
		FastWalker<COUNT> w;
		w.start(root, miss_t, ray);
		while (!w.iterate_staged(nodes_m1, depth, stack, s_nodes_m1, n_staged)) {}
		h = w.hit;
	}
	else
		h = traverse(nodes_m1, root, depth, miss_t, ray, stack);

	const size_t i = static_cast<size_t>(r) * fr.W + x;
	voxel[i] = h.voxel;
	face[i] = static_cast<uint8_t>(h.face);
	t[i] = h.t;
	if (COUNT) npush[i] = static_cast<uint16_t>(min(h.npush, 65535u));
}

// Variants 14 - 19: experiments in the product kernel's shape -- same tile mapping, same tiers; what differs is the
// round (WALKER: FlatWalker = straight-line round, V4Walker = 128-bit half-node fetch, LeanWalker = the product's), the
// loop shape (LOOP 0: one child load, then descend OR advance, as the product; 1: "while-while", every lane advances
// over empty slots until it holds a child, then the warp descends together; 2: every lane descends while it finds
// children, then advances once), where the parent stack lives (LOCAL_STACK: a local-memory array instead of the
// shared-memory column) and the register budget (MINB resident blocks per SM).
template<int SHIFT>
struct LocalLeanStack
{
	uint32_t* e;                                     // kMaxDepth entries of local memory
	__device__ __forceinline__ void store(float dimf, uint32_t w) const { e[(__float_as_uint(dimf) >> 23) - (127u - kMaxDepth)] = w; }
	__device__ __forceinline__ uint32_t load(float dimf) const { return e[(__float_as_uint(dimf) >> 23) - (127u - kMaxDepth)]; }
};

template<template<bool> class WALKER, bool COUNT, int LOOP, bool LOCAL_STACK, int MINB>
__global__ void __launch_bounds__(256, MINB)
trace_frame_walker_kernel(const Dag g, Camera cam, FrameRows fr,
                          uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* __restrict__ t, uint16_t* __restrict__ npush)
{
	extern __shared__ uint32_t s_stack[];
	int x, r;
	if (!frame_pixel(fr, blockIdx.y, gridDim.y, x, r)) return;
	const int y = frame_row(fr, r);

	float dx, dy, dz;
	camera_ray(cam, x, y, dx, dy, dz);
	const Ray ray = ray_setup(g.rt, cam.ox, cam.oy, cam.oz, dx, dy, dz, g.plane_mask);
	Hit h;
	if (fast_path_ok(cam.ox, cam.oy, cam.oz, ray) && lean_path_ok(ray))
	{
		WALKER<COUNT> w;
		w.start(g.root, ray);
		uint32_t lstack[kMaxDepth];
		auto run = [&](auto st) {
			if (LOOP == 1)
			{
				for (;;)
				{
					uint32_t child;
					bool done = false;
					while ((child = w.load_child(g.base_biased)) == 0u)
						if (w.advance(g.miss_t, st)) { done = true; break; }
					if (done || w.descend(child, g.leaf_dimf, st)) break;
				}
			}
			else if (LOOP == 2)
			{
				for (;;)
				{
					uint32_t child;
					bool done = false;
					while ((child = w.load_child(g.base_biased)) != 0u)
						if (w.descend(child, g.leaf_dimf, st)) { done = true; break; }
					if (done || w.advance(g.miss_t, st)) break;
				}
			}
			else
				while (!w.round(g.base_biased, g.leaf_dimf, g.miss_t, st)) {}
		};
		if (LOCAL_STACK) run(LocalLeanStack<0>{ lstack });
		else             run(LeanStack<kLeanShift>{ lean_stack_base(s_stack, g.depth) });
		h = w.hit;
	}
	else
		h = traverse_variant<1, COUNT>(g.nodes_m1, g.root, g.depth, g.miss_t, cam.ox, cam.oy, cam.oz, ray);

	const size_t i = static_cast<size_t>(r) * fr.W + x;
	voxel[i] = h.voxel;
	face[i] = static_cast<uint8_t>(h.face);
	t[i] = h.t;
	if (COUNT) npush[i] = static_cast<uint16_t>(min(h.npush, 65535u));
}

// Variants 24-27: the round-2 walkers and loop shapes again, now WITH the beam start (ort_beam.cuh) -- the product's frame
// kernel with the walker and the loop as parameters.  The beam start removes the coherent rounds (all lanes descend, or all
// advance), which are the ones the branchy round is cheap on; what is left is the split walk near the surface, where the
// straight-line round (FlatWalker) and the other loop shapes might compare differently than they did in
// profiles/r2_loop_shapes.json / r2_v14_straight_line_ncu_full.md.  LOOP: 0 one round() per iteration, 1 advance-while,
// 2 descend-while (= the product).
// GUARD: 0 the product's retry loop around the walk, 1 a slow-path call after the walk (FastWalker from the origin), 2 no
// guard at all (measurement only: what the guard costs).  MINB: resident blocks per SM the register budget allows for.
template<template<bool> class WALKER, bool COUNT, int LOOP, int GUARD = 0, int MINB = 6>
__global__ void __launch_bounds__(256, MINB)
trace_frame_walker_beam_kernel(const Dag g, Camera cam, FrameRows fr,
                               uint32_t* __restrict__ voxel, uint8_t* __restrict__ face, float* t, uint16_t* __restrict__ npush)
{
	extern __shared__ uint32_t s_stack[];
	int x, r;
	const bool inside = frame_pixel(fr, blockIdx.y, gridDim.y, x, r);
	const float tau = read_tile_start(fr, t, x, r);
	if (!inside) return;
	const size_t i = static_cast<size_t>(r) * fr.W + x;
	if (__float_as_uint(tau) == kBeamAllMissBits)
	{
		voxel[i] = 0u;
		face[i] = 6;
		t[i] = g.miss_t;
		if (COUNT) npush[i] = 0;
		return;
	}
	const int y = frame_row(fr, r);
	float dx, dy, dz;
	camera_ray(cam, x, y, dx, dy, dz);
	const Ray ray = ray_setup_camera(g.rt, cam.ox, cam.oy, cam.oz, dx, dy, dz, cam.origin_flags);
	Hit h;
	if ((cam.origin_flags & kOriginInCube) != 0u && lean_path_ok(ray))
	{
		WALKER<COUNT> w;
		const LeanStack<kLeanShift> st{ lean_stack_base(s_stack, g.depth) };
		bool beam_used;
		bool done = lean_start(w, g.root, ray, tau, g.miss_t, beam_used);
		while (!done)
		{
			if (LOOP == 1)
			{
				for (;;)
				{
					uint32_t child;
					bool end = false;
					while ((child = w.load_child(g.base_biased)) == 0u)
						if (w.advance(g.miss_t, st)) { end = true; break; }
					if (end || w.descend(child, g.leaf_dimf, st)) break;
				}
			}
			else if (LOOP == 2)
			{
				for (;;)
				{
					uint32_t child;
					bool end = false;
					while ((child = w.load_child(g.base_biased)) != 0u)
						if (w.descend(child, g.leaf_dimf, st)) { end = true; break; }
					if (end || w.advance(g.miss_t, st)) break;
				}
			}
			else
				while (!w.round(g.base_biased, g.leaf_dimf, g.miss_t, st)) {}
			done = GUARD != 0 || !(beam_used && w.mti == 8u);          // the beam guard (see walk_ray)
			if (!done) { beam_used = false; w.start(g.root, ray); }
		}
		h = w.hit;
		if (GUARD == 1 && beam_used && w.mti == 8u)
			h = traverse_variant<1, COUNT>(g.nodes_m1, g.root, g.depth, g.miss_t, cam.ox, cam.oy, cam.oz, ray);
	}
	else
		h = traverse_variant<1, COUNT>(g.nodes_m1, g.root, g.depth, g.miss_t, cam.ox, cam.oy, cam.oz, ray);

	voxel[i] = h.voxel;
	face[i] = static_cast<uint8_t>(h.face);
	t[i] = h.t;
	if (COUNT) npush[i] = static_cast<uint16_t>(min(h.npush, 65535u));
}

}  // namespace ort

// ------------------------------------------------------------------------------------------------
// dispatch (called from ort_trace_frame_async when an experiment variant / shape option is selected)
// ------------------------------------------------------------------------------------------------

// returns ORT_OK after launching, or -1 when the options do not select an experiment (the caller then launches the
// product kernel)
static int launch_frame_experiment(ort_ctx* c, const ort::Dag& g, const ort::Camera& cam, const ort::FrameRows& fr,
                                   uint32_t* voxel, uint8_t* face, float* t, uint16_t* npush)
{
	const uint32_t* nodes_m1 = g.nodes_m1;
	const ort::RcpTable rt = g.rt;
	const int W = fr.W, rows = fr.rows;
	const dim3 grid((W + 15) / 16, (rows + 15) / 16);
	const int v = c->opt_variant;
	if (v == 5 || v == 6)
	{
		const bool ww = v == 6;
		auto k = npush ? (ww ? ort::trace_frame_tight_kernel<true, true> : ort::trace_frame_tight_kernel<true, false>)
		               : (ww ? ort::trace_frame_tight_kernel<false, true> : ort::trace_frame_tight_kernel<false, false>);
		k<<<grid, 256, 0, c->stream>>>(nodes_m1, g.root, g.depth, g.miss_t, rt, cam, fr, voxel, face, t, npush);
	}
	else if (v == 12)
	{
		unsigned long long* counter = next_counter(c);
		if (cudaMemsetAsync(counter, 0, sizeof(unsigned long long), c->stream) != cudaSuccess) return ORT_ERR_CUDA;
		const unsigned n_tiles = static_cast<unsigned>(grid.x) * grid.y * 8u;
		const unsigned pblocks = grid.x * grid.y < static_cast<unsigned>(c->sm_count * 8) ? grid.x * grid.y : static_cast<unsigned>(c->sm_count * 8);
		if (npush) ort::trace_frame_tiles_kernel<true><<<pblocks, 256, 0, c->stream>>>(nodes_m1, g.root, g.depth, g.miss_t, rt, cam, fr, n_tiles, reinterpret_cast<unsigned int*>(counter), voxel, face, t, npush);
		else       ort::trace_frame_tiles_kernel<false><<<pblocks, 256, 0, c->stream>>>(nodes_m1, g.root, g.depth, g.miss_t, rt, cam, fr, n_tiles, reinterpret_cast<unsigned int*>(counter), voxel, face, t, npush);
	}
	else if (v == 7)
	{
		if (npush) ort::trace_frame_pipe_kernel<true><<<grid, 256, 0, c->stream>>>(nodes_m1, g.base_biased, g.root, g.depth, g.miss_t, rt, cam, fr, voxel, face, t, npush);
		else       ort::trace_frame_pipe_kernel<false><<<grid, 256, 0, c->stream>>>(nodes_m1, g.base_biased, g.root, g.depth, g.miss_t, rt, cam, fr, voxel, face, t, npush);
	}
	else if (v >= 8 && v <= 11 && !npush)
	{
		// probes: 8 = +6 FMA-pipe, 9 = +6 ALU-pipe, 10 = +12 FMA-pipe, 11 = +0 (the same loop shape without extra work)
		auto k = v == 8 ? ort::trace_frame_probe_kernel<6, 0> : v == 9 ? ort::trace_frame_probe_kernel<0, 6>
		       : v == 10 ? ort::trace_frame_probe_kernel<12, 0> : ort::trace_frame_probe_kernel<0, 0>;
		k<<<grid, 256, 0, c->stream>>>(nodes_m1, g.root, g.depth, g.miss_t, rt, cam, fr, voxel, face, t);
	}
	else if (v == 4)
	{
		const int thr = c->opt_low_water > 0 ? c->opt_low_water : 1;
		if (npush) ort::trace_frame_deferred_kernel<true><<<grid, 256, 0, c->stream>>>(nodes_m1, g.root, g.depth, g.miss_t, rt, cam, fr, thr, voxel, face, t, npush);
		else       ort::trace_frame_deferred_kernel<false><<<grid, 256, 0, c->stream>>>(nodes_m1, g.root, g.depth, g.miss_t, rt, cam, fr, thr, voxel, face, t, npush);
	}
	else if (v == 3 && c->index_base == 1)
	{
		// upper levels staged in shared memory: opt_smem_levels = number of node ids to stage (the harness passes
		// the first id of level k+1 from ort_tree_flatten's level offsets, minus one)
		uint32_t n_staged = c->opt_smem_levels > 0 ? static_cast<uint32_t>(c->opt_smem_levels) : 0u;
		if (n_staged > c->n_nodes) n_staged = c->n_nodes;
		if (n_staged > 6144u) n_staged = 6144u;                         // 192 KB of the 227 KB a block may have
		const size_t smem = static_cast<size_t>(n_staged) * 32;
		const dim3 g2((W + 31) / 32, (rows + 31) / 32);
		if (npush)
		{
			if (cudaFuncSetAttribute(ort::trace_frame_staged_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess) return ORT_ERR_CUDA;
			ort::trace_frame_staged_kernel<true><<<g2, 1024, smem, c->stream>>>(nodes_m1, g.root, g.depth, g.miss_t, rt, cam, fr, n_staged, voxel, face, t, npush);
		}
		else
		{
			if (cudaFuncSetAttribute(ort::trace_frame_staged_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess) return ORT_ERR_CUDA;
			ort::trace_frame_staged_kernel<false><<<g2, 1024, smem, c->stream>>>(nodes_m1, g.root, g.depth, g.miss_t, rt, cam, fr, n_staged, voxel, face, t, npush);
		}
	}
	else if (v >= 14 && v <= 19 && lean_capable(c))
	{
		// 14 straight-line round, 15 128-bit fetches, 16 while-while, 17 descend-while, 18 parent stack in local memory,
		// 19 register budget of 6 resident blocks per SM (40 registers)
		const size_t smem = v == 18 ? 0 : ort::lean_smem_bytes(g.depth);
#define ORT_WALKER_KERNEL(W, L, LS, MB) (npush ? ort::trace_frame_walker_kernel<W, true, L, LS, MB> : ort::trace_frame_walker_kernel<W, false, L, LS, MB>)
		auto k = v == 14 ? ORT_WALKER_KERNEL(ort::FlatWalker, 0, false, 1) : v == 15 ? ORT_WALKER_KERNEL(ort::V4Walker, 0, false, 1)
		       : v == 16 ? ORT_WALKER_KERNEL(ort::LeanWalker, 1, false, 1) : v == 17 ? ORT_WALKER_KERNEL(ort::LeanWalker, 2, false, 1)
		       : v == 18 ? ORT_WALKER_KERNEL(ort::LeanWalker, 0, true, 1) : ORT_WALKER_KERNEL(ort::LeanWalker, 0, false, 6);
#undef ORT_WALKER_KERNEL
		k<<<grid, 256, smem, c->stream>>>(g, cam, fr, voxel, face, t, npush);
	}
	else if (v >= 24 && v <= 31 && lean_capable(c))
	{
		// 24 straight-line round, 25 plain round, 26 advance-while, 27 descend-while -- each with the beam start where the launch
		// qualifies for one (else the same walker without: variants 14 / 19-like)
		const int bk = beam_level_any_variant(c, cam, fr, npush != nullptr);
		const size_t smem = ort::lean_smem_bytes(g.depth);
		if (bk)
		{
			const int rc = beam_launch_march(c, bk, cam, fr, t, npush != nullptr);
			if (rc != ORT_OK) return ORT_ERR_CUDA;
#define ORT_BEAM_KERNEL(W, L) (npush ? ort::trace_frame_walker_beam_kernel<W, true, L> : ort::trace_frame_walker_beam_kernel<W, false, L>)
			// 28-31: the product's walker and loop with the guard as a slow-path call / without a guard / other register budgets
#define ORT_BEAM_KERNEL2(G, MB) (npush ? ort::trace_frame_walker_beam_kernel<ort::LeanWalker, true, 2, G, MB> : ort::trace_frame_walker_beam_kernel<ort::LeanWalker, false, 2, G, MB>)
			auto k = v == 24 ? ORT_BEAM_KERNEL(ort::FlatWalker, 0) : v == 25 ? ORT_BEAM_KERNEL(ort::LeanWalker, 0)
			       : v == 26 ? ORT_BEAM_KERNEL(ort::LeanWalker, 1) : v == 27 ? ORT_BEAM_KERNEL(ort::LeanWalker, 2)
			       : v == 28 ? ORT_BEAM_KERNEL2(1, 6) : v == 29 ? ORT_BEAM_KERNEL2(2, 6) : v == 30 ? ORT_BEAM_KERNEL2(0, 5) : ORT_BEAM_KERNEL2(0, 8);
#undef ORT_BEAM_KERNEL2
#undef ORT_BEAM_KERNEL
			k<<<grid, 256, smem, c->stream>>>(g, cam, fr, voxel, face, t, npush);
		}
		else
		{
			// a launch without a beam level (PUSH counts of the reference walk, coarse pixels, ...): the same walker and loop from the origin
#define ORT_WALKER_KERNEL(W, L) (npush ? ort::trace_frame_walker_kernel<W, true, L, false, 6> : ort::trace_frame_walker_kernel<W, false, L, false, 6>)
			auto k = v == 24 ? ORT_WALKER_KERNEL(ort::FlatWalker, 0) : v == 25 ? ORT_WALKER_KERNEL(ort::LeanWalker, 0)
			       : v == 26 ? ORT_WALKER_KERNEL(ort::LeanWalker, 1) : ORT_WALKER_KERNEL(ort::LeanWalker, 2);      // (27-31)
#undef ORT_WALKER_KERNEL
			k<<<grid, 256, smem, c->stream>>>(g, cam, fr, voxel, face, t, npush);
		}
	}
	else if (v == 1 && (c->opt_tile_shape != 0 || c->opt_block == 128 || c->opt_block == 64))
	{
		// block = 16 x 16 pixels by default; options "block" = 128 / 64 (16 x 8 / 16 x 4) and "tile_shape" select other mappings
		const int fblock = c->opt_tile_shape == 0 ? c->opt_block : 256;
		const dim3 fgrid = c->opt_tile_shape == 3 ? dim3((W + 31) / 32, (rows + 7) / 8) : dim3((W + 15) / 16, (rows + fblock / 16 - 1) / (fblock / 16));
		if (npush) ort::trace_frame_shaped_kernel<true><<<fgrid, fblock, 0, c->stream>>>(nodes_m1, g.root, g.depth, g.miss_t, rt, cam, fr, voxel, face, t, npush);
		else       ort::trace_frame_shaped_kernel<false><<<fgrid, fblock, 0, c->stream>>>(nodes_m1, g.root, g.depth, g.miss_t, rt, cam, fr, voxel, face, t, npush);
	}
	else
		return -1;
	++c->launches;
	if (cudaGetLastError() != cudaSuccess) return ORT_ERR_CUDA;
	return ORT_OK;
}
