// ort_query.cuh -- voxels read back from the device DAG: batched at() (ort_voxels_at) and dense boxes (ort_read_voxels),
// DESIGN section 14.
//
// Both walk the mirror as och::h_octree::at (och_h_octree.h:239-258) and och::octree::at (och_octree.cpp:141-160) do:
// from the root, level depth-1 down to 1, child slot = bit l of x | bit l of y << 1 | bit l of z << 2, then the leaf
// row's word of bit 0.  Only the low `depth` bits of a coordinate take part, which is at()'s uint16 cast followed by
// its depth-bit key, so any int32 coordinate wraps exactly as there.
//
// Bounds guard: a walk never loads outside the mirror's rows.  QueryDag::lim is one past the last valid node id
// (n_nodes + index_base), or 0 when the context holds no tree; an interior child 0 or >= lim reads as empty.  That is
// one unsigned compare per level (child - 1 >= lim - 1).  The trace kernels do not check this.
//
// Everything above the __global__ kernels is plain per-point / per-cell code that tests/host_emu/emu_query.cpp compiles
// for the host.
#pragma once

namespace ort {

struct QueryDag
{
	const uint32_t* nodes_m1;   // make_dag's: row of node id i at nodes_m1 + 8 * i (both layouts)
	uint32_t root;              // compact id (h_octree layout) or row 0 (pool layout)
	uint32_t lim;               // valid ids are < lim; 0 = no tree (never uploaded, or an h_octree mirror with root 0)
	int depth;
};

// A box of voxels [x0, x0+nx) x [y0, y0+ny) x [z0, z0+nz) inside the cube, written densely: voxel (x, y, z) at
// ((z - z0) * ny + (y - y0)) * nx + (x - x0).
struct QueryBox
{
	uint32_t x0, y0, z0, nx, ny, nz;
};

// The leaf row holding voxel (x, y, z), or nullptr where the walk meets an empty (or out-of-range) child first.
__device__ __forceinline__ const uint32_t* query_leaf_row(const QueryDag& g, uint32_t x, uint32_t y, uint32_t z)
{
	if (g.root >= g.lim) return nullptr;
	uint32_t node = g.root;
	for (int l = g.depth - 1; l > 0; --l)
	{
		const uint32_t slot = ((x >> l) & 1u) | (((y >> l) & 1u) << 1) | (((z >> l) & 1u) << 2);
		const uint32_t child = __ldg(g.nodes_m1 + (static_cast<size_t>(node) << 3) + slot);
		if (child - 1u >= g.lim - 1u) return nullptr;          // 0 = empty; >= lim: past the mirror's rows
		node = child;
	}
	return g.nodes_m1 + (static_cast<size_t>(node) << 3);
}

// at(x, y, z) on the device mirror
__device__ __forceinline__ uint32_t query_voxel(const QueryDag& g, int32_t x, int32_t y, int32_t z)
{
	const uint32_t ux = static_cast<uint32_t>(x), uy = static_cast<uint32_t>(y), uz = static_cast<uint32_t>(z);
	const uint32_t* row = query_leaf_row(g, ux, uy, uz);
	return row ? __ldg(row + ((ux & 1u) | ((uy & 1u) << 1) | ((uz & 1u) << 2))) : 0u;
}

// the two voxels x, x+1 (x even) of one output row of the box, where they lie inside it
__device__ __forceinline__ void query_store_pair(const QueryBox& b, uint32_t* out, uint32_t x, uint32_t y, uint32_t z, uint32_t v0, uint32_t v1)
{
	if (y < b.y0 || y - b.y0 >= b.ny || z < b.z0 || z - b.z0 >= b.nz) return;
	uint32_t* row = out + (static_cast<size_t>(z - b.z0) * b.ny + (y - b.y0)) * b.nx;
	const bool in0 = x >= b.x0, in1 = x + 1u - b.x0 < b.nx;     // (the cell is cut by the box: x < x0 + nx, x + 1 >= x0)
	if (in0 && in1)
	{
		uint32_t* p = row + (x - b.x0);
		if ((reinterpret_cast<uintptr_t>(p) & 7u) == 0u)
			*reinterpret_cast<uint2*>(p) = make_uint2(v0, v1);
		else
		{
			p[0] = v0;
			p[1] = v1;
		}
	}
	else if (in0)
		row[x - b.x0] = v0;
	else
		row[x + 1u - b.x0] = v1;
}

// The 2 x 2 x 2 leaf cell (cx, cy, cz) -- voxels 2cx .. 2cx+1, ... -- into the box: one descent of depth-1 levels, the
// leaf row as its two 16-byte halves (z = 2cz and z = 2cz + 1; each x-fastest, then y), zeros below an empty subtree.
__device__ __forceinline__ void query_read_cell(const QueryDag& g, const QueryBox& b, uint32_t* out, uint32_t cx, uint32_t cy, uint32_t cz)
{
	const uint32_t x = 2u * cx, y = 2u * cy, z = 2u * cz;
	const uint32_t* row = query_leaf_row(g, x, y, z);
	uint4 lo = { 0u, 0u, 0u, 0u }, hi = { 0u, 0u, 0u, 0u };
	if (row)
	{
		lo = __ldg(reinterpret_cast<const uint4*>(row));
		hi = __ldg(reinterpret_cast<const uint4*>(row) + 1);
	}
	query_store_pair(b, out, x, y, z, lo.x, lo.y);
	query_store_pair(b, out, x, y + 1u, z, lo.z, lo.w);
	query_store_pair(b, out, x, y, z + 1u, hi.x, hi.y);
	query_store_pair(b, out, x, y + 1u, z + 1u, hi.z, hi.w);
}

#ifndef ORT_HOST_EMU

// one thread per point, grid-stride
__global__ void __launch_bounds__(256)
voxels_at_kernel(QueryDag g, const int32_t* __restrict__ xyz, size_t n, uint32_t* __restrict__ out)
{
	const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
	for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
		out[i] = query_voxel(g, __ldg(xyz + 3 * i), __ldg(xyz + 3 * i + 1), __ldg(xyz + 3 * i + 2));
}

// One thread per leaf cell the box cuts.  threadIdx.x / blockIdx.x run along x (consecutive threads store consecutive
// 8-byte pairs of a row); the rows of cells (cy, cz) are shared out over threadIdx.y / blockIdx.y, grid-stride.
// ncx cells along x from cx0, ncy along y from cy0, rows = ncy * ncz in all (< 2^30: the cube has 2^15 cells a side).
__global__ void __launch_bounds__(256)
read_voxels_kernel(QueryDag g, QueryBox b, uint32_t* __restrict__ out, uint32_t cx0, uint32_t ncx, uint32_t cy0, uint32_t ncy, uint32_t cz0, uint32_t rows)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= ncx) return;
	const uint32_t step = gridDim.y * blockDim.y;
	for (uint32_t r = blockIdx.y * blockDim.y + threadIdx.y; r < rows; r += step)
		query_read_cell(g, b, out, cx0 + i, cy0 + r % ncy, cz0 + r / ncy);
}

#endif  // ORT_HOST_EMU

}  // namespace ort
