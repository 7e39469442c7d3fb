// emu_query.cpp -- TEST INFRASTRUCTURE: the per-point and per-cell code of the voxel queries (csrc/ort_query.cuh:
// query_voxel, query_read_cell) compiled for the host through cuda_shim.h, whose __ldg counts every load outside the
// node array.  Built on demand by tests/host_emu/emu_query.py into tests/host_emu/_build/; never part of libort_b200.so.
#include "cuda_shim.h"

struct uint2 { uint32_t x, y; };
static inline uint2 make_uint2(uint32_t x, uint32_t y) { return uint2{ x, y }; }

#include "../../octree_ray_tracing_b200/csrc/ort_query.cuh"

#include <cstddef>

namespace {

// the mirror as the device sees it: n_rows rows; index_base 1 = h_octree compact ids (root = `root`, 0 = no tree),
// 0 = och::octree pool (root = row 0)
ort::QueryDag emu_dag(const uint32_t* nodes8, size_t n_rows, int index_base, uint32_t root, int depth)
{
	g_emu_bounds = EmuBounds{ { reinterpret_cast<const char*>(nodes8), nullptr }, { reinterpret_cast<const char*>(nodes8 + 8 * n_rows), nullptr }, 0 };
	const bool has_root = index_base == 0 || root != 0;
	return ort::QueryDag{ nodes8 - 8 * index_base, index_base ? root : 0u, has_root ? static_cast<uint32_t>(n_rows) + static_cast<uint32_t>(index_base) : 0u, depth };
}

}  // namespace

extern "C" {

// out[i] = query_voxel at xyz[3i..3i+2]; returns the number of loads outside the node array
unsigned long long emu_voxels_at(const uint32_t* nodes8, size_t n_rows, int index_base, uint32_t root, int depth,
                                 const int32_t* xyz, size_t n, uint32_t* out)
{
	const ort::QueryDag g = emu_dag(nodes8, n_rows, index_base, root, depth);
	for (size_t i = 0; i < n; ++i)
		out[i] = ort::query_voxel(g, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]);
	return g_emu_bounds.violations;
}

// the box into out as read_voxels_kernel writes it: query_read_cell for every leaf cell the box cuts
unsigned long long emu_read_voxels(const uint32_t* nodes8, size_t n_rows, int index_base, uint32_t root, int depth,
                                   uint32_t x0, uint32_t y0, uint32_t z0, uint32_t nx, uint32_t ny, uint32_t nz, uint32_t* out)
{
	const ort::QueryDag g = emu_dag(nodes8, n_rows, index_base, root, depth);
	const ort::QueryBox b{ x0, y0, z0, nx, ny, nz };
	for (uint32_t cz = z0 >> 1; cz <= (z0 + nz - 1) >> 1; ++cz)
		for (uint32_t cy = y0 >> 1; cy <= (y0 + ny - 1) >> 1; ++cy)
			for (uint32_t cx = x0 >> 1; cx <= (x0 + nx - 1) >> 1; ++cx)
				ort::query_read_cell(g, b, out, cx, cy, cz);
	return g_emu_bounds.violations;
}

}  // extern "C"
