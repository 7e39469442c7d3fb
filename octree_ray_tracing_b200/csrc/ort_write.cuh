// ort_write.cuh -- a dense box of voxels written into the device DAG (ort_write_voxels, DESIGN section 15).
//
// The result is what ort_tree_flatten returns for a host table holding the old scene with the box replaced.  It reuses
// the builder's intern, numbering and scan kernels (ort_build.cuh) through the content source WriteSrc:
//
//   old DAG, top-down: the distinct old ids reachable at each level (first-occurrence dedup over an array indexed by old
//     id, OldSrc); old_at: the old node at every cell of each level's grid G_l (below).  Children at or past the
//     mirror's rows read as empty, as in ort_query.cuh.
//   bottom-up, l = depth .. 1: one table T_l holds two kinds of entries.  An old node reachable at level l (entry = its
//     position k in the level's list; content = its row with interior children mapped through canon_{l+1}, materialised
//     as mapped_l[k] before the pass), and a touched cell of R_l (entry = kWriteCell | its index in G_l; content = box
//     voxels or old leaf words at the leaf level, the child grid G_{l+1}'s temporary ids above it).  canon_l(old id) is
//     the temporary id of that old node's content.
//   top-down numbering from the new root's temporary id: the builder's frontier pass, unchanged.
//
// Grids.  R_l = the cells of level l that intersect the box (a box of cells); G_1 = R_1 = the root cell and G_l = the
// children of R_{l-1} for l >= 2, so G_l contains R_l plus at most one cell more per side.  A cell of G_l outside R_l
// keeps its old content: its temporary id is canon_l of its old node, filled in after T_l is built.  So a touched cell's
// 8 children are always cells of G_{l+1}, and neither pass ever looks up canon of an id again after its level.
#pragma once

namespace ort {

constexpr uint32_t kWriteCell = 0x80000000u;    // table entry: a cell of G_l (index in the low bits), else an old node's k

// One level's cell grid: G_l's first cell and extent (in cells of the level), temporary ids, old node per cell.
struct WriteGrid
{
	uint32_t ox, oy, oz, gx, gy, gz;
	uint32_t* ids;
	uint32_t* old_at;           // old node id at the cell, 0 = empty (or past the mirror's rows)
	__device__ __forceinline__ size_t index(uint32_t x, uint32_t y, uint32_t z) const { return (static_cast<size_t>(z) * gy + y) * gx + x; }
};

// The old mirror, h_octree layout: row of id i at nodes_m1 + 8 i, valid ids 1 .. lim - 1 (lim = 0: no tree).
struct WriteDag
{
	const uint32_t* nodes_m1;
	uint32_t lim;
	__device__ __forceinline__ uint32_t word(uint32_t node, int c) const { return __ldg(nodes_m1 + (static_cast<size_t>(node) << 3) + c); }
	// interior child c of node: 0 where the row says empty or points past the rows
	__device__ __forceinline__ uint32_t child(uint32_t node, int c) const
	{
		const uint32_t w = word(node, c);
		return w - 1u < lim - 1u ? w : 0u;
	}
};

// The old DAG walked top-down: frontier entries are old ids.
struct OldSrc
{
	WriteDag g;
	__device__ __forceinline__ uint32_t rep(uint32_t t) const { return t; }
	__device__ __forceinline__ uint32_t child(uint32_t e, int c) const { return g.child(e, c); }
};

// Level l of a box write (see the header).
struct WriteSrc
{
	bool leaf;
	BuildInput in;              // the box's voxels, index relative to (bx, by, bz)
	uint32_t bx, by, bz;
	WriteGrid G, C;             // G_l and G_{l+1} (C unused at the leaf level)
	uint32_t rx, ry, rz;        // R_l's first cell within G_l
	uint32_t rgx, rgy, rgz;     // R_l's extent
	WriteDag g;
	const uint32_t* old;        // the old ids reachable at level l, n_old of them
	uint32_t n_old;
	const uint32_t* mapped;     // their contents, 8 words each
	uint32_t* canon;            // canon_l, by old id (written by store)
	const uint32_t* table;      // T_l

	__device__ __forceinline__ size_t items() const { return n_old + static_cast<size_t>(rgx) * rgy * rgz; }
	__device__ __forceinline__ uint32_t entry(size_t i) const
	{
		if (i < n_old) return static_cast<uint32_t>(i);
		const size_t r = i - n_old;
		const uint32_t x = static_cast<uint32_t>(r % rgx), q = static_cast<uint32_t>(r / rgx);
		return kWriteCell | static_cast<uint32_t>(G.index(rx + x, ry + q % rgy, rz + q / rgy));
	}
	// word c of cell e's content
	__device__ __forceinline__ uint32_t cell_word(uint32_t e, int c) const
	{
		const uint32_t i = e & ~kWriteCell;
		const uint32_t x = i % G.gx, q = i / G.gx, y = q % G.gy, z = q / G.gy;
		const uint32_t cx = 2 * (G.ox + x) + (c & 1), cy = 2 * (G.oy + y) + ((c >> 1) & 1), cz = 2 * (G.oz + z) + (c >> 2);
		if (!leaf) return C.ids[C.index(cx - C.ox, cy - C.oy, cz - C.oz)];
		if (cx - bx < in.nx && cy - by < in.ny && cz - bz < in.nz) return in.at(cx - bx, cy - by, cz - bz);
		const uint32_t p = G.old_at[i];
		return p ? g.word(p, c) : 0u;
	}
	__device__ __forceinline__ void content(uint32_t e, uint32_t w[8]) const
	{
		if (e & kWriteCell)
		{
#pragma unroll
			for (int c = 0; c < 8; ++c) w[c] = cell_word(e, c);
		}
		else
		{
			const uint4* m = reinterpret_cast<const uint4*>(mapped + 8 * static_cast<size_t>(e));
			const uint4 lo = m[0], hi = m[1];
			w[0] = lo.x; w[1] = lo.y; w[2] = lo.z; w[3] = lo.w;
			w[4] = hi.x; w[5] = hi.y; w[6] = hi.z; w[7] = hi.w;
		}
	}
	__device__ __forceinline__ void store(size_t i, uint32_t id) const
	{
		if (i < n_old)
			canon[old[i]] = id;
		else
			G.ids[entry(i) & ~kWriteCell] = id;
	}
	__device__ __forceinline__ uint32_t rep(uint32_t t) const { return table[t - 1]; }
	__device__ __forceinline__ uint32_t child(uint32_t e, int c) const
	{
		return (e & kWriteCell) ? cell_word(e, c) : mapped[8 * static_cast<size_t>(e) + c];
	}
};

// old_at of every cell of G (level l >= 2) from its parent's in P = G_{l-1}
__global__ void write_old_at_kernel(WriteGrid P, WriteGrid G, WriteDag g)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= static_cast<size_t>(G.gx) * G.gy * G.gz) return;
	const uint32_t x = static_cast<uint32_t>(i % G.gx), q = static_cast<uint32_t>(i / G.gx), y = q % G.gy, z = q / G.gy;
	const uint32_t ax = G.ox + x, ay = G.oy + y, az = G.oz + z;
	const uint32_t p = P.old_at[P.index((ax >> 1) - P.ox, (ay >> 1) - P.oy, (az >> 1) - P.oz)];
	G.old_at[i] = p ? g.child(p, static_cast<int>((ax & 1u) | ((ay & 1u) << 1) | ((az & 1u) << 2))) : 0u;
}

// mapped_l: the rows of the n old nodes reachable at level l, interior children mapped through canon_{l+1}
__global__ void write_map_kernel(const uint32_t* old, size_t n, WriteDag g, const uint32_t* canon, bool leaf, uint32_t* mapped)
{
	const size_t s = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (s >= 8 * n) return;
	const uint32_t node = old[s >> 3];
	const int c = static_cast<int>(s & 7);
	uint32_t w;
	if (leaf)
		w = g.word(node, c);
	else
	{
		const uint32_t t = g.child(node, c);
		w = t ? canon[t] : 0u;
	}
	mapped[s] = w;
}

// the cells of G_l outside R_l keep their old content: temporary id canon_l of their old node
__global__ void write_fill_kernel(WriteGrid G, uint32_t rx, uint32_t ry, uint32_t rz, uint32_t rgx, uint32_t rgy, uint32_t rgz, const uint32_t* canon)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= static_cast<size_t>(G.gx) * G.gy * G.gz) return;
	const uint32_t x = static_cast<uint32_t>(i % G.gx), q = static_cast<uint32_t>(i / G.gx), y = q % G.gy, z = q / G.gy;
	if (x - rx < rgx && y - ry < rgy && z - rz < rgz) return;        // touched: inserted
	const uint32_t p = G.old_at[i];
	G.ids[i] = p ? canon[p] : 0u;
}

}  // namespace ort
