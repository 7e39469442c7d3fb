// ort_patch.cuh -- a dense box of voxels patched into the device DAG in place (ort_patch_voxels, DESIGN section 16).
//
// Append-only: rows 1 .. n_old are never written; the nodes the box changes are appended as new ids and the root is
// replaced.  The cost is O(cells the box cuts x depth), not O(scene):
//
//   patch index: one open-addressing table per level of row ids keyed by the row's 8 words (rows are immutable, so a
//     compare reads the mirror); ties go to the smallest id.  Built from the reachable DAG by the first patch after the
//     mirror changed by another route, then only appended to.
//   old_at: the old node under every cell of R_l (the cells of level l the box cuts), top-down (write_old_at_kernel).
//   bottom-up, l = depth .. 1, all on the device: R_l's cells are interned in a call-local table (build_insert_kernel over
//     PatchSrc); the first cell of each content (raster order) probes the patch index; the misses are ranked by an
//     exclusive scan and become rows base_l + rank, where base_l (= n_old + 1 + rows appended at lower levels) is read
//     from device memory; every cell gets its final id.  A content of all zeros is id 0 and no row.
//
// Content of a cell of R_l: at the leaf level the box's voxels inside the box and the old leaf row's words outside it;
// above it word c is the final id of child c when that child is in R_{l+1}, else the old node's child c verbatim (an
// untouched subtree is unchanged).  A child at or past the old rows reads as empty (WriteDag::child).
#pragma once

namespace ort {

// One level's patch index: row ids, kBuildEmpty = free.
struct PatchIndex
{
	uint32_t* table;
	uint32_t mask;
};

__device__ __forceinline__ void patch_row(const uint32_t* nodes_m1, uint32_t id, uint32_t w[8])
{
	const uint4* r = reinterpret_cast<const uint4*>(nodes_m1 + (static_cast<size_t>(id) << 3));
	const uint4 lo = __ldg(r), hi = __ldg(r + 1);
	w[0] = lo.x; w[1] = lo.y; w[2] = lo.z; w[3] = lo.w;
	w[4] = hi.x; w[5] = hi.y; w[6] = hi.z; w[7] = hi.w;
}

__device__ __forceinline__ bool patch_row_is(const uint32_t* nodes_m1, uint32_t id, const uint32_t w[8])
{
	uint32_t v[8];
	patch_row(nodes_m1, id, v);
	bool same = true;
#pragma unroll
	for (int c = 0; c < 8; ++c) same &= v[c] == w[c];
	return same;
}

// Enter row id into the index; a row of equal content already there keeps the entry if its id is smaller.
__device__ __forceinline__ void patch_index_insert(PatchIndex ix, const uint32_t* nodes_m1, uint32_t id)
{
	uint32_t w[8];
	patch_row(nodes_m1, id, w);
	uint32_t slot = build_hash(w) & ix.mask;
	for (;;)
	{
		uint32_t e = ix.table[slot];
		if (e == kBuildEmpty)
		{
			e = atomicCAS(ix.table + slot, kBuildEmpty, id);
			if (e == kBuildEmpty) return;
		}
		if (patch_row_is(nodes_m1, e, w))            // (an entry only ever changes to an id of the same content)
		{
			atomicMin(ix.table + slot, id);
			return;
		}
		slot = (slot + 1) & ix.mask;
	}
}

// The id the index holds for content w, 0 when none.
__device__ __forceinline__ uint32_t patch_index_find(PatchIndex ix, const uint32_t* nodes_m1, const uint32_t w[8])
{
	uint32_t slot = build_hash(w) & ix.mask;
	for (;;)
	{
		const uint32_t e = ix.table[slot];
		if (e == kBuildEmpty) return 0u;
		if (patch_row_is(nodes_m1, e, w)) return e;
		slot = (slot + 1) & ix.mask;
	}
}

// index build: the n rows ids[0, n)
__global__ void patch_index_build_kernel(const uint32_t* ids, size_t n, PatchIndex ix, const uint32_t* nodes_m1)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i < n) patch_index_insert(ix, nodes_m1, ids[i]);
}

// index growth: every entry of the old table into the new one
__global__ void patch_index_rehash_kernel(const uint32_t* old_table, size_t old_cap, PatchIndex ix, const uint32_t* nodes_m1)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= old_cap) return;
	const uint32_t e = old_table[i];
	if (e != kBuildEmpty) patch_index_insert(ix, nodes_m1, e);
}

struct PatchIndexSet
{
	PatchIndex ix[kMaxDepth + 1];               // level 1 .. depth
	int depth;
};

// The rows a patch appended enter the index.  first[l] (device memory) is level l's first new id, so level l appended
// first[l] .. first[l - 1] - 1; thread k takes id first[depth] + k.  Nothing enters when the last id passes kIdMask
// (the call is refused).
__global__ void patch_index_append_kernel(const uint32_t* first, PatchIndexSet s, const uint32_t* nodes_m1)
{
	const size_t k = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	const uint32_t end = first[0];
	if (end - 1u > kIdMask) return;
	const uint32_t id = first[s.depth] + static_cast<uint32_t>(k);
	if (id >= end) return;
	int l = s.depth;
	while (id >= first[l - 1]) --l;
	patch_index_insert(s.ix[l], nodes_m1, id);
}

// Level l of a patch (see the header).  R = R_l (ids: temporary, then final), C = R_{l+1} (final ids; unused at the leaf).
struct PatchSrc
{
	bool leaf;
	BuildInput in;              // the box's voxels, index relative to (bx, by, bz)
	uint32_t bx, by, bz;
	WriteGrid R, C;
	WriteDag g;

	__device__ __forceinline__ size_t items() const { return static_cast<size_t>(R.gx) * R.gy * R.gz; }
	__device__ __forceinline__ uint32_t entry(size_t i) const { return static_cast<uint32_t>(i); }
	__device__ __forceinline__ void content(uint32_t e, uint32_t w[8]) const
	{
		const uint32_t x = e % R.gx, q = e / R.gx, y = q % R.gy, z = q / R.gy;
		const uint32_t p = R.old_at[e];
#pragma unroll
		for (int c = 0; c < 8; ++c)
		{
			const uint32_t cx = 2 * (R.ox + x) + (c & 1), cy = 2 * (R.oy + y) + ((c >> 1) & 1), cz = 2 * (R.oz + z) + (c >> 2);
			if (leaf)
				w[c] = cx - bx < in.nx && cy - by < in.ny && cz - bz < in.nz ? in.at(cx - bx, cy - by, cz - bz) : (p ? g.word(p, c) : 0u);
			else
				w[c] = cx - C.ox < C.gx && cy - C.oy < C.gy && cz - C.oz < C.gz ? C.ids[C.index(cx - C.ox, cy - C.oy, cz - C.oz)] : (p ? g.child(p, c) : 0u);
		}
	}
	__device__ __forceinline__ void store(size_t i, uint32_t id) const { R.ids[i] = id; }
};

// Start of a patch: the root cell's old node, and the first id level `depth` appends.
__global__ void patch_begin_kernel(uint32_t* root_old_at, uint32_t old_root, uint32_t* first_id, uint32_t n_old)
{
	*root_old_at = old_root;
	*first_id = n_old + 1;
}

// first[t - 1] = the first cell (raster order) with temporary id t
__global__ void patch_first_kernel(const uint32_t* tmp, size_t n, uint32_t* first)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const uint32_t t = tmp[i];
	if (t) atomicMin(first + (t - 1), static_cast<uint32_t>(i));
}

// The first cell of each content probes the index: hit[i] = the id found (0: none), flag[i] = 1 for a miss.  flag has
// n + 1 entries (the last is 0), so that after the exclusive scan flag[n] is the level's count of new rows.
__global__ void patch_probe_kernel(PatchSrc s, const uint32_t* first, PatchIndex ix, uint32_t* hit, uint32_t* flag)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	const size_t n = s.items();
	if (i > n) return;
	uint32_t f = 0;
	if (i < n)
	{
		const uint32_t t = s.R.ids[i];
		if (t && first[t - 1] == static_cast<uint32_t>(i))
		{
			uint32_t w[8];
			s.content(static_cast<uint32_t>(i), w);
			const uint32_t h = patch_index_find(ix, s.g.nodes_m1, w);
			hit[i] = h;
			f = h == 0u;
		}
	}
	flag[i] = f;
}

// Final ids of R_l and the level's new rows (after the scan: pos = ranks, pos[n] = count).  base[0] is this level's
// first new id; base[-1], the next level's, is base[0] + count.  Rows past `lim` (the mirror's capacity) are not written:
// their ids exceed the id limit and the call is refused.
__global__ void patch_rows_kernel(PatchSrc s, const uint32_t* first, const uint32_t* hit, const uint32_t* pos, uint32_t* base, uint32_t lim,
                                  uint32_t* nodes_m1, uint32_t* root_out)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	const size_t n = s.items();
	const uint32_t b = base[0];
	if (i == 0) base[-1] = b + pos[n];
	if (i >= n) return;
	const uint32_t t = s.R.ids[i];
	uint32_t id = 0;
	if (t)
	{
		const uint32_t f = first[t - 1];
		id = hit[f] ? hit[f] : b + pos[f];
		if (f == static_cast<uint32_t>(i) && !hit[f] && id <= lim)
		{
			uint32_t w[8];
			s.content(static_cast<uint32_t>(i), w);
			uint4* o = reinterpret_cast<uint4*>(nodes_m1 + (static_cast<size_t>(id) << 3));
			o[0] = make_uint4(w[0], w[1], w[2], w[3]);
			o[1] = make_uint4(w[4], w[5], w[6], w[7]);
		}
	}
	s.R.ids[i] = id;
	if (root_out && i == 0) *root_out = id;
}

}  // namespace ort
