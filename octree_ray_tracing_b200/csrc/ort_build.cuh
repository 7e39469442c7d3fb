// ort_build.cuh -- the DAG of a dense voxel grid, built on the GPU (ort_build_voxels, DESIGN section 13).
//
// The result is exactly what ort_tree_flatten returns for a host table holding the same voxels: per level the distinct
// node contents, numbered in the breadth-first order of their first occurrence, root = id 1.  Two phases:
//
//   bottom-up, one level per pass (leaf level `depth` first): every non-empty cell of the level is inserted into a
//     per-level open-addressing table whose entries hold a representative cell.  A thread claims an empty entry with
//     atomicCAS; on a taken entry it compares the full 32 bytes of its content with the representative's, which it
//     reads from the immutable input (leaf level) or child grid (levels above), so no thread ever waits for another.
//     The cell's temporary id is its entry's table slot + 1 (0 = empty cell).
//   top-down, one level per pass (root first): the 8 * n_l child slots of the level's frontier, in final order, give
//     each distinct child the position of its first occurrence (atomicMin); an exclusive scan over the first-occurrence
//     flags yields the next level's final ids and frontier order; the level's rows are written with final child ids.
//
// Hand-written throughout (no CUB / Thrust); deterministic: temporary ids depend on thread timing, final ids do not.
#pragma once

namespace ort {

constexpr uint32_t kBuildEmpty = 0xFFFFFFFFu;
constexpr int kBuildMaxDepth = 11;
constexpr unsigned kScanThreads = 256;
constexpr unsigned kScanItems = 4;                                  // per thread
constexpr unsigned kScanTile = kScanThreads * kScanItems;           // items per block

// One level's cell grid: dims (cells per axis, clipped to the input's extent) and its temporary ids.
struct BuildLevel
{
	uint32_t gx, gy, gz;
	uint32_t* ids;              // gx * gy * gz temporary ids, index (z * gy + y) * gx + x
	uint32_t* table;            // cap entries: representative cell, kBuildEmpty = free
	uint32_t mask;              // cap - 1
};

// The input voxels.  elem_bytes 1 or 4; cells outside [0,nx) x [0,ny) x [0,nz) read as 0.
struct BuildInput
{
	const void* p;
	int elem_bytes;
	uint32_t nx, ny, nz;
	__device__ __forceinline__ uint32_t at(uint32_t x, uint32_t y, uint32_t z) const
	{
		if (x >= nx || y >= ny || z >= nz) return 0u;
		const size_t i = (static_cast<size_t>(z) * ny + y) * nx + x;
		return elem_bytes == 1 ? static_cast<uint32_t>(__ldg(static_cast<const uint8_t*>(p) + i)) : __ldg(static_cast<const uint32_t*>(p) + i);
	}
};

__device__ __forceinline__ void build_decode(uint32_t cell, const BuildLevel& L, uint32_t& x, uint32_t& y, uint32_t& z)
{
	x = cell % L.gx;
	const uint32_t r = cell / L.gx;
	y = r % L.gy;
	z = r / L.gy;
}

// The 8 words of a cell: the voxels below it (leaf level) or the temporary ids of its children (child grid `C`).
// Child c: bit 0 = x, bit 1 = y, bit 2 = z.
__device__ __forceinline__ void build_content(bool leaf, const BuildInput& in, const BuildLevel& C, uint32_t x, uint32_t y, uint32_t z, uint32_t w[8])
{
#pragma unroll
	for (int c = 0; c < 8; ++c)
	{
		const uint32_t cx = 2 * x + (c & 1), cy = 2 * y + ((c >> 1) & 1), cz = 2 * z + (c >> 2);
		if (leaf)
			w[c] = in.at(cx, cy, cz);
		else
			w[c] = (cx < C.gx && cy < C.gy && cz < C.gz) ? C.ids[(static_cast<size_t>(cz) * C.gy + cy) * C.gx + cx] : 0u;
	}
}

__device__ __forceinline__ uint32_t build_hash(const uint32_t w[8])
{
	uint64_t h = 0x9E3779B97F4A7C15ull;
#pragma unroll
	for (int i = 0; i < 8; ++i) { h ^= w[i]; h *= 0xFF51AFD7ED558CCDull; h ^= h >> 29; }
	return static_cast<uint32_t>(h ^ (h >> 32));
}

__device__ __forceinline__ unsigned block_sum(unsigned v)
{
	__shared__ unsigned warp_sums[32];
	for (int o = 16; o; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
	const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
	if (lane == 0) warp_sums[warp] = v;
	__syncthreads();
	unsigned s = 0;
	if (warp == 0)
	{
		s = lane < (blockDim.x >> 5) ? warp_sums[lane] : 0u;
		for (int o = 16; o; o >>= 1) s += __shfl_down_sync(0xFFFFFFFFu, s, o);
	}
	return s;           // valid in thread 0
}

// ---- content sources ------------------------------------------------------------------------------------------------
// The kernels below are shared with the box write (ort_write.cuh) through a content source `Src`:
//   items()            the items one bottom-up pass inserts (a level's cells here)
//   entry(i)           the table entry that stands for item i (its representative value, != kBuildEmpty)
//   content(e, w)      the 8 words of entry e, recomputed from immutable inputs
//   store(i, id)       record item i's temporary id (0 = empty content)
//   rep(t)             the entry of temporary id t (top-down)
//   child(e, c)        word c of entry e's content (top-down, levels above the leaf level)

// The builder's source: level L of the dense grid, its child grid C (levels above the leaf level).
struct DenseSrc
{
	bool leaf;
	BuildInput in;
	BuildLevel L, C;
	__device__ __forceinline__ size_t items() const { return static_cast<size_t>(L.gx) * L.gy * L.gz; }
	__device__ __forceinline__ uint32_t entry(size_t i) const { return static_cast<uint32_t>(i); }
	__device__ __forceinline__ void content(uint32_t e, uint32_t w[8]) const
	{
		uint32_t x, y, z;
		build_decode(e, L, x, y, z);
		build_content(leaf, in, C, x, y, z, w);
	}
	__device__ __forceinline__ void store(size_t i, uint32_t id) const { L.ids[i] = id; }
	__device__ __forceinline__ uint32_t rep(uint32_t t) const { return L.table[t - 1]; }
	__device__ __forceinline__ uint32_t child(uint32_t e, int c) const
	{
		uint32_t x, y, z;
		build_decode(e, L, x, y, z);
		const uint32_t cx = 2 * x + (c & 1), cy = 2 * y + ((c >> 1) & 1), cz = 2 * z + (c >> 2);
		return (cx < C.gx && cy < C.gy && cz < C.gz) ? C.ids[(static_cast<size_t>(cz) * C.gy + cy) * C.gx + cx] : 0u;
	}
};

// Count the items with non-empty content (sizes a level's table).
template<class Src>
__global__ void build_count_kernel(Src src, unsigned long long* count)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	unsigned ne = 0;
	if (i < src.items())
	{
		uint32_t w[8];
		src.content(src.entry(i), w);
		ne = (w[0] | w[1] | w[2] | w[3] | w[4] | w[5] | w[6] | w[7]) != 0u;
	}
	const unsigned s = block_sum(ne);
	if (threadIdx.x == 0 && s) atomicAdd(count, static_cast<unsigned long long>(s));
}

// Bottom-up pass of one level: insert every item with non-empty content into the table (cap = mask + 1 entries), store
// its temporary id (table slot + 1, 0 = empty); count the non-empty items.
template<class Src>
__global__ void build_insert_kernel(Src src, uint32_t* table, uint32_t mask, unsigned long long* nonempty)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	unsigned ne = 0;
	if (i < src.items())
	{
		uint32_t w[8];
		const uint32_t me = src.entry(i);
		src.content(me, w);
		uint32_t id = 0;
		if (w[0] | w[1] | w[2] | w[3] | w[4] | w[5] | w[6] | w[7])
		{
			ne = 1;
			uint32_t slot = build_hash(w) & mask;
			for (;;)
			{
				uint32_t e = table[slot];
				if (e == kBuildEmpty)
				{
					e = atomicCAS(table + slot, kBuildEmpty, me);
					if (e == kBuildEmpty) break;                      // claimed: this item represents its content
				}
				// taken: the same content?  (the full 32 bytes; equal hashes prove nothing)
				uint32_t v[8];
				src.content(e, v);
				bool same = true;
#pragma unroll
				for (int c = 0; c < 8; ++c) same &= v[c] == w[c];
				if (same) break;
				slot = (slot + 1) & mask;
			}
			id = slot + 1;
		}
		src.store(i, id);
	}
	const unsigned s = block_sum(ne);
	if (threadIdx.x == 0 && s) atomicAdd(nonempty, static_cast<unsigned long long>(s));
}

// Distinct contents of a level = claimed table entries.
__global__ void build_count_table_kernel(const uint32_t* table, size_t cap, unsigned long long* count)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	const unsigned s = block_sum(i < cap && table[i] != kBuildEmpty);
	if (threadIdx.x == 0 && s) atomicAdd(count, static_cast<unsigned long long>(s));
}

// Top-down, step 1: the temporary id of child slot s = 8 i + c of frontier node i (ch[s]); first occurrence of each
// distinct child (first[t - 1], indexed by the child level's table slot).
template<class Src>
__global__ void build_children_kernel(const uint32_t* frontier, size_t n_slots, Src src, uint32_t* ch, uint32_t* first)
{
	const size_t s = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (s >= n_slots) return;
	const uint32_t t = src.child(src.rep(frontier[s >> 3]), static_cast<int>(s & 7));
	ch[s] = t;
	if (t) atomicMin(first + (t - 1), static_cast<uint32_t>(s));
}

// step 2: flag[s] = 1 where slot s holds the first occurrence of its child
__global__ void build_flags_kernel(const uint32_t* ch, const uint32_t* first, size_t n_slots, uint32_t* flag)
{
	const size_t s = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (s >= n_slots) return;
	const uint32_t t = ch[s];
	flag[s] = t != 0u && first[t - 1] == static_cast<uint32_t>(s);
}

// step 3 (after the exclusive scan of the flags, pos): the level's rows with final child ids, the next frontier.
// rows = the level's first row in the output; next_base = final id of the next level's first node.  (rows may be ch
// itself: slot s reads ch[s] before it writes rows[s], and no other slot reads it.)
__global__ void build_rows_kernel(const uint32_t* ch, const uint32_t* first, const uint32_t* pos, size_t n_slots, uint32_t next_base,
                                  uint32_t* rows, uint32_t* next_frontier)
{
	const size_t s = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (s >= n_slots) return;
	const uint32_t t = ch[s];
	uint32_t id = 0;
	if (t)
	{
		const uint32_t f = first[t - 1];
		const uint32_t p = pos[f];
		id = next_base + p;
		if (f == static_cast<uint32_t>(s)) next_frontier[p] = t;
	}
	rows[s] = id;
}

// The leaf level's rows: the content of each frontier node's representative.
template<class Src>
__global__ void build_leaf_rows_kernel(const uint32_t* frontier, size_t n, Src src, uint32_t* rows)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) return;
	uint32_t w[8];
	src.content(src.rep(frontier[i]), w);
	uint4* o = reinterpret_cast<uint4*>(rows + 8 * i);
	o[0] = make_uint4(w[0], w[1], w[2], w[3]);
	o[1] = make_uint4(w[4], w[5], w[6], w[7]);
}

// ---- exclusive scan of uint32 (reduce per tile, scan the tile sums, add) ------------------------------------------

// Scans each tile of kScanTile items in place (exclusive) and writes the tile's total to sums[blockIdx.x].
__global__ void __launch_bounds__(kScanThreads) scan_tiles_kernel(uint32_t* a, size_t n, uint32_t* sums)
{
	__shared__ uint32_t warp_tot[kScanThreads / 32];
	const size_t base = static_cast<size_t>(blockIdx.x) * kScanTile + static_cast<size_t>(threadIdx.x) * kScanItems;
	uint32_t v[kScanItems];
	uint32_t own = 0;
#pragma unroll
	for (unsigned k = 0; k < kScanItems; ++k)
	{
		v[k] = base + k < n ? a[base + k] : 0u;
		own += v[k];
	}
	// inclusive scan of the per-thread totals over the warp, then over the warps
	const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
	uint32_t inc = own;
	for (int o = 1; o < 32; o <<= 1)
	{
		const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, inc, o);
		if (lane >= static_cast<unsigned>(o)) inc += u;
	}
	if (lane == 31) warp_tot[warp] = inc;
	__syncthreads();
	if (warp == 0)
	{
		uint32_t w = lane < kScanThreads / 32 ? warp_tot[lane] : 0u;
		for (int o = 1; o < 32; o <<= 1)
		{
			const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, w, o);
			if (lane >= static_cast<unsigned>(o)) w += u;
		}
		if (lane < kScanThreads / 32) warp_tot[lane] = w;        // inclusive over warps
	}
	__syncthreads();
	uint32_t run = inc - own + (warp ? warp_tot[warp - 1] : 0u);
#pragma unroll
	for (unsigned k = 0; k < kScanItems; ++k)
	{
		if (base + k < n) a[base + k] = run;
		run += v[k];
	}
	if (threadIdx.x == kScanThreads - 1) sums[blockIdx.x] = warp_tot[kScanThreads / 32 - 1];
}

__global__ void scan_add_kernel(uint32_t* a, size_t n, const uint32_t* offs)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i < n) a[i] += offs[i / kScanTile];
}

#ifndef ORT_HOST_EMU          // (the host emulation, tests/host_emu/emu_build.cpp, compiles the device code above only)
// scratch words scan_exclusive needs for n items
inline size_t scan_scratch_words(size_t n)
{
	size_t words = 0;
	for (size_t m = n; m > 1;) { m = (m + kScanTile - 1) / kScanTile; words += m; }
	return words + 1;
}

// exclusive prefix sum of a[0, n) in place on `stream`; scratch: scan_scratch_words(n) words
inline void scan_exclusive(uint32_t* a, size_t n, uint32_t* scratch, cudaStream_t stream, uint64_t& launches)
{
	if (n == 0) return;
	const size_t tiles = (n + kScanTile - 1) / kScanTile;
	scan_tiles_kernel<<<static_cast<unsigned>(tiles), kScanThreads, 0, stream>>>(a, n, scratch);
	++launches;
	if (tiles == 1) return;
	scan_exclusive(scratch, tiles, scratch + tiles, stream, launches);
	scan_add_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(a, n, scratch);
	++launches;
}
#endif

}  // namespace ort
