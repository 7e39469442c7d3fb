// ort_fixture.cpp -- headless-harness fixtures: the synthetic terrain the reference's demo builds in
// initialize_h_octree (test_och_h_octree.cpp:767-787), produced by a builder that scales to depth
// 12-14.  Host C++ only.
//
// The reference builds the DAG top-down over the whole solid volume (create_volume, :651-695), then
// patches 3*dim^2 voxels through set() (:776-783) and optionally runs dim^3 noise evaluations to
// carve tunnels (:735-743, :786): minutes at depth 12, hours with tunnels.  Because the DAG is
// content-addressed, the SAME voxel content always yields the same canonical DAG, so this builder
// evaluates the voxel function directly:
//     voxel(x,y,z) = 0            if z > h(x,y)            or carved
//                    2 + grass    if z == h(x,y)
//                    4            if z == h-1 or z == h-2
//                    1            otherwise (stone)
// recursing only where a cell is not trivially empty (above the column maximum) or, without tunnels,
// trivially solid stone (below column minimum - 2; one memoised node per level).  Reference counts
// are then computed top-down as instance counts, which is what the reference's per-instance
// register_node calls add up to (saturating at 2^32-1 instead of wrapping for depth >= 13).
#include "ort_internal.h"
#include "ort_noise.h"
#include "ort_opensimplex.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cctype>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <thread>

namespace {

template<class F>
void parallel_rows(int rows, int nthreads, F f)
{
	if (nthreads <= 1) { for (int r = 0; r < rows; ++r) f(r); return; }
	std::atomic<int> next{ 0 };
	std::vector<std::thread> pool;
	for (int w = 0; w < nthreads; ++w)
		pool.emplace_back([&] { for (int r; (r = next.fetch_add(1)) < rows;) f(r); });
	for (auto& t : pool) t.join();
}

// ---- builder -------------------------------------------------------------------------------

struct Builder
{
	ort_tree* tree;
	int depth, dim;
	const uint16_t* h;
	const uint8_t* grass;
	bool tunnels;
	std::vector<std::vector<uint16_t>> hmin, hmax;    // [k] = min/max over 2^k x 2^k column blocks
	std::vector<uint64_t> carved_own;                 // tunnels: one bit per voxel with z <= zmax (bit y*dim+x of slab z)
	const uint64_t* carved = nullptr;                 // = carved_own.data(), or the caller's bitmap (ort_fixture_carve_gpu)
	std::vector<std::vector<uint8_t>> any;            // [k >= 3]: cell of size 2^k holds at least one carved voxel
	int zmax = -1;

	// the dim^3 noise loop of remove() (:735-743) restricted to z <= max height (voxels above are empty anyway),
	// spread over the host cores
	void precompute_carved(int nthreads)
	{
		const size_t words_per_slab = (static_cast<size_t>(dim) * dim + 63) / 64;
		carved_own.assign(words_per_slab * (zmax + 1), 0);
		parallel_rows(zmax + 1, nthreads, [&](int z) {
			uint64_t* slab = carved_own.data() + words_per_slab * z;
			for (int y = 0; y < dim; ++y)
				for (int x = 0; x < dim; ++x)
					if (z <= h[static_cast<size_t>(y) * dim + x] && ort_noise::carve_test(x, y, z))
					{
						const size_t b = static_cast<size_t>(y) * dim + x;
						slab[b >> 6] |= 1ull << (b & 63);
					}
		});
		carved = carved_own.data();
	}

	// "any carved voxel in the cell" per 8^3 cell from the bitmap, OR-reduced up the levels: cells without carving
	// are built like the tunnel-free terrain (memoised stone, empty above the surface)
	void build_any_pyramid(int nthreads)
	{
		any.assign(depth + 1, {});
		if (depth < 3) return;
		const size_t words_per_slab = (static_cast<size_t>(dim) * dim + 63) / 64;
		const uint8_t* bytes = reinterpret_cast<const uint8_t*>(carved);
		const int w = dim >> 3, nz = (zmax >> 3) + 1;
		any[3].assign(static_cast<size_t>(w) * w * nz, 0);
		parallel_rows(nz, nthreads, [&](int cz) {
			uint8_t* out = any[3].data() + static_cast<size_t>(cz) * w * w;
			for (int z = cz * 8; z < cz * 8 + 8 && z <= zmax; ++z)
			{
				const uint8_t* slab = bytes + words_per_slab * 8 * z;          // byte (y*dim + x) / 8: 8 voxels along x
				for (int y = 0; y < dim; ++y)
				{
					const uint8_t* row = slab + (static_cast<size_t>(y) * dim >> 3);
					uint8_t* orow = out + static_cast<size_t>(y >> 3) * w;
					for (int cx = 0; cx < w; ++cx) orow[cx] |= row[cx];
				}
			}
		});
		for (int k = 4; k <= depth; ++k)
		{
			const int wk = dim >> k, wp = wk * 2, nzk = (zmax >> k) + 1, nzp = (zmax >> (k - 1)) + 1;
			any[k].assign(static_cast<size_t>(wk) * wk * nzk, 0);
			const auto& lo = any[k - 1];
			for (int cz = 0; cz < nzp; ++cz)
				for (int cy = 0; cy < wp; ++cy)
					for (int cx = 0; cx < wp; ++cx)
						if (lo[(static_cast<size_t>(cz) * wp + cy) * wp + cx])
							any[k][(static_cast<size_t>(cz >> 1) * wk + (cy >> 1)) * wk + (cx >> 1)] = 1;
		}
	}

	inline bool cell_carved(int x, int y, int z, int k) const     // may the cell [.., +2^k)^3 (z <= zmax) contain a carved voxel?
	{
		if (k < 3) return true;
		const int wk = dim >> k;
		return any[k][(static_cast<size_t>(z >> k) * wk + (y >> k)) * wk + (x >> k)] != 0;
	}

	inline bool is_carved(int x, int y, int z) const
	{
		const size_t words_per_slab = (static_cast<size_t>(dim) * dim + 63) / 64;
		const size_t b = static_cast<size_t>(y) * dim + x;
		return (carved[words_per_slab * z + (b >> 6)] >> (b & 63)) & 1u;
	}

	inline uint32_t voxel(int x, int y, int z) const
	{
		const int hh = h[static_cast<size_t>(y) * dim + x];
		uint32_t v;
		if (z > hh) return 0;
		if (z == hh) v = 2u + (grass[static_cast<size_t>(y) * dim + x] ? 1u : 0u);
		else if (z >= hh - 2) v = 4u;
		else v = 1u;
		if (tunnels && is_carved(x, y, z)) return 0;
		return v;
	}
};

// Where built nodes go.  TreeSink: straight into the host table.  LocalDag: a private, content-addressed sub-DAG
// with local ids (children of k == 1 nodes are voxel payloads, of k > 1 nodes local ids), merged into the table later.
struct TreeSink
{
	ort_tree* tree;
	bool failed = false;
	uint32_t intern(const uint32_t* n, int)
	{
		const uint32_t id = tree->intern_node(n);
		if (!id) failed = true;
		return id;
	}
};

struct LocalDag
{
	std::vector<uint32_t> words;       // 8 per node, in creation order (children before parents)
	std::vector<uint8_t>  leaf;        // 1: children are voxel payloads
	std::vector<uint8_t>  lvl;         // k = log2(cell size) of the node
	std::vector<uint32_t> slots;       // open addressing -> local id (1-based), 0 = empty
	uint32_t mask = 0;
	bool failed = false;

	static inline uint32_t hash(const uint32_t* n, uint32_t is_leaf)
	{
		uint64_t h = 0x9E3779B97F4A7C15ull + is_leaf;
		for (int i = 0; i < 8; ++i) { h ^= n[i]; h *= 0xFF51AFD7ED558CCDull; h ^= h >> 29; }
		return static_cast<uint32_t>(h ^ (h >> 32));
	}

	void grow()
	{
		const uint32_t cap = slots.empty() ? 1024u : static_cast<uint32_t>(slots.size()) * 2u;
		slots.assign(cap, 0);
		mask = cap - 1;
		for (uint32_t id = 1; id <= leaf.size(); ++id)
		{
			uint32_t p = hash(words.data() + 8 * static_cast<size_t>(id - 1), leaf[id - 1]) & mask;
			while (slots[p]) p = (p + 1) & mask;
			slots[p] = id;
		}
	}

	uint32_t intern(const uint32_t* n, int k)
	{
		if (leaf.size() * 2 >= slots.size()) grow();
		const uint32_t is_leaf = k == 1;
		uint32_t p = hash(n, is_leaf) & mask;
		for (uint32_t id; (id = slots[p]) != 0; p = (p + 1) & mask)
			if (leaf[id - 1] == is_leaf && !std::memcmp(words.data() + 8 * static_cast<size_t>(id - 1), n, 32))
				return id;
		words.insert(words.end(), n, n + 8);
		leaf.push_back(static_cast<uint8_t>(is_leaf));
		lvl.push_back(static_cast<uint8_t>(k));
		return slots[p] = static_cast<uint32_t>(leaf.size());
	}
};

template<class Sink>
struct Walker
{
	const Builder& b;
	Sink& sink;
	uint32_t stone[17] = {};                            // memoised all-stone subtree per cell size 2^k

	uint32_t stone_node(int k)                         // k = log2(cell size) >= 1
	{
		if (stone[k]) return stone[k];
		uint32_t n[8];
		const uint32_t c = k == 1 ? 1u : stone_node(k - 1);
		for (int i = 0; i < 8; ++i) n[i] = c;
		return stone[k] = sink.intern(n, k);
	}

	uint32_t build(int x, int y, int z, int k)         // cell [x,x+2^k) x [y,..) x [z,..); returns node id or 0
	{
		if (sink.failed) return 0;
		const int s = 1 << k;
		const size_t bi = static_cast<size_t>(y >> k) * (b.dim >> k) + (x >> k);
		if (z > b.hmax[k][bi])
			return 0;                                  // entirely above the terrain
		if (z + s - 1 < static_cast<int>(b.hmin[k][bi]) - 2 && !(b.tunnels && b.cell_carved(x, y, z, k)))
			return stone_node(k);                      // entirely plain stone

		uint32_t n[8];
		if (k == 1)
			for (int c = 0; c < 8; ++c) n[c] = b.voxel(x + (c & 1), y + ((c >> 1) & 1), z + (c >> 2));
		else
		{
			const int hs = s >> 1;
			for (int c = 0; c < 8; ++c) n[c] = build(x + (c & 1 ? hs : 0), y + (c & 2 ? hs : 0), z + (c & 4 ? hs : 0), k - 1);
		}
		if (!(n[0] | n[1] | n[2] | n[3] | n[4] | n[5] | n[6] | n[7]))
			return 0;                                  // (only reachable with tunnels: a fully carved cell)
		return sink.intern(n, k);
	}
};

// The volume is cut into 8^3 subcells; the host threads build each subcell's sub-DAG privately (no shared state but
// the read-only maps), then the sub-DAGs are interned into the table one after the other in subcell order -- children
// before parents, local ids translated on the way -- and the three top levels are assembled from the subcell roots.
// Same canonical DAG as the sequential walk; slot numbering depends only on the subcell order, not on thread timing.
uint32_t build_parallel(const Builder& b, ort_tree* tree, int nthreads, bool& failed)
{
	const int ks = b.depth - 3, side = 8, cell = 1 << ks;
	std::vector<LocalDag> dags(static_cast<size_t>(side) * side * side);
	std::vector<uint32_t> local_root(dags.size(), 0);
	parallel_rows(static_cast<int>(dags.size()), nthreads, [&](int i) {
		const int cx = i & 7, cy = (i >> 3) & 7, cz = i >> 6;
		Walker<LocalDag> w{ b, dags[i] };
		local_root[i] = w.build(cx * cell, cy * cell, cz * cell, ks);
	});

	const auto t_par = std::chrono::steady_clock::now();
	if (std::getenv("ORT_FIXTURE_TIMING"))
	{
		size_t tot = 0;
		for (const auto& d : dags) tot += d.leaf.size();
		std::fprintf(stderr, "[ort fixture] %zu local nodes in %zu sub-DAGs\n", tot, dags.size());
	}
	TreeSink sink{ tree };
	std::vector<uint32_t> sub_root(dags.size(), 0), gmap, order;
	constexpr size_t kLook = 12;                       // nodes prepared (children translated, table lines prefetched) ahead of the intern
	uint32_t prep[kLook][8];
	for (size_t i = 0; i < dags.size() && !sink.failed; ++i)
	{
		LocalDag& d = dags[i];
		const size_t n = d.leaf.size();
		gmap.assign(n, 0);
		// level by level (children before parents; the nodes of one level are independent of each other)
		size_t first_of[18] = { 0 };
		for (size_t j = 0; j < n; ++j) ++first_of[d.lvl[j] + 1];
		for (int k = 1; k < 18; ++k) first_of[k] += first_of[k - 1];
		order.resize(n);
		{
			size_t fill[18];
			std::memcpy(fill, first_of, sizeof fill);
			for (size_t j = 0; j < n; ++j) order[fill[d.lvl[j]]++] = static_cast<uint32_t>(j);
		}
		auto prepare = [&](size_t pos) {
			const uint32_t j = order[pos];
			uint32_t* out = prep[pos % kLook];
			std::memcpy(out, d.words.data() + 8 * static_cast<size_t>(j), 32);
			if (!d.leaf[j])
				for (int c = 0; c < 8; ++c) if (out[c]) out[c] = gmap[out[c] - 1];
			tree->prefetch_node(out);
		};
		for (int k = 1; k <= ks && !sink.failed; ++k)
		{
			const size_t lo = first_of[k], hi = first_of[k + 1];
			for (size_t pos = lo; pos < hi && pos < lo + kLook; ++pos) prepare(pos);
			for (size_t pos = lo; pos < hi && !sink.failed; ++pos)
			{
				uint32_t node[8];
				std::memcpy(node, prep[pos % kLook], 32);
				if (pos + kLook < hi) prepare(pos + kLook);
				gmap[order[pos]] = sink.intern(node, 0);
			}
		}
		if (local_root[i]) sub_root[i] = gmap[local_root[i] - 1];
		std::vector<uint32_t>().swap(d.words);
		std::vector<uint32_t>().swap(d.slots);
	}
	// top three levels
	uint32_t lvl[3][64 * 8];
	auto at = [&](int level_side, const uint32_t* src, int x, int y, int z) { return src[(static_cast<size_t>(z) * level_side + y) * level_side + x]; };
	const uint32_t* src = sub_root.data();
	int src_side = 8;
	uint32_t root = 0;
	for (int pass = 0; pass < 3 && !sink.failed; ++pass)
	{
		const int dst_side = src_side / 2;
		uint32_t* dst = lvl[pass];
		for (int z = 0; z < dst_side; ++z)
			for (int y = 0; y < dst_side; ++y)
				for (int x = 0; x < dst_side; ++x)
				{
					uint32_t n[8];
					for (int c = 0; c < 8; ++c) n[c] = at(src_side, src, 2 * x + (c & 1), 2 * y + ((c >> 1) & 1), 2 * z + (c >> 2));
					dst[(static_cast<size_t>(z) * dst_side + y) * dst_side + x] = (n[0] | n[1] | n[2] | n[3] | n[4] | n[5] | n[6] | n[7]) ? sink.intern(n, 0) : 0u;
				}
		src = dst;
		src_side = dst_side;
		root = dst[0];
	}
	failed = sink.failed;
	if (std::getenv("ORT_FIXTURE_TIMING"))
		std::fprintf(stderr, "[ort fixture]   of which merge         %.3f s\n", std::chrono::duration<double>(std::chrono::steady_clock::now() - t_par).count());
	return root;
}

}  // namespace

// refcount(node) = number of instances of the node in the fully expanded tree = what one
// register_node call per instance (the reference's builders) would have produced.
void assign_instance_counts(ort_tree* t, int nthreads)
{
	if (!t->root) return;
	struct Acc
	{
		uint64_t* p; size_t bytes;
		~Acc() { ort_zfree(p, bytes); }
		uint64_t& operator[](size_t i) { return p[i]; }
	} acc{ static_cast<uint64_t*>(ort_zalloc(static_cast<size_t>(t->cap) * 8)), static_cast<size_t>(t->cap) * 8 };
	if (!acc.p) return;
	if (t->depth >= 11)
	{
		void* const ptrs[] = { acc.p };
		ort_prefault(ptrs, &acc.bytes, 1, nthreads);
	}
	std::vector<uint32_t> cur{ t->root - 1 }, next;
	acc[t->root - 1] = 1;
	uint64_t total = 0;
	for (int level = 1; level <= t->depth; ++level)
	{
		next.clear();
		// take this level's counts first: a slot may (rarely) serve on two levels
		std::vector<uint64_t> cnt(cur.size());
		for (size_t i = 0; i < cur.size(); ++i) { cnt[i] = acc[cur[i]]; acc[cur[i]] = 0; }
		for (size_t i = 0; i < cur.size(); ++i)
		{
			// software pipeline over the random slots of the level: node rows far ahead, their children's cells nearer
			if (i + 24 < cur.size())
			{
				__builtin_prefetch(t->nodes + 8 * static_cast<size_t>(cur[i + 24]));
				__builtin_prefetch(t->refcounts + cur[i + 24]);
			}
			if (level != t->depth && i + 8 < cur.size())
			{
				const uint32_t* pn = t->nodes + 8 * static_cast<size_t>(cur[i + 8]);
				for (int c = 0; c < 8; ++c) if (pn[c]) __builtin_prefetch(&acc[pn[c] - 1]);
			}
			const uint32_t slot = cur[i];
			const uint64_t sum = static_cast<uint64_t>(t->refcounts[slot]) + cnt[i];
			t->refcounts[slot] = sum > UINT32_MAX ? UINT32_MAX : static_cast<uint32_t>(sum);
			total += cnt[i];
			if (level == t->depth) continue;
			const uint32_t* n = t->nodes + 8 * static_cast<size_t>(slot);
			for (int c = 0; c < 8; ++c)
				if (n[c])
				{
					if (!acc[n[c] - 1]) next.push_back(n[c] - 1);
					acc[n[c] - 1] += cnt[i];
				}
		}
		cur.swap(next);
	}
	t->nodecnt += static_cast<uint32_t>(total);   // modulo 2^32 like the reference's counter
}

extern "C" {

int ort_parse_voxels(const char* text, size_t len, uint32_t* rgba6, char* names16, int max_voxels)
{
	// och_voxel.cpp:195-305: skip white space, read the name up to ':', then six colours of three hex byte pairs
	if (!text || !rgba6 || max_voxels <= 0)
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_parse_voxels: bad arguments"), -1;
	size_t i = 0;
	int n = 0;
	auto skip_space = [&] { while (i < len && std::isspace(static_cast<unsigned char>(text[i]))) ++i; };
	auto hexval = [](int c) { return c <= '9' ? c - '0' : (c | 0x20) - 'a' + 10; };
	for (;;)
	{
		skip_space();
		if (i >= len) break;
		if (n == max_voxels) break;
		char name[16] = { 0 };
		int k = 0;
		while (i < len && text[i] != ':')
		{
			if (k == 15)
				return ort_fail(nullptr, ORT_ERR_INVALID, "ort_parse_voxels: voxel-names may not exceed 15 characters (voxel %d)", n + 1), -1;
			name[k++] = text[i++];
		}
		if (i >= len)
			return ort_fail(nullptr, ORT_ERR_INVALID, "ort_parse_voxels: input ended unexpectedly in the name of voxel %d", n + 1), -1;
		if (k == 0)
			return ort_fail(nullptr, ORT_ERR_INVALID, "ort_parse_voxels: voxel-names must contain at least one character"), -1;
		++i;   // ':'
		for (int dir = 0; dir < 6; ++dir)
		{
			skip_space();
			uint32_t px = 0xFF000000u;
			for (int byte = 0; byte < 3; ++byte)
			{
				if (i >= len)
					return ort_fail(nullptr, ORT_ERR_INVALID, "ort_parse_voxels: input ended unexpectedly (%s, colour %d)", name, dir + 1), -1;
				if (i + 1 >= len || !std::isxdigit(static_cast<unsigned char>(text[i])) || !std::isxdigit(static_cast<unsigned char>(text[i + 1])))
					return ort_fail(nullptr, ORT_ERR_INVALID, "ort_parse_voxels: non-hex character in colour-value (%s at colour no. %d)", name, dir + 1), -1;
				px |= static_cast<uint32_t>((hexval(text[i]) << 4) | hexval(text[i + 1])) << (8 * byte);
				i += 2;
			}
			rgba6[6 * n + dir] = px;
		}
		if (names16) std::memcpy(names16 + 16 * n, name, 16);
		++n;
	}
	return n;
}

void ort_fixture_heightmap(int depth, uint16_t* heights, int nthreads)
{
	const int dim = 1 << depth;
	parallel_rows(dim, nthreads, [&](int y) {
		for (int x = 0; x < dim; ++x)
		{
			heights[static_cast<size_t>(y) * dim + x] = ort_noise::terrain_height(x, y, dim);
		}
	});
}

void ort_fixture_heightmap_opensimplex(int depth, int64_t seed, uint16_t* heights, int nthreads)
{
	const int dim = 1 << depth;
	const ort_noise::OpenSimplex2 noise(seed);
	parallel_rows(dim, nthreads, [&](int y) {
		for (int x = 0; x < dim; ++x)
			heights[static_cast<size_t>(y) * dim + x] = ort_noise::terrain_height_opensimplex(noise, x, y, dim);
	});
}

void ort_opensimplex2(int64_t seed, const double* xy, size_t n, double* out)
{
	const ort_noise::OpenSimplex2 noise(seed);
	for (size_t i = 0; i < n; ++i) out[i] = noise(xy[2 * i], xy[2 * i + 1]);
}

int ort_fixture_build_terrain(ort_tree* tree, const uint16_t* heights, const uint8_t* grass, int tunnels, int nthreads)
{
	return ort_fixture_build_terrain_ex(tree, heights, grass, tunnels, nthreads, nullptr);
}

int ort_fixture_build_terrain_ex(ort_tree* tree, const uint16_t* heights, const uint8_t* grass, int tunnels, int nthreads, const uint64_t* carved)
{
	if (!tree || !heights || !grass)
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_fixture_build_terrain: bad arguments");

	const bool timing = std::getenv("ORT_FIXTURE_TIMING") != nullptr;
	auto t_prev = std::chrono::steady_clock::now();
	auto lap = [&](const char* what) {
		if (!timing) return;
		const auto now = std::chrono::steady_clock::now();
		std::fprintf(stderr, "[ort fixture] %-22s %.3f s\n", what, std::chrono::duration<double>(now - t_prev).count());
		t_prev = now;
	};
	Builder b;
	b.tree = tree;
	b.depth = tree->depth;
	b.dim = 1 << tree->depth;
	b.h = heights;
	b.grass = grass;
	b.tunnels = tunnels != 0;

	// min / max pyramids over column blocks
	b.hmin.resize(b.depth + 1);
	b.hmax.resize(b.depth + 1);
	b.hmin[0].assign(heights, heights + static_cast<size_t>(b.dim) * b.dim);
	b.hmax[0] = b.hmin[0];
	for (int k = 1; k <= b.depth; ++k)
	{
		const int w = b.dim >> k, pw = w * 2;
		b.hmin[k].resize(static_cast<size_t>(w) * w);
		b.hmax[k].resize(static_cast<size_t>(w) * w);
		for (int y = 0; y < w; ++y)
			for (int x = 0; x < w; ++x)
			{
				const size_t p = static_cast<size_t>(2 * y) * pw + 2 * x;
				const auto& lo = b.hmin[k - 1];
				const auto& hi = b.hmax[k - 1];
				b.hmin[k][static_cast<size_t>(y) * w + x] = std::min(std::min(lo[p], lo[p + 1]), std::min(lo[p + pw], lo[p + pw + 1]));
				b.hmax[k][static_cast<size_t>(y) * w + x] = std::max(std::max(hi[p], hi[p + 1]), std::max(hi[p + pw], hi[p + pw + 1]));
			}
	}

	lap("min/max pyramids");
	if (b.tunnels)
	{
		b.zmax = b.hmax[b.depth][0];
		if (carved) b.carved = carved;
		else b.precompute_carved(nthreads > 0 ? nthreads : 1);
		b.build_any_pyramid(nthreads > 0 ? nthreads : 1);
	}
	lap("tunnel bitmap");
	if (b.depth >= 11) tree->prefault(nthreads > 0 ? nthreads : 1);     // a scene of this size fills the table: zero its pages in parallel
	lap("table page faults");
	bool failed = false;
	if (b.depth >= 7 && nthreads > 1)
		tree->root = build_parallel(b, tree, nthreads, failed);
	else
	{
		TreeSink sink{ tree };
		Walker<TreeSink> w{ b, sink };
		tree->root = w.build(0, 0, 0, b.depth);
		failed = sink.failed;
	}
	if (failed || tree->table_full)
		return ort_fail(nullptr, ORT_ERR_TABLE_FULL, "ort_fixture_build_terrain: node table too full (raise log2_table_capacity)");
	lap("build");
	assign_instance_counts(tree, nthreads > 0 ? nthreads : 1);
	lap("instance counts");
	tree->invalidate_mirror();
	return ORT_OK;
}

}  // extern "C"
