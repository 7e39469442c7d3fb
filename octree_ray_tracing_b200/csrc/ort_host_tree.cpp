// ort_host_tree.cpp -- host side of the drop-in: the reference's reference-counted,
// hash-deduplicated node store (och::h_octree<L,D>, och_h_octree.h:17-288) re-implemented, plus
// what the GPU path adds to it: dirty-slot tracking at the single place the table is written,
// flattening of the live DAG into the compact level-ordered array the kernel reads, and delta
// extraction after edits.  Pure host C++; no CUDA calls except through the C ABI in ort_b200.h.
//
// Slot layout, hash, tag ("cash") rule, probe order, gravestone reuse and refcount arithmetic follow
// the reference exactly, so the ids returned by register_node() and the table contents are the
// same as the reference's for the same call sequence (tests/test_host_tree.py checks this
// slot-for-slot against the oracle).
#include "ort_internal.h"

#include <thread>

#include <atomic>

#if defined(__linux__)
#include <sys/mman.h>
#endif

#include <cstdio>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>
#include <utility>
#include <vector>

namespace {

inline uint32_t fnv1a_signed(const uint32_t* c8)
{
	// och_h_octree.h:52-65 -- the bytes are read through `const char*`, i.e. SIGNED on x86, so
	// bytes >= 0x80 flip the upper 24 hash bits as well.
	const int8_t* b = reinterpret_cast<const int8_t*>(c8);
	uint32_t h = 2166136261u;
	for (int i = 0; i < 32; ++i)
		h = (static_cast<uint32_t>(static_cast<int32_t>(b[i])) ^ h) * 16777619u;
	return h;
}

inline bool same_node(const uint32_t* a, const uint32_t* b)
{
	return std::memcmp(a, b, 32) == 0;
}

inline uint64_t morton3(uint32_t x, uint32_t y, uint32_t z)
{
	// och::z_encode_16 (och_z_order.cpp:191-196): x -> bits 0,3,6.., y -> 1,4,7.., z -> 2,5,8..
	auto spread = [](uint64_t v) {
		v &= 0xFFFFu;
		v = (v | (v << 32)) & 0x001F00000000FFFFull;
		v = (v | (v << 16)) & 0x001F0000FF0000FFull;
		v = (v | (v << 8)) & 0x100F00F00F00F00Full;
		v = (v | (v << 4)) & 0x10C30C30C30C30C3ull;
		v = (v | (v << 2)) & 0x1249249249249249ull;
		return v;
	};
	return spread(x) | (spread(y) << 1) | (spread(z) << 2);
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// construction
// ------------------------------------------------------------------------------------------------

// Zeroed storage for the table arrays.  At L = 24..27 they are 0.6..5 GB of sparsely and randomly accessed memory:
// anonymous mappings come zero-filled for free (no memset pass) and transparent huge pages cut both the page-fault
// count and the TLB misses of every probe.  Small tables use the heap.
namespace { constexpr size_t kBigAlloc = size_t(8) << 20; }

void* ort_zalloc(size_t bytes)
{
	if (bytes < kBigAlloc)
	{
		// 64-byte aligned so that a 32-byte node row never straddles a cache line
		const size_t padded = (bytes + 63) / 64 * 64;
		void* p = std::aligned_alloc(64, padded ? padded : 64);
		if (p) std::memset(p, 0, padded ? padded : 64);
		return p;
	}
#if defined(__linux__)
	void* p = mmap(nullptr, bytes, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
	if (p == MAP_FAILED) return nullptr;
#ifdef MADV_HUGEPAGE
	madvise(p, bytes, MADV_HUGEPAGE);
#endif
	return p;
#else
	return std::calloc(bytes, 1);
#endif
}

void ort_zfree(void* p, size_t bytes)
{
	if (!p) return;
#if defined(__linux__)
	if (bytes >= kBigAlloc) { munmap(p, bytes); return; }
#endif
	std::free(p);
}

ort_tree::ort_tree(int log2cap_, int depth_)
	: log2cap(log2cap_), depth(depth_), cap(1u << log2cap_), idx_mask(((cap - 1u) >> 4) << 4)
{
	const size_t n = cap;
	tags = static_cast<uint8_t*>(ort_zalloc(n));
	refcounts = static_cast<uint32_t*>(ort_zalloc(n * 4));
	nodes = static_cast<uint32_t*>(ort_zalloc(n * 32));
	dirty_bits = static_cast<uint64_t*>(ort_zalloc((n + 63) / 64 * 8));
	id_interior = static_cast<uint32_t*>(ort_zalloc(n * 4));
	id_leaf = static_cast<uint32_t*>(ort_zalloc(n * 4));
	id_level = static_cast<uint8_t*>(ort_zalloc(n));
}

ort_tree::~ort_tree()
{
	const size_t n = cap;
	ort_zfree(tags, n);
	ort_zfree(refcounts, n * 4);
	ort_zfree(nodes, n * 32);
	ort_zfree(dirty_bits, (n + 63) / 64 * 8);
	ort_zfree(id_interior, n * 4);
	ort_zfree(id_leaf, n * 4);
	ort_zfree(id_level, n);
}

// First-touch the table arrays from several threads: the kernel zeroes the (huge) pages in parallel instead of one
// at a time inside the first insert that happens to land on them.  Worth it before bulk builds that will touch the
// whole table anyway (3 s of page-zeroing at L = 26 otherwise); pointless for small or sparsely used tables.
void ort_prefault(void* const* ptrs, const size_t* bytes, int n_ranges, int nthreads)
{
	constexpr size_t kStep = size_t(2) << 20;
	std::vector<std::pair<volatile char*, size_t>> chunks;
	for (int r = 0; r < n_ranges; ++r)
		if (ptrs[r] && bytes[r] >= kBigAlloc)
			for (size_t off = 0; off < bytes[r]; off += kStep)
				chunks.emplace_back(static_cast<volatile char*>(ptrs[r]) + off, std::min(kStep, bytes[r] - off));
	if (chunks.empty()) return;
	if (nthreads < 1) nthreads = 1;
	std::atomic<size_t> next{ 0 };
	auto work = [&] {
		for (size_t i; (i = next.fetch_add(1)) < chunks.size();)
			for (size_t off = 0; off < chunks[i].second; off += 4096)
			{
				const char v = chunks[i].first[off];
				chunks[i].first[off] = v;          // a write, so the page is really allocated; same value, so live data is untouched
			}
	};
	std::vector<std::thread> pool;
	for (int w = 1; w < nthreads; ++w) pool.emplace_back(work);
	work();
	for (auto& th : pool) th.join();
}

void ort_tree::prefault(int nthreads)
{
	const size_t n = cap;
	void* const ptrs[] = { nodes, refcounts, tags, id_interior, id_leaf, id_level };
	const size_t bytes[] = { n * 32, n * 4, n, n * 4, n * 4, n };
	ort_prefault(ptrs, bytes, 6, nthreads);
}

// ------------------------------------------------------------------------------------------------
// table operations (och_h_octree.h:110-288)
// ------------------------------------------------------------------------------------------------

inline void ort_tree::mark_dirty(uint32_t slot)
{
	uint64_t& w = dirty_bits[slot >> 6];
	const uint64_t bit = 1ull << (slot & 63);
	if (!(w & bit))
	{
		w |= bit;
		dirty.push_back(slot);
	}
}

// Probe for `n`.  Returns the slot holding an equal node (found = true) or the slot an insert
// must use (found = false): the LAST gravestone seen on the probe path if any, else the
// terminating empty slot (och_h_octree.h:129-151).
inline uint32_t ort_tree::probe(const uint32_t* n, uint8_t& tag, bool& found) const
{
	const uint32_t h = fnv1a_signed(n);
	uint32_t i = h & idx_mask;                                   // :120 (start slot is 16-aligned)
	tag = static_cast<uint8_t>(h >> log2cap);                    // :122
	if (tag == 0) tag = 1;                                       // :124-127
	else if (tag == 0xFF) tag = 0x7F;

	uint32_t grave = UINT32_MAX;
	for (uint8_t t; (t = tags[i]) != 0; i = (i + 1) & (cap - 1))
	{
		if (t == 0xFF)
			grave = i;
		else if (t == tag && same_node(nodes + 8 * static_cast<size_t>(i), n))
		{
			found = true;
			return i;
		}
	}
	found = false;
	return grave != UINT32_MAX ? grave : i;
}

// Pull the cache lines a probe for `n` will touch first (tag group and the head of its node rows): lets callers
// that know their next few nodes (the fixture merge) overlap the DRAM round trips of a table far larger than the caches.
void ort_tree::prefetch_node(const uint32_t* n) const
{
	const uint32_t i = fnv1a_signed(n) & idx_mask;
	__builtin_prefetch(tags + i);
	__builtin_prefetch(nodes + 8 * static_cast<size_t>(i));
	__builtin_prefetch(nodes + 8 * static_cast<size_t>(i) + 16);
}

uint32_t ort_tree::register_node(const uint32_t* n)
{
	if (fillcnt > static_cast<uint32_t>(static_cast<float>(cap) * 0.9375F))   // :112
	{
		table_full = true;    // the reference prints and exit(0)s here (:114-115); a library reports instead
		return 0;
	}

	uint8_t tag;
	bool found;
	const uint32_t slot = probe(n, tag, found);

	++nodecnt;
	if (found)
	{
		uint32_t& rc = refcounts[slot];
		if (rc != UINT32_MAX) ++rc;                              // saturating (depth >= 13 fixtures); the reference wraps
		return slot + 1;
	}

	++fillcnt;
	tags[slot] = tag;
	std::memcpy(nodes + 8 * static_cast<size_t>(slot), n, 32);  // :155 -- the ONLY write to nodes[] => the delta hook
	refcounts[slot] = 1;
	mark_dirty(slot);
	return slot + 1;
}

// insert-or-find without reference counting; counts are assigned by assign_instance_counts()
uint32_t ort_tree::intern_node(const uint32_t* n)
{
	if (fillcnt > static_cast<uint32_t>(static_cast<float>(cap) * 0.9375F))
	{
		table_full = true;
		return 0;
	}
	uint8_t tag;
	bool found;
	const uint32_t slot = probe(n, tag, found);
	if (!found)
	{
		++fillcnt;
		tags[slot] = tag;
		std::memcpy(nodes + 8 * static_cast<size_t>(slot), n, 32);
		refcounts[slot] = 0;
		mark_dirty(slot);
	}
	return slot + 1;
}

void ort_tree::remove_node(uint32_t idx)
{
	uint32_t& rc = refcounts[idx - 1];
	--nodecnt;
	if (rc == UINT32_MAX)
		return;                                                  // saturated counts are sticky
	if (--rc == 0)
	{
		--fillcnt;
		tags[idx - 1] = 0xFF;                                    // gravestone (:172)
		mark_dirty(idx - 1);                                     // its compact id can be recycled at the next sync
	}
}

void ort_tree::set(uint16_t x, uint16_t y, uint16_t z, uint32_t v)
{
	if (static_cast<uint32_t>(x | y | z) >= (1u << depth))      // :178
		return;

	const uint64_t key = morton3(x, y, z);
	uint32_t path[16];                                           // path[d] = node whose child index is key's digit d
	int d = depth - 1;

	for (uint32_t cur = root; cur != 0 && d >= 0; --d)           // :188-195
	{
		path[d] = cur;
		cur = nodes[8 * static_cast<size_t>(cur - 1) + ((key >> (3 * d)) & 7)];
	}

	const int first_existing = d + 1;                            // digits below this have no node yet
	uint32_t child = v;

	if (first_existing != 0)                                     // :202-217
	{
		if (v == 0)
			return;                                              // removing a voxel that is not there
		for (int k = 0; k < first_existing; ++k)
		{
			uint32_t n[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
			n[(key >> (3 * k)) & 7] = child;
			child = register_node(n);
		}
	}

	for (int k = first_existing; k < depth; ++k)                 // :220-234 path copy-on-write, bottom-up
	{
		remove_node(path[k]);
		uint32_t n[8];
		std::memcpy(n, nodes + 8 * static_cast<size_t>(path[k] - 1), 32);
		n[(key >> (3 * k)) & 7] = child;
		const bool empty = !(n[0] | n[1] | n[2] | n[3] | n[4] | n[5] | n[6] | n[7]);
		child = empty ? 0 : register_node(n);
	}

	root = child;                                                // :236
}

// ------------------------------------------------------------------------------------------------
// bulk box edit (SURVEY 8f-2): the T/Z edit as one operation
// ------------------------------------------------------------------------------------------------
//
// The reference applies a 40^3 edit as 64 000 set() calls, each a root-to-leaf copy-on-write (~0.5 M table inserts
// and as many gravestones, 27-43 ms here, 96-137 ms in the reference).  Because the table is content-addressed, the
// RESULT of that loop is a function of the final voxel content only: the canonical DAG plus, per node, its number
// of instances in the expanded tree (what the refcounts count).  fill_box computes that result directly: it
// recurses only into cells the box cuts, swaps cells the box covers for a memoised uniform subtree (or empty), and
// moves instance counts level by level.  Live nodes, fillcnt, nodecnt, refcounts and traced images equal the
// loop's; slot numbers of NEW nodes may differ (different insertion order, fewer gravestones on the probe paths).

struct ort_tree::BoxEdit
{
	int lo[3], hi[3];
	uint32_t v;
	uint32_t uniform[17];     // memo: subtree of cell size 2^k holding only v
};

// refcount[slot] += delta with the reference's bookkeeping (gravestone at zero, saturation sticky)
void ort_tree::count_one(uint32_t slot, int64_t delta)
{
	uint32_t& rc = refcounts[slot];
	nodecnt += static_cast<uint32_t>(delta);
	if (rc == UINT32_MAX)
		return;
	const int64_t nv = static_cast<int64_t>(rc) + delta;
	if (nv >= static_cast<int64_t>(UINT32_MAX)) { rc = UINT32_MAX; return; }
	rc = nv > 0 ? static_cast<uint32_t>(nv) : 0u;
	if (rc == 0)
	{
		--fillcnt;
		tags[slot] = 0xFF;
		mark_dirty(slot);
	}
}

// one subtree instance rooted at `id` (cell size 2^k) appears (delta > 0) or disappears (delta < 0): every node of
// its DAG gains/loses as many instances as there are paths to it; aggregated per level so shared nodes are visited once
void ort_tree::add_instances(uint32_t id, int k, int64_t delta)
{
	if (!id) return;
	std::vector<std::pair<uint32_t, int64_t>> cur{ { id - 1, delta } }, next;
	for (; k >= 1; --k)
	{
		next.clear();
		for (const auto& [slot, d] : cur)
		{
			if (k > 1)
			{
				const uint32_t* n = nodes + 8 * static_cast<size_t>(slot);
				for (int c = 0; c < 8; ++c)
					if (n[c]) next.emplace_back(n[c] - 1, d);
			}
			count_one(slot, d);
		}
		if (k > 1)
		{
			std::sort(next.begin(), next.end());
			size_t w = 0;
			for (size_t i = 0; i < next.size(); ++i)
			{
				if (w && next[w - 1].first == next[i].first) next[w - 1].second += next[i].second;
				else next[w++] = next[i];
			}
			next.resize(w);
			cur.swap(next);
		}
	}
}

// returns the node that replaces `node` (0 = empty) for the cell [x, x+2^k)^3; instance counts of everything below
// are already moved when it returns, the caller accounts for the returned node itself
uint32_t ort_tree::fill_rec(BoxEdit& e, uint32_t node, int k, int x, int y, int z)
{
	const int s = 1 << k;
	if (x >= e.hi[0] || y >= e.hi[1] || z >= e.hi[2] || x + s <= e.lo[0] || y + s <= e.lo[1] || z + s <= e.lo[2])
		return node;                                              // untouched
	if (x >= e.lo[0] && y >= e.lo[1] && z >= e.lo[2] && x + s <= e.hi[0] && y + s <= e.hi[1] && z + s <= e.hi[2])
	{
		uint32_t u = 0;                                           // covered: uniform subtree (or nothing)
		if (e.v)
		{
			for (int j = 1; j <= k; ++j)
				if (!e.uniform[j])
				{
					uint32_t n[8];
					for (int c = 0; c < 8; ++c) n[c] = j == 1 ? e.v : e.uniform[j - 1];
					e.uniform[j] = intern_node(n);
					if (!e.uniform[j]) return node;               // table full: give up (flag is set)
				}
			u = e.uniform[k];
		}
		if (u == node) return node;
		add_instances(u, k, +1);
		add_instances(node, k, -1);
		return u;
	}

	uint32_t n[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
	if (node) std::memcpy(n, nodes + 8 * static_cast<size_t>(node - 1), 32);
	bool changed = false;
	const int h = s >> 1;
	for (int c = 0; c < 8; ++c)
	{
		const int cx = x + (c & 1 ? h : 0), cy = y + (c & 2 ? h : 0), cz = z + (c & 4 ? h : 0);
		uint32_t nc;
		if (k == 1)
			nc = (cx >= e.lo[0] && cx < e.hi[0] && cy >= e.lo[1] && cy < e.hi[1] && cz >= e.lo[2] && cz < e.hi[2]) ? e.v : n[c];
		else
			nc = fill_rec(e, n[c], k - 1, cx, cy, cz);
		changed |= nc != n[c];
		n[c] = nc;
	}
	if (!changed)
		return node;
	uint32_t out = 0;
	if (n[0] | n[1] | n[2] | n[3] | n[4] | n[5] | n[6] | n[7])
	{
		out = intern_node(n);
		if (!out) return node;
		count_one(out - 1, +1);                                   // the new node first, so that out == node can never die in between
	}
	if (node) count_one(node - 1, -1);
	return out;
}

void ort_tree::fill_box(const int lo[3], const int hi[3], uint32_t v)
{
	BoxEdit e;
	const int dim = 1 << depth;
	for (int a = 0; a < 3; ++a)
	{
		e.lo[a] = lo[a] < 0 ? 0 : lo[a];
		e.hi[a] = hi[a] > dim ? dim : hi[a];
		if (e.lo[a] >= e.hi[a]) return;
	}
	e.v = v;
	std::memset(e.uniform, 0, sizeof e.uniform);
	root = fill_rec(e, root, depth, 0, 0, 0);
}

uint32_t ort_tree::at(int x, int y, int z) const
{
	if (root == 0)                                               // the reference dereferences nodes[-1] here (UB); 0 = air
		return 0;
	const uint64_t key = morton3(static_cast<uint16_t>(x), static_cast<uint16_t>(y), static_cast<uint16_t>(z));
	uint32_t cur = root;
	for (int d = depth - 1; d != 0; --d)
	{
		cur = nodes[8 * static_cast<size_t>(cur - 1) + ((key >> (3 * d)) & 7)];
		if (cur == 0)
			return 0;
	}
	return nodes[8 * static_cast<size_t>(cur - 1) + (key & 7)];
}

void ort_tree::clear()
{
	// :285-288 zeroes only the tags -- root, counters and refcounts keep their values.
	std::memset(tags, 0, cap);
	invalidate_mirror();
}

// ------------------------------------------------------------------------------------------------
// flatten / delta
// ------------------------------------------------------------------------------------------------

void ort_tree::invalidate_mirror()
{
	mirror_valid = false;
}

void ort_tree::reset_ids()
{
	for (uint32_t s : id_owner)
	{
		id_interior[s & 0x7FFFFFFFu] = 0;
		id_leaf[s & 0x7FFFFFFFu] = 0;
	}
	id_owner.clear();
	id_extra.clear();
	free_ids.clear();
	next_id = 1;
}

// Storage of the compact id of (slot, level); assign = the caller is about to hand out an id (claims id_interior for
// this level if it is still unclaimed)
uint32_t& ort_tree::id_ref(uint32_t slot, int level, bool assign)
{
	if (level == depth)
		return id_leaf[slot];
	if (id_interior[slot] == 0u)
	{
		if (assign) id_level[slot] = static_cast<uint8_t>(level);
		if (assign || id_extra.empty()) return id_interior[slot];
		// lookup only: an id for this level may still sit among the extras (the primary was freed, the extra was not)
		auto it = id_extra.find((static_cast<uint64_t>(slot) << 8) | static_cast<uint64_t>(level));
		return it != id_extra.end() ? it->second : id_interior[slot];
	}
	if (id_level[slot] == level)
		return id_interior[slot];
	return id_extra[(static_cast<uint64_t>(slot) << 8) | static_cast<uint64_t>(level)];
}

void ort_tree::clear_dirty()
{
	for (uint32_t s : dirty) dirty_bits[s >> 6] = 0;
	dirty.clear();
}

// Level-ordered (BFS) flatten: ids are handed out in discovery order, so each level occupies a
// contiguous id range, the root is id 1 and the upper levels form a prefix the kernel can stage
// in shared memory.  A slot reached both as an interior node and as a level-`depth` node gets two
// ids (its children mean different things in the two roles).
size_t ort_tree::flatten(uint32_t* level_offsets)
{
	reset_ids();
	flat.clear();
	flat_root = 0;

	if (level_offsets)
		for (int l = 0; l <= depth; ++l) level_offsets[l] = 1;

	if (root == 0)
		return 0;

	flat.reserve((static_cast<size_t>(fillcnt) + 64) * 8);     // (a few slots serve on two levels and get two rows)
	id_owner.reserve(static_cast<size_t>(fillcnt) + 64);
	std::vector<uint32_t> cur, next;
	auto give_id = [&](uint32_t slot, int level) {
		uint32_t& id = id_ref(slot, level, true);
		id = next_id++;
		id_owner.push_back(slot | (level == depth ? 0x80000000u : 0u));
		return id;
	};

	cur.push_back(root - 1);
	give_id(root - 1, 1);
	flat_root = 1;

	for (int level = 1; level <= depth; ++level)
	{
		if (level_offsets) level_offsets[level - 1] = static_cast<uint32_t>(flat.size() / 8 + 1);
		const bool leaf = level == depth;
		next.clear();
		flat.resize(flat.size() + cur.size() * 8);
		uint32_t* out = flat.data() + flat.size() - cur.size() * 8;

		const size_t n_cur = cur.size();
		for (size_t ci = 0; ci < n_cur; ++ci)
		{
			// two-stage software pipeline over the (random) slots of this level: rows far ahead, then -- once a row has
			// arrived -- the id cells of its children
			if (ci + 24 < n_cur) __builtin_prefetch(nodes + 8 * static_cast<size_t>(cur[ci + 24]));
			if (!leaf && ci + 8 < n_cur)
			{
				const uint32_t* pn = nodes + 8 * static_cast<size_t>(cur[ci + 8]);
				for (int c = 0; c < 8; ++c)
					if (pn[c])
					{
						__builtin_prefetch((level + 1 == depth ? id_leaf : id_interior) + (pn[c] - 1));
						if (level + 1 != depth) __builtin_prefetch(id_level + (pn[c] - 1));
					}
			}
			const uint32_t slot = cur[ci];
			const uint32_t* n = nodes + 8 * static_cast<size_t>(slot);
			if (leaf)
				std::memcpy(out, n, 32);
			else
				for (int c = 0; c < 8; ++c)
				{
					uint32_t id = 0;
					if (n[c])
					{
						id = id_ref(n[c] - 1, level + 1, false);
						if (!id)
						{
							id = give_id(n[c] - 1, level + 1);
							next.push_back(n[c] - 1);
						}
					}
					out[c] = id;
				}
			out += 8;
		}
		cur.swap(next);
	}
	if (level_offsets) level_offsets[depth] = static_cast<uint32_t>(flat.size() / 8 + 1);

	return flat.size() / 8;
}

uint32_t ort_tree::delta_visit(uint32_t slot, int level)
{
	const bool leaf = level == depth;
	if (const uint32_t have = id_ref(slot, level, false))
		return have;

	uint32_t id;
	if (!free_ids.empty()) { id = free_ids.back(); free_ids.pop_back(); }
	else id = next_id++;
	id_ref(slot, level, true) = id;
	id_owner.push_back(slot | (leaf ? 0x80000000u : 0u));

	const size_t at = delta_nodes.size();
	delta_ids.push_back(id);
	delta_nodes.resize(at + 8);

	const uint32_t* n = nodes + 8 * static_cast<size_t>(slot);
	if (leaf)
		std::memcpy(delta_nodes.data() + at, n, 32);
	else
		for (int c = 0; c < 8; ++c)
		{
			const uint32_t cid = n[c] ? delta_visit(n[c] - 1, level + 1) : 0;
			delta_nodes[at + c] = cid;   // (delta_nodes may have been reallocated by the recursion)
		}
	return id;
}

// Collect the nodes the device does not have yet.  Invariant used: a node is live iff it is
// reachable from the root (refcount = number of instances in the expanded tree), every insert and
// every death marks its slot dirty, and a changed node implies changed ancestors -- so a walk from
// the root that stops at nodes which still own a compact id visits exactly the new nodes.
bool ort_tree::build_delta()
{
	delta_ids.clear();
	delta_nodes.clear();

	if (!mirror_valid)
		return false;

	// 1. slots written or killed since the last sync lose their compact ids
	for (uint32_t s : dirty)
	{
		if (id_interior[s]) { free_ids.push_back(id_interior[s]); id_interior[s] = 0; }
		if (id_leaf[s]) { free_ids.push_back(id_leaf[s]); id_leaf[s] = 0; }
	}
	if (!id_extra.empty())
		for (auto it = id_extra.begin(); it != id_extra.end();)
		{
			const uint32_t s = static_cast<uint32_t>(it->first >> 8);
			if (dirty_bits[s >> 6] & (1ull << (s & 63)))
			{
				if (it->second) free_ids.push_back(it->second);
				it = id_extra.erase(it);
			}
			else
				++it;
		}
	const size_t n_dirty = dirty.size();
	clear_dirty();

	// 2. walk
	delta_root = root ? delta_visit(root - 1, 1) : 0;

	// id_owner grows by one entry per visit; compact it now and then so it stays O(live)
	if (id_owner.size() > 4 * static_cast<size_t>(fillcnt) + 1024)
	{
		std::vector<uint32_t> keep;
		keep.reserve(fillcnt * 2);
		for (uint32_t e : id_owner)
			if ((e & 0x80000000u ? id_leaf : id_interior)[e & 0x7FFFFFFFu]) keep.push_back(e);
		std::sort(keep.begin(), keep.end());
		keep.erase(std::unique(keep.begin(), keep.end()), keep.end());
		id_owner.swap(keep);
	}

	(void)n_dirty;
	// a delta that replaces most of the tree is better sent as a fresh level-ordered flatten
	if (delta_ids.size() > 1024 && delta_ids.size() * 2 > static_cast<size_t>(fillcnt))
		return false;
	return true;
}

size_t ort_tree::take_delta(const uint32_t** ids, const uint32_t** nodes8, uint32_t* root_out, int* is_full)
{
	if (build_delta())
	{
		*ids = delta_ids.data();
		*nodes8 = delta_nodes.data();
		*root_out = delta_root;
		*is_full = 0;
		return delta_ids.size();
	}
	const size_t n = flatten(nullptr);
	clear_dirty();
	mirror_valid = true;
	*ids = nullptr;
	*nodes8 = flat.data();
	*root_out = flat_root;
	*is_full = 1;
	return n;
}

int ort_tree::sync()
{
	if (!ctx)
		return ORT_ERR_NOT_ATTACHED;
	if (table_full)
		return ORT_ERR_TABLE_FULL;

	if (mirror_valid && dirty.empty() && synced_root_slot == root)
	{
		last_sync_nodes = 0;
		last_sync_full = 0;
		return ORT_OK;
	}

	const uint32_t *ids, *n8;
	uint32_t r;
	int full;
	const size_t n = take_delta(&ids, &n8, &r, &full);
	int rc;
	if (full)
		rc = ort_upload_full(ctx, n8, n, r);
	else
	{
		rc = ort_upload_delta(ctx, ids, n8, n, r);
		if (rc == ORT_ERR_CAPACITY)
		{
			// out of mirror space: re-flatten (drops garbage) and let upload_full grow the mirror
			const size_t m = flatten(nullptr);
			full = 1;
			rc = ort_upload_full(ctx, flat.data(), m, flat_root);
			last_sync_nodes = m;
			last_sync_full = 1;
			if (rc == ORT_OK) synced_root_slot = root; else mirror_valid = false;
			return rc;
		}
	}
	last_sync_nodes = n;
	last_sync_full = full;
	if (rc == ORT_OK) synced_root_slot = root; else mirror_valid = false;
	return rc;
}

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------

extern "C" {

int ort_tree_create(ort_tree** out, int log2cap, int depth)
{
	if (!out || log2cap < 4 || log2cap > 30 || depth < 1 || depth > 16)
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_create: log2_table_capacity in 4..30 and depth in 1..16 required");
	ort_tree* t = new (std::nothrow) ort_tree(log2cap, depth);
	if (!t || !t->tags || !t->refcounts || !t->nodes || !t->dirty_bits || !t->id_interior || !t->id_leaf || !t->id_level)
	{
		delete t;
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_create: out of host memory");
	}
	*out = t;
	return ORT_OK;
}

void ort_tree_destroy(ort_tree* t) { delete t; }

uint32_t ort_tree_register_node(ort_tree* t, const uint32_t c[8]) { return t->register_node(c); }
void     ort_tree_remove_node(ort_tree* t, uint32_t idx) { t->remove_node(idx); }
void     ort_tree_set(ort_tree* t, uint16_t x, uint16_t y, uint16_t z, uint32_t v) { t->set(x, y, z, v); }

void ort_tree_set_many(ort_tree* t, const uint32_t* q, size_t n)
{
	for (size_t i = 0; i < n; ++i)
		t->set(static_cast<uint16_t>(q[4 * i]), static_cast<uint16_t>(q[4 * i + 1]), static_cast<uint16_t>(q[4 * i + 2]), q[4 * i + 3]);
}

void ort_tree_set_box(ort_tree* t, uint16_t cx, uint16_t cy, uint16_t cz, int ext, uint32_t v)
{
	// test_och_h_octree.cpp:408-413 / :427-432: int offsets added to uint16 coordinates, then
	// narrowed back to uint16 by set()'s parameters (so boxes poking out of the cube wrap to >= dim
	// and are ignored by set()'s range check at depth < 16).
	for (int z = -ext / 2; z < (ext + 1) / 2; ++z)
		for (int y = -ext / 2; y < (ext + 1) / 2; ++y)
			for (int x = -ext / 2; x < (ext + 1) / 2; ++x)
				t->set(static_cast<uint16_t>(cx + x), static_cast<uint16_t>(cy + y), static_cast<uint16_t>(cz + z), v);
}

void ort_tree_fill_box(ort_tree* t, int x0, int y0, int z0, int x1, int y1, int z1, uint32_t v)
{
	const int lo[3] = { x0, y0, z0 }, hi[3] = { x1, y1, z1 };
	t->fill_box(lo, hi, v);
}

uint32_t ort_tree_at(const ort_tree* t, int x, int y, int z) { return t->at(x, y, z); }
void     ort_tree_set_root(ort_tree* t, uint32_t idx) { t->root = idx; }
uint32_t ort_tree_get_root(const ort_tree* t) { return t->root; }
uint32_t ort_tree_get_fillcnt(const ort_tree* t) { return t->fillcnt; }
uint32_t ort_tree_get_nodecnt(const ort_tree* t) { return t->nodecnt; }
uint32_t ort_tree_get_max_refcnt(const ort_tree* t) { return t->max_refcnt; }   // never written by the reference either (:99)
void     ort_tree_clear(ort_tree* t) { t->clear(); }
int      ort_tree_table_full(const ort_tree* t) { return t->table_full; }
int      ort_tree_depth(const ort_tree* t) { return t->depth; }
int      ort_tree_log2_capacity(const ort_tree* t) { return t->log2cap; }
const uint32_t* ort_tree_nodes(const ort_tree* t) { return t->nodes; }
const uint8_t*  ort_tree_cashes(const ort_tree* t) { return t->tags; }
const uint32_t* ort_tree_refcounts(const ort_tree* t) { return t->refcounts; }

// The host CPU's RCPSS as a table (the reference's reciprocal, och_h_octree.h:316, is whatever the CPU it runs on
// implements): entry k = RCPSS(1.0 + k * 2^-log2n) for 1.0 <= x < 2.0.  Returns the number of probe inputs (all
// mantissas of [1,2) plus a sample of other exponents) on which the table model -- top log2n mantissa bits decide,
// exponent handled arithmetically, see ort::rcp_model -- disagrees with the instruction: 0 means the GPU will match
// this host bit for bit once the table is passed to ort_set_rcp_table.  -1 on non-x86 builds.
#if defined(__SSE__) || defined(_M_X64) || defined(__x86_64__)
#include <xmmintrin.h>
static inline uint32_t host_rcp_bits(uint32_t x)
{
	float f, r;
	std::memcpy(&f, &x, 4);
	r = _mm_cvtss_f32(_mm_rcp_ss(_mm_set_ss(f)));
	uint32_t b;
	std::memcpy(&b, &r, 4);
	return b;
}
static inline uint32_t model_rcp_bits(const uint32_t* tab, int log2n, uint32_t x)      // the host twin of ort::rcp_model
{
	const uint32_t sign = x & 0x80000000u, e = (x >> 23) & 0xFFu, m = x & 0x7FFFFFu;
	if (e == 255u) return m ? (x | 0x00400000u) : sign;
	if (e == 0u) return sign | 0x7F800000u;
	const uint32_t r = tab[m >> (23 - log2n)];
	const int re = static_cast<int>(r >> 23) - (static_cast<int>(e) - 127);
	if (re <= 0) return sign;
	return sign | (static_cast<uint32_t>(re) << 23) | (r & 0x7FFFFFu);
}
long ort_host_rcp_table(uint32_t* tab, int log2n)
{
	if (!tab || log2n < 1 || log2n > 23) return -1;
	const int sh = 23 - log2n;
	for (uint32_t k = 0; k < (1u << log2n); ++k) tab[k] = host_rcp_bits(0x3F800000u | (k << sh));
	long bad = 0;
	for (uint32_t m = 0; m < (1u << 23); ++m)
	{
		const uint32_t x = 0x3F800000u | m;
		bad += host_rcp_bits(x) != model_rcp_bits(tab, log2n, x);
		bad += host_rcp_bits(x | 0x80000000u) != model_rcp_bits(tab, log2n, x | 0x80000000u);
	}
	for (uint32_t e = 0; e < 256; ++e)
		for (uint32_t m = 0; m < (1u << 23); m += 4099u)
		{
			const uint32_t x = (e << 23) | m;
			bad += host_rcp_bits(x) != model_rcp_bits(tab, log2n, x);
		}
	return bad;
}
// Quick probe used by ort_create: does this CPU's RCPSS reproduce `tab` (one input per table entry, both signs)?
// 1 yes, 0 no.
int ort_host_rcp_matches(const uint32_t* tab, int log2n)
{
	if (!tab || log2n < 1 || log2n > 23) return -1;
	const int sh = 23 - log2n;
	for (uint32_t k = 0; k < (1u << log2n); ++k)
	{
		const uint32_t x = 0x3F800000u | (k << sh) | ((1u << sh) >> 1);      // the middle of the entry's mantissa range
		if (host_rcp_bits(x) != model_rcp_bits(tab, log2n, x)) return 0;
		if (host_rcp_bits(x | 0x80000000u) != model_rcp_bits(tab, log2n, x | 0x80000000u)) return 0;
	}
	return 1;
}
#else
long ort_host_rcp_table(uint32_t*, int) { return -1; }
int ort_host_rcp_matches(const uint32_t*, int) { return -1; }
#endif

// Table dump / load (SURVEY 8f.3).  File = header + one record per occupied slot (live or gravestone), in slot
// order: slot u32, refcount u32, tag u8, 3 pad bytes, 8 children.  Loading restores the exact table -- slots, tags,
// reference counts, root and counters -- so edits continue as if the tree had been built in this process.
namespace {
struct DumpHeader
{
	char     magic[8];          // "ORTTREE1"
	int32_t  log2cap, depth;
	uint32_t root, fillcnt, nodecnt, max_refcnt;
	uint64_t records;
};
struct DumpRecord
{
	uint32_t slot, refcount;
	uint8_t  tag, pad[3];
	uint32_t children[8];
};
}  // namespace

int ort_tree_save(const ort_tree* t, const char* path)
{
	if (!t || !path) return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_save: bad arguments");
	FILE* f = std::fopen(path, "wb");
	if (!f) return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_save: cannot open '%s' for writing", path);
	DumpHeader h{};
	std::memcpy(h.magic, "ORTTREE1", 8);
	h.log2cap = t->log2cap; h.depth = t->depth;
	h.root = t->root; h.fillcnt = t->fillcnt; h.nodecnt = t->nodecnt; h.max_refcnt = t->max_refcnt;
	for (uint32_t s = 0; s < t->cap; ++s) h.records += t->tags[s] != 0;
	bool ok = std::fwrite(&h, sizeof h, 1, f) == 1;
	std::vector<DumpRecord> buf;
	buf.reserve(1 << 16);
	for (uint32_t s = 0; s < t->cap && ok; ++s)
	{
		if (t->tags[s])
		{
			DumpRecord r{};
			r.slot = s; r.refcount = t->refcounts[s]; r.tag = t->tags[s];
			std::memcpy(r.children, t->nodes + 8 * static_cast<size_t>(s), 32);
			buf.push_back(r);
		}
		if (buf.size() == (1u << 16) || (s + 1 == t->cap && !buf.empty()))
		{
			ok = std::fwrite(buf.data(), sizeof(DumpRecord), buf.size(), f) == buf.size();
			buf.clear();
		}
	}
	ok = (std::fclose(f) == 0) && ok;
	return ok ? ORT_OK : ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_save: write to '%s' failed", path);
}

int ort_tree_load(ort_tree* t, const char* path)
{
	if (!t || !path) return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_load: bad arguments");
	FILE* f = std::fopen(path, "rb");
	if (!f) return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_load: cannot open '%s'", path);
	DumpHeader h{};
	if (std::fread(&h, sizeof h, 1, f) != 1 || std::memcmp(h.magic, "ORTTREE1", 8) != 0)
	{
		std::fclose(f);
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_load: '%s' is not a table dump", path);
	}
	if (h.log2cap != t->log2cap || h.depth != t->depth)
	{
		std::fclose(f);
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_load: dump is h_octree<%d,%d>, tree is h_octree<%d,%d>", h.log2cap, h.depth, t->log2cap, t->depth);
	}
	if (h.root > t->cap || h.records > t->cap)
	{
		std::fclose(f);
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_load: '%s' is corrupt (root %u, %llu records for a table of %llu slots)", path, h.root,
		                static_cast<unsigned long long>(h.records), static_cast<unsigned long long>(t->cap));
	}
	std::memset(t->tags, 0, t->cap);
	std::vector<DumpRecord> buf(1 << 16);
	uint64_t left = h.records;
	bool ok = true;
	while (left && ok)
	{
		const size_t n = left < buf.size() ? static_cast<size_t>(left) : buf.size();
		ok = std::fread(buf.data(), sizeof(DumpRecord), n, f) == n;
		for (size_t i = 0; i < n && ok; ++i)
		{
			const DumpRecord& r = buf[i];
			if (r.slot >= t->cap || r.tag == 0) { ok = false; break; }
			t->tags[r.slot] = r.tag;
			t->refcounts[r.slot] = r.refcount;
			std::memcpy(t->nodes + 8 * static_cast<size_t>(r.slot), r.children, 32);
		}
		left -= n;
	}
	std::fclose(f);
	// Nothing in the file is trusted: at(), set() and flatten() follow the root and the interior children as slot + 1
	// indices.  Walk the DAG level by level from the root; every reference above the last level must name an occupied
	// slot of this table.  (A slot can serve at several levels -- content addressing -- hence one visited bit per level.)
	uint64_t occupied = 0, live = 0;
	if (ok)
	{
		for (uint64_t s2 = 0; s2 < t->cap; ++s2)
		{
			occupied += t->tags[s2] != 0;
			live += t->tags[s2] != 0 && t->refcounts[s2] != 0;       // (a gravestone keeps its tag, its count is 0)
		}
		ok = occupied == h.records && (h.root == 0 || (t->tags[h.root - 1] != 0 && t->refcounts[h.root - 1] != 0));
	}
	if (ok && h.root != 0 && t->depth > 1)
	{
		std::vector<uint16_t> seen(t->cap, 0);
		std::vector<uint32_t> cur{ h.root - 1 }, nxt;
		seen[h.root - 1] = 1;
		for (int level = 1; level < t->depth && ok; ++level)
		{
			const uint16_t bit = static_cast<uint16_t>(1u << (level % 16));
			nxt.clear();
			for (const uint32_t slot : cur)
			{
				const uint32_t* ch = t->nodes + 8 * static_cast<size_t>(slot);
				for (int k = 0; k < 8; ++k)
				{
					const uint32_t c = ch[k];
					if (c == 0) continue;
					if (c > t->cap || t->tags[c - 1] == 0 || t->refcounts[c - 1] == 0) { ok = false; break; }
					if (seen[c - 1] & bit) continue;
					seen[c - 1] |= bit;
					nxt.push_back(c - 1);
				}
				if (!ok) break;
			}
			cur.swap(nxt);
		}
	}
	if (!ok)
	{
		std::memset(t->tags, 0, t->cap);
		t->root = 0; t->fillcnt = 0; t->nodecnt = 0;
		t->invalidate_mirror();
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_load: '%s' is truncated or corrupt", path);
	}
	// fillcnt counts the live slots: taken from the table, not from the header
	t->root = h.root; t->fillcnt = static_cast<decltype(t->fillcnt)>(live); t->nodecnt = h.nodecnt; t->max_refcnt = h.max_refcnt;
	t->table_full = false;
	t->clear_dirty();
	t->invalidate_mirror();
	return ORT_OK;
}

// A compact level-ordered DAG (ort_tree_flatten / ort_read_nodes) into an empty table.  A device buffer is read through
// the attached context; a tree without one takes host memory only and makes no CUDA call.  The input is checked in full
// before the table is written: a walk from the root for exactly `depth` levels (so a cyclic input cannot hang it) in
// which every child id must lie in [1, n] and beyond every id of its parent's level, and no reachable row may be empty.
int ort_tree_import(ort_tree* t, const uint32_t* nodes8, size_t n, uint32_t root)
{
	if (!t) return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_import: null tree");
	if (t->root != 0 || t->fillcnt != 0)
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_import: the table is not empty (root %u, %u live nodes)", t->root, t->fillcnt);
	if (n == 0)
		return root == 0 ? ORT_OK : ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_import: root %u of an empty DAG", root);
	if (!nodes8 || root == 0 || root > n || n > UINT32_MAX)
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_import: bad arguments (n=%zu root=%u)", n, root);
	std::vector<uint8_t> keep;
	const uint32_t* rows = static_cast<const uint32_t*>(ort_host_view(t->ctx, nodes8, n * 32, keep));
	if (!rows) return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_import: cannot read the device buffer");

	const int depth = t->depth;
	std::vector<std::vector<uint32_t>> level(depth + 1);      // level[l]: ids reached at level l, in discovery order
	std::vector<uint8_t> seen(n, 0);
	level[1].push_back(root);
	seen[root - 1] = 1;
	for (int l = 1; l <= depth; ++l)
	{
		const uint32_t top = *std::max_element(level[l].begin(), level[l].end());
		for (const uint32_t id : level[l])
		{
			const uint32_t* r = rows + 8 * static_cast<size_t>(id - 1);
			if (!(r[0] | r[1] | r[2] | r[3] | r[4] | r[5] | r[6] | r[7]))
				return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_import: node %u (level %d) is reachable and has no children", id, l);
			if (l == depth) continue;
			for (int c = 0; c < 8; ++c)
			{
				const uint32_t ch = r[c];
				if (!ch) continue;
				if (ch > n)
					return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_import: node %u child %d = %u is out of range (n = %zu)", id, c, ch, n);
				if (ch <= top)
					return ort_fail(nullptr, ORT_ERR_INVALID, "ort_tree_import: node %u (level %d) child %d = %u points to its own level or above", id, l, c, ch);
				if (!seen[ch - 1]) { seen[ch - 1] = 1; level[l + 1].push_back(ch); }
			}
		}
	}

	// bottom-up: children are in the table before their parents
	std::vector<uint32_t> slot_of(n + 1, 0), created;
	for (int l = depth; l >= 1; --l)
		for (const uint32_t id : level[l])
		{
			uint32_t row[8];
			std::memcpy(row, rows + 8 * static_cast<size_t>(id - 1), 32);
			if (l != depth)
				for (int c = 0; c < 8; ++c) if (row[c]) row[c] = slot_of[row[c]];
			const uint32_t before = t->fillcnt;
			const uint32_t s = t->intern_node(row);
			if (!s)
			{
				// table full (flag set, as set() leaves it): take back what this call inserted
				for (const uint32_t k : created) t->tags[k - 1] = 0xFF;
				t->fillcnt = 0;
				t->invalidate_mirror();
				return ort_fail(nullptr, ORT_ERR_TABLE_FULL, "ort_tree_import: the table is full");
			}
			if (t->fillcnt != before) created.push_back(s);
			slot_of[id] = s;
		}
	t->root = slot_of[root];
	assign_instance_counts(t, static_cast<int>(std::max(1u, std::thread::hardware_concurrency())));
	t->invalidate_mirror();
	return ORT_OK;
}

size_t ort_tree_flatten(ort_tree* t, const uint32_t** nodes8, uint32_t* root, uint32_t* level_offsets)
{
	const size_t n = t->flatten(level_offsets);
	// a bare flatten re-numbers the ids, so whatever the device holds is stale afterwards
	t->clear_dirty();
	t->invalidate_mirror();
	if (nodes8) *nodes8 = t->flat.data();
	if (root) *root = t->flat_root;
	return n;
}

int ort_tree_attach(ort_tree* t, ort_ctx* ctx)
{
	t->ctx = ctx;
	t->invalidate_mirror();
	return ORT_OK;
}

int ort_tree_sync(ort_tree* t) { return t->sync(); }

void ort_tree_sync_stats(const ort_tree* t, uint64_t* n, int* full)
{
	if (n) *n = t->last_sync_nodes;
	if (full) *full = t->last_sync_full;
}

size_t ort_tree_take_delta(ort_tree* t, const uint32_t** ids, const uint32_t** nodes8, uint32_t* root, int* is_full)
{
	const size_t n = t->take_delta(ids, nodes8, root, is_full);
	t->synced_root_slot = t->root;
	return n;
}

}  // extern "C"
