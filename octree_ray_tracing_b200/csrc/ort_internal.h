// ort_internal.h -- shared declarations of libort_b200.so's translation units (not installed).
#pragma once

#include "../../include/ort_b200.h"

#include <cstddef>
#include <cstdint>
#include <unordered_map>
#include <vector>

// Records `msg` as the calling thread's last error (and on ctx when given) and returns `code`.
int ort_fail(ort_ctx* ctx, int code, const char* fmt, ...);

// Zero-filled storage for table-sized arrays (anonymous mapping + transparent huge pages above 8 MB, heap below) and
// parallel first-touch of such ranges (the kernel then zeroes the pages on several cores).
void* ort_zalloc(size_t bytes);
void  ort_zfree(void* p, size_t bytes);
void  ort_prefault(void* const* ptrs, const size_t* bytes, int n_ranges, int nthreads);

// `p` itself when it is host memory or ctx is null (no CUDA call is made then), else a host copy of its `bytes` kept in
// `keep`, made on ctx's stream; nullptr when that copy fails.
const void* ort_host_view(ort_ctx* ctx, const void* p, size_t bytes, std::vector<uint8_t>& keep);

// Host node store.  Field meanings follow och::h_octree (och_h_octree.h:70-99).
struct ort_tree
{
	const int      log2cap;
	const int      depth;
	const uint32_t cap;
	const uint32_t idx_mask;        // :32

	uint8_t*  tags = nullptr;       // the reference's `cashes`: 0 empty, 0xFF gravestone, else hash bits
	uint32_t* refcounts = nullptr;
	uint32_t* nodes = nullptr;      // cap * 8 children, 32-B aligned rows

	uint32_t root = 0;
	uint32_t fillcnt = 0;
	uint32_t nodecnt = 0;
	uint32_t max_refcnt = 0;
	bool     table_full = false;

	// ---- device mirror bookkeeping --------------------------------------------------------
	ort_ctx* ctx = nullptr;
	bool     mirror_valid = false;       // ids below describe what the device holds
	uint32_t synced_root_slot = 0;
	uint64_t* dirty_bits = nullptr;      // one bit per slot: written or killed since the last sync
	std::vector<uint32_t> dirty;
	// slot -> compact id.  A node's children mean different things at different levels (ids above the last level,
	// voxel payloads at it) and the table is content-addressed across levels, so the id belongs to (slot, level):
	// id_leaf for level `depth`, id_interior for the first level above it at which the slot was met (recorded in
	// id_level), id_extra[(slot << 8) | level] for the rare slot that also serves at another level.
	uint32_t* id_interior = nullptr;
	uint32_t* id_leaf = nullptr;
	uint8_t*  id_level = nullptr;
	std::unordered_map<uint64_t, uint32_t> id_extra;
	std::vector<uint32_t> id_owner;      // slots that own ids (bit 31 = leaf role), for cheap resets
	std::vector<uint32_t> free_ids;
	uint32_t next_id = 1;

	std::vector<uint32_t> flat;          // last flatten: n * 8
	uint32_t flat_root = 0;
	std::vector<uint32_t> delta_ids, delta_nodes;
	uint32_t delta_root = 0;
	uint64_t last_sync_nodes = 0;
	int      last_sync_full = 0;

	ort_tree(int log2cap, int depth);
	~ort_tree();
	ort_tree(const ort_tree&) = delete;
	ort_tree& operator=(const ort_tree&) = delete;

	uint32_t register_node(const uint32_t* n);
	// insert-or-find WITHOUT touching reference counts (fixture builder; counts are filled in later)
	uint32_t intern_node(const uint32_t* n);
	void     prefetch_node(const uint32_t* n) const;
	void     prefault(int nthreads);
	void     remove_node(uint32_t idx);
	void     set(uint16_t x, uint16_t y, uint16_t z, uint32_t v);
	// bulk edit: every voxel of [lo, hi) (clipped to the cube) becomes v; same content, counts and canonical DAG
	// as the equivalent set() loop, without visiting the voxels one by one
	void     fill_box(const int lo[3], const int hi[3], uint32_t v);
	uint32_t at(int x, int y, int z) const;
	void     clear();

	size_t flatten(uint32_t* level_offsets);
	bool   build_delta();
	size_t take_delta(const uint32_t** ids, const uint32_t** nodes8, uint32_t* root_out, int* is_full);
	int    sync();
	void   invalidate_mirror();
	void   clear_dirty();

private:
	struct BoxEdit;
	uint32_t fill_rec(BoxEdit& e, uint32_t node, int k, int x, int y, int z);
	void     add_instances(uint32_t id, int k, int64_t delta);
	void     count_one(uint32_t slot, int64_t delta);
	void     mark_dirty(uint32_t slot);
	uint32_t probe(const uint32_t* n, uint8_t& tag, bool& found) const;
	void     reset_ids();
	uint32_t delta_visit(uint32_t slot, int level);
	uint32_t& id_ref(uint32_t slot, int level, bool assign);
};

// Adds to every node reachable from t->root its number of instances in the fully expanded tree (what one register_node
// call per instance would have counted), and their sum to nodecnt.  For DAGs interned with intern_node (ort_fixture.cpp).
void assign_instance_counts(ort_tree* t, int nthreads);
