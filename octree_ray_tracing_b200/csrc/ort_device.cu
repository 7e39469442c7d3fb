// ort_device.cu -- device context, host-buffer pipelines and the trace entry points of libort_b200.so (sm_100a).
//
// What lives on the GPU: the live DAG as ONE compact array of 32-byte nodes (two 16-byte halves,
// 16-B aligned) in level order -- root = id 1, then level 2, ... -- so the whole depth-12 terrain
// (~44 MiB) sits contiguously in the 126 MB L2 and the top levels are a contiguous prefix.  The host
// table (ort_host_tree.cpp) stays the owner; edits arrive as (id, node) deltas and are scattered.
#include "ort_internal.h"
#include "ort_rcp_table.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------

static thread_local std::string g_last_error;

// Band schedule of a view (VERDICT r1 item 7 / DESIGN section 12.2).  A frame launch ends when its longest warps do -- rays
// that graze a silhouette run hundreds of rounds -- so the 16-row bands that hold them should be scheduled first, and where
// they are depends on the view.  The trace kernel records, per band, the longest time a warp was busy; the next launch of
// the same view (same camera, same rows) schedules its bands by that measure, most expensive first.  Keyed by view so
// that the cameras of a multi-camera loop do not poison each other.  Results never depend on it: any permutation of the
// bands traces every pixel once.
struct BandMap
{
	bool     used = false;
	uint64_t stamp = 0;                 // last use (eviction)
	float    cam[13] = {};              // pos, rot, fov
	int      geo[6] = {};               // W, H, y0, rows, tile_rows, tile_step
	int      bands = 0;
	uint16_t* d_order[2] = { nullptr, nullptr };   // device schedules: launches read `cur`, a new one is uploaded into the other
	unsigned* d_cost = nullptr;
	unsigned* h_cost = nullptr;         // pinned
	uint16_t* h_order = nullptr;        // pinned, 2 x bands
	cudaEvent_t ev_cost = nullptr;      // the recorded costs have reached h_cost
	cudaEvent_t ev_order = nullptr;     // d_order[cur] has been uploaded
	cudaEvent_t ev_read[2] = { nullptr, nullptr };   // last launch reading d_order[i]
	bool     read_any[2] = { false, false };
	cudaEvent_t ev_up[2] = { nullptr, nullptr };     // the upload of h_order's half i has been executed
	bool     up_any[2] = { false, false };
	int      cur = -1;                  // -1: no schedule yet (band_rotate rule)
	bool     recording = false;
	int      applied = 0;               // schedules uploaded so far
	int      since = 0;                 // launches since the last recording
	int      seen = 0;                  // launches of this view so far
};
constexpr int kBandMaps = 64;

struct ort_ctx
{
	int device = 0;
	int depth = 0;
	cudaStream_t stream = nullptr;      // all kernels + uploads (own stream, or the caller's after ort_set_stream)
	cudaStream_t own_stream = nullptr;
	cudaStream_t copy_stream = nullptr; // D2H of finished chunks, overlapped with the next chunk's kernel
	cudaStream_t h2d_stream = nullptr;  // H2D of the next chunk's rays (host-buffer ort_trace_rays)
	cudaEvent_t  ev_chunk[2] = { nullptr, nullptr };    // kernel of the chunk in slot i done
	cudaEvent_t  ev_copied[2] = { nullptr, nullptr };   // slot i's results have reached the host
	cudaEvent_t  ev_in[2] = { nullptr, nullptr };       // slot i's rays have reached the device
	cudaStream_t aux_stream[3] = { nullptr, nullptr, nullptr };   // chunk kernels of host-buffer frames (their launch tails overlap)
	cudaEvent_t  ev_fork = nullptr, ev_aux[3] = { nullptr, nullptr, nullptr };
	cudaEvent_t  ev_part[8] = {};                         // kernel of chunk k of the current frame done
	bool slot_used[2] = { false, false };
	int  next_slot = 0;

	uint32_t* d_nodes = nullptr;        // cap_nodes * 8
	uint32_t  cap_nodes = 0;
	uint32_t  n_nodes = 0;              // highest compact id in use
	uint32_t  root = 0;
	uint32_t  index_base = 1;           // 1: ids are row+1 (h_octree layout); 0: raw rows, root = row 0 (och::octree pool)
	bool      has_root = false;
	float     miss_t = __builtin_inff();// hit_time of a MISS: INFINITY (och_h_octree.h:429) or 0.0F (och_octree.cpp:302)

	uint32_t* d_palette = nullptr;      // 6 colours per voxel type (olc::Pixel::n packing), shading epilogue
	uint32_t  n_palette = 0;
	uint32_t  exit_rgba = 0xFFFEBF00u;  // olc::Pixel{0x00,0xBF,0xFE} (test_och_h_octree.cpp:76)
	uint32_t  inside_rgba = 0xFF07193Fu;// olc::Pixel{0x3F,0x19,0x07} (:77)

	uint32_t* d_rcp = nullptr;
	int       rcp_log2n = 0;

	// staging (grown on demand)
	void*  d_stage = nullptr;  size_t d_stage_bytes = 0;   // device side of host-pointer calls

	// beam start (ort_beam.cuh): per level k one byte grid of the current DAG, built on demand by the first frame launch
	// that needs it.  Two buffers per level, used in turn, so that launches still reading the grid of the previous DAG
	// version (on other streams) are not overwritten by a rebuild.  Level kBeamFineLevel is the refinement's grid.
	uint8_t* d_beam_skip[9][2] = {};    // levels 0 .. ort::kBeamFineLevel
	int      beam_gen[9] = {};          // buffer of level k in use
	bool     beam_valid[9] = {};        // grid of level k describes the current DAG
	uint8_t* d_beam_tmp = nullptr;      // occupancy + pyramid scratch of a build (largest level)
	cudaEvent_t ev_beam = nullptr;      // last grid build done (builds share the scratch; launches on other streams wait for their grid)
	bool     beam_built_once = false;
	double   rcp_eps = 0;               // largest relative error of the reciprocal table in use
	int      rcp_sig_bits = 24;         // most significant bits any of its entries has
	BandMap band_maps[kBandMaps];
	uint64_t band_stamp = 0;
	int opt_band_order = 1;             // 1: frame launches schedule their bands by the costs recorded for the same view (BandMap)
	uint64_t band_schedules = 0;        // schedules applied so far
	int opt_beam = 1;                   // 1: camera frames of the lean tier start at their tile's beam bound
	int opt_beam_level = 0;             // 0: the finest level the tile size allows, tiles refining on level 8; else forced, no refinement (measurement)
	int opt_count_beam = 0;             // 1: launches that return PUSH counts use the beam start too (the launch's level alone); 2: with the level-8 refinement
	int opt_beam_after = 2;             // frame launches a DAG version must have seen before a grid is built for it (edit loops: see beam_level_for_launch)
	int beam_dag_age = 0;               // frame calls that have met the current DAG version (saturating)
	uint64_t frame_call_seq = 0;        // public frame calls so far (a host-buffer frame is one call, however many chunk launches it makes)
	uint64_t beam_seen_seq = 0;
	bool frame_call_nested = false;
	uint64_t beam_builds = 0;
	uint64_t build_bytes = 0;           // device bytes the last successful ort_build_voxels allocated (its peak)

	unsigned long long* d_counters = nullptr; // work counters of the persistent kernels: a ring, one per launch (kCounterRing)
	unsigned next_counter = 0;
	int max_blocks_rays = 0, max_blocks_frame = 0;

	uint64_t launches = 0;
	int opt_variant = 13;               // 0 = traverse(), 1 = round 1's FastWalker, 13 = round 2's tiers (LeanWalker first); others: ORT_EXPERIMENTS builds
	int rcp_host_status = -1;           // 1: this host's RCPPS equals the built-in table, 0: it differs (warned once), -1: not probed
	int opt_smem_levels = -1;
	int opt_block = 256;
	int opt_tile_shape = 0;
	int opt_persist_blocks = 1;         // explicit rays, persistent kernel: 1 = uncapped build (default), 6 / 8 = builds capped for that many resident blocks per SM
	int opt_band_rotate = -1;           // frames: the 16-row band that is scheduled first; -1 = the horizon band (horizon_band())
	int opt_zero_copy = 0;              // pinned host outputs: 1 = the kernel stores straight into mapped host memory
	int opt_frame_chunks = 0;           // host-buffer frames: launches per frame (0 = automatic)
	int opt_defer_sync = 0;             // host-buffer calls return once enqueued; ort_sync() completes them
	int opt_rays_chunk = 1 << 20;       // rays per pipeline stage of host-buffer ort_trace_rays
	int opt_low_water = 20;             // persistent kernels refill when <= this many lanes are busy
	int opt_rays_variant = 2;           // explicit rays: 2 = persistent refill
	int sm_count = 0;
	std::string last_error;
};

int ort_fail(ort_ctx* ctx, int code, const char* fmt, ...)
{
	char buf[512];
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(buf, sizeof buf, fmt, ap);
	va_end(ap);
	g_last_error = buf;
	if (ctx) ctx->last_error = buf;
	return code;
}

#define ORT_CUDA(ctx, call)                                                                                  \
	do {                                                                                                     \
		cudaError_t e_ = (call);                                                                             \
		if (e_ != cudaSuccess)                                                                               \
			return ort_fail(ctx, ORT_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
	} while (0)

namespace {

struct DeviceGuard
{
	int prev = -1;
	explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
	~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

bool is_device_ptr(const void* p)
{
	if (!p) return false;
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
	return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// device alias of a pinned (page-locked, mapped) host allocation, nullptr for anything else
void* mapped_host_alias(const void* p)
{
	if (!p) return nullptr;
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
	return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}

int ensure_dstage(ort_ctx* c, size_t bytes)
{
	if (bytes <= c->d_stage_bytes) return ORT_OK;
	if (c->d_stage)
	{
		cudaStreamSynchronize(c->stream); cudaStreamSynchronize(c->copy_stream); cudaStreamSynchronize(c->h2d_stream);
		cudaFree(c->d_stage); c->d_stage = nullptr; c->d_stage_bytes = 0;
	}
	c->slot_used[0] = c->slot_used[1] = false;
	ORT_CUDA(c, cudaMalloc(&c->d_stage, bytes));
	c->d_stage_bytes = bytes;
	return ORT_OK;
}

// the two pipeline slots of the device staging buffer: halves of the current capacity, so that a slot of an
// earlier (possibly still draining, see opt_defer_sync) call and a slot of this call never overlap
inline char* stage_slot(ort_ctx* c, int slot) { return static_cast<char*>(c->d_stage) + slot * (c->d_stage_bytes / 2 / 256 * 256); }

// end of a host-buffer call: wait for the results unless the caller asked to collect them with ort_sync()
int finish_host_call(ort_ctx* c)
{
	if (c->opt_defer_sync) return ORT_OK;
	ORT_CUDA(c, cudaStreamSynchronize(c->copy_stream));
	ORT_CUDA(c, cudaStreamSynchronize(c->stream));
	return ORT_OK;
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// every public entry point starts here: a successful call leaves no stale error message behind
inline void enter(ort_ctx* c)
{
	g_last_error.clear();
	if (c) c->last_error.clear();
}

constexpr unsigned kCounterRing = 64;      // persistent launches that may be in flight at once (on any streams)

// the work counter of the next persistent launch (the caller zeroes it on the launch's stream)
inline unsigned long long* next_counter(ort_ctx* c)
{
	return c->d_counters + (c->next_counter++ % kCounterRing);
}

// LeanWalker's slot words are node * 8 + 2^23-magic + index in 32 bits: ids stay below 0x16A00000
inline bool lean_capable(const ort_ctx* c) { return c->n_nodes < 0x16000000u; }

void band_map_release(BandMap& m)
{
	cudaFree(m.d_order[0]); cudaFree(m.d_order[1]); cudaFree(m.d_cost);
	if (m.h_cost) cudaFreeHost(m.h_cost);
	if (m.h_order) cudaFreeHost(m.h_order);
	if (m.ev_cost) cudaEventDestroy(m.ev_cost);
	if (m.ev_order) cudaEventDestroy(m.ev_order);
	for (int i = 0; i < 2; ++i) if (m.ev_read[i]) cudaEventDestroy(m.ev_read[i]);
	for (int i = 0; i < 2; ++i) if (m.ev_up[i]) cudaEventDestroy(m.ev_up[i]);
	m = BandMap{};
}

// the DAG changed: every beam grid is out of date (rebuilt by the next frame launch that wants one)
inline void beam_invalidate(ort_ctx* c)
{
	for (bool& v : c->beam_valid) v = false;
	c->beam_dag_age = 0;
}

}  // namespace

#include "ort_kernels.cuh"
#include "ort_build.cuh"

static_assert(ort::kBeamFineLevel == 8, "ort_ctx holds the beam grids of levels 0 .. 8");

namespace {

ort::Dag make_dag(const ort_ctx* c)
{
	ort::Dag g;
	g.nodes_m1 = c->d_nodes - 8 * static_cast<ptrdiff_t>(c->index_base);
	g.base_biased = static_cast<unsigned long long>(reinterpret_cast<uintptr_t>(g.nodes_m1)) - 4ull * ort::kMagicBits;
	g.root = c->root;
	g.depth = c->depth;
	g.leaf_dimf = std::ldexp(1.0F, -c->depth);
	g.miss_t = c->miss_t;
	g.plane_mask = (1u << (23 - c->depth)) - 1u;
	g.rt = ort::RcpTable{ c->d_rcp, 23 - c->rcp_log2n };
	return g;
}

// the walk a launch uses: the selected variant, with the lean tiers falling back to round 1's walker for DAGs beyond
// the lean id range
inline int walk_variant(const ort_ctx* c)
{
	if (c->opt_variant == 0) return 0;
	if (c->opt_variant == 1 || !lean_capable(c)) return 1;
	return ort::kLean;
}

// Beam start of a frame launch (ort_beam.cuh).  Returns the level of the grid the launch's tiles can be bounded with, or 0
// when the launch runs without: option off, another walk selected, PUSH counts wanted (they count the reference's
// rounds), a tile geometry the bound does not cover (warp tiles other than 8 x 4 pixels, cyclic tiles whose height is not
// a multiple of 4 rows: the 4 rows of a warp tile would not be neighbours in the frame), an origin outside the lean
// tier, a camera without a bound, or pixels too large for the coarsest grid.
int beam_level(const ort_ctx* c, const ort::Camera& cam, const ort::FrameRows& fr, bool counting)
{
	if (!c->opt_beam || c->opt_zero_copy || walk_variant(c) != ort::kLean || (counting && !c->opt_count_beam)) return 0;
	if (fr.tile_shape != 0 || (fr.tile_step > 1 && fr.tile_rows % 4 != 0)) return 0;
	if ((cam.origin_flags & ort::kOriginInCube) == 0u) return 0;
	const double radius = ort::beam_tile_radius(cam, c->rcp_eps);
	if (radius < 0) return 0;
	int k = ort::beam_level_for(radius, c->depth, ort::beam_t_max(cam.ox, cam.oy, cam.oz, c->rcp_eps));
	if (k && c->opt_beam_level >= ort::kBeamMinLevel && c->opt_beam_level < k) k = c->opt_beam_level;      // (only coarser: stays a bound)
	return k;
}

// What a frame launch does.  A grid costs ~9 small launches per DAG version; a loop that edits the DAG every other frame
// (BASELINE config 4: 1080p frames of 0.14 ms) would pay that again and again for frames too small to earn it back
// (measured: 0.140 -> 0.187 ms per frame).  So a DAG version gets its grid only once it has been traced
// by opt_beam_after frame calls without one: an edit loop never builds, a steady scene loses two frames.
int beam_level_for_launch(ort_ctx* c, const ort::Camera& cam, const ort::FrameRows& fr, bool counting)
{
	const int k = beam_level(c, cam, fr, counting);
	if (!k) return 0;
	if (c->beam_valid[k]) return k;
	if (c->beam_seen_seq != c->frame_call_seq)
	{
		c->beam_seen_seq = c->frame_call_seq;
		if (c->beam_dag_age <= c->opt_beam_after) ++c->beam_dag_age;      // the current call included
	}
	return c->beam_dag_age > c->opt_beam_after ? k : 0;
}

// Refinement of a launch that runs with the level-k grid (ort_beam.cuh, item 2): the time limit of its tiles' level-8
// march, or 0 when it has none (a forced level, a launch level below 7, a DAG shallower than 8, a launch that returns PUSH
// counts unless option count_beam is 2: with count_beam 1 the counts stay those of the launch-level start alone).
float beam_fine_limit(const ort_ctx* c, const ort::Camera& cam, int k, bool counting)
{
	if (c->opt_beam_level >= ort::kBeamMinLevel || (counting && c->opt_count_beam < 2)) return 0.0f;
	return ort::beam_fine_t_limit(ort::beam_tile_radius(cam, c->rcp_eps), c->depth, k);
}

// the same for the experiment kernels that bring their own walker (ORT_EXPERIMENTS builds): the selected variant is not
// the product's, everything else decides as above
int beam_level_any_variant(ort_ctx* c, const ort::Camera& cam, const ort::FrameRows& fr, bool counting)
{
	const int keep = c->opt_variant;
	c->opt_variant = ort::kLean;
	const int k = beam_level_for_launch(c, cam, fr, counting);
	c->opt_variant = keep;
	return k;
}

// Build the level-k grid of the current DAG into its spare buffer (on the launch stream, after the previous build).
int beam_build_grid(ort_ctx* c, int k)
{
	const size_t cells = static_cast<size_t>(1) << (3 * k);
	if (!c->d_beam_tmp)
	{
		// occupancy of the finest level + the pyramid levels 1 .. kBeamFineLevel
		size_t bytes = static_cast<size_t>(1) << (3 * ort::kBeamFineLevel);
		for (int j = 1; j <= ort::kBeamFineLevel; ++j) bytes += static_cast<size_t>(1) << (3 * j);
		ORT_CUDA(c, cudaMalloc(&c->d_beam_tmp, bytes));
	}
	const int gen = c->beam_gen[k] ^ 1;
	if (!c->d_beam_skip[k][gen]) ORT_CUDA(c, cudaMalloc(&c->d_beam_skip[k][gen], cells));
	// builds share the scratch: one after the other, whatever streams ask for them
	if (c->beam_built_once) ORT_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_beam, 0));
	uint8_t* occ = c->d_beam_tmp;
	uint8_t* pyr = c->d_beam_tmp + (static_cast<size_t>(1) << (3 * ort::kBeamFineLevel));
	size_t off[ort::kBeamFineLevel + 2] = {};
	for (int j = 1; j <= k; ++j) off[j + 1] = off[j] + (static_cast<size_t>(1) << (3 * j));      // level j at off[j]
	const ort::Dag dag = make_dag(c);
	const unsigned blocks = static_cast<unsigned>((cells + 255) / 256);
	ort::beam_occupancy_kernel<<<blocks, 256, 0, c->stream>>>(dag.nodes_m1, dag.root, k, occ);
	ort::beam_dilate_kernel<<<blocks, 256, 0, c->stream>>>(occ, k, pyr + off[k]);
	for (int j = k - 1; j >= 1; --j)
		ort::beam_reduce_kernel<<<static_cast<unsigned>(((static_cast<size_t>(1) << (3 * j)) + 255) / 256), 256, 0, c->stream>>>(pyr + off[j + 1], j, pyr + off[j]);
	ort::beam_skip_kernel<<<blocks, 256, 0, c->stream>>>(pyr, k, c->d_beam_skip[k][gen]);
	c->launches += 3 + (k - 1);
	ORT_CUDA(c, cudaGetLastError());
	ORT_CUDA(c, cudaEventRecord(c->ev_beam, c->stream));
	c->beam_built_once = true;
	c->beam_gen[k] = gen;
	c->beam_valid[k] = true;
	return ORT_OK;
}

// Make the level-k grid (and with `fine` the refinement's level-8 grid) describe the current DAG; on return the launch
// stream is ordered after the build.  The grids one call builds count as one build (ort_beam_builds).
int beam_ensure_grid(ort_ctx* c, int k, bool fine = false)
{
	bool built = false;
	for (const int level : { k, fine ? ort::kBeamFineLevel : k })
		if (!c->beam_valid[level])
		{
			const int rc = beam_build_grid(c, level);
			if (rc != ORT_OK) return rc;
			built = true;
		}
	if (built)
	{
		++c->beam_builds;
		return ORT_OK;
	}
	// built earlier, possibly on another stream
	ORT_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_beam, 0));
	return ORT_OK;
}

// the march over the tiles of one frame launch; `tile_word` = the output array that carries the start times
int beam_launch_march(ort_ctx* c, int k, const ort::Camera& cam, const ort::FrameRows& fr, float* tile_word, bool counting)
{
	const float fine_t = beam_fine_limit(c, cam, k, counting);
	const int rc = beam_ensure_grid(c, k, fine_t > 0.0f);
	if (rc != ORT_OK) return rc;
	const unsigned tiles = static_cast<unsigned>(((fr.W + 7) / 8) * ((fr.rows + 3) / 4));
	const float min_comp = ort::beam_certify_min_comp(cam, ort::beam_tile_radius(cam, c->rcp_eps), c->rcp_sig_bits);
	const int kf = ort::kBeamFineLevel;
	ort::beam_start_kernel<<<(tiles + 127) / 128, 128, 0, c->stream>>>(ort::BeamGrid{ c->d_beam_skip[k][c->beam_gen[k]], k },
	                                                                   ort::BeamGrid{ c->d_beam_skip[kf][c->beam_gen[kf]], kf }, fine_t, cam, fr, min_comp, tile_word);
	++c->launches;
	ORT_CUDA(c, cudaGetLastError());
	return ORT_OK;
}

// The band map of a view: found, or a slot taken over (a free one, else the least recently used).  A slot's buffers and
// events are created once and kept across views, so that a moving camera -- a new view every frame -- costs a lookup and
// nothing else.  nullptr when the launch has more bands than a slot holds or memory is short.
constexpr int kBandCap = 2048;          // bands a slot can hold (32 768 rows)

BandMap* band_map_for(ort_ctx* c, const ort::Camera& cam, const ort::FrameRows& fr)
{
	const float key[13] = { cam.ox, cam.oy, cam.oz, cam.r[0], cam.r[1], cam.r[2], cam.r[3], cam.r[4], cam.r[5], cam.r[6], cam.r[7], cam.r[8], cam.fov };
	const int geo[6] = { fr.W, fr.H, fr.y0, fr.rows, fr.tile_rows, fr.tile_step };
	const int bands = (fr.rows + 15) / 16;
	if (bands > kBandCap) return nullptr;
	BandMap* pick = nullptr;
	for (BandMap& m : c->band_maps)
		if (m.used && !std::memcmp(m.cam, key, sizeof key) && !std::memcmp(m.geo, geo, sizeof geo))
		{
			m.stamp = ++c->band_stamp;
			return &m;
		}
	for (BandMap& m : c->band_maps)
		if (!m.used) { pick = &m; break; }
	if (!pick)
	{
		pick = &c->band_maps[0];
		for (BandMap& m : c->band_maps)
			if (m.stamp < pick->stamp) pick = &m;
	}
	BandMap& m = *pick;
	if (m.used)
	{
		// the view that leaves may still have launches and copies in flight on its buffers
		if (m.recording) cudaEventSynchronize(m.ev_cost);
		for (int i = 0; i < 2; ++i) if (m.read_any[i]) cudaEventSynchronize(m.ev_read[i]);
		for (int i = 0; i < 2; ++i) if (m.up_any[i]) cudaEventSynchronize(m.ev_up[i]);
	}
	if (!m.d_cost)
	{
		const bool ok = cudaMalloc(&m.d_order[0], kBandCap * 2) == cudaSuccess && cudaMalloc(&m.d_order[1], kBandCap * 2) == cudaSuccess &&
		          cudaMalloc(&m.d_cost, kBandCap * 4) == cudaSuccess && cudaHostAlloc(&m.h_cost, kBandCap * 4, cudaHostAllocDefault) == cudaSuccess &&
		          cudaHostAlloc(&m.h_order, kBandCap * 4, cudaHostAllocDefault) == cudaSuccess &&
		          cudaEventCreateWithFlags(&m.ev_cost, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&m.ev_order, cudaEventDisableTiming) == cudaSuccess &&
		          cudaEventCreateWithFlags(&m.ev_read[0], cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&m.ev_read[1], cudaEventDisableTiming) == cudaSuccess &&
		          cudaEventCreateWithFlags(&m.ev_up[0], cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&m.ev_up[1], cudaEventDisableTiming) == cudaSuccess;
		if (!ok)
		{
			cudaGetLastError();
			band_map_release(m);
			return nullptr;
		}
	}
	m.used = true;
	m.stamp = ++c->band_stamp;
	std::memcpy(m.cam, key, sizeof key);
	std::memcpy(m.geo, geo, sizeof geo);
	m.bands = bands;
	m.read_any[0] = m.read_any[1] = false;
	m.up_any[0] = m.up_any[1] = false;
	m.cur = -1;
	m.recording = false;
	m.applied = 0;
	m.since = 0;
	m.seen = 0;
	return &m;
}

// Before a frame launch: apply the newest recorded schedule of the view (fr.band_order) and decide whether this launch
// records (fr.band_cost).  Costs are recorded by the first launches of a view and refreshed now and then.
void band_map_before(ort_ctx* c, BandMap* m, ort::FrameRows& fr, bool may_record)
{
	// (the pinned half the next schedule is written to must have been read by its previous upload: a copy still queued on
	// a stalled stream would otherwise pick up a half-written permutation)
	const int nxt = m->cur == 0 ? 1 : 0;
	if (m->recording && cudaEventQuery(m->ev_cost) == cudaSuccess && (!m->up_any[nxt] || cudaEventQuery(m->ev_up[nxt]) == cudaSuccess))
	{
		m->recording = false;
		// most expensive band first (stable: equal costs keep the band_rotate order they were measured in)
		const int nb = m->bands;
		uint16_t* ho = m->h_order + static_cast<size_t>(nxt) * kBandCap;
		std::vector<int> idx(nb);
		for (int b = 0; b < nb; ++b) idx[b] = (b + fr.band_rotate) % nb;
		std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return m->h_cost[a] > m->h_cost[b]; });
		for (int b = 0; b < nb; ++b) ho[b] = static_cast<uint16_t>(idx[b]);
		// the device buffer may still be read by launches of two schedules ago; the upload waits for them
		bool fine = true;
		if (m->read_any[nxt]) fine = cudaStreamWaitEvent(c->stream, m->ev_read[nxt], 0) == cudaSuccess;
		fine = fine && cudaMemcpyAsync(m->d_order[nxt], ho, nb * 2, cudaMemcpyHostToDevice, c->stream) == cudaSuccess &&
		       cudaEventRecord(m->ev_up[nxt], c->stream) == cudaSuccess && cudaEventRecord(m->ev_order, c->stream) == cudaSuccess;
		if (fine)
		{
			m->up_any[nxt] = true;
			m->cur = nxt;
			++m->applied;
			++c->band_schedules;
		}
		else
			cudaGetLastError();
	}
	if (m->cur >= 0)
	{
		if (cudaStreamWaitEvent(c->stream, m->ev_order, 0) == cudaSuccess)      // uploaded on whatever stream asked first
			fr.band_order = m->d_order[m->cur];
		else
			cudaGetLastError();
	}
	++m->since;
	++m->seen;
	// (a view seen for the first time records nothing: a camera that moves every frame never comes back to it)
	if (may_record && !m->recording && m->seen >= 2 && (m->applied < 2 || m->since >= 64))
	{
		if (cudaMemsetAsync(m->d_cost, 0, m->bands * 4, c->stream) == cudaSuccess)
			fr.band_cost = m->d_cost;
		else
			cudaGetLastError();
	}
}

void band_map_after(ort_ctx* c, BandMap* m, const ort::FrameRows& fr)
{
	if (fr.band_order)
	{
		const int i = fr.band_order == m->d_order[0] ? 0 : 1;
		if (cudaEventRecord(m->ev_read[i], c->stream) == cudaSuccess) m->read_any[i] = true;
	}
	if (fr.band_cost)
	{
		if (cudaMemcpyAsync(m->h_cost, m->d_cost, m->bands * 4, cudaMemcpyDeviceToHost, c->stream) == cudaSuccess &&
		    cudaEventRecord(m->ev_cost, c->stream) == cudaSuccess)
		{
			m->recording = true;
			m->since = 0;
		}
		else
			cudaGetLastError();
	}
}

}  // namespace

#ifdef ORT_EXPERIMENTS
#include "ort_experiments.cuh"
#endif


// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------

extern "C" {

const char* ort_version(void)
{
#ifdef ORT_EXPERIMENTS
	return "ort_b200 0.2 (sm_100a, +experiments)";
#else
	return "ort_b200 0.2 (sm_100a)";
#endif
}

const char* ort_last_error(const ort_ctx* ctx)
{
	if (ctx && !ctx->last_error.empty()) return ctx->last_error.c_str();
	return g_last_error.c_str();
}

int ort_create(ort_ctx** out, int device, int depth, uint32_t node_capacity)
{
	enter(nullptr);
	if (!out || depth < 1 || depth > ort::kMaxDepth)
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_create: depth must be 1..%d", ort::kMaxDepth);
	*out = nullptr;

	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
	{
		cudaGetLastError();
		return ort_fail(nullptr, ORT_ERR_NO_DEVICE, "ort_create: no CUDA device is visible; this library has no CPU path");
	}
	if (device < 0 || device >= ndev)
		return ort_fail(nullptr, ORT_ERR_INVALID, "ort_create: device %d out of range (%d visible)", device, ndev);

	cudaDeviceProp prop;
	ORT_CUDA(nullptr, cudaGetDeviceProperties(&prop, device));
	if (prop.major != 10)
		return ort_fail(nullptr, ORT_ERR_NO_DEVICE, "ort_create: device %d is sm_%d%d; this library carries sm_100a code only", device, prop.major, prop.minor);

	DeviceGuard g(device);
	ort_ctx* c = new (std::nothrow) ort_ctx;
	if (!c) return ort_fail(nullptr, ORT_ERR_INVALID, "ort_create: out of host memory");
	c->device = device;
	c->depth = depth;
	c->sm_count = prop.multiProcessorCount;

	// everything below may fail half-way: ort_destroy() releases whatever exists by then
	const int rc = [&]() -> int {
		ORT_CUDA(nullptr, cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
		c->stream = c->own_stream;
		ORT_CUDA(nullptr, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
		ORT_CUDA(nullptr, cudaStreamCreateWithFlags(&c->h2d_stream, cudaStreamNonBlocking));
		ORT_CUDA(nullptr, cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
		ORT_CUDA(nullptr, cudaEventCreateWithFlags(&c->ev_beam, cudaEventDisableTiming));
		for (int i = 0; i < 3; ++i)
		{
			ORT_CUDA(nullptr, cudaStreamCreateWithFlags(&c->aux_stream[i], cudaStreamNonBlocking));
			ORT_CUDA(nullptr, cudaEventCreateWithFlags(&c->ev_aux[i], cudaEventDisableTiming));
		}
		for (int i = 0; i < 8; ++i)
			ORT_CUDA(nullptr, cudaEventCreateWithFlags(&c->ev_part[i], cudaEventDisableTiming));
		for (int i = 0; i < 2; ++i)
		{
			ORT_CUDA(nullptr, cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming));
			ORT_CUDA(nullptr, cudaEventCreateWithFlags(&c->ev_chunk[i], cudaEventDisableTiming));
			ORT_CUDA(nullptr, cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
		}

		if (node_capacity < 64) node_capacity = 64;
		ORT_CUDA(nullptr, cudaMalloc(&c->d_nodes, static_cast<size_t>(node_capacity) * 32));
		c->cap_nodes = node_capacity;

		ORT_CUDA(nullptr, cudaMalloc(&c->d_counters, sizeof(unsigned long long) * kCounterRing));
		{
			const size_t smem = ort::lean_smem_bytes(depth);
			int b = 0;
			ORT_CUDA(nullptr, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, ort::trace_persistent_kernel<false, false>, 256, smem));
			c->max_blocks_rays = b * c->sm_count;
			ORT_CUDA(nullptr, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, ort::trace_persistent_kernel<false, true>, 256, smem));
			c->max_blocks_frame = b * c->sm_count;
		}
		return ort_set_rcp_table(c, ort_rcp_table_default, ORT_RCP_TABLE_LOG2N);
	}();
	if (rc != ORT_OK)
	{
		const std::string keep = g_last_error;
		ort_destroy(c);
		g_last_error = keep;
		return rc;
	}

	// The built-in RCPPS table is the one Intel's instruction yields.  A reference running on another vendor's CPU
	// computes other reciprocals, and a "drop-in" that silently disagreed with the host it runs next to would be a
	// trap: probe this host's instruction once and say so (ort_host_rcp_table() + ort_set_rcp_table() fix it).
	c->rcp_host_status = ort_host_rcp_matches(ort_rcp_table_default, ORT_RCP_TABLE_LOG2N);
	if (c->rcp_host_status == 0)
	{
		static bool warned = false;
		if (!warned)
		{
			warned = true;
			std::fprintf(stderr, "ort_b200: warning: this host's RCPPS differs from the built-in reciprocal table; GPU results will match a reference "
			                     "run on an Intel host, not on this one.  Call ort_host_rcp_table() and ort_set_rcp_table() to match this host.\n");
		}
	}
	*out = c;
	return ORT_OK;
}

int ort_rcp_host_status(const ort_ctx* c) { return c ? c->rcp_host_status : -1; }

int ort_destroy(ort_ctx* c)
{
	if (!c) return ORT_OK;
	DeviceGuard g(c->device);
	cudaDeviceSynchronize();                   // launches may be in flight on streams the caller handed over (ort_set_stream)
	if (c->stream) cudaStreamSynchronize(c->stream);
	if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
	if (c->h2d_stream) cudaStreamSynchronize(c->h2d_stream);
	cudaFree(c->d_nodes);
	cudaFree(c->d_rcp);
	cudaFree(c->d_palette);
	cudaFree(c->d_counters);
	cudaFree(c->d_stage);
	for (BandMap& m : c->band_maps) band_map_release(m);
	cudaFree(c->d_beam_tmp);
	for (int k = 0; k <= ort::kBeamFineLevel; ++k) { cudaFree(c->d_beam_skip[k][0]); cudaFree(c->d_beam_skip[k][1]); }
	if (c->ev_beam) cudaEventDestroy(c->ev_beam);
	for (int i = 0; i < 2; ++i)
	{
		if (c->ev_chunk[i]) cudaEventDestroy(c->ev_chunk[i]);
		if (c->ev_in[i]) cudaEventDestroy(c->ev_in[i]);
		if (c->ev_copied[i]) cudaEventDestroy(c->ev_copied[i]);
	}
	if (c->own_stream) cudaStreamDestroy(c->own_stream);
	if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
	if (c->h2d_stream) cudaStreamDestroy(c->h2d_stream);
	for (int i = 0; i < 3; ++i)
	{
		if (c->aux_stream[i]) { cudaStreamSynchronize(c->aux_stream[i]); cudaStreamDestroy(c->aux_stream[i]); }
		if (c->ev_aux[i]) cudaEventDestroy(c->ev_aux[i]);
	}
	if (c->ev_fork) cudaEventDestroy(c->ev_fork);
	for (int i = 0; i < 8; ++i) if (c->ev_part[i]) cudaEventDestroy(c->ev_part[i]);
	delete c;
	return ORT_OK;
}

int ort_set_rcp_table(ort_ctx* c, const uint32_t* tab, int log2n)
{
	enter(c);
	if (!c || !tab || log2n < 1 || log2n > 23)
		return ort_fail(c, ORT_ERR_INVALID, "ort_set_rcp_table: need a table of 2^1..2^23 entries");
	DeviceGuard g(c->device);
	ORT_CUDA(c, cudaStreamSynchronize(c->stream));
	{
		// every entry is the reciprocal of a number in [1, 2): exponent field 126 or 127 (ort::rcp_model relies on it)
		std::vector<uint32_t> host(static_cast<size_t>(1) << log2n);
		ORT_CUDA(c, cudaMemcpy(host.data(), tab, host.size() * 4, cudaMemcpyDefault));
		for (size_t k = 0; k < host.size(); ++k)
			if (((host[k] >> 23) | 1u) != 127u)
				return ort_fail(c, ORT_ERR_INVALID, "ort_set_rcp_table: entry %zu (0x%08x) is not in (0.5, 1]: not a reciprocal table of [1, 2)", k, host[k]);
		c->rcp_eps = ort::rcp_table_rel_error(host.data(), log2n);      // the beam start's bound widens with the table's error
		c->rcp_sig_bits = ort::rcp_table_sig_bits(host.data(), log2n);
	}
	if (c->rcp_log2n != log2n)
	{
		cudaFree(c->d_rcp);
		c->d_rcp = nullptr;
		ORT_CUDA(c, cudaMalloc(&c->d_rcp, sizeof(uint32_t) << log2n));
		c->rcp_log2n = log2n;
	}
	ORT_CUDA(c, cudaMemcpy(c->d_rcp, tab, sizeof(uint32_t) << log2n, cudaMemcpyDefault));
	return ORT_OK;
}

int ort_upload_full(ort_ctx* c, const uint32_t* nodes8, size_t n, uint32_t root)
{
	enter(c);
	if (!c || (n && !nodes8) || root > n || n > ort::kIdMask)
		return ort_fail(c, ORT_ERR_INVALID, "ort_upload_full: bad arguments (n=%zu root=%u)", n, root);
	DeviceGuard g(c->device);
	// A full upload replaces (and may reallocate) the array every launch in flight reads -- on the context's streams and on
	// any stream the caller handed over with ort_set_stream since: wait for the whole device, not for one stream.
	ORT_CUDA(c, cudaDeviceSynchronize());
	if (n > c->cap_nodes)
	{
		// grow with head-room for the deltas that will follow
		size_t want = n + n / 4 + 4096;
		if (want > ort::kIdMask) want = ort::kIdMask;   // compact ids are 29-bit (FastWalker: 3 bits of each stack entry carry the child index)
		cudaFree(c->d_nodes);
		c->d_nodes = nullptr;
		c->cap_nodes = 0;
		ORT_CUDA(c, cudaMalloc(&c->d_nodes, want * 32));
		c->cap_nodes = static_cast<uint32_t>(want);
	}
	if (n)
		ORT_CUDA(c, cudaMemcpyAsync(c->d_nodes, nodes8, n * 32, cudaMemcpyDefault, c->stream));
	ORT_CUDA(c, cudaStreamSynchronize(c->stream));   // the source may be reused by the caller right away
	c->n_nodes = static_cast<uint32_t>(n);
	c->root = root;
	c->index_base = 1;
	c->has_root = root != 0;
	c->miss_t = __builtin_inff();
	beam_invalidate(c);
	return ORT_OK;
}

int ort_upload_pool(ort_ctx* c, const uint32_t* nodes8, size_t n)
{
	if (!c || !nodes8 || n == 0 || n > ort::kIdMask)
		return ort_fail(c, ORT_ERR_INVALID, "ort_upload_pool: bad arguments (n=%zu)", n);
	const int rc = ort_upload_full(c, nodes8, n, 1);      // same copy; then switch the addressing to raw rows
	if (rc != ORT_OK) return rc;
	c->root = 0;
	c->index_base = 0;
	c->has_root = true;
	c->miss_t = 0.0F;                                     // och_octree.cpp:302
	beam_invalidate(c);
	return ORT_OK;
}

int ort_upload_delta(ort_ctx* c, const uint32_t* ids, const uint32_t* nodes8, size_t n, uint32_t root)
{
	enter(c);
	if (!c || (n && (!ids || !nodes8)))
		return ort_fail(c, ORT_ERR_INVALID, "ort_upload_delta: bad arguments");
	DeviceGuard g(c->device);

	uint32_t max_id = c->n_nodes;
	const bool dev_src = n && is_device_ptr(ids);
	if (n && dev_src != is_device_ptr(nodes8))
		return ort_fail(c, ORT_ERR_INVALID, "ort_upload_delta: ids and nodes8 must both be host or both be device pointers");
	if (n && (reinterpret_cast<uintptr_t>(nodes8) & 3u))
		return ort_fail(c, ORT_ERR_INVALID, "ort_upload_delta: nodes8 must be 4-byte aligned");
	if (n)
	{
		// ids are validated on the host either way (deltas are small: a few thousand entries)
		std::vector<uint32_t> tmp;
		const uint32_t* hid = ids;
		if (dev_src)
		{
			tmp.resize(n);
			ORT_CUDA(c, cudaMemcpy(tmp.data(), ids, n * 4, cudaMemcpyDeviceToHost));
			hid = tmp.data();
		}
		for (size_t i = 0; i < n; ++i)
		{
			if (hid[i] == 0) return ort_fail(c, ORT_ERR_INVALID, "ort_upload_delta: id 0 at entry %zu", i);
			if (hid[i] > max_id) max_id = hid[i];
		}
	}
	if (max_id > c->cap_nodes || root > c->cap_nodes)
		return ort_fail(c, ORT_ERR_CAPACITY, "ort_upload_delta: id %u exceeds the mirror capacity %u", max_id, c->cap_nodes);

	if (n)
	{
		const uint32_t* d_ids = ids;
		const uint32_t* d_src = nodes8;
		if (!dev_src)
		{
			// [ids | pad to 16 B | nodes] through the device staging buffer
			const size_t off = align_up(n * 4, 16);
			int rc = ensure_dstage(c, off + n * 32);
			if (rc != ORT_OK) return rc;
			// the staging buffer may still hold results of deferred host-buffer calls that are on their way out
			for (int i = 0; i < 2; ++i)
				if (c->slot_used[i]) ORT_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_copied[i], 0));
			char* base = static_cast<char*>(c->d_stage);
			ORT_CUDA(c, cudaMemcpyAsync(base, ids, n * 4, cudaMemcpyHostToDevice, c->stream));
			ORT_CUDA(c, cudaMemcpyAsync(base + off, nodes8, n * 32, cudaMemcpyHostToDevice, c->stream));
			d_ids = reinterpret_cast<const uint32_t*>(base);
			d_src = reinterpret_cast<const uint32_t*>(base + off);
		}
		const uint32_t threads = 256, blocks = static_cast<uint32_t>((2 * n + threads - 1) / threads);
		// (the kernel reads the source rows word by word: a device-side [ids | nodes] payload puts them at any 4-byte offset)
		ort::scatter_nodes_kernel<<<blocks, threads, 0, c->stream>>>(reinterpret_cast<uint4*>(c->d_nodes), d_ids, d_src, static_cast<uint32_t>(n));
		++c->launches;
		ORT_CUDA(c, cudaGetLastError());
		// host sources may be reused by the caller; device sources usually belong to a caching allocator that knows
		// nothing about this stream -- either way the scatter has read them when the call returns
		ORT_CUDA(c, cudaStreamSynchronize(c->stream));
	}
	c->n_nodes = max_id;
	bool changed = n != 0;
	if (c->index_base == 1)
	{
		changed = changed || c->root != root;
		c->root = root;
		c->has_root = root != 0;
	}
	if (changed) beam_invalidate(c);            // (an empty delta -- a per-frame sync without edits -- leaves the grids alone)
	return ORT_OK;
}

// ------------------------------------------------------------------------------------------------
// DAG of a dense voxel grid (ort_build.cuh, DESIGN section 13)
// ------------------------------------------------------------------------------------------------

}  // extern "C"

namespace {

// device allocations of one build, released however the build ends; `bytes` counts them (nothing is freed before the
// end, so that is the build's peak)
struct BuildTemps
{
	std::vector<void*> ptrs;
	uint64_t bytes = 0;
	~BuildTemps() { for (void* p : ptrs) cudaFree(p); }
	template<class T> cudaError_t alloc(T** p, size_t count)
	{
		void* q = nullptr;
		const size_t b = count ? count * sizeof(T) : sizeof(T);
		const cudaError_t e = cudaMalloc(&q, b);
		if (e == cudaSuccess) { ptrs.push_back(q); bytes += b; }
		*p = static_cast<T*>(q);
		return e;
	}
};

inline unsigned blocks_for(size_t n, unsigned threads = 256) { return static_cast<unsigned>((n + threads - 1) / threads); }

inline size_t pow2_at_least(size_t v)
{
	size_t p = 64;
	while (p < v) p <<= 1;
	return p;
}

int build_voxels(ort_ctx* c, const void* voxels, int elem_bytes, uint32_t nx, uint32_t ny, uint32_t nz, size_t* n_out, uint32_t* level_offsets)
{
	const int D = c->depth;
	cudaStream_t st = c->stream;
	BuildTemps tmp;

	// the input, on this device
	const void* src = voxels;
	{
		cudaPointerAttributes a;
		const bool dev = cudaPointerGetAttributes(&a, voxels) == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged);
		cudaGetLastError();
		if (dev && a.type == cudaMemoryTypeDevice && a.device != c->device)
			return ort_fail(c, ORT_ERR_INVALID, "ort_build_voxels: the voxels live on device %d, the context on device %d", a.device, c->device);
		if (dev && (reinterpret_cast<uintptr_t>(voxels) & static_cast<uintptr_t>(elem_bytes - 1)))
			return ort_fail(c, ORT_ERR_INVALID, "ort_build_voxels: a device source of %d-byte elements must be %d-byte aligned", elem_bytes, elem_bytes);
		if (!dev)
		{
			const size_t bytes = static_cast<size_t>(nx) * ny * nz * elem_bytes;
			void* d = nullptr;
			ORT_CUDA(c, tmp.alloc(reinterpret_cast<uint8_t**>(&d), bytes));
			ORT_CUDA(c, cudaMemcpyAsync(d, voxels, bytes, cudaMemcpyDefault, st));
			src = d;
		}
	}
	const ort::BuildInput in{ src, elem_bytes, nx, ny, nz };

	// level grids, clipped to the input's extent: level l has cells of side 2^(D-l+1) voxels
	ort::BuildLevel lv[ort::kBuildMaxDepth + 2] = {};
	size_t cap[ort::kBuildMaxDepth + 2] = {};
	{
		uint32_t gx = (nx + 1) / 2, gy = (ny + 1) / 2, gz = (nz + 1) / 2;
		for (int l = D; l >= 1; --l)
		{
			lv[l].gx = gx; lv[l].gy = gy; lv[l].gz = gz;
			ORT_CUDA(c, tmp.alloc(&lv[l].ids, static_cast<size_t>(gx) * gy * gz));
			gx = (gx + 1) / 2; gy = (gy + 1) / 2; gz = (gz + 1) / 2;
		}
	}
	unsigned long long* d_cnt = nullptr;                       // [0] leaf non-empty, [l] non-empty of level l, [D+1+l] distinct
	ORT_CUDA(c, tmp.alloc(&d_cnt, 2 * (D + 1)));
	ORT_CUDA(c, cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long) * 2 * (D + 1), st));
	unsigned long long h_cnt[2 * (ort::kBuildMaxDepth + 1)] = {};

	// bottom-up: a level's distinct contents are at most its non-empty cells, which are at most the level below's
	ort::build_count_leaf_kernel<<<blocks_for(static_cast<size_t>(lv[D].gx) * lv[D].gy * lv[D].gz), 256, 0, st>>>(in, lv[D], d_cnt);
	++c->launches;
	ORT_CUDA(c, cudaMemcpyAsync(h_cnt, d_cnt, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
	ORT_CUDA(c, cudaStreamSynchronize(st));
	size_t bound = static_cast<size_t>(h_cnt[0]);
	for (int l = D; l >= 1; --l)
	{
		const size_t cells = static_cast<size_t>(lv[l].gx) * lv[l].gy * lv[l].gz;
		cap[l] = pow2_at_least(2 * std::min(bound, cells));      // load factor <= 1/2
		ORT_CUDA(c, tmp.alloc(&lv[l].table, cap[l]));
		lv[l].mask = static_cast<uint32_t>(cap[l] - 1);
		ORT_CUDA(c, cudaMemsetAsync(lv[l].table, 0xFF, cap[l] * 4, st));
		ort::build_insert_kernel<<<blocks_for(cells), 256, 0, st>>>(l == D, in, lv[l], l == D ? lv[l] : lv[l + 1], d_cnt + l);
		ort::build_count_table_kernel<<<blocks_for(cap[l]), 256, 0, st>>>(lv[l].table, cap[l], d_cnt + D + 1 + l);
		c->launches += 2;
		ORT_CUDA(c, cudaGetLastError());
		ORT_CUDA(c, cudaMemcpyAsync(h_cnt + l, d_cnt + l, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
		ORT_CUDA(c, cudaStreamSynchronize(st));
		bound = static_cast<size_t>(h_cnt[l]);
	}
	ORT_CUDA(c, cudaMemcpyAsync(h_cnt + D + 1, d_cnt + D + 1, sizeof(unsigned long long) * (D + 1), cudaMemcpyDeviceToHost, st));
	ORT_CUDA(c, cudaStreamSynchronize(st));

	// final ids: level l holds ids base[l] .. base[l] + n[l] - 1
	size_t n_lvl[ort::kBuildMaxDepth + 2] = {}, base[ort::kBuildMaxDepth + 2] = {};
	size_t total = 0;
	for (int l = 1; l <= D; ++l)
	{
		n_lvl[l] = static_cast<size_t>(h_cnt[D + 1 + l]);
		base[l] = 1 + total;
		total += n_lvl[l];
	}
	if (total > ort::kIdMask)
		return ort_fail(c, ORT_ERR_CAPACITY, "ort_build_voxels: the grid's DAG has %zu nodes, more than the %u compact ids allow", total, ort::kIdMask);

	// the output rows: straight into a new mirror when the current one is too small, else a temporary copied over
	uint32_t* out = nullptr;
	size_t out_cap = 0;
	struct NewMirror { uint32_t* p = nullptr; ~NewMirror() { cudaFree(p); } } fresh;
	if (total > c->cap_nodes)
	{
		out_cap = std::min<size_t>(total + total / 4 + 4096, ort::kIdMask);      // head-room for the deltas that follow, as ort_upload_full
		ORT_CUDA(c, cudaMalloc(&fresh.p, out_cap * 32));
		out = fresh.p;
	}
	else if (total)
		ORT_CUDA(c, tmp.alloc(&out, total * 8));

	if (total)
	{
		// top-down: scratch sized for the widest level
		size_t max_slots = 0, max_cap = 0;
		for (int l = 1; l < D; ++l) { max_slots = std::max(max_slots, 8 * n_lvl[l]); max_cap = std::max(max_cap, cap[l + 1]); }
		uint32_t *ch = nullptr, *pos = nullptr, *first = nullptr, *scratch = nullptr;
		uint32_t* frontier[ort::kBuildMaxDepth + 2] = {};
		for (int l = 1; l <= D; ++l) ORT_CUDA(c, tmp.alloc(&frontier[l], n_lvl[l]));
		if (max_slots)
		{
			ORT_CUDA(c, tmp.alloc(&ch, max_slots));
			ORT_CUDA(c, tmp.alloc(&pos, max_slots));
			ORT_CUDA(c, tmp.alloc(&first, max_cap));
			ORT_CUDA(c, tmp.alloc(&scratch, ort::scan_scratch_words(max_slots)));
		}
		ORT_CUDA(c, cudaMemcpyAsync(frontier[1], lv[1].ids, 4, cudaMemcpyDeviceToDevice, st));     // the root cell's temporary id
		for (int l = 1; l < D; ++l)
		{
			const size_t slots = 8 * n_lvl[l];
			ORT_CUDA(c, cudaMemsetAsync(first, 0xFF, cap[l + 1] * 4, st));
			ort::build_children_kernel<<<blocks_for(slots), 256, 0, st>>>(frontier[l], slots, lv[l], lv[l + 1], ch, first);
			ort::build_flags_kernel<<<blocks_for(slots), 256, 0, st>>>(ch, first, slots, pos);
			c->launches += 2;
			ort::scan_exclusive(pos, slots, scratch, st, c->launches);
			ort::build_rows_kernel<<<blocks_for(slots), 256, 0, st>>>(ch, first, pos, slots, static_cast<uint32_t>(base[l + 1]),
			                                                          out + 8 * (base[l] - 1), frontier[l + 1]);
			++c->launches;
			ORT_CUDA(c, cudaGetLastError());
		}
		ort::build_leaf_rows_kernel<<<blocks_for(n_lvl[D]), 256, 0, st>>>(frontier[D], n_lvl[D], in, lv[D], out + 8 * (base[D] - 1));
		++c->launches;
		ORT_CUDA(c, cudaGetLastError());
	}
	ORT_CUDA(c, cudaStreamSynchronize(st));

	// install, as ort_upload_full does: every launch in flight reads the array that is replaced
	ORT_CUDA(c, cudaDeviceSynchronize());
	if (out_cap)
	{
		cudaFree(c->d_nodes);
		c->d_nodes = out;
		c->cap_nodes = static_cast<uint32_t>(out_cap);
		fresh.p = nullptr;                                         // (owned by the context now)
	}
	else if (total)
	{
		ORT_CUDA(c, cudaMemcpyAsync(c->d_nodes, out, total * 32, cudaMemcpyDeviceToDevice, st));
		ORT_CUDA(c, cudaStreamSynchronize(st));
	}
	c->n_nodes = static_cast<uint32_t>(total);
	c->root = total ? 1u : 0u;
	c->index_base = 1;
	c->has_root = total != 0;
	c->miss_t = __builtin_inff();
	beam_invalidate(c);
	c->build_bytes = tmp.bytes + out_cap * 32;
	if (n_out) *n_out = total;
	if (level_offsets)
	{
		for (int l = 1; l <= D; ++l) level_offsets[l - 1] = static_cast<uint32_t>(base[l]);
		level_offsets[D] = static_cast<uint32_t>(total + 1);
	}
	return ORT_OK;
}

}  // namespace

extern "C" {

int ort_build_voxels(ort_ctx* c, const void* voxels, int elem_bytes, int nx, int ny, int nz, size_t* n_nodes, uint32_t* level_offsets)
{
	enter(c);
	if (!c) return ort_fail(c, ORT_ERR_INVALID, "ort_build_voxels: null context");
	if (c->depth > ort::kBuildMaxDepth)
		return ort_fail(c, ORT_ERR_INVALID, "ort_build_voxels: context depth %d; the builder takes depth <= %d", c->depth, ort::kBuildMaxDepth);
	const int dim = 1 << c->depth;
	if (!voxels || (elem_bytes != 1 && elem_bytes != 4) || nx < 1 || ny < 1 || nz < 1 || nx > dim || ny > dim || nz > dim)
		return ort_fail(c, ORT_ERR_INVALID, "ort_build_voxels: bad arguments (voxels=%p elem_bytes=%d extent %d x %d x %d, 1..%d per axis)",
		                voxels, elem_bytes, nx, ny, nz, dim);
	DeviceGuard g(c->device);
	const int rc = build_voxels(c, voxels, elem_bytes, static_cast<uint32_t>(nx), static_cast<uint32_t>(ny), static_cast<uint32_t>(nz), n_nodes, level_offsets);
	if (rc != ORT_OK) cudaGetLastError();       // (an allocation that failed leaves its error behind for the next check)
	return rc;
}

int ort_read_nodes(ort_ctx* c, uint32_t first, size_t n, uint32_t* nodes8)
{
	enter(c);
	if (!c || (n && (!nodes8 || first == 0 || static_cast<size_t>(first) - 1 + n > c->n_nodes)))
		return ort_fail(c, ORT_ERR_INVALID, "ort_read_nodes: bad arguments (first=%u n=%zu, %u rows in the mirror)", first, n, c ? c->n_nodes : 0u);
	if (!n) return ORT_OK;
	DeviceGuard g(c->device);
	ORT_CUDA(c, cudaMemcpyAsync(nodes8, c->d_nodes + 8 * (static_cast<size_t>(first) - 1), n * 32, cudaMemcpyDefault, c->stream));
	ORT_CUDA(c, cudaStreamSynchronize(c->stream));
	return ORT_OK;
}

uint64_t ort_build_bytes(const ort_ctx* c) { return c ? c->build_bytes : 0; }

}  // extern "C"

// Host copy of a buffer that may live on a device (ort_tree_import), made on the context's stream: the buffer itself
// when it is host memory or there is no context (a tree without one makes no CUDA call), nullptr when the copy fails.
const void* ort_host_view(ort_ctx* c, const void* p, size_t bytes, std::vector<uint8_t>& keep)
{
	if (!c || !p) return p;
	DeviceGuard g(c->device);
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return p; }
	if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) return p;
	keep.resize(bytes);
	if (cudaMemcpyAsync(keep.data(), p, bytes, cudaMemcpyDefault, c->stream) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess)
	{
		cudaGetLastError();
		return nullptr;
	}
	return keep.data();
}

extern "C" {

// ------------------------------------------------------------------------------------------------
// trace
// ------------------------------------------------------------------------------------------------

static ort::Camera make_camera(const ort_ctx* c, const float pos[3], const float rot[9], float fov_factor, int W, int H);

// Which 16-row band of the launch should be scheduled first.  A launch ends when its longest rays do, and those are
// the grazing rays at the top of the downward-looking part of the picture (farthest terrain); rows above the horizon
// leave the cube after a few rounds.  Top-to-bottom block order is right when the whole strip looks down (the far
// terrain comes first); with the horizon inside the strip the cheap sky rows would go first and the long rays start
// late (pose A: SMs busy 70 % of the launch).  So: start at the first band whose centre ray points below the horizon
// (z is up in the reference's world, test_och_h_octree.cpp:767-787) and wrap around to the sky at the end.  Any
// rotation is valid; this one only shortens the launch tail (pose A: 0.58 -> 0.51 ms per 4K frame).
static int horizon_band(const ort::Camera& cam, int W, int y0, int rows, int tile_rows, int tile_step)
{
	const int bands = (rows + 15) / 16;
	const float u = cam.aspect * (cam.vfx * static_cast<float>(W / 2) - 1.0F);
	for (int b = 0; b < bands; ++b)
	{
		const int r = b * 16 + 8 < rows ? b * 16 + 8 : rows - 1;
		const int y = tile_step == 1 ? y0 + r : y0 + (r / tile_rows) * tile_rows * tile_step + r % tile_rows;
		const float v = cam.vfy * static_cast<float>(y) - 1.0F;
		const float rv = u * cam.r[3] + v * cam.r[4] + cam.fov * cam.r[5];        // ray z = -rv * rm (ort::camera_ray)
		if (rv > 0.0F) return b;
	}
	return 0;
}

static ort::Camera make_camera(const ort_ctx* c, const float pos[3], const float rot[9], float fov_factor, int W, int H)
{
	ort::Camera cam;
	cam.ox = pos[0]; cam.oy = pos[1]; cam.oz = pos[2];
	for (int i = 0; i < 9; ++i) cam.r[i] = rot[i];
	cam.fov = fov_factor;
	cam.aspect = static_cast<float>(W) / static_cast<float>(H);   // test_och_h_octree.cpp:89
	cam.vfx = 2.0F / static_cast<float>(W);                       // :91
	cam.vfy = 2.0F / static_cast<float>(H);                       // :93
	cam.origin_flags = ort::camera_origin_flags(pos[0], pos[1], pos[2], (1u << (23 - c->depth)) - 1u);
	return cam;
}

static int launch_miss(ort_ctx* c, size_t n, uint32_t* v, uint8_t* f, float* t, uint16_t* np)
{
	if (!n) return ORT_OK;
	// root 0: every ray is a MISS of the h_octree kind (the callers' guard, test_och_h_octree.cpp:443)
	ort::fill_miss_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->stream>>>(v, f, t, np, __builtin_inff(), n);
	++c->launches;
	ORT_CUDA(c, cudaGetLastError());
	return ORT_OK;
}

static int bad_variant(ort_ctx* c)
{
#ifdef ORT_EXPERIMENTS
	return ort_fail(c, ORT_ERR_INVALID, "variant %d is not a frame kernel of this build", c->opt_variant);
#else
	return ort_fail(c, ORT_ERR_INVALID, "variant %d is an experiment kernel: this library was built without ORT_EXPERIMENTS (use libort_b200_exp.so)", c->opt_variant);
#endif
}

int ort_trace_rays_async(ort_ctx* c, const float* o3, int o_stride, const float* d3, size_t n,
                         uint32_t* voxel, uint8_t* face, float* t, uint16_t* npush)
{
	enter(c);
	if (!c || (n && (!o3 || !d3 || !voxel || !face || !t)) || (o_stride != 0 && o_stride != 3))
		return ort_fail(c, ORT_ERR_INVALID, "ort_trace_rays: bad arguments");
	if (!n) return ORT_OK;
	DeviceGuard g(c->device);
	if (!c->has_root)
		return launch_miss(c, n, voxel, face, t, npush);
	const ort::Dag dag = make_dag(c);
	const size_t smem = ort::lean_smem_bytes(c->depth);
	if (c->opt_rays_variant == 2 && c->opt_variant != 0 && lean_capable(c))
	{
		// persistent warps with lane refill; every launch draws from its own counter of the ring, zeroed on the launch's
		// stream, so launches on different caller streams (ort_set_stream) do not interfere
		unsigned long long* counter = next_counter(c);
		ORT_CUDA(c, cudaMemsetAsync(counter, 0, sizeof(unsigned long long), c->stream));
		const unsigned long long need = (n + 255) / 256;
		const ort::Camera cam0{};
		const ort::FrameRows fr0{};
		// the uncapped build is the default (16.7 M incoherent rays: 1.58 ms; capped for 6 / 8 resident blocks per SM: 1.67 / 1.83 ms,
		// profiles/r2_config3_rays_vs_reference.json)
		const int per_sm = npush ? 0 : (c->opt_persist_blocks == 8 ? 8 : (c->opt_persist_blocks == 6 ? 6 : 0));
		const unsigned long long cap_blocks = per_sm ? static_cast<unsigned long long>(c->sm_count) * per_sm : static_cast<unsigned long long>(c->max_blocks_rays);
		const unsigned pb = static_cast<unsigned>(need < cap_blocks ? need : cap_blocks);
		if (npush)            ort::trace_persistent_kernel<true, false><<<pb, 256, smem, c->stream>>>(dag, o3, o_stride, d3, cam0, fr0, n, counter, c->opt_low_water, voxel, face, t, npush);
		else if (per_sm == 0) ort::trace_persistent_kernel<false, false><<<pb, 256, smem, c->stream>>>(dag, o3, o_stride, d3, cam0, fr0, n, counter, c->opt_low_water, voxel, face, t, npush);
		else if (per_sm == 6) ort::trace_persistent_kernel<false, false, 6><<<pb, 256, smem, c->stream>>>(dag, o3, o_stride, d3, cam0, fr0, n, counter, c->opt_low_water, voxel, face, t, npush);
		else                  ort::trace_persistent_kernel<false, false, 8><<<pb, 256, smem, c->stream>>>(dag, o3, o_stride, d3, cam0, fr0, n, counter, c->opt_low_water, voxel, face, t, npush);
		++c->launches;
		ORT_CUDA(c, cudaGetLastError());
		return ORT_OK;
	}
	const unsigned blocks = static_cast<unsigned>((n + 255) / 256);
#define ORT_LAUNCH_RAYS(V, C) ort::trace_rays_kernel<V, C><<<blocks, 256, (V) == ort::kLean ? smem : 0, c->stream>>>(dag, o3, o_stride, d3, n, voxel, face, t, npush)
	switch (walk_variant(c))
	{
	case 0:  if (npush) ORT_LAUNCH_RAYS(0, true); else ORT_LAUNCH_RAYS(0, false); break;
	case 1:  if (npush) ORT_LAUNCH_RAYS(1, true); else ORT_LAUNCH_RAYS(1, false); break;
	default: if (npush) ORT_LAUNCH_RAYS(ort::kLean, true); else ORT_LAUNCH_RAYS(ort::kLean, false); break;
	}
#undef ORT_LAUNCH_RAYS
	++c->launches;
	ORT_CUDA(c, cudaGetLastError());
	return ORT_OK;
}

static bool frame_args_ok(const float* pos, const float* rot, int W, int H, int y0, int rows, int tile_rows, int tile_step)
{
	return pos && rot && W > 0 && H > 0 && rows >= 0 && tile_rows > 0 && tile_step > 0 && y0 >= 0;
}

int ort_trace_frame_async(ort_ctx* c, const float pos[3], const float rot[9], float fov_factor,
                          int W, int H, int y0, int rows, int tile_rows, int tile_step,
                          uint32_t* voxel, uint8_t* face, float* t, uint16_t* npush)
{
	enter(c);
	if (!c || !frame_args_ok(pos, rot, W, H, y0, rows, tile_rows, tile_step) || (rows && (!voxel || !face || !t)))
		return ort_fail(c, ORT_ERR_INVALID, "ort_trace_frame: bad arguments");
	if (!rows) return ORT_OK;
	DeviceGuard g(c->device);
	if (!c->frame_call_nested) ++c->frame_call_seq;
	const size_t n = static_cast<size_t>(rows) * W;
	if (!c->has_root)
		return launch_miss(c, n, voxel, face, t, npush);
	const ort::Dag dag = make_dag(c);
	const ort::Camera cam = make_camera(c, pos, rot, fov_factor, W, H);
	const int rotate = c->opt_band_rotate >= 0 ? c->opt_band_rotate % ((rows + 15) / 16) : horizon_band(cam, W, y0, rows, tile_rows, tile_step);
	ort::FrameRows fr{ W, H, y0, rows, tile_rows, tile_step, c->opt_tile_shape, rotate, ort::tile_shift_of(tile_rows) };
	const dim3 grid((W + 15) / 16, (rows + 15) / 16);
	const size_t smem = ort::lean_smem_bytes(c->depth);
	if (c->opt_variant == 2 && lean_capable(c))
	{
		// the persistent lane-refill kernel over the pixels of the strip (in 8 x 4 tile order)
		unsigned long long* counter = next_counter(c);
		ORT_CUDA(c, cudaMemsetAsync(counter, 0, sizeof(unsigned long long), c->stream));
		const unsigned long long tiles = static_cast<unsigned long long>((W + 7) / 8) * ((rows + 3) / 4);
		const unsigned long long np = tiles * 32ull, need = (np + 255) / 256;
		const unsigned pblocks = static_cast<unsigned>(need < static_cast<unsigned long long>(c->max_blocks_frame) ? need : c->max_blocks_frame);
		if (npush) ort::trace_persistent_kernel<true, true><<<pblocks, 256, smem, c->stream>>>(dag, nullptr, 0, nullptr, cam, fr, np, counter, c->opt_low_water, voxel, face, t, npush);
		else       ort::trace_persistent_kernel<false, true><<<pblocks, 256, smem, c->stream>>>(dag, nullptr, 0, nullptr, cam, fr, np, counter, c->opt_low_water, voxel, face, t, npush);
		++c->launches;
		ORT_CUDA(c, cudaGetLastError());
		return ORT_OK;
	}
#ifdef ORT_EXPERIMENTS
	{
		const int rc = launch_frame_experiment(c, dag, cam, fr, voxel, face, t, npush);
		if (rc == ORT_ERR_CUDA) return ort_fail(c, ORT_ERR_CUDA, "experiment variant %d: launch failed: %s", c->opt_variant, cudaGetErrorString(cudaGetLastError()));
		if (rc == ORT_OK) return ORT_OK;
	}
#endif
	if (c->opt_variant != 0 && c->opt_variant != 1 && c->opt_variant != 2 && c->opt_variant != ort::kLean)
		return bad_variant(c);
	const int bk = beam_level_for_launch(c, cam, fr, npush != nullptr);
	if (bk)
	{
		const int rc = beam_launch_march(c, bk, cam, fr, t, npush != nullptr);
		if (rc != ORT_OK) return rc;
	}
	// band schedule of this view (launches of 8 bands and more; the frame kernels of the product walks)
	BandMap* bm = (c->opt_band_order && c->opt_band_rotate < 0 && grid.y >= 8 && grid.y < 65536 && c->opt_tile_shape == 0 && walk_variant(c) == ort::kLean)
	                  ? band_map_for(c, cam, fr) : nullptr;
	if (bm) band_map_before(c, bm, fr, npush == nullptr);
#define ORT_LAUNCH_FRAME(V, C, B) ort::trace_frame_kernel<V, C, B><<<grid, 256, (V) == ort::kLean ? smem : 0, c->stream>>>(dag, cam, fr, voxel, face, t, npush)
	switch (walk_variant(c))
	{
	case 0:  if (npush) ORT_LAUNCH_FRAME(0, true, false); else ORT_LAUNCH_FRAME(0, false, false); break;
	case 1:  if (npush) ORT_LAUNCH_FRAME(1, true, false); else ORT_LAUNCH_FRAME(1, false, false); break;
	default:
		if (fr.band_cost)
		{
			// (recording launches return no PUSH counts: band_map_before() leaves those alone)
			if (bk) ort::trace_frame_kernel<ort::kLean, false, true, true><<<grid, 256, smem, c->stream>>>(dag, cam, fr, voxel, face, t, npush);
			else    ort::trace_frame_kernel<ort::kLean, false, false, true><<<grid, 256, smem, c->stream>>>(dag, cam, fr, voxel, face, t, npush);
		}
		else if (bk) { if (npush) ORT_LAUNCH_FRAME(ort::kLean, true, true); else ORT_LAUNCH_FRAME(ort::kLean, false, true); }
		else         { if (npush) ORT_LAUNCH_FRAME(ort::kLean, true, false); else ORT_LAUNCH_FRAME(ort::kLean, false, false); }
		break;
	}
#undef ORT_LAUNCH_FRAME
	++c->launches;
	ORT_CUDA(c, cudaGetLastError());
	if (bm) band_map_after(c, bm, fr);
	return ORT_OK;
}

int ort_trace_frames_async(ort_ctx* c, const ort_frame_job* jobs, int n_jobs)
{
	enter(c);
	if (!c || n_jobs < 0 || (n_jobs && !jobs))
		return ort_fail(c, ORT_ERR_INVALID, "ort_trace_frames_async: bad arguments");
	DeviceGuard g(c->device);
	for (int i = 0; i < n_jobs; ++i)
	{
		const ort_frame_job& j = jobs[i];
		if (!frame_args_ok(j.pos, j.rot, j.W, j.H, j.y0, j.rows, j.tile_rows, j.tile_step) || (j.rows && (!j.voxel || !j.face || !j.t)))
			return ort_fail(c, ORT_ERR_INVALID, "ort_trace_frames_async: bad job %d", i);
	}
	if (!c->has_root)
	{
		for (int i = 0; i < n_jobs; ++i)
		{
			const int rc = launch_miss(c, static_cast<size_t>(jobs[i].rows) * jobs[i].W, jobs[i].voxel, jobs[i].face, jobs[i].t, jobs[i].npush);
			if (rc != ORT_OK) return rc;
		}
		return ORT_OK;
	}
	if (c->opt_variant != 0 && c->opt_variant != 1 && c->opt_variant != ort::kLean)
		return ort_fail(c, ORT_ERR_INVALID, "ort_trace_frames_async: the batched launch exists for variants 0, 1 and 13 (selected: %d)", c->opt_variant);
	const ort::Dag dag = make_dag(c);
	const size_t smem = ort::lean_smem_bytes(c->depth);
	++c->frame_call_seq;
	int i = 0;
	while (i < n_jobs)
	{
		// the next batch: up to kMaxJobs non-empty jobs, consumed in order
		ort::FrameJobBatch batch{};
		int n = 0;
		unsigned gx = 0, gy = 0;
		for (; i < n_jobs && n < ort::kMaxJobs; ++i)
		{
			const ort_frame_job& j = jobs[i];
			if (!j.rows) continue;
			ort::FrameJob& d = batch.job[n++];
			d.cam = make_camera(c, j.pos, j.rot, j.fov_factor, j.W, j.H);
			const int rotate = c->opt_band_rotate >= 0 ? c->opt_band_rotate % ((j.rows + 15) / 16) : horizon_band(d.cam, j.W, j.y0, j.rows, j.tile_rows, j.tile_step);
			d.fr = ort::FrameRows{ j.W, j.H, j.y0, j.rows, j.tile_rows, j.tile_step, 0, rotate, ort::tile_shift_of(j.tile_rows) };
			d.voxel = j.voxel; d.face = j.face; d.t = j.t; d.npush = j.npush;
			d.beam_k = 0;
			d.beam_fine_t = 0.0f;
			gx = std::max(gx, static_cast<unsigned>((j.W + 15) / 16));
			gy = std::max(gy, static_cast<unsigned>((j.rows + 15) / 16));
		}
		if (!n) break;
		bool count = false;
		for (int k = 0; k < n; ++k) count |= batch.job[k].npush != nullptr;
		// beam start: all or nothing per batch (one kernel instantiation per launch)
		bool beam = true;
		unsigned max_tiles = 0;
		for (int k = 0; k < n && beam; ++k)
		{
			ort::FrameJob& d = batch.job[k];
			d.beam_k = beam_level_for_launch(c, d.cam, d.fr, count);
			d.beam_min_comp = ort::beam_certify_min_comp(d.cam, ort::beam_tile_radius(d.cam, c->rcp_eps), c->rcp_sig_bits);
			d.beam_fine_t = beam_fine_limit(c, d.cam, d.beam_k, count);
			beam = d.beam_k != 0;
			max_tiles = std::max(max_tiles, static_cast<unsigned>(((d.fr.W + 7) / 8) * ((d.fr.rows + 3) / 4)));
		}
		if (beam)
		{
			ort::BeamGridSet grids{};
			for (int k = 0; k < n; ++k)
			{
				const int bk = batch.job[k].beam_k, kf = ort::kBeamFineLevel;
				const bool fine = batch.job[k].beam_fine_t > 0.0f;
				const int rc = beam_ensure_grid(c, bk, fine);
				if (rc != ORT_OK) return rc;
				grids.skip[bk] = c->d_beam_skip[bk][c->beam_gen[bk]];
				if (fine) grids.skip[kf] = c->d_beam_skip[kf][c->beam_gen[kf]];
			}
			ort::beam_start_batch_kernel<<<dim3((max_tiles + 127) / 128, static_cast<unsigned>(n)), 128, 0, c->stream>>>(grids, batch);
			++c->launches;
			ORT_CUDA(c, cudaGetLastError());
		}
		else
			for (int k = 0; k < n; ++k) { batch.job[k].beam_k = 0; batch.job[k].beam_fine_t = 0.0f; }
		const dim3 bgrid(gx, gy, static_cast<unsigned>(n));
#define ORT_LAUNCH_BATCH(V, C, B) ort::trace_frames_kernel<V, C, B><<<bgrid, 256, (V) == ort::kLean ? smem : 0, c->stream>>>(dag, batch)
		switch (walk_variant(c))
		{
		case 0:  if (count) ORT_LAUNCH_BATCH(0, true, false); else ORT_LAUNCH_BATCH(0, false, false); break;
		case 1:  if (count) ORT_LAUNCH_BATCH(1, true, false); else ORT_LAUNCH_BATCH(1, false, false); break;
		default:
			if (beam) { if (count) ORT_LAUNCH_BATCH(ort::kLean, true, true); else ORT_LAUNCH_BATCH(ort::kLean, false, true); }
			else      { if (count) ORT_LAUNCH_BATCH(ort::kLean, true, false); else ORT_LAUNCH_BATCH(ort::kLean, false, false); }
			break;
		}
#undef ORT_LAUNCH_BATCH
		++c->launches;
		ORT_CUDA(c, cudaGetLastError());
	}
	return ORT_OK;
}

// Device layout of one staged result block of n rays: voxel[n] | t[n] | npush[n] | face[n], each 256-B aligned.
struct StageLayout
{
	size_t off_v, off_t, off_np, off_f, total;
	explicit StageLayout(size_t n)
	{
		off_v = 0;
		off_t = align_up(off_v + n * 4, 256);
		off_np = align_up(off_t + n * 4, 256);
		off_f = align_up(off_np + n * 2, 256);
		total = align_up(off_f + n, 256);
	}
};

static int launch_frame_rgba(ort_ctx* c, const float pos[3], const float rot[9], float fov_factor,
                             int W, int H, int y0, int rows, int tile_rows, int tile_step, uint32_t* d_rgba);

// Host outputs of a frame call (rgba != nullptr: shaded pixels, else voxel / face / t [/ npush]).
//   * The rows are cut into kChunks chunks (borders on multiples of 16 rows and of tile_rows); a small first chunk gets
//     the copy engine going early.  Each chunk is its own launch, on the auxiliary streams in turn, so the latency
//     tail of one launch (a few grazing rays with hundreds of PUSHes) overlaps the bulk of the next instead of
//     adding up; chunk k's results travel to the host on copy_stream as soon as its kernel is done.
//   * Staging holds the whole frame, twice: with opt_defer_sync the next call's kernels run while this call's
//     results are still crossing PCIe (9 B per ray at ~57 GB/s is slower than the trace).
//   * ctx->stream is joined to the chunk kernels, so whatever the caller enqueues next (a delta upload) stays ordered.
static int frame_to_host(ort_ctx* c, const float pos[3], const float rot[9], float fov_factor,
                         int W, int H, int y0, int rows, int tile_rows, int tile_step,
                         uint32_t* voxel, uint8_t* face, float* t, uint16_t* npush, uint32_t* rgba)
{
	// chunk borders: a short first chunk, then growing ones (triangular weights).  Synchronous calls default to 8
	// chunks; with opt_defer_sync the copy of one frame hides behind the next frame's kernels anyway, so 2 do.
	constexpr int kMaxChunks = 8;
	int kChunks = c->opt_frame_chunks > 0 ? c->opt_frame_chunks : (c->opt_defer_sync ? 2 : 8);
	if (kChunks > kMaxChunks) kChunks = kMaxChunks;
	int gcd_ = 16, b_ = tile_rows;
	while (b_) { const int r_ = gcd_ % b_; gcd_ = b_; b_ = r_; }
	const int q = 16 / gcd_ * tile_rows;                              // lcm(16, tile_rows)
	int bounds[kMaxChunks + 1] = { 0 };
	bounds[kChunks] = rows;
	const int wsum = kChunks * (kChunks + 1) / 2;
	for (int k = 0, acc = 0; k < kChunks - 1; ++k)
	{
		acc += k + 1;
		const int r = static_cast<int>(static_cast<long long>(rows) * acc / wsum) / q * q;
		bounds[k + 1] = r < bounds[k] ? bounds[k] : r;
	}

	const size_t n_all = static_cast<size_t>(rows) * W;
	const StageLayout L(n_all);
	const size_t slot_bytes = rgba ? align_up(n_all * 4, 256) : L.total;
	int rc = ensure_dstage(c, 2 * slot_bytes);
	if (rc != ORT_OK) return rc;
	const int slot = c->next_slot;
	c->next_slot ^= 1;
	char* sb = stage_slot(c, slot);

	cudaStream_t user = c->stream;
	ORT_CUDA(c, cudaEventRecord(c->ev_fork, user));
	for (int i = 0; i < 3; ++i)
	{
		ORT_CUDA(c, cudaStreamWaitEvent(c->aux_stream[i], c->ev_fork, 0));
		if (c->slot_used[slot])
			ORT_CUDA(c, cudaStreamWaitEvent(c->aux_stream[i], c->ev_copied[slot], 0));   // the slot's previous frame has left
	}
	const int n_streams = 3;
	int launched = 0;
	++c->frame_call_seq;                      // the chunks below are one frame call
	struct Nested { ort_ctx* c; explicit Nested(ort_ctx* c_) : c(c_) { c->frame_call_nested = true; } ~Nested() { c->frame_call_nested = false; } } nested(c);
	for (int k = 0; k < kChunks; ++k)
	{
		const int r0 = bounds[k], nr = bounds[k + 1] - bounds[k];
		if (nr <= 0) continue;
		const size_t n = static_cast<size_t>(nr) * W, first = static_cast<size_t>(r0) * W;
		// rows r0.. of this call: same mapping with the chunk's first frame row as origin (r0 is a multiple of tile_rows)
		const int cy0 = y0 + (r0 / tile_rows) * tile_rows * tile_step;
		cudaStream_t ks = c->aux_stream[launched % n_streams];
		++launched;
		c->stream = ks;
		if (rgba)
			rc = launch_frame_rgba(c, pos, rot, fov_factor, W, H, cy0, nr, tile_rows, tile_step, reinterpret_cast<uint32_t*>(sb) + first);
		else
			rc = ort_trace_frame_async(c, pos, rot, fov_factor, W, H, cy0, nr, tile_rows, tile_step,
			                           reinterpret_cast<uint32_t*>(sb + L.off_v) + first, reinterpret_cast<uint8_t*>(sb + L.off_f) + first,
			                           reinterpret_cast<float*>(sb + L.off_t) + first, npush ? reinterpret_cast<uint16_t*>(sb + L.off_np) + first : nullptr);
		c->stream = user;
		if (rc != ORT_OK) return rc;
		ORT_CUDA(c, cudaEventRecord(c->ev_part[k], ks));
		ORT_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->ev_part[k], 0));
		if (rgba)
			ORT_CUDA(c, cudaMemcpyAsync(rgba + first, reinterpret_cast<uint32_t*>(sb) + first, n * 4, cudaMemcpyDeviceToHost, c->copy_stream));
		else
		{
			ORT_CUDA(c, cudaMemcpyAsync(voxel + first, reinterpret_cast<uint32_t*>(sb + L.off_v) + first, n * 4, cudaMemcpyDeviceToHost, c->copy_stream));
			ORT_CUDA(c, cudaMemcpyAsync(t + first, reinterpret_cast<float*>(sb + L.off_t) + first, n * 4, cudaMemcpyDeviceToHost, c->copy_stream));
			ORT_CUDA(c, cudaMemcpyAsync(face + first, reinterpret_cast<uint8_t*>(sb + L.off_f) + first, n, cudaMemcpyDeviceToHost, c->copy_stream));
			if (npush) ORT_CUDA(c, cudaMemcpyAsync(npush + first, reinterpret_cast<uint16_t*>(sb + L.off_np) + first, n * 2, cudaMemcpyDeviceToHost, c->copy_stream));
		}
	}
	ORT_CUDA(c, cudaEventRecord(c->ev_copied[slot], c->copy_stream));
	ORT_CUDA(c, cudaEventRecord(c->ev_chunk[slot], c->copy_stream));      // (slot protocol of ort_trace_rays: "kernel done" is implied)
	c->slot_used[slot] = true;
	for (int i = 0; i < 3 && i < launched; ++i)
	{
		ORT_CUDA(c, cudaEventRecord(c->ev_aux[i], c->aux_stream[i]));
		ORT_CUDA(c, cudaStreamWaitEvent(user, c->ev_aux[i], 0));
	}
	return finish_host_call(c);
}

int ort_trace_rays(ort_ctx* c, const float* o3, int o_stride, const float* d3, size_t n,
                   uint32_t* voxel, uint8_t* face, float* t, uint16_t* npush)
{
	enter(c);
	if (!c) return ort_fail(c, ORT_ERR_INVALID, "ort_trace_rays: null context");
	if (!n) return ORT_OK;
	if (!o3 || !d3 || !voxel || !face || !t || (o_stride != 0 && o_stride != 3))
		return ort_fail(c, ORT_ERR_INVALID, "ort_trace_rays: bad arguments");
	DeviceGuard g(c->device);

	const bool in_dev = is_device_ptr(d3), out_dev = is_device_ptr(voxel);
	if (in_dev && out_dev)
	{
		int rc = ort_trace_rays_async(c, o3, o_stride, d3, n, voxel, face, t, npush);
		if (rc != ORT_OK) return rc;
		ORT_CUDA(c, cudaStreamSynchronize(c->stream));
		return ORT_OK;
	}

	// Host buffers: the rays are cut into chunks of opt_rays_chunk; chunk k+1's rays go H2D (h2d_stream) while
	// chunk k is traced (stream) and chunk k-1's results go D2H (copy_stream) -- PCIe is full duplex, so the call
	// costs about max(24 B/ray up, 9 B/ray down, kernel) instead of their sum.  Two staging slots.
	const size_t chunk = static_cast<size_t>(c->opt_rays_chunk > 4096 ? c->opt_rays_chunk : 4096);
	const size_t cn = n < chunk ? n : chunk;
	const StageLayout L(cn);
	const size_t off_d = L.total, off_o = align_up(off_d + cn * 12, 256);
	const size_t slot_bytes = align_up(off_o + (o_stride ? cn * 12 : 12), 256);
	int rc = ensure_dstage(c, 2 * slot_bytes);
	if (rc != ORT_OK) return rc;

	for (size_t first = 0; first < n; first += cn)
	{
		const size_t m = n - first < cn ? n - first : cn;
		const int slot = c->next_slot;
		c->next_slot ^= 1;
		char* base = stage_slot(c, slot);
		const float* dd = d3 + first * 3;
		const float* dorg = o_stride ? o3 + first * 3 : o3;
		if (!in_dev)
		{
			if (c->slot_used[slot])
			{
				ORT_CUDA(c, cudaStreamWaitEvent(c->h2d_stream, c->ev_chunk[slot], 0));    // the slot's previous kernel has read its rays
				ORT_CUDA(c, cudaStreamWaitEvent(c->h2d_stream, c->ev_copied[slot], 0));   // (and its results have left)
			}
			ORT_CUDA(c, cudaMemcpyAsync(base + off_d, dd, m * 12, cudaMemcpyHostToDevice, c->h2d_stream));
			ORT_CUDA(c, cudaMemcpyAsync(base + off_o, dorg, o_stride ? m * 12 : 12, cudaMemcpyHostToDevice, c->h2d_stream));
			ORT_CUDA(c, cudaEventRecord(c->ev_in[slot], c->h2d_stream));
			ORT_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_in[slot], 0));
			dd = reinterpret_cast<const float*>(base + off_d);
			dorg = reinterpret_cast<const float*>(base + off_o);
		}
		if (!out_dev && c->slot_used[slot])
			ORT_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_copied[slot], 0));
		uint32_t* dv = out_dev ? voxel + first : reinterpret_cast<uint32_t*>(base + L.off_v);
		float*    dt = out_dev ? t + first : reinterpret_cast<float*>(base + L.off_t);
		uint8_t*  df = out_dev ? face + first : reinterpret_cast<uint8_t*>(base + L.off_f);
		uint16_t* dn = !npush ? nullptr : (out_dev ? npush + first : reinterpret_cast<uint16_t*>(base + L.off_np));

		rc = ort_trace_rays_async(c, dorg, o_stride, dd, m, dv, df, dt, dn);
		if (rc != ORT_OK) return rc;
		ORT_CUDA(c, cudaEventRecord(c->ev_chunk[slot], c->stream));
		if (!out_dev)
		{
			ORT_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->ev_chunk[slot], 0));
			ORT_CUDA(c, cudaMemcpyAsync(voxel + first, dv, m * 4, cudaMemcpyDeviceToHost, c->copy_stream));
			ORT_CUDA(c, cudaMemcpyAsync(t + first, dt, m * 4, cudaMemcpyDeviceToHost, c->copy_stream));
			ORT_CUDA(c, cudaMemcpyAsync(face + first, df, m, cudaMemcpyDeviceToHost, c->copy_stream));
			if (npush) ORT_CUDA(c, cudaMemcpyAsync(npush + first, dn, m * 2, cudaMemcpyDeviceToHost, c->copy_stream));
		}
		ORT_CUDA(c, cudaEventRecord(c->ev_copied[slot], c->copy_stream));
		c->slot_used[slot] = true;
	}
	return finish_host_call(c);
}

int ort_trace_frame(ort_ctx* c, const float pos[3], const float rot[9], float fov_factor,
                    int W, int H, int y0, int rows, int tile_rows, int tile_step,
                    uint32_t* voxel, uint8_t* face, float* t, uint16_t* npush)
{
	enter(c);
	if (!c) return ort_fail(c, ORT_ERR_INVALID, "ort_trace_frame: null context");
	if (rows == 0) return ORT_OK;
	if (!voxel || !face || !t || !frame_args_ok(pos, rot, W, H, y0, rows, tile_rows, tile_step))
		return ort_fail(c, ORT_ERR_INVALID, "ort_trace_frame: bad arguments");
	DeviceGuard g(c->device);

	if (is_device_ptr(voxel))
	{
		int rc = ort_trace_frame_async(c, pos, rot, fov_factor, W, H, y0, rows, tile_rows, tile_step, voxel, face, t, npush);
		if (rc != ORT_OK) return rc;
		ORT_CUDA(c, cudaStreamSynchronize(c->stream));
		return ORT_OK;
	}

	if (c->opt_zero_copy)
	{
		// pinned outputs: the kernel's stores go over PCIe as they are produced -- no staging, no copy engine
		uint32_t* zv = static_cast<uint32_t*>(mapped_host_alias(voxel));
		uint8_t*  zf = static_cast<uint8_t*>(mapped_host_alias(face));
		float*    zt = static_cast<float*>(mapped_host_alias(t));
		uint16_t* zn = npush ? static_cast<uint16_t*>(mapped_host_alias(npush)) : nullptr;
		if (zv && zf && zt && (!npush || zn))
		{
			int rc = ort_trace_frame_async(c, pos, rot, fov_factor, W, H, y0, rows, tile_rows, tile_step, zv, zf, zt, zn);
			if (rc != ORT_OK) return rc;
			ORT_CUDA(c, cudaStreamSynchronize(c->stream));
			return ORT_OK;
		}
	}

	return frame_to_host(c, pos, rot, fov_factor, W, H, y0, rows, tile_rows, tile_step, voxel, face, t, npush, nullptr);
}

int ort_set_palette(ort_ctx* c, const uint32_t* rgba6, uint32_t n_voxels, uint32_t exit_rgba, uint32_t inside_rgba)
{
	enter(c);
	if (!c || (n_voxels && !rgba6))
		return ort_fail(c, ORT_ERR_INVALID, "ort_set_palette: bad arguments");
	DeviceGuard g(c->device);
	ORT_CUDA(c, cudaStreamSynchronize(c->stream));
	cudaFree(c->d_palette);
	c->d_palette = nullptr;
	c->n_palette = 0;
	if (n_voxels)
	{
		ORT_CUDA(c, cudaMalloc(&c->d_palette, static_cast<size_t>(n_voxels) * 24));
		ORT_CUDA(c, cudaMemcpy(c->d_palette, rgba6, static_cast<size_t>(n_voxels) * 24, cudaMemcpyDefault));
		c->n_palette = n_voxels;
	}
	c->exit_rgba = exit_rgba;
	c->inside_rgba = inside_rgba;
	return ORT_OK;
}

static int launch_frame_rgba(ort_ctx* c, const float pos[3], const float rot[9], float fov_factor,
                             int W, int H, int y0, int rows, int tile_rows, int tile_step, uint32_t* d_rgba)
{
	const ort::Palette pal{ c->d_palette, c->n_palette, c->exit_rgba, c->inside_rgba };
	const dim3 grid((W + 15) / 16, (rows + 15) / 16);
	if (!c->has_root)
	{
		// empty tree: every pixel is sky (update_image's first branch, test_och_h_octree.cpp:443-446)
		const size_t n = static_cast<size_t>(rows) * W;
		ort::fill_u32_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->stream>>>(d_rgba, c->exit_rgba, n);
		++c->launches;
		ORT_CUDA(c, cudaGetLastError());
		return ORT_OK;
	}
	const ort::Dag dag = make_dag(c);
	const ort::Camera cam = make_camera(c, pos, rot, fov_factor, W, H);
	const int rotate = c->opt_band_rotate >= 0 ? c->opt_band_rotate % ((rows + 15) / 16) : horizon_band(cam, W, y0, rows, tile_rows, tile_step);
	const ort::FrameRows fr{ W, H, y0, rows, tile_rows, tile_step, 0, rotate, ort::tile_shift_of(tile_rows) };
	const int bk = beam_level_for_launch(c, cam, fr, false);
	if (bk)
	{
		const int rc = beam_launch_march(c, bk, cam, fr, reinterpret_cast<float*>(d_rgba), false);
		if (rc != ORT_OK) return rc;
	}
	switch (walk_variant(c))
	{
	case 0:  ort::trace_frame_rgba_kernel<0><<<grid, 256, 0, c->stream>>>(dag, cam, fr, pal, d_rgba); break;
	case 1:  ort::trace_frame_rgba_kernel<1><<<grid, 256, 0, c->stream>>>(dag, cam, fr, pal, d_rgba); break;
	default:
		if (bk) ort::trace_frame_rgba_kernel<ort::kLean, true><<<grid, 256, ort::lean_smem_bytes(c->depth), c->stream>>>(dag, cam, fr, pal, d_rgba);
		else    ort::trace_frame_rgba_kernel<ort::kLean, false><<<grid, 256, ort::lean_smem_bytes(c->depth), c->stream>>>(dag, cam, fr, pal, d_rgba);
		break;
	}
	++c->launches;
	ORT_CUDA(c, cudaGetLastError());
	return ORT_OK;
}

int ort_trace_frame_rgba(ort_ctx* c, const float pos[3], const float rot[9], float fov_factor,
                         int W, int H, int y0, int rows, int tile_rows, int tile_step, uint32_t* rgba)
{
	enter(c);
	if (!c || !pos || !rot || !rgba || W <= 0 || H <= 0 || rows < 0 || tile_rows <= 0 || tile_step <= 0 || y0 < 0)
		return ort_fail(c, ORT_ERR_INVALID, "ort_trace_frame_rgba: bad arguments");
	if (!rows) return ORT_OK;
	DeviceGuard g(c->device);
	if (is_device_ptr(rgba))
	{
		++c->frame_call_seq;
		return launch_frame_rgba(c, pos, rot, fov_factor, W, H, y0, rows, tile_rows, tile_step, rgba);   // enqueue only
	}

	if (c->opt_zero_copy)
		if (uint32_t* z = static_cast<uint32_t*>(mapped_host_alias(rgba)))
		{
			++c->frame_call_seq;
			int rc = launch_frame_rgba(c, pos, rot, fov_factor, W, H, y0, rows, tile_rows, tile_step, z);
			if (rc != ORT_OK) return rc;
			ORT_CUDA(c, cudaStreamSynchronize(c->stream));
			return ORT_OK;
		}

	return frame_to_host(c, pos, rot, fov_factor, W, H, y0, rows, tile_rows, tile_step, nullptr, nullptr, nullptr, nullptr, rgba);
}

int ort_fixture_heightmap_gpu(ort_ctx* c, int depth, uint16_t* heights)
{
	enter(c);
	if (!c || !heights || depth < 1 || depth > 15)
		return ort_fail(c, ORT_ERR_INVALID, "ort_fixture_heightmap_gpu: bad arguments");
	DeviceGuard g(c->device);
	const int dim = 1 << depth;
	const size_t bytes = static_cast<size_t>(dim) * dim * 2;
	const bool dev_out = is_device_ptr(heights);
	uint16_t* d = heights;
	if (!dev_out)
	{
		int rc = ensure_dstage(c, bytes);
		if (rc != ORT_OK) return rc;
		ORT_CUDA(c, cudaStreamSynchronize(c->copy_stream));      // the staging buffer may still be draining (opt_defer_sync)
		d = static_cast<uint16_t*>(c->d_stage);
	}
	const dim3 grid((dim + 255) / 256, dim);
	ort::fixture_heightmap_kernel<<<grid, 256, 0, c->stream>>>(d, dim);
	++c->launches;
	ORT_CUDA(c, cudaGetLastError());
	if (!dev_out)
		ORT_CUDA(c, cudaMemcpyAsync(heights, d, bytes, cudaMemcpyDeviceToHost, c->stream));
	ORT_CUDA(c, cudaStreamSynchronize(c->stream));
	return ORT_OK;
}

int ort_fixture_carve_gpu(ort_ctx* c, int depth, const uint16_t* heights, int zmax, uint64_t* carved)
{
	enter(c);
	if (!c || !heights || !carved || depth < 5 || depth > 15 || zmax < 0 || zmax >= (1 << depth))
		return ort_fail(c, ORT_ERR_INVALID, "ort_fixture_carve_gpu: bad arguments (depth must be 5..15)");
	DeviceGuard g(c->device);
	const int dim = 1 << depth;
	const size_t words64_per_slab = (static_cast<size_t>(dim) * dim + 63) / 64;
	const size_t h_bytes = static_cast<size_t>(dim) * dim * 2;
	const size_t out_bytes = words64_per_slab * 8 * (static_cast<size_t>(zmax) + 1);
	const bool dev_h = is_device_ptr(heights), dev_out = is_device_ptr(carved);

	uint16_t* d_h = nullptr;
	uint32_t* d_bits = nullptr;
	if (!dev_h)
	{
		ORT_CUDA(c, cudaMalloc(&d_h, h_bytes));
		ORT_CUDA(c, cudaMemcpyAsync(d_h, heights, h_bytes, cudaMemcpyHostToDevice, c->stream));
	}
	if (!dev_out)
	{
		const cudaError_t e = cudaMalloc(&d_bits, out_bytes);
		if (e != cudaSuccess) { cudaFree(d_h); return ort_fail(c, ORT_ERR_CUDA, "ort_fixture_carve_gpu: %zu bytes for the carve bitmap: %s", out_bytes, cudaGetErrorString(e)); }
	}
	uint32_t* bits = dev_out ? reinterpret_cast<uint32_t*>(carved) : d_bits;
	// z goes into gridDim.z (<= 65535) in slices
	for (int z0 = 0; z0 <= zmax; z0 += 32768)
	{
		const int nz = zmax + 1 - z0 < 32768 ? zmax + 1 - z0 : 32768;
		const dim3 grid((dim + 255) / 256, dim, nz);
		ort::fixture_carve_kernel<<<grid, 256, 0, c->stream>>>(dev_h ? heights : d_h, dim, bits + static_cast<size_t>(z0) * words64_per_slab * 2, words64_per_slab * 2);
		++c->launches;
	}
	cudaError_t e = cudaGetLastError();
	if (e == cudaSuccess && !dev_out) e = cudaMemcpyAsync(carved, d_bits, out_bytes, cudaMemcpyDeviceToHost, c->stream);
	if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
	cudaFree(d_h);
	cudaFree(d_bits);
	if (e != cudaSuccess)
		return ort_fail(c, ORT_ERR_CUDA, "ort_fixture_carve_gpu: %s", cudaGetErrorString(e));
	return ORT_OK;
}

int ort_sync(ort_ctx* c)
{
	enter(c);
	if (!c) return ort_fail(c, ORT_ERR_INVALID, "ort_sync: null context");
	DeviceGuard g(c->device);
	ORT_CUDA(c, cudaStreamSynchronize(c->h2d_stream));
	ORT_CUDA(c, cudaStreamSynchronize(c->stream));
	ORT_CUDA(c, cudaStreamSynchronize(c->copy_stream));
	return ORT_OK;
}

void*    ort_stream(ort_ctx* c) { return c ? c->stream : nullptr; }

int ort_set_stream(ort_ctx* c, void* stream)
{
	if (!c) return ort_fail(c, ORT_ERR_INVALID, "ort_set_stream: null context");
	c->stream = stream ? static_cast<cudaStream_t>(stream) : c->own_stream;
	return ORT_OK;
}
int      ort_device(const ort_ctx* c) { return c ? c->device : -1; }
uint32_t ort_node_count(const ort_ctx* c) { return c ? c->n_nodes : 0; }
uint32_t ort_root(const ort_ctx* c) { return c ? c->root : 0; }
uint64_t ort_launch_count(const ort_ctx* c) { return c ? c->launches : 0; }

int ort_set_option(ort_ctx* c, const char* key, int value)
{
	enter(c);
	if (!c || !key) return ort_fail(c, ORT_ERR_INVALID, "ort_set_option: bad arguments");
	if (!std::strcmp(key, "variant")) c->opt_variant = value;
	else if (!std::strcmp(key, "smem_levels")) c->opt_smem_levels = value;
	else if (!std::strcmp(key, "block")) c->opt_block = value;
	else if (!std::strcmp(key, "low_water")) c->opt_low_water = value;
	else if (!std::strcmp(key, "tile_shape")) c->opt_tile_shape = value;
	else if (!std::strcmp(key, "zero_copy")) c->opt_zero_copy = value;
	else if (!std::strcmp(key, "band_rotate")) c->opt_band_rotate = value;
	else if (!std::strcmp(key, "persist_blocks")) c->opt_persist_blocks = value;
	else if (!std::strcmp(key, "l1_carveout"))
	{
		// measurement: shared-memory carve-out (percent) of the default frame kernels; they use no shared memory, so 0
		// asks for the largest L1
		DeviceGuard g(c->device);
		ORT_CUDA(c, cudaFuncSetAttribute(ort::trace_frame_kernel<1, false>, cudaFuncAttributePreferredSharedMemoryCarveout, value));
		ORT_CUDA(c, cudaFuncSetAttribute(ort::trace_frame_kernel<ort::kLean, false>, cudaFuncAttributePreferredSharedMemoryCarveout, value));
	}
	else if (!std::strcmp(key, "band_order")) c->opt_band_order = value;
	else if (!std::strcmp(key, "beam")) c->opt_beam = value;
	else if (!std::strcmp(key, "beam_level")) c->opt_beam_level = value;
	else if (!std::strcmp(key, "count_beam")) c->opt_count_beam = value;
	else if (!std::strcmp(key, "beam_after")) c->opt_beam_after = value;
	else if (!std::strcmp(key, "defer_sync")) c->opt_defer_sync = value;
	else if (!std::strcmp(key, "frame_chunks")) c->opt_frame_chunks = value;
	else if (!std::strcmp(key, "rays_chunk")) c->opt_rays_chunk = value;
	else if (!std::strcmp(key, "rays_variant")) c->opt_rays_variant = value;
	else return ort_fail(c, ORT_ERR_INVALID, "ort_set_option: unknown key '%s'", key);
	return ORT_OK;
}

int ort_beam_level(ort_ctx* c, const float pos[3], const float rot[9], float fov_factor, int W, int H)
{
	enter(c);
	if (!c || !pos || !rot || W <= 0 || H <= 0) return 0;
	const ort::Camera cam = make_camera(c, pos, rot, fov_factor, W, H);
	const ort::FrameRows fr{ W, H, 0, H, 1, 1, c->opt_tile_shape, 0, 0 };
	return beam_level(c, cam, fr, false);
}

int ort_beam_grid(ort_ctx* c, int level, uint8_t* skip_out)
{
	enter(c);
	if (!c || !skip_out || level < 1 || level > ort::kBeamFineLevel || level > c->depth)
		return ort_fail(c, ORT_ERR_INVALID, "ort_beam_grid: level must be 1..min(depth, %d)", ort::kBeamFineLevel);
	if (!c->has_root)
		return ort_fail(c, ORT_ERR_INVALID, "ort_beam_grid: no DAG on the device");
	DeviceGuard g(c->device);
	const int rc = beam_ensure_grid(c, level);
	if (rc != ORT_OK) return rc;
	ORT_CUDA(c, cudaMemcpyAsync(skip_out, c->d_beam_skip[level][c->beam_gen[level]], static_cast<size_t>(1) << (3 * level), cudaMemcpyDeviceToHost, c->stream));
	ORT_CUDA(c, cudaStreamSynchronize(c->stream));
	return ORT_OK;
}

uint64_t ort_beam_builds(const ort_ctx* c) { return c ? c->beam_builds : 0; }
uint64_t ort_band_schedules(const ort_ctx* c) { return c ? c->band_schedules : 0; }

int ort_measure_gather_peak(ort_ctx* c, size_t bytes, double* gb_per_s)
{
	enter(c);
	if (!c || !gb_per_s || bytes < (1u << 20))
		return ort_fail(c, ORT_ERR_INVALID, "ort_measure_gather_peak: need a context, an output and >= 1 MiB");
	DeviceGuard g(c->device);
	uint32_t* buf = nullptr;
	ORT_CUDA(c, cudaMalloc(&buf, bytes + 4));
	ORT_CUDA(c, cudaMemsetAsync(buf, 0x5A, bytes + 4, c->stream));
	const uint32_t n_sectors = static_cast<uint32_t>(bytes / 32);
	const uint32_t blocks = static_cast<uint32_t>(c->sm_count) * 8u, iters = 256;
	cudaEvent_t a, b;
	ORT_CUDA(c, cudaEventCreate(&a));
	ORT_CUDA(c, cudaEventCreate(&b));
	float best = 1e30f;
	for (int rep = 0; rep < 6; ++rep)                                         // rep 0 warms L2
	{
		ORT_CUDA(c, cudaEventRecord(a, c->stream));
		ort::gather_peak_kernel<<<blocks, 256, 0, c->stream>>>(buf, n_sectors, iters, buf + bytes / 4);
		++c->launches;
		ORT_CUDA(c, cudaEventRecord(b, c->stream));
		ORT_CUDA(c, cudaEventSynchronize(b));
		float ms = 0;
		ORT_CUDA(c, cudaEventElapsedTime(&ms, a, b));
		if (rep && ms < best) best = ms;
	}
	cudaEventDestroy(a);
	cudaEventDestroy(b);
	cudaFree(buf);
	const double loads = static_cast<double>(blocks) * 256.0 * iters * 8.0;
	*gb_per_s = loads * 32.0 / (best * 1e-3) / 1e9;
	return ORT_OK;
}

int ort_host_alloc(void** out, size_t bytes)
{
	if (!out) return ort_fail(nullptr, ORT_ERR_INVALID, "ort_host_alloc: null out");
	ORT_CUDA(nullptr, cudaHostAlloc(out, bytes, cudaHostAllocDefault));
	return ORT_OK;
}

int ort_host_free(void* p)
{
	if (p) ORT_CUDA(nullptr, cudaFreeHost(p));
	return ORT_OK;
}

void ort_camera_coeffs(float yaw, float pitch, float rot[9], float* fov_factor)
{
	// test_och_h_octree.cpp:95-115; roll (a) is fixed at 0 there, so sin_a = 0 and cos_a = 1
	const float fov = 1.25F;
	if (fov_factor) *fov_factor = 1 / tanf(fov / 2);
	const float sa = 0, ca = 1;
	const float sb = sinf(yaw), cb = cosf(yaw);
	const float sc = sinf(pitch), cc = cosf(pitch);
	rot[0] = ca * cb;
	rot[1] = ca * sb * sc - sa * cc;
	rot[2] = ca * sb * cc + sa * sc;
	rot[3] = sa * cb;
	rot[4] = sa * sb * sc + ca * cc;
	rot[5] = sa * sb * cc - ca * sc;
	rot[6] = -sb;
	rot[7] = cb * sc;
	rot[8] = cb * cc;
}

}  // extern "C"

#include "ort_mg.cuh"
