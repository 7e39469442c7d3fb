/* ort_b200.h -- C ABI of the B200-native h_octree trace path (libort_b200.so).
 *
 * Drop-in boundary for the ONE hot path of AlexanderRipar/Octree_Ray_Tracing: the adapted
 * Laine-Karras traversal behind och::h_octree<L,D>::sse_trace and the node store it reads.
 * The reference has no FFI of its own; its boundary is the C++ member API of och::h_octree
 * (och_h_octree.h:17-452) plus the call sites in test_och_h_octree.cpp.  Every entry point
 * below names the reference interface it replaces (paths relative to
 * /root/reference/Octree_Ray_Tracing/).  include/och_h_octree_b200.hpp rebuilds the
 * reference's C++ class on top of this ABI; INTEGRATION.md shows the binding.
 *
 * Conventions: opaque handles, plain pointers and sizes, int error codes (0 = ORT_OK), no
 * exceptions cross the boundary, no CPU fallback -- every trace entry point fails with
 * ORT_ERR_CUDA / ORT_ERR_NO_DEVICE when no sm_100 device is usable.  A handle is driven by one
 * host thread at a time; different handles may be driven concurrently.
 */
#ifndef ORT_B200_H
#define ORT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ort_ctx  ort_ctx;   /* device side: node mirror + streams of ONE GPU                */
typedef struct ort_tree ort_tree;  /* host side:   the reference's node_hashtable, re-implemented  */
typedef struct ort_octree ort_octree; /* host side: och::octree's node pool, re-implemented          */

enum
{
	ORT_OK = 0,
	ORT_ERR_INVALID = 1,     /* bad argument                                                      */
	ORT_ERR_CUDA = 2,        /* a CUDA call failed; see ort_last_error()                          */
	ORT_ERR_NO_DEVICE = 3,   /* no CUDA device / not an sm_100 part                               */
	ORT_ERR_TABLE_FULL = 4,  /* host table above 93.75 % fill (reference: printf + exit(0), och_h_octree.h:112-116) */
	ORT_ERR_CAPACITY = 5,    /* device mirror too small for this upload                           */
	ORT_ERR_NOT_ATTACHED = 6 /* tree operation needs a device context                             */
};

/* face codes = och::direction (och_tree_helper.h:7-18) */
enum
{
	ORT_FACE_X_POS = 0, ORT_FACE_Y_POS = 1, ORT_FACE_Z_POS = 2,
	ORT_FACE_X_NEG = 3, ORT_FACE_Y_NEG = 4, ORT_FACE_Z_NEG = 5,
	ORT_FACE_EXIT = 6, ORT_FACE_INSIDE = 7, ORT_FACE_ERROR = 8
};

const char* ort_version(void);
/* message of the last failing call on this thread (ctx may be NULL) */
const char* ort_last_error(const ort_ctx* ctx);

/* ================================================================================================
 * Device context
 * ============================================================================================== */

/* Replaces: construction of the table the tracer reads (och_h_octree.h:93).  Allocates the
 * device node mirror (node_capacity nodes of 32 B, 16-B aligned halves) on `device` and loads
 * the built-in reciprocal table.  depth = tree depth D (1..16). */
int ort_create(ort_ctx** out, int device, int depth, uint32_t node_capacity);
int ort_destroy(ort_ctx* ctx);

/* Replaces: the CPU's RCPPS used at och_h_octree.h:316.  tab has 1<<log2n entries (log2n 1..23):
 * the RCPPS result bit patterns for 1.0 <= x < 2.0 indexed by the top log2n mantissa bits; other
 * exponents, zeros, infinities follow the rule documented at oc_rcp_table_bits (DESIGN.md §rcp).
 * The built-in default is the 2048-entry table of Intel's RCPPS (csrc/ort_rcp_table.h). */
int ort_set_rcp_table(ort_ctx* ctx, const uint32_t* tab, int log2n);
/* Derive that table from the CPU this process runs on (x86 RCPSS), for hosts whose reciprocal differs from the
 * built-in Intel table: fills tab[1 << log2n] and returns how many probe inputs the table model gets wrong (0 = the
 * GPU trace will equal this host's CPU trace bit for bit after ort_set_rcp_table(ctx, tab, log2n)); -1 if the build
 * has no RCPSS.  log2n = 11 suffices on Intel; try larger values until the return value is 0 elsewhere. */
long ort_host_rcp_table(uint32_t* tab, int log2n);
/* Does this host's RCPSS reproduce `tab` (probed on one input per entry, both signs)?  1 yes, 0 no, -1 no RCPSS in this
 * build.  ort_create() runs this probe against the built-in table and warns once on stderr when it fails, because the
 * GPU would then disagree with a reference running on this very host; ort_rcp_host_status() returns what it found. */
int ort_host_rcp_matches(const uint32_t* tab, int log2n);
int ort_rcp_host_status(const ort_ctx* ctx);

/* Replaces: the tracer's view of table->nodes[] / root_idx (och_h_octree.h:82, :95, :344).
 * nodes8 = n_nodes * 8 uint32 in COMPACT numbering: node id i (1-based) is row i-1; interior
 * children are compact ids, children of level-`depth` nodes are voxel payloads; 0 = empty.
 * root = compact id of the root, 0 = empty tree (every ray then misses, as the reference's
 * callers arrange: test_och_h_octree.cpp:443, :535).  Host or device pointers; a device source is
 * read on the context's own stream, so whatever produced it (an NCCL broadcast, a copy on
 * another stream) must have completed -- synchronise the producer first. */
int ort_upload_full(ort_ctx* ctx, const uint32_t* nodes8, size_t n_nodes, uint32_t root);
/* Replaces: the writes at och_h_octree.h:155 between two frames.  Scatters n nodes to compact
 * ids ids[i] (1-based) and installs the new root. */
int ort_upload_delta(ort_ctx* ctx, const uint32_t* ids, const uint32_t* nodes8, size_t n, uint32_t root);

/* Replaces: the tracer's view of och::octree::_table (och_octree.h:32, och_octree.cpp:217).  nodes8 = the pool's
 * first n_nodes rows; row 0 is the root, child values are raw row numbers, 0 = empty.  Switches the context to the
 * pool layout: the walk starts at row 0 and a MISS reports hit_time 0.0F (och_octree.cpp:302) instead of INFINITY.
 * ort_upload_delta afterwards addresses rows as id = row + 1 (its root argument is ignored in this layout). */
int ort_upload_pool(ort_ctx* ctx, const uint32_t* nodes8, size_t n_nodes);

/* Build the DAG of a dense voxel grid on ctx's GPU and install it as the device mirror, like ort_upload_full.
 * voxels: nx*ny*nz unsigned elements of elem_bytes (1 or 4), index (z*ny + y)*nx + x = voxel (x, y, z); 0 = empty, cells
 * outside the grid are empty.  Host or device pointer (a device source must be complete: synchronise its producer).
 * The mirror afterwards holds exactly what ort_tree_flatten returns for a table holding these voxels: root id 1 (0 and
 * n = 0 for an empty grid), level_offsets (optional, depth+1 entries) as ort_tree_flatten's.  ctx depth <= 11.
 * ORT_ERR_INVALID for bad arguments, ORT_ERR_CAPACITY for a DAG beyond the 2^29 - 1 compact ids, ORT_ERR_CUDA when
 * device memory runs out; after any failure the previous mirror is still installed.  A device source of 4-byte
 * elements must be 4-byte aligned. */
int ort_build_voxels(ort_ctx* ctx, const void* voxels, int elem_bytes, int nx, int ny, int nz,
                     size_t* n_nodes, uint32_t* level_offsets);
/* Write the box [x0, x0+nx) x [y0, y0+ny) x [z0, z0+nz) of voxels into the DAG on ctx's GPU and install the result as
 * the mirror.  voxels: nx*ny*nz elements of elem_bytes (1 or 4), voxel (x, y, z) of the box at index
 * ((z-z0)*ny + (y-y0))*nx + (x-x0) -- the layout ort_read_voxels writes and ort_build_voxels reads; 0 erases.  Every
 * voxel outside the box keeps the value ort_voxels_at returned before the call.  The mirror afterwards holds exactly
 * what ort_tree_flatten returns for a table holding the resulting voxels (root id 1, or 0 and n = 0 when the scene became
 * empty; level_offsets, optional, depth+1 entries, as ort_build_voxels'), whatever form the previous mirror had: built,
 * fully uploaded, after deltas with unreachable rows, or never uploaded to.  The box does not wrap: 0 <= x0, 1 <= nx <=
 * 2048 and x0 + nx <= 2^depth on each axis; context depth 1..16.  Host (pageable or pinned) or device source; a device
 * source must be complete and, for 4-byte elements, 4-byte aligned.  ORT_ERR_INVALID for bad arguments, a box outside
 * the cube, a source on another device, a misaligned device source or a context in the och::octree pool layout;
 * ORT_ERR_CAPACITY for a result beyond the 2^29 - 1 compact ids; ORT_ERR_CUDA when device memory runs out.  After any
 * failure the previous mirror is still installed.  Returns once the new mirror is installed (as ort_build_voxels).  A
 * host table attached to ctx no longer describes the mirror afterwards. */
int ort_write_voxels(ort_ctx* ctx, int x0, int y0, int z0, const void* voxels, int elem_bytes,
                     int nx, int ny, int nz, size_t* n_nodes, uint32_t* level_offsets);
/* Patch the box [x0, x0+nx) x [y0, y0+ny) x [z0, z0+nz) of voxels into the DAG on ctx's GPU in place, at a cost that
 * grows with the box (cells it cuts x depth), not with the scene.  Same voxel contract as ort_write_voxels (layout,
 * 1- or 4-byte elements, host or device source, 0 erases, every voxel outside the box keeps what ort_voxels_at returned),
 * with at most 512 voxels per axis; bigger boxes go through ort_write_voxels or several patches.
 * Mirror contract (unlike ort_write_voxels, the result is not ort_tree_flatten's form):
 *   - rows 1 .. n_old (n_old = ort_node_count before the call) are not modified.  New rows are appended as ids
 *     n_old+1 .. n_old+*n_added (n_added optional), the root is replaced and ort_node_count grows by *n_added.
 *   - no duplicates: no appended row has the content of a row the patch index holds at the same level, and no two
 *     appended rows of one level are equal.  The patch index holds the rows reachable from the root when it was built
 *     (by the first patch after the mirror changed by any other call) plus every row appended since.  So when the
 *     reachable DAG had no duplicates, it has none afterwards: its reachable node count is ort_tree_flatten's n.
 *   - deterministic numbering: new ids are assigned level by level from the leaf level up to the root level; within a
 *     level in the raster order (x fastest, then y, then z) of the first cell of the level that the box cuts and that
 *     has each new content.  Where several index rows hold the same content, the smallest id is used.  The same
 *     patches on the same mirror give byte-identical mirrors on any GPU, so replicas stay identical without rows sent.
 *   - a content of all zeros is id 0 and no row: a scene that becomes empty has root 0, and its rows stay.
 *   Garbage rows accumulate over a long session; ort_write_voxels of any box returns the mirror to ort_tree_flatten's form.
 * Frames queued before the call (async launches, defer_sync host frames, work on a caller's stream) trace the old scene:
 * they read rows <= n_old only.  The call does not wait for the device unless the mirror must grow (reallocated as in
 * ort_upload_full) or the index is built or grown; it ends with one small readback on ort_stream(ctx).
 * ORT_ERR_INVALID for bad arguments, a box outside the cube or wider than 512, a source on another device, a misaligned
 * device source or the och::octree pool layout; ORT_ERR_CAPACITY when an appended id would pass 2^29 - 1 (rows written
 * past n_old are then simply unused); ORT_ERR_CUDA when device memory runs out.  After any failure the rows, root,
 * ort_node_count and later frames are unchanged.  ort_build_bytes is not changed.  A host table attached to ctx no
 * longer describes the mirror afterwards. */
int ort_patch_voxels(ort_ctx* ctx, int x0, int y0, int z0, const void* voxels, int elem_bytes,
                     int nx, int ny, int nz, size_t* n_added);
/* Copy n rows of the device mirror, starting at compact id first (1-based), to nodes8 (host or device). */
int ort_read_nodes(ort_ctx* ctx, uint32_t first, size_t n, uint32_t* nodes8);
/* Device bytes the last successful ort_build_voxels or ort_write_voxels allocated: its temporaries plus a new mirror if it
 * had to grow one (nothing is freed before the call ends, so this is its peak on top of what the context held). */
uint64_t ort_build_bytes(const ort_ctx* ctx);

/* Replaces: n calls of at(x, y, z) (och_h_octree.h:239-258; och::octree::at, och_octree.cpp:141-160) on the DAG
 * currently on ctx's device, in either layout (h_octree compact ids or och::octree pool rows).  xyz: n triples x, y, z;
 * out[i] = the voxel at triple i, bit for bit what at() returns on a table holding the mirrored DAG.  Coordinate rule
 * (at()'s): each coordinate is cast to uint16 and only its low `depth` bits choose the cell, so negative coordinates and
 * coordinates >= 2^depth (or >= 65536) wrap around the cube.  A context that holds no tree (never uploaded to, or an
 * h_octree mirror with root 0) reads 0 everywhere; a pool mirror is walked from row 0.  A child id past the mirror's
 * rows reads as empty: the walk never loads outside them.
 * Pointers may be host (pageable or pinned) or device memory, in any mix; device buffers must be 4-byte aligned.  With
 * both on the device the call only enqueues on ort_stream(ctx); otherwise it returns when out holds the result (host
 * buffers go through device staging in chunks of at most 64 MiB).  n == 0 does nothing.  ORT_ERR_INVALID for a null
 * context, a null buffer with n > 0 or a misaligned device buffer. */
int ort_voxels_at(ort_ctx* ctx, const int32_t* xyz, size_t n, uint32_t* out);
/* The voxels of the box [x0, x0+nx) x [y0, y0+ny) x [z0, z0+nz) of the device DAG, as uint32.
 * Index (z*ny + y)*nx + x relative to the box origin, the layout ort_build_voxels reads.  The box does not wrap: it
 * needs 0 <= x0, nx >= 1 and x0 + nx <= 2^depth on each axis, else ORT_ERR_INVALID and nothing is written.  Same
 * content rules, pointers and completion as ort_voxels_at; a host output is staged in chunks of whole output rows of at
 * most 64 MiB, so a large box never needs a device buffer of its size. */
int ort_read_voxels(ort_ctx* ctx, int x0, int y0, int z0, int nx, int ny, int nz, uint32_t* out);

/* Replaces: N calls of sse_trace(ox,oy,oz,dx,dy,dz, direction&, uint32_t&, float&) const
 * (och_h_octree.h:292-447).  o3: origins, 3 floats each, o_stride = 3, or ONE shared origin with
 * o_stride = 0.  d3: n directions.  Outputs per ray: voxel = hit_voxel, face = hit_direction,
 * t = hit_time.  All pointers may be host (pageable or pinned) or device pointers.  Host buffers
 * run as a three-stage pipeline over chunks of "rays_chunk" rays (ort_set_option): chunk k+1's
 * rays go up while chunk k is traced and chunk k-1's results come down (pin the buffers -- e.g.
 * ort_host_alloc -- for the copies to overlap).  npush (optional, may be NULL) receives each
 * ray's number of child-slot loads (PUSH evaluations), saturated to 65535. */
int ort_trace_rays(ort_ctx* ctx, const float* o3, int o_stride, const float* d3, size_t n,
                   uint32_t* voxel, uint8_t* face, float* t, uint16_t* npush);

/* Replaces: tree_camera::update_position + the update_image pixel loop
 * (test_och_h_octree.cpp:87-138, :437-457) for rows of a W x H frame: rays are generated in the
 * kernel from pos / rot[9] (t_x_fx .. t_z_fz, :107-115) / fov_factor (:97) and traced.
 * Rows: local row r (0 <= r < rows) is frame row  y0 + (r / tile_rows) * tile_rows * tile_step
 * + r % tile_rows  -- tile_step = 1 gives the contiguous strip [y0, y0+rows); tile_step = N with
 * y0 = rank * tile_rows gives rank's share of a cyclic strip partition over N GPUs.
 * Outputs are rows * W entries in local row order, pixel index = x + r * W.  npush as above.
 * Host outputs: the rows are traced in a few chunks whose kernels overlap on internal streams and
 * whose results are copied to the host as each chunk finishes; the call returns when everything
 * has arrived -- unless option "defer_sync" is set, in which case it returns once the work is
 * queued and ort_sync() completes it (a frame loop then traces frame k+1 while frame k's results
 * are still crossing PCIe; use one set of host buffers per frame in flight). */
int ort_trace_frame(ort_ctx* ctx, const float pos[3], const float rot[9], float fov_factor,
                    int W, int H, int y0, int rows, int tile_rows, int tile_step,
                    uint32_t* voxel, uint8_t* face, float* t, uint16_t* npush);

/* Enqueue-only form for device output buffers: no synchronisation, no staging; work is queued on
 * the context's stream (see ort_stream).  Same semantics otherwise. */
int ort_trace_frame_async(ort_ctx* ctx, const float pos[3], const float rot[9], float fov_factor,
                          int W, int H, int y0, int rows, int tile_rows, int tile_step,
                          uint32_t* d_voxel, uint8_t* d_face, float* d_t, uint16_t* d_npush);
int ort_trace_rays_async(ort_ctx* ctx, const float* d_o3, int o_stride, const float* d_d3, size_t n,
                         uint32_t* d_voxel, uint8_t* d_face, float* d_t, uint16_t* d_npush);

/* Several frame jobs in one launch -- strips of different frames, the views of a multi-camera rig, the frames of a
 * step.  Every launch ends with the latency tail of its longest rays; a batch exposes that tail once instead of once
 * per job (8 GPUs x 1/8-frame strips: 91 % -> 9x % of linear).  Fields as the arguments of ort_trace_frame_async;
 * outputs are device pointers, npush may be NULL.  Enqueue only, on ort_stream(ctx). */
typedef struct ort_frame_job
{
	float pos[3];
	float rot[9];
	float fov_factor;
	int   W, H, y0, rows, tile_rows, tile_step;
	uint32_t* voxel;
	uint8_t*  face;
	float*    t;
	uint16_t* npush;
} ort_frame_job;
int ort_trace_frames_async(ort_ctx* ctx, const ort_frame_job* jobs, int n_jobs);

/* Replaces: och::voxel_data::get_colours() as trace_pixel uses it (test_och_h_octree.cpp:84) plus the sky / inside
 * colours (:76-77).  rgba6 = 6 colours per voxel type in face order x+,y+,z+,x-,y-,z-, packed like olc::Pixel::n
 * (r | g<<8 | b<<16 | a<<24); voxel type v uses rgba6[6*(v-1) .. 6*(v-1)+5]. */
int ort_set_palette(ort_ctx* ctx, const uint32_t* rgba6, uint32_t n_voxels, uint32_t exit_rgba, uint32_t inside_rgba);
/* Parse the reference's voxels.txt format (och_voxel.h:8-27, och_voxel.cpp:195-305): "Name:" followed by six RRGGBB
 * colours, repeated.  Writes up to max_voxels * 6 packed colours (alpha 0xFF) and names (16 bytes each, may be
 * NULL); returns the number of voxel types found, or -1 with ort_last_error set on a malformed file. */
int ort_parse_voxels(const char* text, size_t len, uint32_t* rgba6, char* names16, int max_voxels);
/* Replaces: update_image (test_och_h_octree.cpp:437-457) including the colour lookup of trace_pixel (:64-85): one
 * uint32 pixel per ray, same row addressing as ort_trace_frame.  rgba may be a host pointer (chunked, overlapped
 * D2H, returns when the pixels are there) or a device pointer (enqueue only on ort_stream). */
int ort_trace_frame_rgba(ort_ctx* ctx, const float pos[3], const float rot[9], float fov_factor,
                         int W, int H, int y0, int rows, int tile_rows, int tile_step, uint32_t* rgba);

/* ==============================================================================================
 * Multi-GPU (SURVEY 8e): one process per GPU, the DAG replicated, a frame cut into cyclic tile strips -- rank r
 * traces tiles r, r + world, ... (tile_rows rows each) with ort_trace_frame(y0 = r * tile_rows, tile_step = world).
 * The trace needs no exchange.  NCCL (loaded at run time, libnccl.so.2) carries exactly two things: the DAG / its edit
 * deltas from the rank that owns the host table, and the finished strips to the rank that consumes the frame --
 * the multi-GPU form of update_image's single frame (test_och_h_octree.cpp:437-457).
 * ============================================================================================== */
typedef struct ort_mg ort_mg;
/* 128 bytes identifying the job: created on one rank, shipped to the others by the application (any channel). */
int ort_mg_unique_id(void* id128);
/* Collective: the communicator of ctx's GPU, rank of world.  world == 1 needs neither NCCL nor an id. */
int ort_mg_create(ort_mg** out, ort_ctx* ctx, int rank, int world, const void* id128);
int ort_mg_destroy(ort_mg* mg);
int ort_mg_rank(const ort_mg* mg);
int ort_mg_world(const ort_mg* mg);
int ort_mg_nccl_version(void);                       /* 0 when NCCL cannot be loaded */
/* rows of rank's strip of an H-row frame (the frame's last tile may be short) */
int ort_mg_strip_rows(int rank, int world, int H, int tile_rows);
/* Collective: ship one update -- a full flatten (is_full) or a delta (ids + rows), as ort_tree_take_delta yields it --
 * from rank src (host pointers, read there only) to every rank's context.  Replaces the upload half of
 * ort_tree_sync for a replicated DAG. */
int ort_mg_broadcast_update(ort_mg* mg, const uint32_t* ids, const uint32_t* nodes8, size_t n, uint32_t root, int is_full, int src);
/* Collective: trace this rank's strips of a W x H frame and gather the frame on rank dst, whose voxel / face / t are
 * device buffers of W * H entries (ignored on the other ranks).  W % 4 == 0.  Enqueue only: the trace runs on
 * ort_stream(ctx), send / receive / unpack on the communicator's own stream, strips in a ring of blocks, so the
 * traces of the next frames overlap the wire time of these.  ort_mg_sync() returns when every frame queued so far
 * is complete. */
int ort_mg_trace_frame_gather(ort_mg* mg, const float pos[3], const float rot[9], float fov_factor, int W, int H, int tile_rows, int dst,
                              uint32_t* voxel, uint8_t* face, float* t);
/* The same for a sequence of frames in one call (the cameras of a rig, the frames of a step); fields as the arguments above. */
typedef struct ort_mg_frame_job
{
	float pos[3];
	float rot[9];
	float fov_factor;
	int   W, H, tile_rows, dst;
	uint32_t* voxel;
	uint8_t*  face;
	float*    t;
} ort_mg_frame_job;
int ort_mg_trace_frames_gather(ort_mg* mg, const ort_mg_frame_job* jobs, int n_jobs);
/* Collective setting: frames per wire operation.  1 (default): the strips of every frame leave as soon as they are traced
 * (lowest latency).  n > 1: the strips of n consecutive frames leave in ONE NCCL group -- fewer, larger, all-to-all-shaped
 * exchanges that NCCL spreads over all peers and channels at once (highest throughput when many frames are in flight);
 * ort_mg_flush() sends a partial group, ort_mg_sync() flushes and waits. */
int ort_mg_set_group(ort_mg* mg, int frames);
int ort_mg_flush(ort_mg* mg);
/* Collective setting: how the strips travel.  1 (default): peer copies -- every rank maps the other ranks' receive rings
 * (CUDA IPC) and a strip block moves with one cudaMemcpyAsync on the copy engines over NVLink, no SM involved; NCCL
 * carries one 4-byte all-reduce per wire operation for the ordering.  Falls back to 0 where CUDA IPC is unavailable.
 * 0: NCCL ncclSend / ncclRecv (its copy kernels share the SMs with the trace kernels).  ort_mg_transport() returns what
 * is in use after the first frame.  The environment variable ORT_MG_TRANSPORT presets it. */
int ort_mg_set_transport(ort_mg* mg, int transport);
int ort_mg_transport(const ort_mg* mg);
/* Streams the strips are traced on in turn (1..8; default 4, 8 from five ranks on): a strip launch ends with the latency
 * tail of its longest rays, and only launches on different streams overlap that tail with the bulk of the next one. */
int ort_mg_set_trace_streams(ort_mg* mg, int n);
int ort_mg_sync(ort_mg* mg);
void* ort_mg_stream(ort_mg* mg);                     /* the cudaStream_t of the gather (for event timing) */
double ort_mg_wire_bytes(const ort_mg* mg);          /* bytes this rank has sent + received for gathers so far */
uint64_t ort_mg_wire_ops(const ort_mg* mg);          /* NCCL groups issued for gathers so far */

int   ort_sync(ort_ctx* ctx);
void* ort_stream(ort_ctx* ctx);                 /* the cudaStream_t all work of ctx is queued on */
/* Queue subsequent work of ctx on the caller's cudaStream_t (NULL: back to the context's own stream).  Lets a
 * harness keep several frames in flight (one stream each) so that the tail of one launch -- a handful of grazing
 * rays with hundreds of PUSHes -- overlaps the bulk of the next.  The caller orders uploads against traces. */
int   ort_set_stream(ort_ctx* ctx, void* stream);
int   ort_device(const ort_ctx* ctx);
uint32_t ort_node_count(const ort_ctx* ctx);    /* highest compact id in use on the device */
uint32_t ort_root(const ort_ctx* ctx);
/* number of kernels of this library launched on ctx since creation (bench.py's gpu_launches) */
uint64_t ort_launch_count(const ort_ctx* ctx);
/* Options.  Behaviour: "defer_sync" (host-buffer trace calls return once queued; ort_sync() collects),
 * "frame_chunks" (launches per host-buffer frame, 0 = automatic: 8, or 2 with defer_sync), "rays_chunk" (rays per
 * pipeline stage of host-buffer ort_trace_rays, default 2^20), "zero_copy" (kernels store straight into pinned host
 * outputs; measured slower than the copy engine, off by default), "band_rotate" (which 16-row band of a frame launch
 * is scheduled first; -1 = automatic: the first band that looks below the horizon, so the long grazing rays start
 * early and the cheap sky rows fill the end of the launch).  Kernel selection for A/B measurements: "variant"
 * (frames: 0 baseline walk, 1 fast walk = default, 2 persistent lane-refill, 3 upper levels staged in shared memory,
 * 4 deferred phases, 5 tight bookkeeping, 6 while-while), "rays_variant" (explicit rays: 1 one thread per ray,
 * 2 persistent lane-refill = default), "low_water", "smem_levels", "tile_shape", "block".
 * Beam start of camera frames (csrc/ort_beam.cuh): "beam" (1 = default: every 8 x 4 pixel tile of a frame launch starts
 * its rays at a lower bound of their hit times taken from a coarse grid of the DAG, and rays that provably leave the
 * cube unhindered end as a MISS without a round -- same outputs bit for bit, fewer PUSH rounds; 0 = every ray walks from
 * its origin like och_h_octree.h:292-447), "beam_after" (default 2: a DAG version gets its grid once it has been traced
 * that many times without one, so that a loop which edits the DAG every other frame never pays for grids it cannot use;
 * 0 = build at the first frame; where the pixels are fine enough, tiles of DAGs of depth 8 and more then refine their start
 * on a level-8 grid built with it), "beam_level" (force a coarser grid level and no refinement, measurement), "count_beam"
 * (launches that return PUSH counts normally walk from the origin so that the counts are the reference's; 1 = they
 * use the beam start of the launch's level and count the loads issued then; 2 = they refine on level 8 too, as the
 * frame launches without counts do).
 * Band schedule: "band_order" (1 = default: a frame launch of a view that has been traced before -- same camera, same
 * rows -- schedules its 16-row bands by what they cost last time, most expensive first, so that the long rays of a view
 * start early; 0 = the "band_rotate" rule only).  Outputs never depend on it. */
int ort_set_option(ort_ctx* ctx, const char* key, int value);

/* Introspection of the beam start.  ort_beam_level: the grid level (3..7) frame launches of this camera geometry would
 * use on ctx, 0 = they run without a beam start (pixels too coarse for the coarsest grid, rot not a rotation, option
 * off, ...); tiles may refine on level 8 beyond it.  ort_beam_grid: the level-`level` grid (1..8) of the DAG currently on the device, (2^level)^3 bytes to host
 * memory, index (z * N + y) * N + x: 0 = some cell among the 27 around this one holds a voxel, j > 0 = the level-j cell
 * around this one has no such cell.  Both are for tests and tools; tracing needs neither. */
int ort_beam_level(ort_ctx* ctx, const float pos[3], const float rot[9], float fov_factor, int W, int H);
int ort_beam_grid(ort_ctx* ctx, int level, uint8_t* skip_out);
/* number of beam grid builds on ctx since creation (one per DAG version and level in use; a launch's level and the level-8
 * grid of its refinement, built together, count as one) */
uint64_t ort_beam_builds(const ort_ctx* ctx);
/* number of band schedules applied on ctx since creation (option "band_order", default 1: a frame launch records what each
 * 16-row band cost, the next launches of the same view -- same camera, same rows -- schedule the most expensive bands
 * first; results do not depend on it) */
uint64_t ort_band_schedules(const ort_ctx* ctx);

/* Diagnostic for roofline reports: throughput of random 32-byte-sector gathers (independent 4-byte loads, 8 in
 * flight per thread, full occupancy) over a `bytes`-sized buffer on ctx's GPU, in GB/s of sectors moved.  With
 * bytes = the DAG's size (L2-resident) this is the memory-side ceiling of the traversal. */
int ort_measure_gather_peak(ort_ctx* ctx, size_t bytes, double* gb_per_s);

/* pinned host memory for callers that want zero staging */
int ort_host_alloc(void** out, size_t bytes);
int ort_host_free(void* p);

/* rot[9], fov_factor from yaw (dir.x) and pitch (dir.y) exactly as update_position computes
 * them on the host (test_och_h_octree.cpp:95-115). */
void ort_camera_coeffs(float yaw, float pitch, float rot[9], float* fov_factor);

/* ================================================================================================
 * Host node store -- och::h_octree<Log2_table_capacity, Depth> (och_h_octree.h:17-288)
 * ============================================================================================== */

int      ort_tree_create(ort_tree** out, int log2_table_capacity, int depth);
void     ort_tree_destroy(ort_tree* tree);
/* register_node (:110-160): returns slot+1, or 0 with the table-full flag set */
uint32_t ort_tree_register_node(ort_tree* tree, const uint32_t children[8]);
void     ort_tree_remove_node(ort_tree* tree, uint32_t idx);                               /* :162-174 */
void     ort_tree_set(ort_tree* tree, uint16_t x, uint16_t y, uint16_t z, uint32_t v);     /* :176-237 */
/* n x (x, y, z, v) uint32 quadruples applied in order */
void     ort_tree_set_many(ort_tree* tree, const uint32_t* xyzv, size_t n);
/* the T / Z edit (test_och_h_octree.cpp:408-413, :427-432): set() over the box
 * [cx-ext/2, cx+(ext+1)/2) x ... in the reference's z, y, x loop order, uint16 wrap-around included */
void     ort_tree_set_box(ort_tree* tree, uint16_t cx, uint16_t cy, uint16_t cz, int ext, uint32_t v);
/* Bulk form of the same edit: every voxel of [x0,x1) x [y0,y1) x [z0,z1) (clipped to the cube) becomes v in ONE
 * pass over the cells the box cuts.  Voxel content, live nodes, fillcnt, nodecnt, refcounts and traced images equal
 * those of the set() loop; only the slot numbers handed to NEW nodes may differ (insertion order).  ~100x faster. */
void     ort_tree_fill_box(ort_tree* tree, int x0, int y0, int z0, int x1, int y1, int z1, uint32_t v);
/* Table dump / load: the occupied slots (children, tag, reference count) plus root and counters, so that a scene
 * built once (depth 14: seconds to minutes) restarts instantly and keeps accepting edits.  The loading tree must
 * have the dump's log2_table_capacity and depth.  (No counterpart in the reference; SURVEY 8f.3.) */
int      ort_tree_save(const ort_tree* tree, const char* path);
int      ort_tree_load(ort_tree* tree, const char* path);
uint32_t ort_tree_at(const ort_tree* tree, int x, int y, int z);                           /* :239-258 */
void     ort_tree_set_root(ort_tree* tree, uint32_t idx);                                  /* :260-263 */
uint32_t ort_tree_get_root(const ort_tree* tree);                                          /* :265-268 */
uint32_t ort_tree_get_fillcnt(const ort_tree* tree);                                       /* :270-273 */
uint32_t ort_tree_get_nodecnt(const ort_tree* tree);                                       /* :275-278 */
uint32_t ort_tree_get_max_refcnt(const ort_tree* tree);                                    /* :280-283 */
void     ort_tree_clear(ort_tree* tree);                                                   /* :285-288 */
int      ort_tree_table_full(const ort_tree* tree);
int      ort_tree_depth(const ort_tree* tree);
int      ort_tree_log2_capacity(const ort_tree* tree);
/* raw views of the table (cap*8 uint32, cap bytes, cap uint32) for inspection / parity tests */
const uint32_t* ort_tree_nodes(const ort_tree* tree);
const uint8_t*  ort_tree_cashes(const ort_tree* tree);
const uint32_t* ort_tree_refcounts(const ort_tree* tree);

/* Flatten the live DAG into compact, level-ordered numbering (root = id 1, then level 2, ...).
 * Returns the node count; *nodes8 (n*8 uint32) stays owned by the tree and is valid until the
 * next flatten/sync.  level_offsets (optional, depth+1 entries) receives the first id of each
 * level (entry depth = n+1).  Pure host code. */
size_t   ort_tree_flatten(ort_tree* tree, const uint32_t** nodes8, uint32_t* root, uint32_t* level_offsets);
/* Register a compact level-ordered DAG (as ort_tree_flatten / ort_read_nodes give it) in an EMPTY table: nodes interned
 * bottom-up, reference counts = instance counts (as the fixture builder assigns them), fillcnt / nodecnt accordingly;
 * the next ort_tree_sync is a full upload.  Host pointer, or device pointer when the tree is attached to a context (the
 * copy runs on that context's stream; a tree without a context makes no CUDA call).  ORT_ERR_INVALID for a non-empty table or a
 * malformed DAG (child id out of range or at the wrong level, an all-zero reachable row); ORT_ERR_TABLE_FULL as set(). */
int      ort_tree_import(ort_tree* tree, const uint32_t* nodes8, size_t n, uint32_t root);

/* Bind a device context: subsequent ort_tree_sync() calls mirror the table into it. */
int      ort_tree_attach(ort_tree* tree, ort_ctx* ctx);
/* Bring the device mirror up to date with the host table: a full level-ordered upload the first
 * time (or when more than half of the live nodes changed), otherwise a delta holding only the
 * nodes created since the last sync.  Cheap when nothing changed. */
int      ort_tree_sync(ort_tree* tree);
/* statistics of the last ort_tree_sync: nodes uploaded, 1 if it was a full upload */
void     ort_tree_sync_stats(const ort_tree* tree, uint64_t* nodes_uploaded, int* was_full);
/* Build the pending delta WITHOUT a device (for multi-GPU broadcast and CPU tests): returns n and
 * pointers (owned by the tree) to ids[n], nodes8[n*8] and the new compact root; is_full = 1 means
 * the buffers hold a full flatten instead.  The delta is consumed (marked as applied). */
size_t   ort_tree_take_delta(ort_tree* tree, const uint32_t** ids, const uint32_t** nodes8, uint32_t* root, int* is_full);

/* ================================================================================================
 * Host node pool -- och::octree (och_octree.h:10-69, och_octree.cpp:14-165)
 * ============================================================================================== */

int      ort_octree_create(ort_octree** out, int depth, uint32_t table_capacity);              /* och_octree.cpp:14 */
void     ort_octree_destroy(ort_octree* tree);
void     ort_octree_set(ort_octree* tree, int16_t x, int16_t y, int16_t z, uint32_t vx);       /* :74-91  */
void     ort_octree_unset(ort_octree* tree, int16_t x, int16_t y, int16_t z);                  /* :93-139 */
uint32_t ort_octree_at(const ort_octree* tree, int16_t x, int16_t y, int16_t z);               /* :141-160 */
int      ort_octree_get_node_cnt(const ort_octree* tree);                                      /* :162-165 */
/* n x (x, y, z, v, kind) int32 applied in order; kind 0 = set, 1 = unset */
void     ort_octree_apply(ort_octree* tree, const int32_t* ops, size_t n);
/* 1 once alloc() ran out of pool rows (the reference prints "Too many allocations" and exits, :50-54) */
int      ort_octree_failed(const ort_octree* tree);
int      ort_octree_depth(const ort_octree* tree);
uint32_t ort_octree_table_capacity(const ort_octree* tree);
const uint32_t* ort_octree_nodes(const ort_octree* tree);                                      /* _table, cap * 8 */
int      ort_octree_attach(ort_octree* tree, ort_ctx* ctx);
/* mirror the pool into the attached context: whole used prefix the first time, then only the rows edits touched */
int      ort_octree_sync(ort_octree* tree);
void     ort_octree_sync_stats(const ort_octree* tree, uint64_t* nodes_uploaded, int* was_full);

/* ================================================================================================
 * Headless harness fixtures (replaces initialize_h_octree and friends,
 * test_och_h_octree.cpp:561-598, :651-695, :767-787)
 * ============================================================================================== */

/* heights[y*dim+x] = get_terrain_heigth(x, y) with och::simplex_n(0.5F) (:561-566) */
void ort_fixture_heightmap(int depth, uint16_t* heights, int nthreads);
/* The demo's alternative terrain noise: heights[y*dim+x] = get_terrain_heigth(x, y) with the commented line
 * `terrain_noise.Evaluate(px, py)` (test_och_h_octree.cpp:568), terrain_noise = OpenSimplexNoise(seed), seed 8789 in the
 * demo (:33); 2-D OpenSimplex as vendored by the reference (opensimplex.h:222-289, :338-386), double precision. */
void ort_fixture_heightmap_opensimplex(int depth, int64_t seed, uint16_t* heights, int nthreads);
/* OpenSimplexNoise(seed).Evaluate(x, y) for n points (xy = n pairs) -- the function the heightmap above samples */
void ort_opensimplex2(int64_t seed, const double* xy, size_t n, double* out);
/* Same voxel content as initialize_h_octree (solid stone below the heightmap, grass/dark-grass
 * top chosen by grass[y*dim+x], two dirt layers, optional simplex tunnels) but built bottom-up
 * with memoisation, so depth 12-14 take seconds.  The DAG is canonical, so it equals the
 * reference's up to slot numbering.  Returns ORT_OK or ORT_ERR_TABLE_FULL. */
int  ort_fixture_build_terrain(ort_tree* tree, const uint16_t* heights, const uint8_t* grass, int tunnels, int nthreads);
/* Same, with the tunnel bitmap supplied by the caller (NULL: computed on the host threads).  carved: one bit per
 * voxel for z <= max(heights): bit (y*dim + x) of slab z, slabs of (dim*dim + 63)/64 uint64 words; set = removed by
 * remove(tree, splatter_noise(-0.5F, .., 1/16)) (test_och_h_octree.cpp:735-743, :755-763, :786). */
int  ort_fixture_build_terrain_ex(ort_tree* tree, const uint16_t* heights, const uint8_t* grass, int tunnels, int nthreads, const uint64_t* carved);
/* The fixture's noise evaluations on the GPU (SURVEY 8f.3), bit-identical to the host versions: the heightmap
 * (get_terrain_heigth over the map, :561-566) and the tunnel bitmap in the layout above (depth 5..15; the dim^3 loop
 * of :735-743 restricted to z <= zmax).  Outputs may be host or device pointers. */
int  ort_fixture_heightmap_gpu(ort_ctx* ctx, int depth, uint16_t* heights);
int  ort_fixture_carve_gpu(ort_ctx* ctx, int depth, const uint16_t* heights, int zmax, uint64_t* carved);

#ifdef __cplusplus
}
#endif

#endif /* ORT_B200_H */
