/*
 * vx_b200.h -- C ABI of libvx_b200.so: the B200 (sm_100a) implementation of the
 * per-frame voxel pipeline of gatewaytofredom/differential_projection_voxel_renderer
 * (Rust crate `voxel_engine` 0.1.0): binary greedy meshing of 32^3 chunks, chunk
 * frustum / screen-rect culling, differential projection of the axis-aligned quad
 * vertices and the span (scanline) rasterizer with depth buffer and 8x8
 * micro-textured, per-face-lit shading.
 *
 * The reference has no FFI: its boundary is the crate's public Rust API.  Every
 * entry point below names the Rust item it stands in for (file:line relative to
 * /root/reference/); INTEGRATION.md shows the `extern "C"` block and the thin
 * `impl BinaryGreedyMesher` / `impl Rasterizer` shims a maintainer adds.
 *
 * Conventions
 *   - plain pointers + sizes, POD structs, no C++/torch types;
 *   - every call returns VX_OK (0) or a negative VX_ERR_*; there is NO CPU
 *     fallback: without a usable CUDA device the context cannot be created and
 *     every other call fails with VX_ERR_NO_DEVICE / VX_ERR_INVALID;
 *   - host pointers unless the name says `_device` / `d_`;
 *   - a VxContext owns one CUDA device + stream; calls on one context are
 *     serialised by the caller (like `&mut Rasterizer`), different contexts are
 *     independent (one per GPU / per thread);
 *   - matrices are 16 f32, column-major (glam `Mat4::to_cols_array`).
 */
#ifndef VX_B200_H
#define VX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define VX_API __attribute__((visibility("default")))
#else
#define VX_API
#endif

#define VX_CHUNK_SIZE 32
#define VX_CHUNK_VOLUME 32768

enum {
    VX_OK = 0,
    VX_ERR_INVALID = -1,   /* bad argument */
    VX_ERR_NO_DEVICE = -2, /* no CUDA device / wrong architecture */
    VX_ERR_CUDA = -3,      /* CUDA runtime error, see vx_last_error */
    VX_ERR_CAPACITY = -4,  /* an internal limit was exceeded (e.g. > 2^21 visible quads) */
    VX_ERR_OOM = -5
};

/* neighbour codes for `neighbors` (N x 6, order +X,-X,+Y,-Y,+Z,-Z = FaceDir, mesh.rs:136-143) */
#define VX_NBR_NONE (-1)          /* no chunk: border faces exposed (binary_greedy.rs:314) */
#define VX_NBR_UNIFORM_AIR (-2)   /* Uniform non-solid neighbour (binary_greedy.rs:305-313) */
#define VX_NBR_UNIFORM_SOLID (-3) /* Uniform solid neighbour */

typedef struct VxContext VxContext;
typedef struct VxMeshBatch VxMeshBatch; /* device-resident meshes of a batch of chunks */

/* `Quad` mesh.rs:245-250 (x = row, y = col/bit, width = rows, height = run length) */
typedef struct { uint8_t x, y, width, height; } VxQuad;

/* `Vertex` mesh.rs:46-58 (8 bytes) */
typedef struct { uint8_t x, y, z, block_type, light, packed; uint16_t padding; } VxVertex;

/* `MicroTexture` x4 = `TextureAtlas` texture.rs:5-13,56-79 */
typedef struct {
    uint32_t palette[4][16];
    uint8_t indices[4][32];
} VxAtlas;

/* Per-frame configuration: Rasterizer pub fields (rasterizer.rs:335-341), ShadingConfig
 * (shading.rs:9-31), framebuffer size and clear colour (main.rs:393). */
typedef struct {
    int32_t width, height;
    uint32_t clear_color;
    int32_t backface_culling;
    int32_t enable_shading;
    float light_dir[3];
    float ambient, diffuse;
    /* Rows [stripe_y0, stripe_y0 + stripe_rows) are rendered and returned (a FrameSlice,
     * framebuffer.rs:16-23).  stripe_rows == 0 means the whole frame.  Screen-space
     * mapping always uses the full `height` (PixelTarget::full_height). */
    int32_t stripe_y0, stripe_rows;
    /* 0: exact reference vertex arithmetic VP*(offset+local) (rasterizer.rs:1177-1185);
     * 1: differential projection base + x*c0 + y*c1 + z*c2 (differential_projection.rs:69). */
    int32_t differential_projection;
    /* 1: vx_render_frame_device only enqueues the frame (no host synchronisation); scratch overflow and
     * statistics are then reported by vx_frame_stats(). */
    int32_t async_submit;
    /* 1: bracket each frame kernel with CUDA events on the context's stream (cull, setup, raster); read the
     * durations with vx_frame_kernel_times().  2: additionally record the raster work-item timeline
     * (vx_frame_trace). */
    int32_t profile_kernels;
    /* 1: render_frame_macrotile semantics (macrotile_renderer.rs:51-170, macrotile.rs:179-224): no near-depth sort --
     * meshes are drawn in list order, those whose screen box covers more than 25 % of the frame (large primitives)
     * after all others -- and every 128-pixel macrotile column is its own PixelTarget, i.e. a span's interpolation
     * restarts at the column's first pixel (rasterizer.rs:1404-1432 with rect_x0 = the tile's x0).
     * profile_kernels = 2 acts like 1 in this mode. */
    int32_t macrotile;
    /* 1: the chunk-level occlusion pass of render_frame (main.rs:501-526 over OcclusionBuffer, occlusion.rs:60-153;
     * off in the reference's default run, main.rs:112): survivors front to back, a mesh at least two chunks away whose
     * every grid cell already holds a depth nearer than near_depth - 0.005 is dropped, every other one marks its
     * screen rect into the grid at its near depth.  Grid = occlusion_grid_w x occlusion_grid_h cells over the full
     * frame (128 x 72, main.rs:46-47; at most 12288 cells).  Ignored by vx_render_mesh and in macrotile mode. */
    int32_t occlusion_culling;
    int32_t occlusion_grid_w, occlusion_grid_h;
    /* Hint: frames the caller keeps in flight on this device at the same time (contexts used as lanes, see
     * vx_render_frame_begin); 0 or 1 = this frame has the GPU to itself.  It only changes how finely the raster work of a
     * frame is cut (a frame that shares the GPU with others is cut coarser: fewer, larger work items = fewer instructions
     * for the same pixels), never the result. */
    int32_t frames_in_flight;
} VxFrameConfig;

typedef struct {
    int32_t n_chunks;
    int32_t n_meshes;     /* chunks with has_mesh != 0 */
    int64_t total_quads;  /* length of the quad stream (after vx_mesh_batch_update it includes replaced, dead quads) */
} VxMeshBatchInfo;

/* Raw device pointers of a batch (for zero-copy interop, e.g. NCCL all-gather of quad
 * streams between ranks).  Valid until vx_mesh_batch_release. */
typedef struct {
    uint8_t *d_quads;          /* 3 bytes per TinyQuad (mesh.rs:273-342) */
    uint32_t *d_quad_base;     /* [N] first quad of chunk i */
    uint32_t *d_quad_count;    /* [N] */
    uint32_t *d_slice_offsets; /* [N][6][33] relative to quad_base; [f][32] = end of face f */
    int32_t *d_face_aabb;      /* [N][6][6] FaceList min.xyz,max.xyz (mesh.rs:347-397) */
    uint8_t *d_has_mesh;       /* [N] Option<ChunkMesh>::is_some */
    int32_t *d_positions;      /* [N][3] chunk coordinates */
} VxMeshBatchDevice;

typedef struct {
    int32_t n_input;          /* meshes considered */
    int32_t n_survivors;      /* after filter B */
    int32_t n_quads;          /* quads of the survivors */
    int32_t n_triangles;      /* triangles after near clip + backface cull */
    int32_t n_bin_entries;    /* (triangle, stripe) pairs */
    int32_t n_kernel_launches;
    int32_t reserved[2];
} VxFrameStats;

/* ---- context ---------------------------------------------------------- */
VX_API int vx_context_create(int device_id, VxContext **out);
VX_API void vx_context_destroy(VxContext *ctx);
VX_API const char *vx_error_string(int code);
/* last CUDA / validation message recorded on this context (empty string if none) */
VX_API const char *vx_last_error(const VxContext *ctx);
VX_API int vx_device_synchronize(VxContext *ctx);
/* CUDA stream the context launches on (cudaStream_t as void*), for event timing */
VX_API void *vx_context_stream(VxContext *ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
VX_API int64_t vx_context_launch_count(const VxContext *ctx);

/* Page-locked host memory mapped into the device address space (cudaHostAllocMapped | Portable).  Frame buffers
 * allocated here (or with cudaHostAlloc / cudaHostRegister by the caller) are written directly by the raster kernel
 * when passed to vx_render_frame: no staging copy, the PCIe writes overlap rasterization.  The Rust side backs
 * `Framebuffer::color_buffer` / `depth_buffer` (framebuffer.rs:197-245) with it. */
VX_API int vx_host_alloc(VxContext *ctx, size_t bytes, void **out);
VX_API void vx_host_free(VxContext *ctx, void *p);

/* ---- one process per GPU: peer-mapped buffers and cross-GPU hand-off flags ----------------------------------
 * The reference gives each Rayon worker a disjoint `&mut` stripe of ONE framebuffer (framebuffer.rs:392-431,
 * main.rs:581-597).  Across GPUs the composed frame lives in one GPU's memory; the other processes map it with CUDA
 * IPC and pass the mapped pointer (offset to their stripe's first row) to vx_render_frame_into, so the raster kernel's
 * write-out stores the stripe over NVLink -- no staging copy and no collective.  Per frame only a 32-bit counter per
 * rank crosses the link:
 *   vx_device_alloc / vx_device_free   zero-filled device memory with its own allocation (exportable)
 *   vx_ipc_export / vx_ipc_open / vx_ipc_close   64-byte handle of such an allocation / mapping in another process
 *   vx_signal_flags  enqueue on ctx's stream: after everything already enqueued has completed, publish `value` into
 *                    each of the n (<= 32) flag words (d_flags = HOST array of n device addresses, local or
 *                    peer-mapped), release semantics at system scope
 *   vx_wait_flags    enqueue: one warp polls n flag words of THIS GPU (`stride_words` apart) until all have reached
 *                    `value` (wrap-safe >=), or timeout_us (<= 0: 2 s) passes -- then the status is set, nothing hangs
 *   vx_wait_status   synchronises the stream; VX_ERR_CUDA + *timed_out = 1 if a wait since the last call timed out */
VX_API int vx_device_alloc(VxContext *ctx, size_t bytes, void **d_out);
VX_API int vx_device_free(VxContext *ctx, void *d_ptr);
VX_API int vx_ipc_export(VxContext *ctx, void *d_ptr, uint8_t handle_out[64]);
VX_API int vx_ipc_open(VxContext *ctx, const uint8_t handle[64], void **d_out);
VX_API int vx_ipc_close(VxContext *ctx, void *d_ptr);
VX_API int vx_signal_flags(VxContext *ctx, uint32_t *const *d_flags, int32_t n, uint32_t value);
VX_API int vx_wait_flags(VxContext *ctx, const uint32_t *d_flags, int32_t n, int32_t stride_words, uint32_t value, int32_t timeout_us);
/* vx_wait_flags followed by vx_signal_flags in ONE kernel (the composing GPU's per-frame step: every stripe has
 * arrived -> hand the buffer of an older frame back to all ranks). */
VX_API int vx_wait_then_signal(VxContext *ctx, const uint32_t *d_wait_flags, int32_t n_wait, int32_t stride_words, uint32_t wait_value,
                        uint32_t *const *d_signal_flags, int32_t n_signal, uint32_t signal_value, int32_t timeout_us);
VX_API int vx_wait_status(VxContext *ctx, int32_t *timed_out);

/* ---- terrain generation (the step before meshing) -------------------- */

/* Improved 2-D gradient noise tables + the constants of chunk.rs:173-177 (scale 0.01, amplitude 20). */
typedef struct {
    int32_t perm[512];   /* permutation table, doubled (perm[i + 256] == perm[i]), entries 0..255 */
    double grad[8][2];   /* gradient directions */
    double scale, amplitude;
} VxTerrainParams;

/* Chunk::generate_terrain (chunk.rs:114-207) for n chunk positions, on the device: d_voxels_out (device, n x 32768,
 * 16-byte aligned) receives the voxels of the Varied chunks (zeros for Uniform ones), uniform_flags_out (host, n)
 * 0 = Varied, 1 = Uniform(Air), 4 = Uniform(Stone) -- the encoding vx_mesh_chunks takes.  Feeding the result to
 * vx_mesh_chunks_device removes the 32 KiB/chunk upload of a whole-world re-mesh.  The arithmetic reproduces this
 * repo's host generator (worldgen.py) bit for bit; the reference's own noise crate is not available offline, so its
 * exact heights are not claimed (DESIGN.md 5). */
VX_API int vx_generate_terrain(VxContext *ctx, const int32_t *positions, int32_t n, const VxTerrainParams *params, uint8_t *d_voxels_out,
                        uint8_t *uniform_flags_out);

/* ---- streaming world (SURVEY 8f N2): World::update (world.rs:57-100) and the mesh cache of the frame loop
 * (main.rs:225-280) with the voxels resident on the device.  A world batch has `capacity` chunk slots; the host
 * (differential_projection_voxel_renderer_b200/world.py mirrors `World`) decides which lattice position lives in
 * which slot, the device holds voxels, Uniform flags, neighbour table and meshes.  A slot without a chunk is
 * "uniform air without neighbours": it has no mesh and is an absent neighbour (faces towards it are exposed,
 * binary_greedy.rs:127-168 with a missing map entry). ---- */
VX_API int vx_world_batch_create(VxContext *ctx, int32_t capacity, VxMeshBatch **out);
/* More slots for a world batch; everything loaded stays (voxels, flags, neighbour rows, meshes, quad stream).  The
 * reference's chunk map grows without bound while the camera moves (world.rs:84-87 returns before the unload step on
 * every frame that hits max_chunks_per_frame) and World::set_view_distance widens the sphere at run time
 * (world.rs:181-198, called from main.rs:168-176). */
VX_API int vx_world_batch_grow(VxContext *ctx, VxMeshBatch *b, int32_t new_capacity);
/* positions (n x 3, may be NULL) and neighbour rows (n x 6: slot of the chunk in direction +X,-X,+Y,-Y,+Z,-Z or
 * VX_NBR_NONE; may be NULL) of the listed slots. */
VX_API int vx_world_batch_assign(VxContext *ctx, VxMeshBatch *b, const int32_t *slots, int32_t n, const int32_t *positions,
                          const int32_t *neighbors);
/* Chunk::generate_terrain (chunk.rs:114-207, as vx_generate_terrain) for n new chunks straight into their slots:
 * voxels, Uniform flag and position.  uniform_flags_out (n bytes, may be NULL) returns 0 / 1 + block type. */
VX_API int vx_world_batch_generate(VxContext *ctx, VxMeshBatch *b, const int32_t *slots, int32_t n, const int32_t *positions,
                            const VxTerrainParams *params, uint8_t *uniform_flags_out);
/* chunks.retain(..) / mesh_cache.retain(..) (world.rs:92-97, main.rs:275): the slots become empty. */
VX_API int vx_world_batch_unload(VxContext *ctx, VxMeshBatch *b, const int32_t *slots, int32_t n);
/* mesh_chunk_in_indexed_world (binary_greedy.rs:127) for exactly the listed slots (main.rs:255-272); every other
 * mesh stays as it is, even if its neighbourhood changed since it was built -- the reference's cache is stale in
 * the same way.  Quads are appended to the stream; when it is full the live quads are compacted (copied, not
 * re-meshed). */
VX_API int vx_world_batch_remesh(VxContext *ctx, VxMeshBatch *b, const int32_t *slots, int32_t n);
/* Block edits: voxel voxel_index[i] (= z*1024 + y*32 + x inside the chunk) of slot slots[i] becomes block_types[i]
 * (0..3), for n edits in list order -- when several edits name the same voxel, the last one wins.  A Uniform slot becomes
 * Varied on its first edit: its 32 KiB are filled with its block type, its flag becomes 0, then the edits land (a chunk
 * that ends up all air is still Varied; the mesher gives it no mesh, which draws like Uniform air).  Nothing is
 * re-meshed: call vx_world_batch_remesh for the chunks whose meshes can change (the edited chunk, and the neighbour across
 * each face on which an edited voxel lies).  Edit loaded slots only: an absent slot that is edited anyway becomes a
 * Varied air chunk holding the edits, at whatever position its row last held, and stays so until the slot is generated
 * again.  Stream ordered; synchronises before it returns. */
VX_API int vx_world_batch_set_blocks(VxContext *ctx, VxMeshBatch *b, const int32_t *slots, const int32_t *voxel_index,
                                     const uint8_t *block_types, int32_t n);

/* ---- ray casting through a world batch (picking) -------------------------------------------------------------------
 * One ray per thread, an Amanatides-Woo walk over the voxels the world batch holds; the exact semantics, which the CPU
 * oracle (tests/ray_oracle.c: vxo_raycast) restates statement for statement, so that both give identical bits:
 *   - ray i: origin o (f32 x 3, world units: voxel (x,y,z) occupies [x,x+1) x [y,y+1) x [z,z+1)), direction d (f32 x 3,
 *     used as given, not normalised), start slot = the slot of the chunk that holds floor(o); the point at parameter t is
 *     o + t*d.  max_t is one value per call.
 *   - VX_RAY_INVALID: a non-finite component of o or d, d == (0,0,0), |o| >= 2^24 on some axis, max_t outside [0, 1e4]
 *     (or NaN), a start slot outside [0, capacity) (-1 = "not loaded"), or a start slot whose position row is not the
 *     floor division by 32 of the start voxel v = (floorf(o.x), floorf(o.y), floorf(o.z)).
 *   - step on each axis: the sign of d (no step where the component is 0).  The parameter of the next voxel face on an
 *     axis is computed in closed form whenever it is needed, tnext = ((float)plane - o) / d, with plane = v + 1 when
 *     stepping up and plane = v when stepping down (v = the current voxel on that axis) -- never accumulated.
 *   - the walk: if the current voxel is solid (type != 0) the ray hits it.  Else take the axis with the smallest tnext,
 *     ties x before y before z; tnext > max_t -> VX_RAY_MISS; step the voxel on that axis; leaving the chunk through a
 *     neighbour entry < 0 (VX_NBR_NONE: nothing loaded there) -> VX_RAY_LEFT_WORLD; else repeat in the new voxel.
 *   - a Uniform chunk (flag != 0) has no voxel rows: a Uniform solid chunk is solid everywhere (type flag - 1; a ray that
 *     enters it hits the entered voxel), a Uniform air chunk is walked without voxel loads.
 *   - a hit reports status VX_RAY_HIT, the slot, the world voxel, its block type, t = the tnext of the step that entered
 *     the voxel and face = the FaceDir (0..5 = +X,-X,+Y,-Y,+Z,-Z) of the hit voxel's face the ray crossed: a step towards
 *     +x enters through -X, face 1.  An origin inside a solid voxel is a hit with t = 0 and face -1.  (A ray that starts
 *     on a voxel face and steps down crosses that face at once, t = -0.0f.)
 *   - every other status leaves slot = -1, voxel = (0,0,0), face = -1, t = 0, block_type = 0.
 * The walk takes at most sum over the stepping axes of (floor(|d_axis| * max_t) + 3) steps (the planes within max_t, one
 * for rounding, one for an origin on a face), so no ray runs unbounded; a -DVX_DEBUG_CHECKS build checks that bound inside
 * the kernel, and vx_world_raycast then fails with VX_ERR_CUDA if a ray since the last call exceeded it. */
enum { VX_RAY_HIT = 0, VX_RAY_MISS = 1, VX_RAY_LEFT_WORLD = 2, VX_RAY_INVALID = 3 };
typedef struct {
    int32_t status;   /* VX_RAY_* */
    int32_t slot;     /* -1 unless hit */
    int32_t voxel[3]; /* world voxel coordinates */
    int32_t face;     /* FaceDir entered, -1 = origin inside a solid voxel */
    float t;
    uint8_t block_type, pad[3];
} VxRayHit; /* 32 bytes */
/* n rays from host arrays (origins / dirs n x 3 f32, start_slots n) into hits_out (n, host).  VX_ERR_INVALID for a batch
 * that is not a world batch, a start slot outside [-1, capacity) or a missing array; a bad ray is reported through its
 * status.  Synchronises before it returns. */
VX_API int vx_world_raycast(VxContext *ctx, const VxMeshBatch *b, const float *origins, const float *dirs, const int32_t *start_slots,
                            int32_t n, float max_t, VxRayHit *hits_out);
/* The same kernel on arrays resident on the context's device; asynchronous on the context's stream.  Every bad ray,
 * including a start slot out of range, is reported through its status (VX_ERR_INVALID only for a batch that is not a
 * world batch or a missing array). */
VX_API int vx_world_raycast_device(VxContext *ctx, const VxMeshBatch *b, const float *d_origins, const float *d_dirs,
                                   const int32_t *d_start_slots, int32_t n, float max_t, VxRayHit *d_hits_out);

/* ---- meshing ---------------------------------------------------------- */

/* BinaryGreedyMesher::mesh_world (binary_greedy.rs:62-78) / mesh_chunk_in_world (:83) /
 * mesh_chunk_in_indexed_world (:127) / mesh_chunk (:55, neighbors == NULL).
 *   voxels        N x 32768 u8, index = z*1024 + y*32 + x (chunk.rs:52), values 0..3
 *   positions     N x 3 chunk coordinates (kept with the batch for rendering)
 *   neighbors     N x 6: index into this batch, or VX_NBR_*; NULL = all VX_NBR_NONE
 *   uniform_flags N: 0 = Varied, else 1 + block_type of a Uniform chunk (-> no mesh,
 *                 binary_greedy.rs:87); NULL = all Varied.  A neighbour index that points
 *                 at a Uniform chunk is treated by its block type (:305-313).
 * Host -> device copy, mesh kernel; the result stays on the device. */
VX_API int vx_mesh_chunks(VxContext *ctx, const uint8_t *voxels, const int32_t *positions, const int32_t *neighbors,
                   const uint8_t *uniform_flags, int32_t n_chunks, VxMeshBatch **out);
/* Incremental re-mesh of a batch created by vx_mesh_chunks (which keeps a device copy of the world with the batch):
 * the reference re-meshes an edited chunk and invalidates its six neighbours (main.rs:225-280, world.rs:57-100).
 *   chunk_ids      n_ids edited chunks (indices into the batch)
 *   voxels         n_ids x 32768 new voxel data, uniform_flags n_ids (as vx_mesh_chunks) or NULL = all Varied
 * The edited chunks and the neighbours listed for them at creation are re-meshed in place (*n_remeshed of them); new
 * quads are appended to the quad stream, the replaced ones become dead space.  When the stream runs out of room the
 * live quads are compacted (copied, not re-meshed).  Every other chunk's mesh is untouched. */
VX_API int vx_mesh_batch_update(VxContext *ctx, VxMeshBatch *batch, const int32_t *chunk_ids, int32_t n_ids, const uint8_t *voxels,
                         const uint8_t *uniform_flags, int32_t *n_remeshed);
/* Same with all four arrays already resident on the context's device. */
VX_API int vx_mesh_chunks_device(VxContext *ctx, const uint8_t *d_voxels, const int32_t *d_positions,
                          const int32_t *d_neighbors, const uint8_t *d_uniform_flags, int32_t n_chunks,
                          VxMeshBatch **out);
/* Chunk-sharded meshing (one rank of a multi-GPU remesh sweep, SURVEY.md 8e): mesh only the chunks listed in
 * d_subset (ids into the n_chunks-sized arrays, e.g. every world_size-th sorted chunk id).  The voxel / neighbour
 * arrays are the whole world (replicated), so neighbour halos need no exchange; the batch has n_subset chunks in
 * subset order.  *batch_inout == NULL: create it; else re-mesh into it (steady state, no allocation, no sync). */
VX_API int vx_mesh_chunk_subset_device(VxContext *ctx, const uint8_t *d_voxels, const int32_t *d_positions,
                                const int32_t *d_neighbors, const uint8_t *d_uniform_flags, int32_t n_chunks,
                                const int32_t *d_subset, int32_t n_subset, VxMeshBatch **batch_inout);
/* Re-mesh into an existing batch of the same n_chunks (steady-state remesh sweep: no allocation). */
VX_API int vx_remesh_chunks_device(VxContext *ctx, const uint8_t *d_voxels, const int32_t *d_neighbors,
                            const uint8_t *d_uniform_flags, VxMeshBatch *batch);
VX_API int vx_mesh_batch_info(VxContext *ctx, const VxMeshBatch *b, VxMeshBatchInfo *info);
VX_API int vx_mesh_batch_device(const VxMeshBatch *b, VxMeshBatchDevice *out);
/* Copy a batch to host arrays (any pointer may be NULL to skip it).  Sizes: quads 3*total_quads,
 * quad_base/quad_count N, slice_offsets N*6*33, face_aabb N*36, has_mesh N. */
VX_API int vx_mesh_batch_download(VxContext *ctx, const VxMeshBatch *b, uint8_t *quads, uint32_t *quad_base,
                           uint32_t *quad_count, uint32_t *slice_offsets, int32_t *face_aabb, uint8_t *has_mesh);
/* Build a device batch from host mesh arrays (meshes produced elsewhere, e.g. gathered
 * from the other ranks of a chunk-sharded remesh). */
VX_API int vx_mesh_batch_upload(VxContext *ctx, const uint8_t *quads, int64_t total_quads, const uint32_t *quad_base,
                         const uint32_t *quad_count, const uint32_t *slice_offsets, const int32_t *face_aabb,
                         const uint8_t *has_mesh, const int32_t *positions, int32_t n_chunks, VxMeshBatch **out);
/* Chunk-sharded meshing across GPUs, exchange step (BinaryGreedyMesher::mesh_world returns EVERY mesh to its caller,
 * binary_greedy.rs:62-78): rank r meshes the chunks k with k % world == r (vx_mesh_chunk_subset_device; row j of the
 * shard = chunk r + j * world).  vx_shard_layout fixes one block layout for all ranks (sections quad_base / quad_count /
 * slice_offsets / face_aabb / has_mesh / quad stream, 16-byte aligned; host-only helper), vx_mesh_shard_pack copies a
 * shard into its block, the caller all-gathers the blocks (one NCCL collective over NVLink; rank r's block at
 * d_blocks + r * rank_stride) and vx_mesh_batch_assemble_shards builds the batch in chunk order on every rank:
 * shard_quads[r] (host) = quads in rank r's stream.  The assembled quad stream is the concatenation of the shard
 * streams; per-chunk quad lists stay bit-identical.  *batch_inout NULL: a new batch; else re-filled in place. */
typedef struct {
    int64_t rank_stride;  /* bytes per block */
    int64_t off_quad_base, off_quad_count, off_slice_offsets, off_face_aabb, off_has_mesh, off_quads;
    int64_t quads_capacity; /* quads a block's stream section holds */
    int32_t rows_per_rank;  /* ceil(n_chunks / world) */
    int32_t reserved;
} VxShardLayout;
VX_API int vx_shard_layout(int32_t rows_per_rank, int64_t max_shard_quads, VxShardLayout *out);
VX_API int vx_mesh_shard_pack(VxContext *ctx, const VxMeshBatch *shard, const VxShardLayout *layout, uint8_t *d_block);
VX_API int vx_mesh_batch_assemble_shards(VxContext *ctx, int32_t n_chunks, int32_t world, const uint8_t *d_blocks,
                                  const VxShardLayout *layout, const int64_t *shard_quads, const int32_t *d_positions,
                                  VxMeshBatch **batch_inout);
/* The same exchange without a host round trip, for the steady state of a re-mesh sweep (block capacity known from an
 * earlier sweep): _pack_async copies the whole quad section the block has room for plus the shard's quad total (a u64 at
 * off_quads - 16 of the block); _assemble_shards_async reads the totals from the gathered blocks on the device, so nothing
 * is read back between the mesh kernel, the all-gather and the assembled batch.  A shard that outgrew its block sets the
 * batch's overflow flag: the next vx_mesh_batch_info on the assembled batch fails with VX_ERR_CAPACITY and the caller goes
 * through the synchronous pair once to size the blocks anew. */
VX_API int vx_mesh_shard_pack_async(VxContext *ctx, const VxMeshBatch *shard, const VxShardLayout *layout, uint8_t *d_block);
VX_API int vx_mesh_batch_assemble_shards_async(VxContext *ctx, int32_t n_chunks, int32_t world, const uint8_t *d_blocks,
                                        const VxShardLayout *layout, const int32_t *d_positions, VxMeshBatch **batch_inout);
VX_API void vx_mesh_batch_release(VxContext *ctx, VxMeshBatch *b);

/* BinaryGreedyMesher::greedy_mesh_slice (binary_greedy.rs:675) for n_slices masks of 32 rows.
 * out: up to 512 quads per slice at out[i*512 ...], n_out[i] quads. */
VX_API int vx_greedy_mesh_slices(VxContext *ctx, const uint32_t *masks, int32_t n_slices, VxQuad *out, int32_t *n_out);

/* ---- culling ---------------------------------------------------------- */

/* World::get_visible_chunks_frustum (world.rs:118-146) with Frustum::from_view_projection /
 * intersects_aabb (camera/mod.rs:123-183).  visible_out[i] in {0,1}. */
VX_API int vx_cull_chunks(VxContext *ctx, const int32_t *positions, int32_t n, const float vp[16], const float cam_pos[3],
                   int32_t view_distance, int32_t frustum_culling, uint8_t *visible_out);

/* culling::apply_horizon_culling (culling.rs:40-119) with HorizonCullingConfig (:16-36; defaults bins 128,
 * base_margin 0.1, margin_dist_factor 0.05, min_dist_chunks 2.0).  centers: n_centers x 3 VisibleMesh centres
 * (main.rs:286-290); order_inout: n mesh ids -> the kept ids, stably sorted front to back; *n_kept of them.
 * Optional stage: main.rs does not call it (:368-377).  atan2 is evaluated in f64 and rounded (the reference uses the
 * platform libm): a mesh within an ulp of a bin boundary may land in the neighbouring bin. */
VX_API int vx_horizon_cull(VxContext *ctx, const float cam_pos[3], const float *centers, int32_t n_centers, int32_t *order_inout,
                    int32_t n, int32_t bins, float base_margin, float margin_dist_factor, float min_dist_chunks,
                    int32_t *n_kept);

/* ---- rendering -------------------------------------------------------- */

VX_API void vx_default_frame_config(VxFrameConfig *cfg, int32_t width, int32_t height);
VX_API void vx_default_atlas(VxAtlas *atlas); /* TextureAtlas::default texture.rs:60-79 */
/* Rasterizer::new_with_atlas (rasterizer.rs:357): atlas used by later render calls. */
VX_API int vx_set_atlas(VxContext *ctx, const VxAtlas *atlas);

/* main.rs RedrawRequested steady state (:283-297, :368-377) + render_frame (:379-608):
 * VisibleMesh list -> distance sort -> AABB projection / reject (filter B) -> near-depth sort ->
 * [occlusion pass :501-526 when cfg->occlusion_culling] -> project + clip + backface-cull every quad ->
 * stripe-binned span rasterization -> framebuffer.  cfg->macrotile selects render_frame_macrotile's order instead.
 *   mesh_ids      chunks of `batch` that passed filter A (caller order = tie-break order), or NULL
 *                 with n_meshes < 0 to run filter A on the device over the batch's own positions
 *                 (view_distance then required)
 *   color_out     rows x width u32 ARGB (may be NULL), depth_out rows x width f32 (may be NULL),
 *                 rows = stripe_rows or height.  Device-mapped page-locked buffers (vx_host_alloc) are written in
 *                 place by the kernel; other host memory is filled by a copy from the device framebuffer
 *   survivors_out draw order (capacity n_meshes / n_chunks; entries past *n_survivors are undefined), may be NULL;
 *                 meshes dropped by filter B or by the occlusion pass are not in it */
VX_API int vx_render_frame(VxContext *ctx, const VxMeshBatch *batch, const int32_t *mesh_ids, int32_t n_meshes,
                    const float vp[16], const float cam_pos[3], int32_t view_distance, const VxFrameConfig *cfg,
                    uint32_t *color_out, float *depth_out, int32_t *survivors_out, int32_t *n_survivors);
/* Pipelined vx_render_frame: the reference's loop presents frame k while the next iteration is already under way
 * (main.rs:320-336).  _begin enqueues one whole frame -- draw-list upload, cull / setup / raster, read-back of the
 * statistics and the draw order -- and returns a ticket without waiting for the GPU; _end(ticket) blocks until THAT
 * frame is complete in color_out / depth_out and hands out its draw order.  At most two frames are in flight
 * (begin k+1 may precede end k), so each needs its own buffers, and the buffers must be page-locked memory
 * (vx_host_alloc): the frame is rendered into a device buffer of its in-flight slot and leaves through the copy engine
 * on a second stream, so the PCIe transfer of frame k runs beside the kernels of frame k+1 (steady-state period =
 * max(render, transfer)).  The frame's statistics and draw order are written into the slot by the frame's own kernels
 * and travel with it, so the context's next frame never waits for a transfer.  A frame whose scratch overflowed is
 * re-rendered synchronously inside _end, with the cfg and the atlas (vx_set_atlas) the frame had at _begin, so the
 * result is always the same as vx_render_frame's.
 * Frames in flight ON THE DEVICE: contexts are independent (stream + frame scratch each), so a caller that deals its
 * frames round-robin over L contexts of one device ("lanes") lets the kernels of different frames overlap -- one frame
 * is three dependent latency-bound kernels and leaves most of the GPU idle; L = 3 raises the device's frame throughput
 * by half.  Nothing else is needed: any batch can be rendered through any context of its device. */
VX_API int vx_render_frame_begin(VxContext *ctx, const VxMeshBatch *batch, const int32_t *mesh_ids, int32_t n_meshes,
                          const float vp[16], const float cam_pos[3], int32_t view_distance, const VxFrameConfig *cfg,
                          uint32_t *color_out, float *depth_out, int32_t *ticket);
VX_API int vx_render_frame_end(VxContext *ctx, int32_t ticket, int32_t *survivors_out, int32_t *n_survivors);
/* Device-resident variant: nothing is copied back; the frame stays in the context's framebuffer
 * (see vx_framebuffer_device).  Used with CUDA-event timing and for multi-GPU composition. */
VX_API int vx_render_frame_device(VxContext *ctx, const VxMeshBatch *batch, const int32_t *d_mesh_ids, int32_t n_meshes,
                           const float vp[16], const float cam_pos[3], int32_t view_distance,
                           const VxFrameConfig *cfg);
/* As vx_render_frame_device, but the frame (rows x width, tightly packed) is written to caller-provided memory the
 * device can address: device memory of this GPU, peer memory of another GPU (stripe composition without a copy), or
 * device-mapped page-locked host memory.  NULL = the context's own buffer for that plane. */
VX_API int vx_render_frame_into(VxContext *ctx, const VxMeshBatch *batch, const int32_t *d_mesh_ids, int32_t n_meshes,
                         const float vp[16], const float cam_pos[3], int32_t view_distance, const VxFrameConfig *cfg,
                         uint32_t *d_color_dst, float *d_depth_dst);
/* Stripe of a frame that is composed on another GPU (one process per GPU; framebuffer.rs:392-431 hands disjoint
 * `&mut` stripes of ONE framebuffer to the workers): as vx_render_frame_into with d_color_dst / d_depth_dst pointing
 * into the peer-mapped frame (vx_ipc_open), plus the hand-off inside the frame's own kernels -- before its first store
 * the kernel waits until *d_wait_flag (a word in THIS GPU's memory, written by the composing GPU when it has consumed
 * the frame that last used the buffer) has reached wait_value; after its last store the last CTA publishes signal_value
 * into *d_signal_flag (the composing GPU's arrival word for this rank) with release semantics at system scope.  Either
 * pointer may be NULL.  (The wait itself is done by one thread of the setup kernel, which the raster kernel follows.)  On
 * the composing GPU the same kernel can also do the per-frame bookkeeping (see the struct).  Always asynchronous (like
 * cfg->async_submit = 1); a wait that exceeds timeout_us (<= 0: 2 s) is reported by vx_frame_stats, nothing hangs. */
typedef struct {
    const uint32_t *d_wait_flag;
    uint32_t wait_value;
    uint32_t *d_signal_flag;
    uint32_t signal_value;
    int32_t timeout_us;
    /* Composing GPU only (else n_arrive = 0): the kernel's CTA 0, once it is out of work, marks *d_signal_flag (this rank's
     * own arrival word), waits until the n_arrive
     * arrival words of THIS GPU (arrive_stride_words apart) have reached arrive_value -- every rank's stripe of the frame
     * is then in place when the kernel ends -- and publishes release_value into the n_release (<= 32) acknowledgement
     * words listed in release_flags (HOST array of device addresses, local or peer-mapped): the buffer of frame
     * release_value - 1 may be overwritten.  This replaces the separate vx_wait_then_signal launch. */
    int32_t n_arrive, arrive_stride_words;
    const uint32_t *d_arrive_flags;
    uint32_t arrive_value, release_value;
    int32_t n_release;
    /* 1 (ranks other than the composing one): publish signal_value from a 1-thread kernel enqueued behind the raster kernel
     * instead of from the raster kernel's last CTA.  The fused publish makes every raster CTA fence its peer stores at
     * system scope before it leaves; with several frames in flight on the GPU those idle SM slots cost more than the extra
     * launch (measured at N = 2: 34.5 -> 29.9 us per frame). */
    int32_t signal_after;
    uint32_t *const *release_flags;
} VxStripeSync;
VX_API int vx_render_frame_stripe(VxContext *ctx, const VxMeshBatch *batch, const int32_t *d_mesh_ids, int32_t n_meshes,
                           const float vp[16], const float cam_pos[3], int32_t view_distance, const VxFrameConfig *cfg,
                           uint32_t *d_color_dst, float *d_depth_dst, const VxStripeSync *sync);
/* Device pointers of the last rendered frame: colour (u32) and depth (f32), rows x width. */
VX_API int vx_framebuffer_device(VxContext *ctx, uint32_t **d_color, float **d_depth, int32_t *rows, int32_t *width);
VX_API int vx_frame_stats(VxContext *ctx, VxFrameStats *out);
/* Diagnostics: the raw 32-word control block of the last frame -- [0] survivors, [1] quads, [2] triangles kept, [3] bin
 * entries, [4] overflow bits (1 triangle slots, 2 a tile bin, 8 more than 2^21 quads, 16 big-triangle list, 32 raster
 * work items, 64 bounds check of a VX_DEBUG_CHECKS build, 128 stripe hand-off timeout, 256 setup units; a synchronous frame
 * grows the scratch behind 1, 2, 32 and 256 and renders again, so its own word reads 0 unless the frame failed), [5] fullest
 * bin, [6] big triangles (bounding box over more than 64 tiles), [7] setup units,
 * [8] meshes culled by the occlusion pass, [9] raster work items, [12] items the plan wanted, [13] second near-clip
 * pieces, [14] (triangle, row, column block) tasks binned, [16..24] items per plan class, [25] raster CTAs that
 * finished. */
VX_API int vx_frame_counters(VxContext *ctx, uint32_t out[32]);
/* CUDA-event durations (ms) of the last frame rendered with profile_kernels != 0:
 * [0] cull, [1] rank + project/clip/setup + binning, [2] unused (0), [3] work-item plan + span raster + write-out. */
VX_API int vx_frame_kernel_times(VxContext *ctx, float ms_out[4]);
/* Diagnostics: timeline of the raster work items of the last frame rendered with profile_kernels = 2.
 * out: 14 x u64 per item = tile, part | parts << 16, start ns, end ns (%globaltimer), SM id, source entries,
 * keys-ready ns, first-expansion ns, first-task-round ns, then for thread 0's first task the clock cycles spent on
 * record load, edge setup, span setup + jump, pixel walk, and its pixel count. */
VX_API int vx_frame_trace(VxContext *ctx, uint64_t *out, int32_t cap_items, int32_t *n_items);
/* Same for the setup kernel: 12 x u64 per CTA = start, ranked, projected, binned, done (ns), tiles in the unit's box,
 * triangles kept, units processed, counted, ranges reserved (ns), 2 unused.  CTAs that had no unit stay all-zero. */
VX_API int vx_frame_setup_trace(VxContext *ctx, uint64_t *out, int32_t cap_ctas, int32_t *n_ctas);
/* Diagnostics: triangles binned per 128x8 tile in the last frame (row-major tile grid, ntx x nty). */
VX_API int vx_frame_bin_counts(VxContext *ctx, uint32_t *counts_out, int32_t cap, int32_t *ntx, int32_t *nty);
/* Same layout: the (row, 16-pixel column block) tasks the tile's entries expand to -- with the entry counts the cost model of
 * the work-balanced stripe split (a stripe costs ~ entries + tasks / 5 on top of what every stripe costs). */
VX_API int vx_frame_bin_tasks(VxContext *ctx, uint32_t *tasks_out, int32_t cap, int32_t *ntx, int32_t *nty);

/* render_frame_macrotile (macrotile_renderer.rs:51-170; MacroTileBins::add_mesh macrotile.rs:179-224, MacroTile as
 * PixelTarget :300-343): clear, project_mesh_aabb per mesh of the caller's list (:175-250, the arithmetic of filter B),
 * per 128x128 macrotile the binned meshes in list order and then the large primitives (> 25 % of the screen) through
 * the span rasterizer with the tile as target, tile colours flushed to color_out (W x H).  = vx_render_frame with
 * cfg.macrotile = 1 and no distance / near-depth sort.  tile_depth_out (W x H, may be NULL) receives the tiles' depth
 * buffers, which the reference drops (its framebuffer depth stays +inf).  projected_out (n_meshes entries, may be
 * NULL): the meshes that passed project_mesh_aabb in draw order -- list order, large primitives last;
 * *n_projected = the reference's return value.  The Hi-Z buffer argument of the reference is only cleared there
 * and never consulted, so it has no counterpart.  A mesh is assumed to stay inside its projected chunk box (the
 * reference bins by that box; geometry of a chunk cannot leave it). */
VX_API int vx_render_frame_macrotile(VxContext *ctx, const VxMeshBatch *batch, const int32_t *mesh_ids, int32_t n_meshes,
                              const float vp[16], const VxFrameConfig *cfg, uint32_t *color_out, float *tile_depth_out,
                              int32_t *projected_out, int32_t *n_projected);

/* SpanWalkerRasterizer::rasterize_projected_packet (span_walker.rs:116-283) + FrameSlice::fill_span (:412-441) over n
 * projected quads in submission order (ProjectedPackets concatenated, differential_projection.rs:295-304: NDC boxes,
 * constant depth, block type; visible[i] = bit i of visibility_mask, NULL = all visible): rows whose centre lies in
 * the screen box, columns round(x_min) .. round(x_max + 0.001), flat colour per block type (:386-396), depth test
 * `<` against the existing contents of the W x H host framebuffer (read-modify-write).  The viewport of the walker
 * and the framebuffer have the same size, as everywhere in the reference. */
VX_API int vx_span_walk_quads(VxContext *ctx, const float *x_min, const float *y_min, const float *x_max, const float *y_max,
                       const float *depth_near, const uint8_t *block_type, const uint8_t *visible, int32_t n, int32_t width,
                       int32_t height, uint32_t *color_inout, float *depth_inout);
/* Same on device-resident data: d_boxes = x_min[n], y_min[n], x_max[n], y_max[n], depth_near[n]; d_types =
 * block_type[n], visible[n]; d_color / d_depth = W x H framebuffer in device memory.  Asynchronous on the context's
 * stream. */
VX_API int vx_span_walk_quads_device(VxContext *ctx, const float *d_boxes, const uint8_t *d_types, int32_t n, int32_t width,
                              int32_t height, uint32_t *d_color, float *d_depth);
/* FrameSlice::fill_span (span_walker.rs:412-441) for n spans in submission order: pixels [x_start, x_end) of row y
 * after the reference's clamps, depth test `<`.  A row outside the framebuffer is VX_ERR_INVALID (the reference
 * would index out of bounds). */
VX_API int vx_fill_spans(VxContext *ctx, const int32_t *y, const int32_t *x_start, const int32_t *x_end, const float *depth,
                  const uint32_t *color, int32_t n, int32_t width, int32_t height, uint32_t *color_inout, float *depth_inout);

/* The Hyper-Pipeline (SURVEY 3.3; tests/span_walker_fuzz_tests.rs:158-173, benches/differential_projection.rs) for a
 * list of meshes of a batch, device-resident end to end: ChunkFacePackets::from_chunk_mesh (face_packets.rs:122-174:
 * packets of 32 consecutive quads per face) -> PacketPipeline::process_chunk_packets (packet_pipeline.rs:69-142: one
 * FaceBasis per packet from the packet's first quad, packet-level backface test normal.z < 0, scalar projection
 * project_single_scalar with exact division, frustum mask :279-293) -> SpanWalkerRasterizer::rasterize_projected_packet
 * per packet, all in mesh-list order.  W x H host framebuffer, read-modify-write.  *n_visible_quads (may be NULL) =
 * quads that passed the backface and frustum tests.  The reference's AVX2 projection (reciprocal + Newton step) is not
 * reproduced; this is its scalar path. */
VX_API int vx_hyper_pipeline_render(VxContext *ctx, const VxMeshBatch *batch, const int32_t *mesh_ids, int32_t n_meshes,
                             const float vp[16], int32_t width, int32_t height, uint32_t *color_inout, float *depth_inout,
                             int32_t *n_visible_quads);

/* Rasterizer::render_mesh / render_mesh_into_slice / render_mesh_into_tile (rasterizer.rs:385-431)
 * for one mesh into a caller framebuffer (W x H host arrays, read-modify-write: depth-tested against
 * the existing contents).  rect = PixelTarget::rect() = (x0, y0, w, h). */
VX_API int vx_render_mesh(VxContext *ctx, const VxMeshBatch *batch, int32_t mesh_id, const float vp[16],
                   const VxFrameConfig *cfg, const int32_t rect[4], uint32_t *color_inout, float *depth_inout);

/* Rasterizer::render_mesh_tiny_quads(mesh, view_proj, target, use_span_renderer) (rasterizer.rs:782-929), the pub
 * generic both mesh paths go through.  use_span_renderer != 0: vx_render_mesh.  0: the barycentric rasterizer
 * render_tiny_quad / render_triangle_from_clip_textured (:932-1071, :1881-2107): box of the clipped triangle
 * intersected with the framebuffer and rect, `area < 0.1` triangles dropped, edge functions advanced by one rounded
 * add per pixel and per row from the box's top-left pixel centre, coverage w0, w1, w2 >= 0, depth and perspective-
 * correct texel from the barycentric weights.  W x H host arrays, read-modify-write; exact vertex arithmetic only
 * (cfg->differential_projection is ignored on this path). */
VX_API int vx_render_mesh_tiny_quads(VxContext *ctx, const VxMeshBatch *batch, int32_t mesh_id, const float vp[16],
                              const VxFrameConfig *cfg, const int32_t rect[4], int32_t use_span_renderer,
                              uint32_t *color_inout, float *depth_inout);
/* Rasterizer::render_mesh_with_up (rasterizer.rs:399-411): the whole framebuffer; the span renderer when the camera
 * is level (|camera_up.y| >= 0.995, is_camera_level :377-382), the barycentric one otherwise. */
VX_API int vx_render_mesh_with_up(VxContext *ctx, const VxMeshBatch *batch, int32_t mesh_id, const float vp[16],
                           const VxFrameConfig *cfg, const float camera_up[3], uint32_t *color_inout, float *depth_inout);

/* ---- hyper-pipeline pieces ------------------------------------------- */

/* `FacePacket32` face_packets.rs:13-25: up to 32 quads of one face direction, structure of arrays, 32-byte aligned. */
typedef struct {
    uint8_t len;
    uint8_t u_min[32], v_min[32], u_len[32], v_len[32];
    uint8_t axis_pos[32];   /* slice + 1 for positive faces, slice for negative ones (:146-151) */
    uint8_t block_type[32];
    uint8_t pad[31];        /* align(32): sizeof == 224 */
} VxFacePacket32;

/* ChunkFacePackets::from_chunk_mesh (face_packets.rs:122-174) for one mesh of a batch: packets of face 0 first, then
 * face 1 ... (FaceDir order), n_packets_per_face[f] of them; packets_out must hold their sum (<= cap_packets, else
 * VX_ERR_CAPACITY with the sizes filled in).  The arrays of a packet feed vx_project_packet directly. */
VX_API int vx_face_packets(VxContext *ctx, const VxMeshBatch *batch, int32_t mesh_id, VxFacePacket32 *packets_out, int32_t cap_packets,
                    int32_t n_packets_per_face[6]);

/* FaceBasis::from_face_direction (differential_projection.rs:37-62) for n (face, chunk, slice) triples.
 * basis_out: n x 16 f32 = origin, tangent, bitangent, normal. */
VX_API int vx_face_basis(VxContext *ctx, const int32_t *faces, const int32_t *chunk_pos, const uint8_t *slice_idx, int32_t n,
                  const float vp[16], float *basis_out);
/* FaceBasis::project_packet_bounds_simd / project_single_scalar (differential_projection.rs:92-196) for
 * n quads sharing one basis (SoA u8 arrays as FacePacket32, face_packets.rs:13-25), exact division.
 * Outputs n f32 each: NDC x_min, y_min, x_max, y_max, depth_near (ProjectedPacket :295-304). */
VX_API int vx_project_packet(VxContext *ctx, const float basis[16], const uint8_t *u_min, const uint8_t *v_min,
                      const uint8_t *u_len, const uint8_t *v_len, int32_t n, float *x_min, float *y_min,
                      float *x_max, float *y_max, float *depth_near);
/* simd_vertex::decompress_and_transform_vertices (simd_vertex.rs:24): out4 = n x 4 clip-space f32. */
VX_API int vx_transform_vertices(VxContext *ctx, const VxVertex *verts, int32_t n, const float offset[3], const float vp[16],
                          float *out4);
/* Clip-space corners of the quads of one mesh exactly as the raster path computes them
 * (rasterizer.rs:1092-1185): out = n_quads x 4 x 4 f32; mode as VxFrameConfig.differential_projection. */
VX_API int vx_project_mesh_vertices(VxContext *ctx, const VxMeshBatch *batch, int32_t mesh_id, const float vp[16],
                             int32_t differential, float *out, int64_t cap_quads);

/* ---- self tests ------------------------------------------------------- */

/* The raster kernels divide with an inlined, branch-free copy of nvcc's IEEE division fast path behind an explicit
 * exponent guard (vx_math.cuh: vx_div_fast).  This runs it against the `/` operator on n_pairs pseudo-random operand
 * pairs (mode 0: any bit patterns, 1: magnitudes of the raster path, 2: short mantissas; 3: the texel-lookup variant
 * vx_div_texel, compared on the texel index) and returns
 * counters_out = {mismatches among guard-accepted pairs (must be 0), pairs sent to the fallback, pairs tested}. */
VX_API int vx_selftest_division(VxContext *ctx, uint64_t seed, uint64_t n_pairs, int32_t mode, uint64_t counters_out[3]);

#ifdef __cplusplus
}
#endif
#endif
