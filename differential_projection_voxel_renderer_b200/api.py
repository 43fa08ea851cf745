"""Host-side mirror of the reference crate's public meshing / rendering API, on top of the C ABI.

Same names and argument meaning as the Rust items they stand in for (citations relative to
/root/reference/src/): `BinaryGreedyMesher` (meshing/binary_greedy.rs:50-168,675-683), `ChunkMesh` / `TinyQuad`
(meshing/mesh.rs:273-687), `Framebuffer` (rendering/framebuffer.rs:197-245), `Rasterizer`
(rendering/rasterizer.rs:335-431), `Frustum` (camera/mod.rs:111-183), `FaceBasis`
(rendering/differential_projection.rs:18-82), `decompress_and_transform_vertices` (rendering/simd_vertex.rs:24),
`render_frame` (main.rs:379-608).  Every call runs on the GPU through libvx_b200.so; nothing here falls back to
the CPU (and nothing here touches oracle/).
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import VxAtlas, VxError, VxFrameConfig, VxFrameStats, VxMeshBatchDevice, VxMeshBatchInfo, VxTerrainParams

CHUNK_SIZE = 32
CHUNK_VOLUME = 32768
FACE_DIRS = ("PosX", "NegX", "PosY", "NegY", "PosZ", "NegZ")  # mesh.rs:136-143


def _p(a):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


class Context:
    """One CUDA device + stream (VxContext)."""

    def __init__(self, device: int = 0):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.vx_context_create(int(device), C.byref(h))
        if rc != 0:
            raise VxError(rc, self.lib.vx_error_string(rc).decode())
        self.handle = h
        self.device = int(device)
        self._host_allocs = []
        self._atlas = bytes(_default_atlas_cached())  # the atlas the context holds (vx_context_create loads the default one)

    def check(self, rc: int):
        if rc != 0:
            detail = self.lib.vx_last_error(self.handle).decode()
            raise VxError(rc, f"{self.lib.vx_error_string(rc).decode()}: {detail}")

    def synchronize(self):
        self.check(self.lib.vx_device_synchronize(self.handle))

    @property
    def stream(self) -> int:
        return int(self.lib.vx_context_stream(self.handle) or 0)

    @property
    def launch_count(self) -> int:
        return int(self.lib.vx_context_launch_count(self.handle))

    def set_atlas(self, atlas: VxAtlas):
        self.check(self.lib.vx_set_atlas(self.handle, C.byref(atlas)))
        self._atlas = bytes(atlas)

    def holds_atlas(self, atlas: VxAtlas) -> bool:
        """True if the last atlas loaded through set_atlas (or the default one of a new context) equals `atlas`."""
        return self._atlas == bytes(atlas)

    def host_array(self, shape, dtype) -> np.ndarray:
        """Array in device-mapped page-locked host memory (vx_host_alloc): passed as color_out / depth_out of
        render_frame it is written by the raster kernel directly.  Lives until the context is closed."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        p = C.c_void_p()
        self.check(self.lib.vx_host_alloc(self.handle, n, C.byref(p)))
        self._host_allocs.append(p)
        buf = (C.c_char * max(n, 1)).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def close(self):
        if getattr(self, "handle", None):
            for p in getattr(self, "_host_allocs", []):
                self.lib.vx_host_free(self.handle, p)
            self._host_allocs = []
            self.lib.vx_context_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


class FrameLanes:
    """Frames in flight on the device: `lanes` contexts on one GPU (a stream and a frame scratch each; the first may be an
    existing context), dealt out round-robin.  One frame is a chain of three dependent, latency-bound kernels that leaves
    most of the GPU's issue slots idle; frames of different lanes are independent (each lane plans its raster work from
    its own previous frame), so their kernels run side by side and the device's frame throughput rises by about a half
    (1280x720 view distance 12 on a B200: 74 us per frame alone, 43 us with three lanes, 34 us with eight).  A lane is just a VxContext:
    the C-ABI side of this is vx_context_create called `lanes` times."""

    def __init__(self, device: int = 0, lanes: int = 3, first: Optional[Context] = None):
        if lanes < 1:
            raise ValueError("lanes must be >= 1")
        self.ctxs: List[Context] = [first or Context(device)] + [Context(device) for _ in range(lanes - 1)]
        self._owned = self.ctxs[(1 if first is not None else 0):]
        self._next = 0

    def __len__(self):
        return len(self.ctxs)

    def __getitem__(self, i) -> Context:
        return self.ctxs[i]

    def next(self) -> Context:
        """The context the next frame goes to."""
        c = self.ctxs[self._next % len(self.ctxs)]
        self._next += 1
        return c

    def set_atlas(self, atlas: VxAtlas):
        for c in self.ctxs:
            c.set_atlas(atlas)

    def synchronize(self):
        for c in self.ctxs:
            c.synchronize()

    @property
    def launch_count(self) -> int:
        return sum(c.launch_count for c in self.ctxs)

    def close(self):
        for c in self._owned:
            c.close()
        self._owned = []


def default_frame_config(width: int, height: int) -> VxFrameConfig:
    cfg = VxFrameConfig()
    _lib.load().vx_default_frame_config(C.byref(cfg), width, height)
    return cfg


def default_atlas() -> VxAtlas:
    a = VxAtlas()
    _lib.load().vx_default_atlas(C.byref(a))
    return a


_default_atlas: Optional[VxAtlas] = None


def _default_atlas_cached() -> VxAtlas:
    global _default_atlas
    if _default_atlas is None:
        _default_atlas = default_atlas()
    return _default_atlas


def unpack_quads(q3: np.ndarray) -> np.ndarray:
    """(n,3) u8 TinyQuads -> (n,5) [u, v, w, h, block_type]  (TinyQuad accessors, mesh.rs:309-341)."""
    q3 = np.asarray(q3, dtype=np.uint8).reshape(-1, 3).astype(np.int32)
    u = q3[:, 0] & 0x1F
    v = ((q3[:, 0] >> 5) & 7) | ((q3[:, 1] & 3) << 3)
    w = ((q3[:, 1] >> 2) & 0x3F) + 1
    h = (q3[:, 2] & 0x3F) + 1
    bt = (q3[:, 2] >> 6) & 3
    return np.stack([u, v, w, h, bt], axis=1)


class ChunkMesh:
    """Host view of one chunk's mesh (mesh.rs:422-436): 6 FaceLists x 32 slice lists of TinyQuads."""

    def __init__(self, chunk_position, quads, slice_offsets, face_aabb):
        self.chunk_position = np.asarray(chunk_position, dtype=np.int32)
        self.quads = quads                    # (n,3) u8 in reference order
        self.slice_offsets = slice_offsets    # (6,33) u32
        self.face_aabb = face_aabb            # (6,6) i32: min.xyz, max.xyz

    def quad_count(self) -> int:  # mesh.rs:591
        return int(self.quads.shape[0])

    def is_empty(self) -> bool:  # mesh.rs:586
        return self.quad_count() == 0

    def slice_quads(self, face: int, slice_idx: int) -> np.ndarray:
        a, b = int(self.slice_offsets[face, slice_idx]), int(self.slice_offsets[face, slice_idx + 1])
        return self.quads[a:b]

    def face_quad_count(self, face: int) -> int:
        return int(self.slice_offsets[face, 32] - self.slice_offsets[face, 0])

    def world_offset(self) -> np.ndarray:  # mesh.rs:483-485
        return (self.chunk_position * CHUNK_SIZE).astype(np.float32)


class MeshBatch:
    """Device-resident meshes of a batch of chunks (VxMeshBatch)."""

    def __init__(self, ctx: Context, handle):
        self.ctx = ctx
        self.handle = handle
        self._host = None
        self._n_chunks = None

    def info(self) -> VxMeshBatchInfo:
        info = VxMeshBatchInfo()
        self.ctx.check(self.ctx.lib.vx_mesh_batch_info(self.ctx.handle, self.handle, C.byref(info)))
        return info

    def device_pointers(self) -> VxMeshBatchDevice:
        d = VxMeshBatchDevice()
        self.ctx.check(self.ctx.lib.vx_mesh_batch_device(self.handle, C.byref(d)))
        return d

    def download(self):
        """-> dict of host arrays: quads (Q,3), quad_base, quad_count, slice_offsets (N,6,33), face_aabb (N,6,6), has_mesh."""
        info = self.info()
        n, q = info.n_chunks, int(info.total_quads)
        out = {
            "quads": np.zeros((q, 3), dtype=np.uint8),
            "quad_base": np.zeros(n, dtype=np.uint32),
            "quad_count": np.zeros(n, dtype=np.uint32),
            "slice_offsets": np.zeros((n, 6, 33), dtype=np.uint32),
            "face_aabb": np.zeros((n, 6, 6), dtype=np.int32),
            "has_mesh": np.zeros(n, dtype=np.uint8),
        }
        self.ctx.check(self.ctx.lib.vx_mesh_batch_download(
            self.ctx.handle, self.handle, _p(out["quads"]), _p(out["quad_base"]), _p(out["quad_count"]),
            _p(out["slice_offsets"]), _p(out["face_aabb"]), _p(out["has_mesh"])))
        self._host = out
        return out

    def chunk_quads(self, i: int) -> np.ndarray:
        h = self._host or self.download()
        b, c = int(h["quad_base"][i]), int(h["quad_count"][i])
        return h["quads"][b:b + c]

    def chunk_mesh(self, i: int, position=(0, 0, 0)) -> Optional[ChunkMesh]:
        h = self._host or self.download()
        if not h["has_mesh"][i]:
            return None
        return ChunkMesh(position, self.chunk_quads(i), h["slice_offsets"][i], h["face_aabb"][i])

    def update(self, chunk_ids, voxels, uniform_flags=None) -> int:
        """Re-mesh edited chunks (and the six neighbours of each, main.rs:225-280) in place: vx_mesh_batch_update.
        voxels: (len(chunk_ids), 32768) new data.  Returns the number of chunks re-meshed."""
        ids = np.ascontiguousarray(chunk_ids, dtype=np.int32).reshape(-1)
        vox = np.ascontiguousarray(voxels, dtype=np.uint8).reshape(ids.shape[0], CHUNK_VOLUME)
        uf = None if uniform_flags is None else np.ascontiguousarray(uniform_flags, dtype=np.uint8).reshape(ids.shape[0])
        n = C.c_int32(0)
        self.ctx.check(self.ctx.lib.vx_mesh_batch_update(self.ctx.handle, self.handle, _p(ids), ids.shape[0], _p(vox), _p(uf), C.byref(n)))
        self._host = None
        return int(n.value)

    def release(self):
        if self.handle:
            self.ctx.lib.vx_mesh_batch_release(self.ctx.handle, self.handle)
            self.handle = None

    def __del__(self):
        try:
            if self.ctx.handle:
                self.release()
        except Exception:
            pass


def upload_mesh_batch(ctx: Context, quads, quad_base, quad_count, slice_offsets, face_aabb, has_mesh, positions) -> MeshBatch:
    quads = np.ascontiguousarray(quads, dtype=np.uint8).reshape(-1)
    n = int(np.asarray(quad_base).shape[0])
    arrs = [np.ascontiguousarray(quad_base, dtype=np.uint32), np.ascontiguousarray(quad_count, dtype=np.uint32),
            np.ascontiguousarray(slice_offsets, dtype=np.uint32), np.ascontiguousarray(face_aabb, dtype=np.int32),
            np.ascontiguousarray(has_mesh, dtype=np.uint8), np.ascontiguousarray(positions, dtype=np.int32)]
    h = C.c_void_p()
    ctx.check(ctx.lib.vx_mesh_batch_upload(ctx.handle, _p(quads), C.c_int64(quads.size // 3), *[_p(a) for a in arrs], n, C.byref(h)))
    return MeshBatch(ctx, h)


def terrain_params(seed: int = 12345) -> VxTerrainParams:
    """noise 0.9.0 Perlin::new(seed) tables (permutation table doubled, the four diagonal gradients twice) +
    chunk.rs:173-177 constants."""
    from . import worldgen
    tp = VxTerrainParams()
    perm = worldgen._perm_table(seed)
    for i in range(512):
        tp.perm[i] = int(perm[i])
    for i in range(8):
        tp.grad[i][0] = float(worldgen._GRAD2[i, 0])
        tp.grad[i][1] = float(worldgen._GRAD2[i, 1])
    tp.scale = 0.01
    tp.amplitude = 20.0
    return tp


def generate_terrain(positions, d_voxels: int, ctx: Optional[Context] = None, params: Optional[VxTerrainParams] = None) -> np.ndarray:
    """Chunk::generate_terrain (chunk.rs:114-207) on the device: fills the device array at d_voxels (n x 32768 u8) and
    returns the uniform flags (n,) u8."""
    ctx = ctx or default_context()
    positions = np.ascontiguousarray(positions, dtype=np.int32).reshape(-1, 3)
    params = params or terrain_params()
    flags = np.zeros(positions.shape[0], dtype=np.uint8)
    ctx.check(ctx.lib.vx_generate_terrain(ctx.handle, _p(positions), positions.shape[0], C.byref(params), C.c_void_p(d_voxels), _p(flags)))
    return flags


class BinaryGreedyMesher:
    """binary_greedy.rs:50.  Stateless; methods take an optional Context (default: device 0)."""

    @staticmethod
    def mesh_batch(voxels, positions=None, neighbors=None, uniform_flags=None, ctx: Optional[Context] = None,
                   validate: bool = True) -> MeshBatch:
        """Batched form of mesh_world / mesh_chunk_in_indexed_world (binary_greedy.rs:62-168): N x 32768 voxels."""
        ctx = ctx or default_context()
        voxels = np.ascontiguousarray(voxels, dtype=np.uint8).reshape(-1, CHUNK_VOLUME)
        n = voxels.shape[0]
        if validate and voxels.size and int(voxels.max()) > 3:  # a host-side scan of the whole array: skip it for trusted input
            raise VxError(_lib.VX_ERR_INVALID, "voxel values must be BlockType 0..3 (block_type.rs:6-11)")
        positions = None if positions is None else np.ascontiguousarray(positions, dtype=np.int32).reshape(n, 3)
        neighbors = None if neighbors is None else np.ascontiguousarray(neighbors, dtype=np.int32).reshape(n, 6)
        uniform_flags = None if uniform_flags is None else np.ascontiguousarray(uniform_flags, dtype=np.uint8).reshape(n)
        h = C.c_void_p()
        ctx.check(ctx.lib.vx_mesh_chunks(ctx.handle, _p(voxels), _p(positions), _p(neighbors), _p(uniform_flags), n, C.byref(h)))
        return MeshBatch(ctx, h)

    @staticmethod
    def mesh_batch_subset(d_voxels: int, d_positions: int, d_neighbors: int, d_uniform_flags: int, n_chunks: int,
                          d_subset: int, n_subset: int, ctx: Context, batch: Optional[MeshBatch] = None) -> MeshBatch:
        """One rank's share of a chunk-sharded remesh (vx_mesh_chunk_subset_device): device pointers of the replicated
        world arrays + the chunk ids to mesh.  Pass the returned batch back in to re-mesh without allocating."""
        h = batch.handle if batch is not None else C.c_void_p()
        ctx.check(ctx.lib.vx_mesh_chunk_subset_device(ctx.handle, C.c_void_p(d_voxels), C.c_void_p(d_positions or None),
                                                      C.c_void_p(d_neighbors or None), C.c_void_p(d_uniform_flags or None),
                                                      int(n_chunks), C.c_void_p(d_subset), int(n_subset), C.byref(h)))
        if batch is not None:
            batch._host = None
            return batch
        return MeshBatch(ctx, h)

    @staticmethod
    def mesh_chunk(voxels, position=(0, 0, 0), ctx: Optional[Context] = None) -> Optional[ChunkMesh]:
        """binary_greedy.rs:55: no neighbour information, borders are air."""
        b = BinaryGreedyMesher.mesh_batch(np.asarray(voxels).reshape(1, CHUNK_VOLUME), [position], None, None, ctx)
        try:
            return b.chunk_mesh(0, position)
        finally:
            b.release()

    @staticmethod
    def mesh_world(voxels, positions, uniform_flags=None, ctx: Optional[Context] = None):
        """binary_greedy.rs:62-78: meshes in input order, Uniform / empty chunks skipped; neighbours resolved by position."""
        positions = np.ascontiguousarray(positions, dtype=np.int32).reshape(-1, 3)
        index = {tuple(p): i for i, p in enumerate(positions.tolist())}
        offs = [(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]
        nb = np.full((positions.shape[0], 6), -1, dtype=np.int32)
        for i, p in enumerate(positions.tolist()):
            for f, o in enumerate(offs):
                j = index.get((p[0] + o[0], p[1] + o[1], p[2] + o[2]))
                if j is not None:
                    nb[i, f] = j
        b = BinaryGreedyMesher.mesh_batch(voxels, positions, nb, uniform_flags, ctx)
        try:
            b.download()
            return [m for m in (b.chunk_mesh(i, positions[i]) for i in range(positions.shape[0])) if m is not None]
        finally:
            b.release()

    @staticmethod
    def greedy_mesh_slice(mask, ctx: Optional[Context] = None) -> np.ndarray:
        """binary_greedy.rs:675: [u32;32] -> (n,4) u8 quads (x=row, y=col, width, height)."""
        return BinaryGreedyMesher.greedy_mesh_slices(np.asarray(mask).reshape(1, 32), ctx)[0]

    @staticmethod
    def greedy_mesh_slices(masks, ctx: Optional[Context] = None):
        ctx = ctx or default_context()
        masks = np.ascontiguousarray(masks, dtype=np.uint32).reshape(-1, 32)
        n = masks.shape[0]
        out = np.zeros((n, 512, 4), dtype=np.uint8)
        cnt = np.zeros(n, dtype=np.int32)
        ctx.check(ctx.lib.vx_greedy_mesh_slices(ctx.handle, _p(masks), n, _p(out), _p(cnt)))
        return [out[i, :cnt[i]].copy() for i in range(n)]


class Frustum:
    """camera/mod.rs:111-183 evaluated on the device through vx_cull_chunks."""

    def __init__(self, view_projection, ctx: Optional[Context] = None):
        self.vp = np.ascontiguousarray(view_projection, dtype=np.float32).reshape(16)
        self.ctx = ctx or default_context()

    @classmethod
    def from_view_projection(cls, vp, ctx: Optional[Context] = None) -> "Frustum":
        return cls(vp, ctx)


def get_visible_chunks_frustum(positions, camera_position, view_projection, view_distance: int,
                               frustum_culling: bool = True, ctx: Optional[Context] = None) -> np.ndarray:
    """World::get_visible_chunks_frustum (world.rs:118-146) -> (N,) u8 visibility flags."""
    ctx = ctx or default_context()
    positions = np.ascontiguousarray(positions, dtype=np.int32).reshape(-1, 3)
    vp = np.ascontiguousarray(view_projection, dtype=np.float32).reshape(16)
    cam = np.ascontiguousarray(camera_position, dtype=np.float32).reshape(3)
    out = np.zeros(positions.shape[0], dtype=np.uint8)
    ctx.check(ctx.lib.vx_cull_chunks(ctx.handle, _p(positions), positions.shape[0], _p(vp), _p(cam), int(view_distance),
                                     1 if frustum_culling else 0, _p(out)))
    return out


def apply_horizon_culling(camera_position, centers, order=None, bins: int = 128, base_margin: float = 0.1,
                          margin_dist_factor: float = 0.05, min_dist_chunks: float = 2.0, ctx: Optional[Context] = None) -> np.ndarray:
    """culling::apply_horizon_culling (culling.rs:40-119): centers (N,3) VisibleMesh centres, order = candidate ids
    (default: all).  Returns the kept ids, stably sorted front to back."""
    ctx = ctx or default_context()
    centers = np.ascontiguousarray(centers, dtype=np.float32).reshape(-1, 3)
    cam = np.ascontiguousarray(camera_position, dtype=np.float32).reshape(3)
    order = np.arange(centers.shape[0], dtype=np.int32) if order is None else np.ascontiguousarray(order, dtype=np.int32).copy()
    nk = C.c_int32(0)
    ctx.check(ctx.lib.vx_horizon_cull(ctx.handle, _p(cam), _p(centers), centers.shape[0], _p(order), order.shape[0], int(bins),
                                      float(base_margin), float(margin_dist_factor), float(min_dist_chunks), C.byref(nk)))
    return order[:nk.value].copy()


class Framebuffer:
    """framebuffer.rs:197-245: ARGB colour + f32 depth, row-major."""

    def __init__(self, width: int, height: int):
        self.width = int(width)
        self.height = int(height)
        self.color_buffer = np.zeros((self.height, self.width), dtype=np.uint32)
        self.depth_buffer = np.full((self.height, self.width), np.inf, dtype=np.float32)

    def clear(self, clear_color: int):  # framebuffer.rs:219
        self.color_buffer[...] = np.uint32(clear_color)
        self.depth_buffer[...] = np.inf

    def fill_spans(self, y, x_start, x_end, depth, color, ctx: Optional[Context] = None):
        """FrameSlice::fill_span (span_walker.rs:412-441) for n spans in order: pixels [x_start, x_end) of row y, depth test `<`."""
        ctx = ctx or default_context()
        ya, xs, xe = (np.ascontiguousarray(a, dtype=np.int32).ravel() for a in (y, x_start, x_end))
        d = np.ascontiguousarray(depth, dtype=np.float32).ravel()
        c = np.ascontiguousarray(color, dtype=np.uint32).ravel()
        if not (ya.size == xs.size == xe.size == d.size == c.size):
            raise ValueError("fill_spans: arrays of different length")
        ctx.check(ctx.lib.vx_fill_spans(ctx.handle, _p(ya), _p(xs), _p(xe), _p(d), _p(c), int(ya.size), self.width, self.height,
                                        _p(self.color_buffer), _p(self.depth_buffer)))

    def fill_span(self, y: int, x_start: int, x_end: int, depth: float, color: int, ctx: Optional[Context] = None):
        self.fill_spans([y], [x_start], [x_end], [depth], [color], ctx)


class SpanWalkerRasterizer:
    """span_walker.rs:97-396: flat-colour rasterizer of projected axis-aligned quads (the Hyper-Pipeline's last stage)."""

    BLOCK_COLORS = (0x00000000, 0x00FF00FF, 0x8B4513FF, 0x808080FF)  # get_block_color :386-396

    def __init__(self, viewport_width: int, viewport_height: int, ctx: Optional[Context] = None):
        self.viewport_width = int(viewport_width)
        self.viewport_height = int(viewport_height)
        self.ctx = ctx or default_context()

    def rasterize_projected_packet(self, x_min, y_min, x_max, y_max, depth_near, block_type, framebuffer: Framebuffer, visible=None):
        """rasterize_projected_packet :116 for n quads (any number of ProjectedPackets concatenated; `visible` = the bits
        of their visibility masks, None = all).  The framebuffer must have the walker's viewport size."""
        if (framebuffer.width, framebuffer.height) != (self.viewport_width, self.viewport_height):
            raise ValueError("framebuffer and viewport sizes differ")
        f = [np.ascontiguousarray(a, dtype=np.float32).ravel() for a in (x_min, y_min, x_max, y_max, depth_near)]
        bt = np.ascontiguousarray(block_type, dtype=np.uint8).ravel()
        vis = None if visible is None else np.ascontiguousarray(visible, dtype=np.uint8).ravel()
        n = int(bt.size)
        if any(a.size != n for a in f) or (vis is not None and vis.size != n):
            raise ValueError("rasterize_projected_packet: arrays of different length")
        self.ctx.check(self.ctx.lib.vx_span_walk_quads(self.ctx.handle, _p(f[0]), _p(f[1]), _p(f[2]), _p(f[3]), _p(f[4]), _p(bt), _p(vis), n,
                                                       framebuffer.width, framebuffer.height, _p(framebuffer.color_buffer),
                                                       _p(framebuffer.depth_buffer)))


class ShadingConfig:
    """ShadingConfig (shading.rs:21-31): face lighting = clamp(ambient + diffuse * max(normal . light_dir, 0), 0, 1).
    The defaults are ShadingConfig::default, the same values vx_default_frame_config writes."""

    def __init__(self, light_dir=None, ambient: Optional[float] = None, diffuse: Optional[float] = None):
        d = default_frame_config(1, 1)
        self.light_dir = tuple(float(x) for x in (d.light_dir if light_dir is None else light_dir))
        self.ambient = float(d.ambient if ambient is None else ambient)
        self.diffuse = float(d.diffuse if diffuse is None else diffuse)

    def apply(self, cfg: VxFrameConfig) -> VxFrameConfig:
        cfg.light_dir[0], cfg.light_dir[1], cfg.light_dir[2] = self.light_dir
        cfg.ambient, cfg.diffuse = self.ambient, self.diffuse
        return cfg


class Rasterizer:
    """rasterizer.rs:335-431.  pub fields: backface_culling, shading, enable_shading, atlas.

    Each Rasterizer draws with its own atlas (None: the default atlas, as Rasterizer::new); several of them may share a
    context.  The context holds one atlas at a time, so a draw loads this Rasterizer's atlas first when the context
    holds another one (vx_set_atlas; the next frame then rebuilds the colour table)."""

    def __init__(self, ctx: Optional[Context] = None, atlas: Optional[VxAtlas] = None):
        self.ctx = ctx or default_context()
        self.backface_culling = True
        self.shading = ShadingConfig()
        self.enable_shading = True
        self.atlas = atlas  # new_with_atlas rasterizer.rs:357
        self.differential_projection = False

    def _cfg(self, w, h) -> VxFrameConfig:
        cfg = self.shading.apply(default_frame_config(w, h))
        cfg.backface_culling = 1 if self.backface_culling else 0
        cfg.enable_shading = 1 if self.enable_shading else 0
        cfg.differential_projection = 1 if self.differential_projection else 0
        atlas = self.atlas if self.atlas is not None else _default_atlas_cached()
        if not self.ctx.holds_atlas(atlas):
            self.ctx.set_atlas(atlas)
        return cfg

    def _render(self, batch: MeshBatch, mesh_id: int, view_proj, fb: Framebuffer, rect):
        vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
        rect = np.ascontiguousarray(rect, dtype=np.int32)
        cfg = self._cfg(fb.width, fb.height)
        self.ctx.check(self.ctx.lib.vx_render_mesh(self.ctx.handle, batch.handle, int(mesh_id), _p(vp), C.byref(cfg), _p(rect),
                                                   _p(fb.color_buffer), _p(fb.depth_buffer)))

    def render_mesh(self, batch: MeshBatch, mesh_id: int, view_proj, framebuffer: Framebuffer):
        """rasterizer.rs:385: whole framebuffer (one stripe)."""
        self._render(batch, mesh_id, view_proj, framebuffer, (0, 0, framebuffer.width, framebuffer.height))

    def render_mesh_into_slice(self, batch: MeshBatch, mesh_id: int, view_proj, framebuffer: Framebuffer, y0: int, rows: int):
        """rasterizer.rs:413: FrameSlice = rows [y0, y0+rows) of the framebuffer."""
        self._render(batch, mesh_id, view_proj, framebuffer, (0, y0, framebuffer.width, rows))

    def render_mesh_into_tile(self, batch: MeshBatch, mesh_id: int, view_proj, framebuffer: Framebuffer, x0, y0, tw, th):
        """rasterizer.rs:423: FrameTile rectangle."""
        self._render(batch, mesh_id, view_proj, framebuffer, (x0, y0, tw, th))

    def render_mesh_with_up(self, batch: MeshBatch, mesh_id: int, view_proj, framebuffer: Framebuffer, camera_up):
        """rasterizer.rs:399: whole framebuffer; span renderer iff the camera is level (|up.y| >= 0.995), else barycentric."""
        vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
        up = np.ascontiguousarray(camera_up, dtype=np.float32).reshape(3)
        cfg = self._cfg(framebuffer.width, framebuffer.height)
        self.ctx.check(self.ctx.lib.vx_render_mesh_with_up(self.ctx.handle, batch.handle, int(mesh_id), _p(vp), C.byref(cfg), _p(up),
                                                           _p(framebuffer.color_buffer), _p(framebuffer.depth_buffer)))

    def render_mesh_tiny_quads(self, batch: MeshBatch, mesh_id: int, view_proj, framebuffer: Framebuffer, rect, use_span_renderer: bool):
        """rasterizer.rs:782: target = rect (x0, y0, w, h) of the framebuffer; use_span_renderer False = barycentric path."""
        vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
        rect = np.ascontiguousarray(rect, dtype=np.int32).reshape(4)
        cfg = self._cfg(framebuffer.width, framebuffer.height)
        self.ctx.check(self.ctx.lib.vx_render_mesh_tiny_quads(self.ctx.handle, batch.handle, int(mesh_id), _p(vp), C.byref(cfg), _p(rect),
                                                              1 if use_span_renderer else 0, _p(framebuffer.color_buffer),
                                                              _p(framebuffer.depth_buffer)))


def render_frame(batch: MeshBatch, view_proj, camera_position, cfg: VxFrameConfig, mesh_ids=None, view_distance: int = 0,
                 color_out=None, depth_out=None, want_depth: bool = True, ctx: Optional[Context] = None, survivors_out=None):
    """main.rs:379-608 (+ :283-297, :368-377).  Returns (color (rows,W) u32, depth (rows,W) f32 or None, survivors i32).
    color_out / depth_out allocated with Context.host_array (device-mapped page-locked memory) are written by the
    raster kernel in place; ordinary arrays are filled by a device-to-host copy."""
    ctx = ctx or batch.ctx
    vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
    cam = np.ascontiguousarray(camera_position, dtype=np.float32).reshape(3)
    rows = cfg.stripe_rows if cfg.stripe_rows > 0 else cfg.height
    if color_out is None:
        color_out = np.empty((rows, cfg.width), dtype=np.uint32)
    if depth_out is None and want_depth:
        depth_out = np.empty((rows, cfg.width), dtype=np.float32)
    if mesh_ids is not None:
        mesh_ids = np.ascontiguousarray(mesh_ids, dtype=np.int32)
        n = int(mesh_ids.shape[0])
        cap = max(1, n)
    else:
        n = -1
        if batch._n_chunks is None:
            batch._n_chunks = int(batch.info().n_chunks)
        cap = max(1, batch._n_chunks)
    surv = survivors_out if survivors_out is not None else np.empty(cap, dtype=np.int32)
    ns = C.c_int32(0)
    ctx.check(ctx.lib.vx_render_frame(ctx.handle, batch.handle, _p(mesh_ids), n, _p(vp), _p(cam), int(view_distance), C.byref(cfg),
                                      _p(color_out), _p(depth_out), _p(surv), C.byref(ns)))
    return color_out, depth_out, (surv[:ns.value] if survivors_out is not None else surv[:ns.value].copy())


# ---- picking (vx_world_raycast) ------------------------------------------------------------------------------------

RAY_HIT_DTYPE = np.dtype([("status", "<i4"), ("slot", "<i4"), ("voxel", "<i4", (3,)), ("face", "<i4"), ("t", "<f4"),
                          ("block_type", "u1"), ("pad", "u1", (3,))])  # VxRayHit, 32 bytes
assert RAY_HIT_DTYPE.itemsize == C.sizeof(_lib.VxRayHit)

# ---- region edits (vx_world_batch_fill_regions) ---------------------------------------------------------------------

REGION_OP_DTYPE = np.dtype([("radius_sq", "<i8"), ("shape", "<i4"), ("a", "<i4", (3,)), ("b", "<i4", (3,)), ("block_type", "u1"),
                            ("replace_mask", "u1"), ("pad", "u1", (2,))])  # VxRegionOp, 40 bytes
assert REGION_OP_DTYPE.itemsize == C.sizeof(_lib.VxRegionOp)

# ---- copy and paste (vx_world_batch_copy_region, vx_world_batch_paste) ------------------------------------------------

PASTE_SKIP = _lib.PASTE_SKIP
PASTE_OP_DTYPE = np.dtype([("offset", "<i8"), ("origin", "<i4", (3,)), ("dims", "<i4", (3,)), ("replace_mask", "u1"),
                           ("pad", "u1", (7,))])  # VxPasteOp, 40 bytes
assert PASTE_OP_DTYPE.itemsize == C.sizeof(_lib.VxPasteOp)


def pixel_rays(view_proj, camera_position, pixels, width: int, height: int):
    """Rays from the camera through pixel centres, for vx_world_raycast: origin = camera_position, direction = the pixel
    centre (the rasterizer's convention: ndc.x = (px + 0.5) / W * 2 - 1, ndc.y = 1 - (py + 0.5) / H * 2) unprojected at the
    far plane (ndc.z = 1) through the inverse view-projection, in float64, normalised, then rounded to f32.
    pixels: (n, 2) (px, py).  Returns (origins (n, 3) f32, dirs (n, 3) f32)."""
    m = np.asarray(view_proj, dtype=np.float32).reshape(4, 4).T.astype(np.float64)  # column-major -> row-major
    px = np.asarray(pixels, dtype=np.float64).reshape(-1, 2)
    n = px.shape[0]
    ndc = np.empty((n, 4), dtype=np.float64)
    ndc[:, 0] = (px[:, 0] + 0.5) / width * 2.0 - 1.0
    ndc[:, 1] = 1.0 - (px[:, 1] + 0.5) / height * 2.0
    ndc[:, 2] = 1.0
    ndc[:, 3] = 1.0
    far = ndc @ np.linalg.inv(m).T
    cam = np.asarray(camera_position, dtype=np.float32).reshape(3)
    d = far[:, :3] / far[:, 3:4] - cam.astype(np.float64)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.repeat(cam.reshape(1, 3), n, axis=0), d.astype(np.float32)


def hyper_pipeline_render(batch: MeshBatch, mesh_ids, view_proj, framebuffer: Framebuffer, ctx: Optional[Context] = None) -> int:
    """The Hyper-Pipeline for a list of meshes (vx_hyper_pipeline_render): face packets -> PacketPipeline
    (packet_pipeline.rs:69-142) -> span walker, into `framebuffer` (read-modify-write).  Returns the quads that passed the
    packet backface test and the frustum mask."""
    ctx = ctx or batch.ctx
    vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
    ids = np.ascontiguousarray(mesh_ids, dtype=np.int32).ravel()
    n = C.c_int32(0)
    ctx.check(ctx.lib.vx_hyper_pipeline_render(ctx.handle, batch.handle, _p(ids), int(ids.size), _p(vp), framebuffer.width, framebuffer.height,
                                               _p(framebuffer.color_buffer), _p(framebuffer.depth_buffer), C.byref(n)))
    return int(n.value)


def render_frame_macrotile(batch: MeshBatch, mesh_ids, view_proj, cfg: VxFrameConfig, want_tile_depth: bool = True,
                           ctx: Optional[Context] = None):
    """render_frame_macrotile (macrotile_renderer.rs:51-170).  Returns (color (H,W) u32, tile depth (H,W) f32 or None --
    the reference drops it --, projected mesh ids in draw order: list order, large primitives last)."""
    ctx = ctx or batch.ctx
    vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
    ids = np.ascontiguousarray(mesh_ids, dtype=np.int32).ravel()
    color = np.empty((cfg.height, cfg.width), dtype=np.uint32)
    depth = np.empty((cfg.height, cfg.width), dtype=np.float32) if want_tile_depth else None
    proj = np.empty(max(1, ids.size), dtype=np.int32)
    n = C.c_int32(0)
    ctx.check(ctx.lib.vx_render_frame_macrotile(ctx.handle, batch.handle, _p(ids), int(ids.size), _p(vp), C.byref(cfg), _p(color), _p(depth),
                                                _p(proj), C.byref(n)))
    return color, depth, proj[:n.value].copy()


class FrameLoop:
    """The state main.rs keeps across iterations of its frame loop -- framebuffer, depth buffer, draw list
    (main.rs:283-297, :379-608) -- bound once, so a frame costs one C-ABI call (vx_render_frame) and nothing else:
    the ARGB frame (and depth, if asked for) lands in device-mapped page-locked host arrays written by the raster
    kernel in place.  render() returns views of those arrays, valid until the next render()."""

    def __init__(self, batch: MeshBatch, cfg: VxFrameConfig, view_distance: int = 0, want_depth: bool = False,
                 ctx: Optional[Context] = None, lanes: int = 1):
        self.ctx = ctx or batch.ctx
        self.batch = batch
        self.cfg = cfg
        self.lanes = FrameLanes(self.ctx.device, lanes, first=self.ctx)  # submit() deals frames over these
        rows = cfg.stripe_rows if cfg.stripe_rows > 0 else cfg.height
        self.color = self.ctx.host_array((rows, cfg.width), np.uint32)
        self.depth = self.ctx.host_array((rows, cfg.width), np.float32) if want_depth else None
        if batch._n_chunks is None:
            batch._n_chunks = int(batch.info().n_chunks)
        self.survivors = np.empty(max(1, batch._n_chunks), dtype=np.int32)
        self._vp = np.zeros(16, dtype=np.float32)
        self._cam = np.zeros(3, dtype=np.float32)
        self._ns = C.c_int32(0)
        self._fn = self.ctx.lib.vx_render_frame
        self._args = (self.ctx.handle, batch.handle, None, -1, self._vp.ctypes.data, self._cam.ctypes.data, int(view_distance),
                      C.byref(cfg), self.color.ctypes.data, self.depth.ctypes.data if want_depth else None,
                      self.survivors.ctypes.data, C.byref(self._ns))

    def render(self, view_proj, camera_position):
        """One frame: returns (color, depth or None, survivors) like render_frame."""
        self._vp[:] = np.asarray(view_proj, dtype=np.float32).reshape(16)
        self._cam[:] = camera_position
        rc = self._fn(*self._args)
        if rc != 0:
            self.ctx.check(rc)
        return self.color, self.depth, self.survivors[:self._ns.value]

    # ---- pipelined use (vx_render_frame_begin / _end): frame k + 1 is enqueued before the host waits for frame k, the
    #      way main.rs:320-336 presents one frame while the next loop iteration is already running -------------------------
    def _buffer_sets(self):
        """Two (colour, depth, survivors) sets per lane: a lane may have two frames in flight."""
        if getattr(self, "_sets", None) is None:
            rows = self.color.shape[0]
            self._sets = []
            for li, lane in enumerate(self.lanes.ctxs):
                pair = []
                for j in range(2):
                    if li == 0 and j == 0:
                        pair.append((self.color, self.depth, self.survivors))
                    else:
                        pair.append((lane.host_array((rows, self.cfg.width), np.uint32),
                                     lane.host_array((rows, self.cfg.width), np.float32) if self.depth is not None else None,
                                     np.empty_like(self.survivors)))
                self._sets.append(pair)
            self._ticket = C.c_int32(0)
            self._n_submitted = 0
            self._pending = {}  # ticket -> (lane index, the lane's own ticket, buffer set)
        return self._sets

    @property
    def max_in_flight(self) -> int:
        return 2 * len(self.lanes)

    def submit(self, view_proj, camera_position) -> int:
        """Enqueue one frame without waiting for it; returns its ticket.  Frames go to the lanes round-robin, each lane
        takes two, so at most 2 * lanes frames may be in flight (wait() for the oldest before submitting more)."""
        sets = self._buffer_sets()
        self._vp[:] = np.asarray(view_proj, dtype=np.float32).reshape(16)
        self._cam[:] = camera_position
        a = self._args
        k = self._n_submitted
        if len(self.lanes) > 1:  # tell the library that this frame shares the GPU (coarser raster work items); cfg may have changed
            if getattr(self, "_cfg_lanes", None) is None:
                self._cfg_lanes = VxFrameConfig()
            C.memmove(C.byref(self._cfg_lanes), C.byref(self.cfg), C.sizeof(VxFrameConfig))
            self._cfg_lanes.frames_in_flight = len(self.lanes)
            a = a[:7] + (C.byref(self._cfg_lanes),) + a[8:]
        li = k % len(self.lanes)
        lane = self.lanes[li]
        j = (k // len(self.lanes)) & 1
        color, depth, _ = sets[li][j]
        rc = lane.lib.vx_render_frame_begin(lane.handle, a[1], None, -1, a[4], a[5], a[6], a[7], color.ctypes.data,
                                            depth.ctypes.data if depth is not None else None, C.byref(self._ticket))
        if rc != 0:
            lane.check(rc)
        self._n_submitted = k + 1
        self._pending[k] = (li, int(self._ticket.value), j)
        return k

    def wait(self, ticket: int):
        """Block until the frame `ticket` is complete in host memory: returns (color, depth or None, survivors) -- views
        that stay valid until 2 * lanes more frames have been submitted."""
        sets = self._buffer_sets()
        if ticket not in self._pending:
            raise VxError(-1, "FrameLoop.wait: unknown ticket")
        li, lane_ticket, j = self._pending.pop(ticket)
        lane = self.lanes[li]
        color, depth, surv = sets[li][j]
        rc = lane.lib.vx_render_frame_end(lane.handle, lane_ticket, surv.ctypes.data, C.byref(self._ns))
        if rc != 0:
            lane.check(rc)
        return color, depth, surv[:self._ns.value]

    def close(self):
        self.lanes.close()


def render_frame_device(batch: MeshBatch, view_proj, camera_position, cfg: VxFrameConfig, view_distance: int,
                        ctx: Optional[Context] = None):
    """Device-resident frame: filter A on the device over the batch's chunks, nothing copied back."""
    ctx = ctx or batch.ctx
    st = getattr(ctx, "_rfd_state", None)
    if st is None:  # the argument buffers are kept per context: the host side of a frame has to stay at a few microseconds
        vp_a, cam_a = np.zeros(16, dtype=np.float32), np.zeros(3, dtype=np.float32)
        st = ctx._rfd_state = [vp_a, cam_a, _p(vp_a), _p(cam_a), ctx.lib.vx_render_frame_device, None, None]
    if view_proj is not st[5] or camera_position is not st[6]:
        st[0][:] = np.asarray(view_proj, dtype=np.float32).reshape(16)
        st[1][:] = camera_position
        # immutable inputs (tuples) are recognised by identity next time; arrays may be changed in place by the caller
        st[5] = view_proj if isinstance(view_proj, tuple) else None
        st[6] = camera_position if isinstance(camera_position, tuple) else None
    rc = st[4](ctx.handle, batch.handle, None, -1, st[2], st[3], int(view_distance), C.byref(cfg))
    if rc != 0:
        ctx.check(rc)


def render_frame_into(batch: MeshBatch, view_proj, camera_position, cfg: VxFrameConfig, view_distance: int, d_color: int,
                      d_depth: int = 0, ctx: Optional[Context] = None):
    """vx_render_frame_into: like render_frame_device, the frame goes to the given device-addressable pointers."""
    ctx = ctx or batch.ctx
    vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
    cam = np.ascontiguousarray(camera_position, dtype=np.float32).reshape(3)
    ctx.check(ctx.lib.vx_render_frame_into(ctx.handle, batch.handle, None, -1, _p(vp), _p(cam), int(view_distance), C.byref(cfg),
                                           C.c_void_p(d_color or None), C.c_void_p(d_depth or None)))


def frame_stats(ctx: Context) -> VxFrameStats:
    st = VxFrameStats()
    ctx.check(ctx.lib.vx_frame_stats(ctx.handle, C.byref(st)))
    return st


def frame_kernel_times(ctx: Context) -> np.ndarray:
    """ms of [cull+sort, setup, bin fill, raster] for the last frame rendered with cfg.profile_kernels = 1."""
    out = np.zeros(4, dtype=np.float32)
    ctx.check(ctx.lib.vx_frame_kernel_times(ctx.handle, _p(out)))
    return out


def frame_bin_counts(ctx: Context) -> np.ndarray:
    """(nty, ntx) triangles binned per 128x8 tile in the last frame."""
    out = np.zeros(1 << 16, dtype=np.uint32)
    ntx, nty = C.c_int32(), C.c_int32()
    ctx.check(ctx.lib.vx_frame_bin_counts(ctx.handle, _p(out), out.size, C.byref(ntx), C.byref(nty)))
    return out[:ntx.value * nty.value].reshape(nty.value, ntx.value).copy()


def frame_bin_tasks(ctx: Context) -> np.ndarray:
    """(nty, ntx) (row, 16-pixel column block) tasks per 128x8 tile in the last frame: with frame_bin_counts the cost model
    of the work-balanced stripe split (sharding.stripe_band_cost)."""
    out = np.zeros(1 << 16, dtype=np.uint32)
    ntx, nty = C.c_int32(), C.c_int32()
    ctx.check(ctx.lib.vx_frame_bin_tasks(ctx.handle, _p(out), out.size, C.byref(ntx), C.byref(nty)))
    return out[:ntx.value * nty.value].reshape(nty.value, ntx.value).copy()


def framebuffer_device(ctx: Context):
    dc, dd, rows, width = C.c_void_p(), C.c_void_p(), C.c_int32(), C.c_int32()
    ctx.check(ctx.lib.vx_framebuffer_device(ctx.handle, C.byref(dc), C.byref(dd), C.byref(rows), C.byref(width)))
    return dc.value, dd.value, rows.value, width.value


def face_packets(batch: MeshBatch, mesh_id: int, ctx: Optional[Context] = None):
    """ChunkFacePackets::from_chunk_mesh (face_packets.rs:122-174): list of 6 lists of dicts with the SoA arrays of each
    FacePacket32 (len, u_min, v_min, u_len, v_len, axis_pos, block_type as u8 arrays of 32)."""
    ctx = ctx or batch.ctx
    per_face = (C.c_int32 * 6)()
    h = batch._host or batch.download()
    cap = max(1, (int(h["quad_count"][mesh_id]) + 31) // 32 + 6)
    arr = (_lib.VxFacePacket32 * cap)()
    ctx.check(ctx.lib.vx_face_packets(ctx.handle, batch.handle, int(mesh_id), arr, cap, per_face))
    out, k = [], 0
    for f in range(6):
        lst = []
        for _ in range(per_face[f]):
            pk = arr[k]
            lst.append({"len": int(pk.len), **{name: np.ctypeslib.as_array(getattr(pk, name)).copy()
                                               for name in ("u_min", "v_min", "u_len", "v_len", "axis_pos", "block_type")}})
            k += 1
        out.append(lst)
    return out


class FaceBasis:
    """differential_projection.rs:18-82: origin, tangent, bitangent, normal in clip space."""

    def __init__(self, m: np.ndarray):
        self.origin, self.tangent, self.bitangent, self.normal = m[0], m[1], m[2], m[3]
        self.matrix = m

    @classmethod
    def from_face_direction(cls, face_dir: int, chunk_pos, slice_idx: int, view_proj, ctx: Optional[Context] = None) -> "FaceBasis":
        return face_bases([face_dir], [chunk_pos], [slice_idx], view_proj, ctx)[0]

    def is_front_facing(self) -> bool:  # differential_projection.rs:78-82
        return bool(self.normal[2] < 0.0)

    def project_packet_bounds(self, u_min, v_min, u_len, v_len, ctx: Optional[Context] = None):
        """project_packet_bounds_simd / project_single_scalar (:92-196) -> x_min, y_min, x_max, y_max, depth_near (NDC)."""
        ctx = ctx or default_context()
        arrs = [np.ascontiguousarray(a, dtype=np.uint8) for a in (u_min, v_min, u_len, v_len)]
        n = int(arrs[0].shape[0])
        outs = [np.zeros(n, dtype=np.float32) for _ in range(5)]
        basis = np.ascontiguousarray(self.matrix, dtype=np.float32)
        ctx.check(ctx.lib.vx_project_packet(ctx.handle, _p(basis), *[_p(a) for a in arrs], n, *[_p(o) for o in outs]))
        return outs


def face_bases(faces: Sequence[int], chunk_pos, slice_idx, view_proj, ctx: Optional[Context] = None):
    ctx = ctx or default_context()
    faces = np.ascontiguousarray(faces, dtype=np.int32)
    n = int(faces.shape[0])
    cp = np.ascontiguousarray(chunk_pos, dtype=np.int32).reshape(n, 3)
    sl = np.ascontiguousarray(slice_idx, dtype=np.uint8).reshape(n)
    vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
    out = np.zeros((n, 4, 4), dtype=np.float32)
    ctx.check(ctx.lib.vx_face_basis(ctx.handle, _p(faces), _p(cp), _p(sl), n, _p(vp), _p(out)))
    return [FaceBasis(out[i]) for i in range(n)]


def decompress_and_transform_vertices(vertices, chunk_offset, view_proj, ctx: Optional[Context] = None) -> np.ndarray:
    """simd_vertex.rs:24: (n,8) u8 Vertex records -> (n,4) clip-space f32."""
    ctx = ctx or default_context()
    v = np.ascontiguousarray(vertices, dtype=np.uint8).reshape(-1, 8)
    off = np.ascontiguousarray(chunk_offset, dtype=np.float32).reshape(3)
    vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
    out = np.zeros((v.shape[0], 4), dtype=np.float32)
    ctx.check(ctx.lib.vx_transform_vertices(ctx.handle, _p(v), v.shape[0], _p(off), _p(vp), _p(out)))
    return out


def project_mesh_vertices(batch: MeshBatch, mesh_id: int, view_proj, differential: bool, ctx: Optional[Context] = None) -> np.ndarray:
    """Clip-space corners (n_quads,4,4) of a mesh's quads as the raster setup computes them (rasterizer.rs:1092-1185)."""
    ctx = ctx or batch.ctx
    h = batch._host or batch.download()
    n = int(h["quad_count"][mesh_id])
    out = np.zeros((max(n, 1), 4, 4), dtype=np.float32)
    vp = np.ascontiguousarray(view_proj, dtype=np.float32).reshape(16)
    ctx.check(ctx.lib.vx_project_mesh_vertices(ctx.handle, batch.handle, int(mesh_id), _p(vp), 1 if differential else 0, _p(out), C.c_int64(max(n, 1))))
    return out[:n]
