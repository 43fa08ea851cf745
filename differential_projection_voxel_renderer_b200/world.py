"""Host mirror of the reference's streaming world and of the mesh cache its frame loop keeps.

`World` / `WorldConfig` follow /root/reference/src/world.rs:8-215 (same names, same update order, same per-frame
generation cap and unload hysteresis); `MeshCache` follows the chunk-to-mesh bookkeeping of the frame loop,
/root/reference/src/main.rs:216-297.  The voxels, the neighbour table and the meshes live on the device in a world
batch (vx_world_batch_*, include/vx_b200.h): the host only decides which lattice position occupies which slot.
Nothing here generates, meshes or draws on the CPU.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Iterable, List, Optional, Tuple

import numpy as np

from . import _lib, api
from ._lib import VxTerrainParams

Pos = Tuple[int, int, int]
CHUNK_SIZE = 32
FACE_OFFSETS = ((1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1))  # FaceDir order, mesh.rs:136-143
NBR_NONE = -1


class WorldConfig:
    """world.rs:8-27."""

    def __init__(self, view_distance: int = 8, frustum_culling: bool = True, max_chunks_per_frame: int = 4):
        self.view_distance = int(view_distance)
        self.frustum_culling = bool(frustum_culling)
        self.max_chunks_per_frame = int(max_chunks_per_frame)


def world_to_chunk_pos(world_pos) -> Pos:
    """world.rs:201-207: (world_pos / CHUNK_SIZE as f32).floor() as i32, component-wise in f32."""
    p = np.asarray(world_pos, dtype=np.float32)
    c = np.floor(p / np.float32(CHUNK_SIZE))
    return int(c[0]), int(c[1]), int(c[2])


def sphere_capacity(view_distance: int) -> int:
    """Lattice points within the unload radius view_distance + 2 (world.rs:91): the most chunks the world can hold."""
    r = view_distance + 2
    g = np.arange(-r, r + 1)
    x, y, z = np.meshgrid(g, g, g, indexing="ij")
    return int(((x * x + y * y + z * z) <= r * r).sum())


class _DeviceWorld:
    """The vx_world_batch_* calls and vx_world_raycast; tests substitute a recorder for it to check the host logic without a
    GPU."""

    def __init__(self, ctx: api.Context, capacity: int, terrain: VxTerrainParams):
        self.ctx = ctx
        self.terrain = terrain
        h = C.c_void_p()
        ctx.check(ctx.lib.vx_world_batch_create(ctx.handle, int(capacity), C.byref(h)))
        self.batch = api.MeshBatch(ctx, h)
        self.batch._n_chunks = int(capacity)

    def generate(self, slots: np.ndarray, positions: np.ndarray) -> np.ndarray:
        flags = np.zeros(slots.size, dtype=np.uint8)
        self.ctx.check(self.ctx.lib.vx_world_batch_generate(self.ctx.handle, self.batch.handle, api._p(slots), int(slots.size),
                                                            api._p(positions), C.byref(self.terrain), api._p(flags)))
        return flags

    def assign(self, slots: np.ndarray, neighbors: np.ndarray):
        self.ctx.check(self.ctx.lib.vx_world_batch_assign(self.ctx.handle, self.batch.handle, api._p(slots), int(slots.size), None,
                                                          api._p(neighbors)))

    def grow(self, capacity: int):
        self.ctx.check(self.ctx.lib.vx_world_batch_grow(self.ctx.handle, self.batch.handle, int(capacity)))
        self.batch._n_chunks = int(capacity)
        self.batch._host = None

    def unload(self, slots: np.ndarray):
        self.ctx.check(self.ctx.lib.vx_world_batch_unload(self.ctx.handle, self.batch.handle, api._p(slots), int(slots.size)))

    def remesh(self, slots: np.ndarray):
        self.ctx.check(self.ctx.lib.vx_world_batch_remesh(self.ctx.handle, self.batch.handle, api._p(slots), int(slots.size)))

    def set_blocks(self, slots: np.ndarray, voxel_index: np.ndarray, block_types: np.ndarray):
        self.ctx.check(self.ctx.lib.vx_world_batch_set_blocks(self.ctx.handle, self.batch.handle, api._p(slots), api._p(voxel_index),
                                                              api._p(block_types), int(slots.size)))

    def raycast(self, origins: np.ndarray, dirs: np.ndarray, start_slots: np.ndarray, max_t: float) -> np.ndarray:
        hits = np.zeros(start_slots.size, dtype=api.RAY_HIT_DTYPE)
        self.ctx.check(self.ctx.lib.vx_world_raycast(self.ctx.handle, self.batch.handle, api._p(origins), api._p(dirs), api._p(start_slots),
                                                     int(start_slots.size), float(max_t), api._p(hits)))
        return hits


class World:
    """world.rs:30-215 with device-resident chunks: `chunks` maps a lattice position to its slot in the world batch."""

    def __init__(self, config: Optional[WorldConfig] = None, ctx: Optional[api.Context] = None, capacity: Optional[int] = None,
                 terrain: Optional[VxTerrainParams] = None, device=None):
        self.config = config or WorldConfig()
        self.capacity = int(capacity) if capacity is not None else sphere_capacity(self.config.view_distance)
        self.device = device if device is not None else _DeviceWorld(ctx or api.default_context(), self.capacity,
                                                                     terrain or api.terrain_params())
        self.chunks: Dict[Pos, int] = {}
        self.uniform_flags: Dict[Pos, int] = {}   # 0 Varied, 1 + block type Uniform (chunk.rs:127-134)
        # block edits by chunk position: voxel index (z*1024 + y*32 + x) -> block type; kept while the chunk is unloaded and
        # applied again when it is generated anew
        self.edits: Dict[Pos, Dict[int, int]] = {}
        self._free: List[int] = list(range(self.capacity - 1, -1, -1))
        self.last_camera_chunk: Optional[Pos] = None
        self.generated_last_update: List[Pos] = []
        self.unloaded_last_update: List[Pos] = []

    # ---- bookkeeping ---------------------------------------------------------------------------------------------
    @property
    def batch(self) -> api.MeshBatch:
        return self.device.batch

    def contains_chunk(self, pos: Pos) -> bool:  # world.rs:171-173
        return tuple(pos) in self.chunks

    def chunk_count(self) -> int:  # world.rs:166-168
        return len(self.chunks)

    def get_all_chunks(self) -> List[Pos]:  # world.rs:176-178, in (x, y, z) order (the reference's HashMap order is arbitrary)
        return sorted(self.chunks)

    def _neighbor_row(self, pos: Pos) -> List[int]:
        return [self.chunks.get((pos[0] + o[0], pos[1] + o[1], pos[2] + o[2]), NBR_NONE) for o in FACE_OFFSETS]

    def _push_neighbor_rows(self, positions: Iterable[Pos]):
        todo = sorted(set(p for p in positions if p in self.chunks))
        if not todo:
            return
        slots = np.array([self.chunks[p] for p in todo], dtype=np.int32)
        rows = np.array([self._neighbor_row(p) for p in todo], dtype=np.int32).reshape(-1, 6)
        self.device.assign(slots, rows)

    # ---- World::update world.rs:57-100 ------------------------------------------------------------------------------
    def update(self, camera_position) -> bool:
        """Generate the missing chunks inside the view sphere in the reference's scan order (x, then y, then z), at most
        max_chunks_per_frame of them -- hitting the cap returns before the unload step, exactly like the reference --
        then unload everything beyond view_distance + 2.  Returns True if chunks were generated."""
        camera_chunk = world_to_chunk_pos(camera_position)
        self.last_camera_chunk = camera_chunk
        vd = self.config.view_distance
        vd_sq = np.float32(vd * vd)
        new: List[Pos] = []
        hit_cap = False
        for cx in range(camera_chunk[0] - vd, camera_chunk[0] + vd + 1):
            for cy in range(camera_chunk[1] - vd, camera_chunk[1] + vd + 1):
                for cz in range(camera_chunk[2] - vd, camera_chunk[2] + vd + 1):
                    dx, dy, dz = cx - camera_chunk[0], cy - camera_chunk[1], cz - camera_chunk[2]
                    if np.float32(dx * dx + dy * dy + dz * dz) > vd_sq:
                        continue
                    pos = (cx, cy, cz)
                    if pos not in self.chunks and pos not in new:
                        new.append(pos)
                        if len(new) >= self.config.max_chunks_per_frame:
                            hit_cap = True
                            break
                if hit_cap:
                    break
            if hit_cap:
                break
        self._load(new)
        self.generated_last_update = new
        self.unloaded_last_update = []
        if hit_cap:
            return True
        unload_sq = np.float32((vd + 2) * (vd + 2))
        gone = [p for p in self.chunks
                if np.float32((p[0] - camera_chunk[0]) ** 2 + (p[1] - camera_chunk[1]) ** 2 + (p[2] - camera_chunk[2]) ** 2) > unload_sq]
        self._unload(sorted(gone))
        self.unloaded_last_update = sorted(gone)
        return len(new) > 0

    def get_or_generate_chunk(self, pos: Pos) -> int:  # world.rs:49-53
        pos = tuple(pos)
        if pos not in self.chunks:
            self._load([pos])
        return self.chunks[pos]

    def _load(self, new: List[Pos]):
        if not new:
            return
        if len(new) > len(self._free):
            # The reference's HashMap just grows: a camera that keeps moving hits max_chunks_per_frame every frame, returns
            # before the unload step (world.rs:84-87) and so never unloads.  Grow the device batch the same way.
            self._grow(max(2 * self.capacity, self.capacity + len(new)))
        slots = np.array([self._free.pop() for _ in new], dtype=np.int32)
        for p, s in zip(new, slots.tolist()):
            self.chunks[p] = s
        flags = self.device.generate(slots, np.array(new, dtype=np.int32).reshape(-1, 3))
        for p, f in zip(new, flags.tolist()):
            self.uniform_flags[p] = int(f)
        edited = [p for p in new if p in self.edits]
        if edited:
            self._apply_edits([(p, i, t) for p in edited for i, t in self.edits[p].items()])
        touched = list(new)
        for p in new:  # the chunks next to a new one now have a neighbour there
            touched += [(p[0] + o[0], p[1] + o[1], p[2] + o[2]) for o in FACE_OFFSETS]
        self._push_neighbor_rows(touched)

    def _grow(self, capacity: int):
        if capacity <= self.capacity:
            return
        self.device.grow(capacity)
        self._free = list(range(capacity - 1, self.capacity - 1, -1)) + self._free
        self.capacity = capacity

    def set_view_distance(self, view_distance: int):  # world.rs:181-184 (main.rs:168-176 calls it at run time)
        self.config.view_distance = max(1, int(view_distance))

    def view_distance(self) -> int:  # world.rs:187-189
        return self.config.view_distance

    def clear(self):  # world.rs:192-195
        self._unload(sorted(self.chunks))
        self.last_camera_chunk = None

    def _unload(self, gone: List[Pos]):
        if not gone:
            return
        slots = np.array([self.chunks[p] for p in gone], dtype=np.int32)
        for p in gone:
            self._free.append(self.chunks.pop(p))
            self.uniform_flags.pop(p, None)
        self.device.unload(slots)
        touched = []
        for p in gone:  # their neighbours lose the reference to the slot (it will be reused)
            touched += [(p[0] + o[0], p[1] + o[1], p[2] + o[2]) for o in FACE_OFFSETS]
        self._push_neighbor_rows(touched)

    # ---- block edits and picking (vx_world_batch_set_blocks, vx_world_raycast) ---------------------------------------------
    def _apply_edits(self, edits: List[Tuple[Pos, int, int]]):
        for p, _, _ in edits:
            self.uniform_flags[p] = 0  # a Uniform chunk becomes Varied on its first edit
        self.device.set_blocks(np.array([self.chunks[p] for p, _, _ in edits], dtype=np.int32),
                               np.array([i for _, i, _ in edits], dtype=np.int32), np.array([t for _, _, t in edits], dtype=np.uint8))

    def set_blocks(self, world_xyz, block_types) -> List[Pos]:
        """Set the blocks at world voxel coordinates world_xyz (n, 3) to block_types (n,) or one type for all (0 = air .. 3);
        when a voxel is listed twice the last entry wins.  Every chunk must be loaded (KeyError otherwise, before anything
        changes).  The edits are recorded in `edits` and come back when a chunk is unloaded and generated again.  Nothing is
        re-meshed: returns the positions whose meshes may change -- the edited chunks and the loaded neighbour across each
        face on which an edited voxel lies (the mesher reads a neighbour only on the shared border plane) -- for
        MeshCache.refresh."""
        xyz = np.asarray(world_xyz, dtype=np.int64).reshape(-1, 3)
        types = np.broadcast_to(np.asarray(block_types, dtype=np.int64).reshape(-1), (xyz.shape[0],))
        if types.size and (types.min() < 0 or types.max() > 3):
            raise ValueError("block types are 0..3")
        cpos, local = xyz >> 5, xyz & 31
        index = local[:, 2] * 1024 + local[:, 1] * 32 + local[:, 0]
        edits = [(tuple(int(c) for c in cp), int(i), int(t)) for cp, i, t in zip(cpos, index, types)]
        missing = sorted({p for p, _, _ in edits if p not in self.chunks})
        if missing:
            raise KeyError(f"set_blocks: chunks not loaded: {missing}")
        if not edits:
            return []
        for p, i, t in edits:
            self.edits.setdefault(p, {})[i] = t
        self._apply_edits(edits)
        dirty = set()
        for (p, _, _), lp in zip(edits, local.tolist()):
            dirty.add(p)
            for a in range(3):
                for border, face in ((31, 2 * a), (0, 2 * a + 1)):
                    if lp[a] == border:
                        o = FACE_OFFSETS[face]
                        q = (p[0] + o[0], p[1] + o[1], p[2] + o[2])
                        if q in self.chunks:
                            dirty.add(q)
        return sorted(dirty)

    def start_slots(self, origins) -> np.ndarray:
        """Slot of the chunk that holds each origin (world_to_chunk_pos), -1 where it is not loaded or not finite."""
        o = np.asarray(origins, dtype=np.float32).reshape(-1, 3)
        slots = np.full(o.shape[0], -1, dtype=np.int32)
        with np.errstate(invalid="ignore", over="ignore"):
            c = np.floor(o / np.float32(CHUNK_SIZE))
        ok = np.isfinite(c).all(axis=1) & (np.abs(c) < 2.0 ** 30).all(axis=1)
        if ok.any():
            uniq, inv = np.unique(c[ok].astype(np.int64), axis=0, return_inverse=True)
            found = np.array([self.chunks.get((int(u[0]), int(u[1]), int(u[2])), -1) for u in uniq], dtype=np.int32)
            slots[ok] = found[inv.reshape(-1)]
        return slots

    def raycast(self, origins, dirs, max_t: float) -> Dict[str, np.ndarray]:
        """vx_world_raycast (semantics in include/vx_b200.h) for rays starting in loaded chunks (others are RAY_INVALID).
        Returns arrays per ray: status (RAY_HIT / _MISS / _LEFT_WORLD / _INVALID), chunk (the chunk position), local and
        voxel (the hit voxel inside its chunk and in the world), face (FaceDir the ray entered through, -1 = the origin is
        inside a solid voxel), block_type, t (o + t*d is the entry point) and distance (t * |d|; inf unless hit), plus
        the raw VxRayHit records as `hits`."""
        o = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, 3)
        hits = self.device.raycast(o, d, self.start_slots(o), float(max_t))
        hit = hits["status"] == _lib.RAY_HIT
        vox = hits["voxel"].astype(np.int32)
        dist = np.where(hit, hits["t"].astype(np.float64) * np.linalg.norm(d.astype(np.float64), axis=1), np.inf)
        return {"status": hits["status"].copy(), "chunk": vox >> 5, "local": vox & 31, "voxel": vox, "face": hits["face"].copy(),
                "block_type": hits["block_type"].copy(), "t": hits["t"].copy(), "distance": dist, "hits": hits}

    def pick(self, camera_position, view_proj, pixels, width: int, height: int, max_distance: float) -> Dict[str, np.ndarray]:
        """What is under each pixel (n, 2) of a width x height frame: raycast along api.pixel_rays (unit directions, so
        t is the distance from the camera), at most max_distance (<= 1e4) far."""
        origins, dirs = api.pixel_rays(view_proj, camera_position, pixels, width, height)
        return self.raycast(origins, dirs, max_distance)

    # ---- visibility world.rs:103-146 --------------------------------------------------------------------------------
    def get_visible_chunks(self, camera_position) -> List[Pos]:
        cc = world_to_chunk_pos(camera_position)
        vd_sq = np.float32(self.config.view_distance * self.config.view_distance)
        return [p for p in self.get_all_chunks()
                if np.float32((p[0] - cc[0]) ** 2 + (p[1] - cc[1]) ** 2 + (p[2] - cc[2]) ** 2) <= vd_sq]

    def get_visible_chunks_frustum(self, camera_position, view_proj=None) -> List[Pos]:
        """world.rs:118-146: view distance and (when frustum_culling is on and a view-projection is given) the frustum
        test of the chunk box, evaluated on the device (vx_cull_chunks); positions in (x, y, z) order."""
        allp = self.get_all_chunks()
        if not allp:
            return []
        if view_proj is None or not self.config.frustum_culling:
            return self.get_visible_chunks(camera_position)
        pos = np.array(allp, dtype=np.int32).reshape(-1, 3)
        vis = api.get_visible_chunks_frustum(pos, camera_position, view_proj, self.config.view_distance, True, self.device.ctx)
        return [p for p, v in zip(allp, vis.tolist()) if v]


class MeshCache:
    """The mesh bookkeeping of the frame loop, main.rs:224-280: a chunk is meshed when it first becomes visible, the
    already meshed neighbours of a newly meshed chunk are re-meshed with it (their border faces may have become
    internal), nothing else is ever re-meshed, and meshes of unloaded chunks are dropped."""

    def __init__(self, world: World):
        self.world = world
        self.cached: set = set()          # positions with an entry (Some(mesh) or None) in mesh_cache
        self.meshed_last_frame: List[Pos] = []

    def update(self, visible_chunks: Iterable[Pos]) -> List[Pos]:
        w = self.world
        to_mesh: List[Pos] = []
        for pos in visible_chunks:
            if pos not in self.cached:
                to_mesh.append(pos)
                for o in FACE_OFFSETS:
                    npos = (pos[0] + o[0], pos[1] + o[1], pos[2] + o[2])
                    if w.contains_chunk(npos) and npos in self.cached:
                        to_mesh.append(npos)
        to_mesh = sorted(set(to_mesh))  # sort_by_key + dedup, main.rs:257-258
        to_mesh = [p for p in to_mesh if w.contains_chunk(p)]  # index.get(..) main.rs:267
        if to_mesh:
            w.device.remesh(np.array([w.chunks[p] for p in to_mesh], dtype=np.int32))
            self.cached.update(to_mesh)
        self.cached = {p for p in self.cached if w.contains_chunk(p)}  # main.rs:275
        self.meshed_last_frame = to_mesh
        return to_mesh

    def refresh(self, positions: Iterable[Pos]) -> List[Pos]:
        """Re-mesh, in one vx_world_batch_remesh call, those of `positions` (e.g. World.set_blocks' result) that have a
        cache entry; the others are meshed when they first become visible.  Returns the re-meshed positions."""
        w = self.world
        todo = sorted({tuple(p) for p in positions} & self.cached)
        todo = [p for p in todo if w.contains_chunk(p)]
        if todo:
            w.device.remesh(np.array([w.chunks[p] for p in todo], dtype=np.int32))
        return todo

    def visible_mesh_slots(self, visible_chunks: Iterable[Pos]) -> np.ndarray:
        """Slots of the visible chunks that have a cache entry, in (x, y, z) order: the mesh_ids of vx_render_frame
        (chunks whose entry is None -- Uniform or empty -- are skipped by the device through has_mesh)."""
        return np.array([self.world.chunks[p] for p in sorted(visible_chunks) if p in self.cached], dtype=np.int32)


def frame(world: World, cache: MeshCache, cam_position, view_proj, cfg, ctx: Optional[api.Context] = None, **render_kw):
    """One iteration of the reference's frame loop, main.rs:216-336 without window and input: world.update, visible
    chunks, mesh-cache maintenance, render_frame over the visible meshes.  Returns render_frame's result."""
    world.update(cam_position)
    visible = world.get_visible_chunks_frustum(cam_position, view_proj)
    cache.update(visible)
    ids = cache.visible_mesh_slots(visible)
    return api.render_frame(world.batch, view_proj, cam_position, cfg, mesh_ids=ids, ctx=ctx or world.device.ctx, **render_kw)
