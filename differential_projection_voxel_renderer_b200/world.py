"""Host mirror of the reference's streaming world and of the mesh cache its frame loop keeps.

`World` / `WorldConfig` follow /root/reference/src/world.rs:8-215 (same names, same update order, same per-frame
generation cap and unload hysteresis); `MeshCache` follows the chunk-to-mesh bookkeeping of the frame loop,
/root/reference/src/main.rs:216-297.  The voxels, the neighbour table and the meshes live on the device in a world
batch (vx_world_batch_*, include/vx_b200.h): the host only decides which lattice position occupies which slot.
Nothing here generates, meshes or draws on the CPU.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Iterable, List, Optional, Tuple

import numpy as np

from . import _lib, api
from ._lib import VxTerrainParams

Pos = Tuple[int, int, int]
CHUNK_SIZE = 32
FACE_OFFSETS = ((1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1))  # FaceDir order, mesh.rs:136-143
NBR_NONE = -1
PASTE_SKIP = _lib.PASTE_SKIP


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


REGION_COORD, REGION_RADIUS_SQ = 1 << 29, 1 << 56  # the bounds of vx_world_batch_fill_regions


def _region_op(shape: int, a, b, radius_sq: int, block_type: int, replace) -> np.ndarray:
    """A checked VxRegionOp record (api.REGION_OP_DTYPE); ValueError for what vx_world_batch_fill_regions would refuse."""
    types = range(4) if replace is None else [int(t) for t in replace]
    if not 0 <= int(block_type) <= 3 or any(not 0 <= t <= 3 for t in types):
        raise ValueError("block types are 0..3")
    a, b = np.asarray(a, dtype=np.int64).reshape(3), np.asarray(b, dtype=np.int64).reshape(3)
    if (np.abs(a) > REGION_COORD).any() or (np.abs(b) > REGION_COORD).any() or int(radius_sq) > REGION_RADIUS_SQ:
        raise ValueError("region coordinates are limited to [-2^29, 2^29] and radius_sq to 2^56")
    op = np.zeros((), dtype=api.REGION_OP_DTYPE)
    op["shape"], op["a"], op["b"], op["radius_sq"] = shape, a, b, int(radius_sq)
    op["block_type"], op["replace_mask"] = int(block_type), sum(1 << t for t in set(types))
    return op


def region_contains(op: np.ndarray, voxels: np.ndarray) -> np.ndarray:
    """Which world voxels (n, 3) lie inside the region of a VxRegionOp record (include/vx_b200.h)."""
    v = np.asarray(voxels, dtype=np.int64).reshape(-1, 3)
    a = op["a"].astype(np.int64)
    if int(op["shape"]) == _lib.REGION_BOX:
        return ((v >= a) & (v <= op["b"].astype(np.int64))).all(axis=1)
    d = v - a
    r = math.isqrt(int(op["radius_sq"]))
    near = (np.abs(d) <= r).all(axis=1)
    return near & ((np.where(near[:, None], d, 0) ** 2).sum(axis=1) <= int(op["radius_sq"]))


PASTE_MAX_DIM = 1024  # the largest extent per axis of vx_world_batch_copy_region / vx_world_batch_paste


def _paste_box(lo, dims) -> Tuple[np.ndarray, np.ndarray]:
    """lo and dims as int64 (3,); ValueError for a box vx_world_batch_copy_region / _paste would refuse."""
    lo, dims = np.asarray(lo, dtype=np.int64).reshape(3), np.asarray(dims, dtype=np.int64).reshape(3)
    if (dims < 1).any() or (dims > PASTE_MAX_DIM).any():
        raise ValueError(f"copy / paste boxes are 1..{PASTE_MAX_DIM} voxels per axis")
    if (np.abs(lo) > REGION_COORD).any() or (np.abs(lo + dims - 1) > REGION_COORD).any():
        raise ValueError("copy / paste coordinates are limited to [-2^29, 2^29]")
    return lo, dims


def _chunk_starts(lo: int, n: int) -> np.ndarray:
    """Indices 0 <= i < n along one axis of a box starting at world voxel lo where a new chunk begins (0 included)."""
    return np.unique(np.concatenate([[0], np.arange((-lo) % CHUNK_SIZE, n, CHUNK_SIZE)])).astype(np.intp)


class _DeviceWorld:
    """The vx_world_batch_* calls (block and region edits included), vx_world_raycast and vx_world_move_boxes; tests
    substitute a recorder for it to check the host logic without a GPU."""

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

    def fill_regions(self, ops: np.ndarray, slots: np.ndarray) -> np.ndarray:
        """ops: api.REGION_OP_DTYPE records; returns the change bits per slot."""
        changed = np.zeros(slots.size, dtype=np.uint8)
        self.ctx.check(self.ctx.lib.vx_world_batch_fill_regions(self.ctx.handle, self.batch.handle, api._p(ops), int(ops.size), api._p(slots),
                                                                int(slots.size), api._p(changed)))
        return changed

    def read_voxels(self, slots: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """The raw voxel rows (n, 32768) and Uniform flags (n,) of the slots."""
        voxels = np.zeros((slots.size, CHUNK_SIZE ** 3), dtype=np.uint8)
        flags = np.zeros(slots.size, dtype=np.uint8)
        self.ctx.check(self.ctx.lib.vx_world_batch_read_voxels(self.ctx.handle, self.batch.handle, api._p(slots), int(slots.size),
                                                               api._p(voxels), api._p(flags)))
        return voxels, flags

    def copy_region(self, lo: np.ndarray, dims: np.ndarray, chunk_slots: np.ndarray) -> np.ndarray:
        """The box lo .. lo + dims - 1 as (dims[2], dims[1], dims[0]) uint8; chunk_slots [cz][cy][cx] (-1 = not loaded)."""
        lo, dims = np.ascontiguousarray(lo, dtype=np.int32), np.ascontiguousarray(dims, dtype=np.int32)
        out = np.empty(tuple(int(d) for d in dims[::-1]), dtype=np.uint8)
        table = np.ascontiguousarray(chunk_slots, dtype=np.int32)
        self.ctx.check(self.ctx.lib.vx_world_batch_copy_region(self.ctx.handle, self.batch.handle, api._p(lo), api._p(dims), api._p(table),
                                                               api._p(out)))
        return out

    def paste(self, ops: np.ndarray, templates: np.ndarray, slots: np.ndarray) -> np.ndarray:
        """ops: api.PASTE_OP_DTYPE records into the uint8 buffer templates; returns the change bits per slot."""
        changed = np.zeros(slots.size, dtype=np.uint8)
        self.ctx.check(self.ctx.lib.vx_world_batch_paste(self.ctx.handle, self.batch.handle, api._p(ops), int(ops.size), api._p(templates),
                                                         C.c_int64(templates.size), api._p(slots), int(slots.size), api._p(changed)))
        return changed

    def raycast(self, origins: np.ndarray, dirs: np.ndarray, start_slots: np.ndarray, max_t: float) -> np.ndarray:
        hits = np.zeros(start_slots.size, dtype=api.RAY_HIT_DTYPE)
        self.ctx.check(self.ctx.lib.vx_world_raycast(self.ctx.handle, self.batch.handle, api._p(origins), api._p(dirs), api._p(start_slots),
                                                     int(start_slots.size), float(max_t), api._p(hits)))
        return hits

    def move_boxes(self, pos: np.ndarray, size: np.ndarray, delta: np.ndarray, slots: np.ndarray) -> np.ndarray:
        """pos (n, 3) and slots (n,) are updated in place; returns the flags (n,)."""
        flags = np.zeros(slots.size, dtype=np.uint32)
        self.ctx.check(self.ctx.lib.vx_world_move_boxes(self.ctx.handle, self.batch.handle, api._p(pos), api._p(size), api._p(delta),
                                                        api._p(slots), int(slots.size), api._p(flags)))
        return flags


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
        # region fills (fill_box / fill_ball; api.REGION_OP_DTYPE records) in issue order, and per chunk position the indices
        # of the fills that changed it: replayed, before `edits`, when the chunk is generated anew
        self.fills: List[np.ndarray] = []
        self._fills_at: Dict[Pos, List[int]] = {}
        # pastes (paste; an api.PASTE_OP_DTYPE record with offset 0 and its own copy of the template) in issue order, how many
        # fills were issued before each, and per chunk position the indices of the pastes that changed it: replayed with the
        # fills, in issue order, before `edits`
        self.pastes: List[Tuple[np.ndarray, np.ndarray]] = []
        self._pastes_after: List[int] = []
        self._pastes_at: Dict[Pos, List[int]] = {}
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
        replay = [p for p in new if p in self._fills_at or p in self._pastes_at]
        if replay:
            self._replay(replay)
        edited = [p for p in new if p in self.edits]
        if edited:
            self._apply_edits([(p, i, t) for p in edited for i, t in self.edits[p].items()])
        touched = list(new)
        for p in new:  # the chunks next to a new one now have a neighbour there
            touched += [(p[0] + o[0], p[1] + o[1], p[2] + o[2]) for o in FACE_OFFSETS]
        self._push_neighbor_rows(touched)

    def _replay(self, positions: List[Pos]):
        """Replay the fills and pastes that changed `positions` (just generated) in issue order: each run of consecutive
        fills in one fill_regions call, each run of consecutive pastes in one paste call, over the positions that one of
        the run's ops changed.  Exact (DESIGN §3.3): both are per-voxel functions of the voxel's old type."""
        fills = sorted({i for p in positions for i in self._fills_at.get(p, ())})
        pastes = sorted({j for p in positions for j in self._pastes_at.get(p, ())})
        # paste j was issued after fills 0 .. _pastes_after[j] - 1, so it sorts between fill _pastes_after[j] - 1 and the next
        order = sorted([(i, 1, i) for i in fills] + [(self._pastes_after[j], 0, j) for j in pastes])
        runs: List[Tuple[int, List[int]]] = []
        for _, is_fill, i in order:
            if runs and runs[-1][0] == is_fill:
                runs[-1][1].append(i)
            else:
                runs.append((is_fill, [i]))
        for is_fill, run in runs:
            at, members = (self._fills_at, set(run)) if is_fill else (self._pastes_at, set(run))
            ps = [p for p in positions if members.intersection(at.get(p, ()))]
            slots = np.array([self.chunks[p] for p in ps], dtype=np.int32)
            if is_fill:
                changed = self.device.fill_regions(np.stack([self.fills[i] for i in run]), slots)
            else:
                ops = np.stack([self.pastes[j][0] for j in run])
                sizes = [self.pastes[j][1].size for j in run]
                ops["offset"] = np.concatenate([[0], np.cumsum(sizes)[:-1]])
                changed = self.device.paste(ops, np.concatenate([self.pastes[j][1].reshape(-1) for j in run]), slots)
            for p, c in zip(ps, changed.tolist()):
                if c & _lib.REGION_CHANGED:
                    self.uniform_flags[p] = 0

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

    # ---- region edits (vx_world_batch_fill_regions) ----------------------------------------------------------------
    def fill_box(self, lo, hi, block_type: int, replace: Optional[Iterable[int]] = None) -> List[Pos]:
        """Set the voxels of the box lo..hi (world voxel coordinates, both corners inclusive) whose type is in `replace` (block
        types; None = all four) to block_type.  See fill_ball for what is returned and kept."""
        op = _region_op(_lib.REGION_BOX, lo, hi, 0, block_type, replace)
        lo, hi = op["a"].astype(np.int64), op["b"].astype(np.int64)
        if (lo > hi).any():
            return []
        return self._fill(op, self._chunks_between(lo >> 5, hi >> 5))

    def fill_ball(self, centre, radius_sq: int, block_type: int, replace: Optional[Iterable[int]] = None) -> List[Pos]:
        """Set the voxels v with |v - centre|^2 <= radius_sq (world voxel coordinates, integers) whose type is in `replace` (block
        types; None = all four) to block_type: carve an explosion with fill_ball(c, r2, 0, replace=(1, 2, 3)).  Exact semantics
        in include/vx_b200.h (vx_world_batch_fill_regions).  Every chunk that holds a voxel of the ball must be loaded
        (KeyError otherwise, before anything changes); a ball with radius_sq < 0 is empty and returns [] without a device
        call.  The fill is recorded and comes back when a chunk is unloaded and generated again (fills first, in issue order,
        then `edits`, into which every fill is folded).  Nothing is re-meshed: returns the positions whose meshes may change --
        the chunks whose voxels or Uniform flag changed and the loaded neighbour across each face on which a voxel changed --
        for MeshCache.refresh."""
        op = _region_op(_lib.REGION_BALL, centre, (0, 0, 0), radius_sq, block_type, replace)
        if int(op["radius_sq"]) < 0:
            return []
        a, r = op["a"].astype(np.int64), math.isqrt(int(op["radius_sq"]))
        box = self._chunks_between((a - r) >> 5, (a + r) >> 5)
        near = np.clip(a, box * CHUNK_SIZE, box * CHUNK_SIZE + CHUNK_SIZE - 1) - a  # the point of each chunk nearest the centre
        return self._fill(op, box[(near * near).sum(axis=1) <= int(op["radius_sq"])])

    def _chunks_between(self, c0: np.ndarray, c1: np.ndarray) -> np.ndarray:
        """Chunk positions c0 .. c1 (inclusive) as (n, 3) int64 in (x, y, z) order; KeyError when the range reaches beyond the
        loaded chunks on some axis (a region's chunks span its whole range on each axis, so one of them is not loaded)."""
        loaded = np.array(list(self.chunks), dtype=np.int64).reshape(-1, 3)
        if loaded.size == 0 or (c0 < loaded.min(axis=0)).any() or (c1 > loaded.max(axis=0)).any():
            raise KeyError(f"fill: chunks {tuple(c0.tolist())} .. {tuple(c1.tolist())} reach beyond the loaded world")
        axes = [np.arange(int(u), int(v) + 1) for u, v in zip(c0, c1)]
        return np.stack(np.meshgrid(*axes, indexing="ij"), axis=-1).reshape(-1, 3)

    def _fill(self, op: np.ndarray, touched: np.ndarray) -> List[Pos]:
        touched = [tuple(int(c) for c in p) for p in touched]
        missing = [p for p in touched if p not in self.chunks]
        if missing:
            raise KeyError(f"fill: chunks not loaded: {missing[:16]}{' ...' if len(missing) > 16 else ''}")
        changed = self.device.fill_regions(op.reshape(1), np.array([self.chunks[p] for p in touched], dtype=np.int32))
        k = len(self.fills)
        self.fills.append(op)
        dirty = set()
        for p, c in zip(touched, changed.tolist()):
            if not c & _lib.REGION_CHANGED:
                continue  # unchanged: replaying the fill there would change nothing but voxels that `edits` sets anyway
            self._fills_at.setdefault(p, []).append(k)
            self.uniform_flags[p] = 0
            dirty.add(p)
            for f, o in enumerate(FACE_OFFSETS):
                q = (p[0] + o[0], p[1] + o[1], p[2] + o[2])
                if (c >> f) & 1 and q in self.chunks:
                    dirty.add(q)
            e = self.edits.get(p)
            if e:  # fold: an edited voxel inside the shape whose type is in the mask now holds block_type
                idx = np.fromiter(e.keys(), dtype=np.int64, count=len(e))
                types = np.fromiter(e.values(), dtype=np.int64, count=len(e))
                v = np.stack([idx & 31, (idx >> 5) & 31, idx >> 10], axis=1) + np.array(p, dtype=np.int64) * CHUNK_SIZE
                hit = region_contains(op, v) & (((int(op["replace_mask"]) >> types) & 1) == 1)
                for i in idx[hit].tolist():
                    e[i] = int(op["block_type"])
        return sorted(dirty)

    # ---- copy and paste (vx_world_batch_copy_region, vx_world_batch_paste) ------------------------------------------
    def copy_region(self, lo, hi) -> np.ndarray:
        """The voxels of the box lo..hi (world voxel coordinates, both corners inclusive, 1..1024 voxels per axis) as uint8
        indexed [z, y, x], PASTE_SKIP where the chunk is not loaded: one device call (vx_world_batch_copy_region).  Unloaded
        space is never an error, so the result can be pasted back as it is."""
        lo = np.asarray(lo, dtype=np.int64).reshape(3)
        lo, dims = _paste_box(lo, np.asarray(hi, dtype=np.int64).reshape(3) - lo + 1)
        c0, c1 = lo >> 5, (lo + dims - 1) >> 5
        table = np.array([[[self.chunks.get((x, y, z), -1) for x in range(c0[0], c1[0] + 1)] for y in range(c0[1], c1[1] + 1)]
                          for z in range(c0[2], c1[2] + 1)], dtype=np.int32)
        return self.device.copy_region(lo, dims, table)

    def paste(self, template, origin, replace: Optional[Iterable[int]] = None) -> List[Pos]:
        """Stamp template ((sz, sy, sx) uint8, indexed [z, y, x]) with byte (0, 0, 0) on world voxel origin: a byte 0..3 sets
        its voxel to that type if the voxel's type is in `replace` (block types; None = all four); PASTE_SKIP leaves it
        alone.  Transparent air is np.where(t == 0, PASTE_SKIP, t); rotations are np.rot90(t, k, axes=(0, 2)).  Exact
        semantics in include/vx_b200.h (vx_world_batch_paste).  Every chunk where the template has a byte other than
        PASTE_SKIP must be loaded (KeyError otherwise, before anything changes); the others are not touched, so a copy
        taken across unloaded space can be pasted back.  The paste is recorded with its own copy of the template and comes
        back when a chunk is unloaded and generated again (with the fills, in issue order, then `edits`, into which every
        paste is folded).  Nothing is re-meshed: returns the positions whose meshes may change, as fill_ball does."""
        t = np.asarray(template)
        if t.ndim != 3 or not np.issubdtype(t.dtype, np.integer):
            raise ValueError("a template is a (sz, sy, sx) array of block types")
        origin, dims = _paste_box(origin, t.shape[::-1])
        if ((t > 3) & (t != PASTE_SKIP)).any() or (t < 0).any():
            raise ValueError("template bytes are block types 0..3 or PASTE_SKIP")
        types = range(4) if replace is None else [int(v) for v in replace]
        if any(not 0 <= v <= 3 for v in types):
            raise ValueError("block types are 0..3")
        t = np.array(t, dtype=np.uint8, order="C")  # the record's own copy
        # the chunks under at least one byte other than PASTE_SKIP
        starts = [_chunk_starts(int(origin[e]), int(dims[e])) for e in range(3)]
        solid = (t != PASTE_SKIP).view(np.uint8)
        for axis, e in ((0, 2), (1, 1), (2, 0)):
            solid = np.maximum.reduceat(solid, starts[e], axis=axis)
        c0 = origin >> 5
        touched = [(int(c0[0] + i), int(c0[1] + j), int(c0[2] + k)) for k, j, i in zip(*np.nonzero(solid))]
        missing = sorted(p for p in touched if p not in self.chunks)
        if missing:
            raise KeyError(f"paste: chunks not loaded: {missing[:16]}{' ...' if len(missing) > 16 else ''}")
        if not touched:
            return []
        op = np.zeros((), dtype=api.PASTE_OP_DTYPE)
        op["origin"], op["dims"], op["replace_mask"] = origin, dims, sum(1 << v for v in set(types))
        changed = self.device.paste(op.reshape(1), t.reshape(-1), np.array([self.chunks[p] for p in touched], dtype=np.int32))
        k = len(self.pastes)
        self.pastes.append((op, t))
        self._pastes_after.append(len(self.fills))
        dirty = set()
        for p, c in zip(touched, changed.tolist()):
            if not c & _lib.REGION_CHANGED:
                continue  # unchanged: replaying the paste there would change nothing but voxels that `edits` sets anyway
            self._pastes_at.setdefault(p, []).append(k)
            self.uniform_flags[p] = 0
            dirty.add(p)
            for f, o in enumerate(FACE_OFFSETS):
                q = (p[0] + o[0], p[1] + o[1], p[2] + o[2])
                if (c >> f) & 1 and q in self.chunks:
                    dirty.add(q)
            e = self.edits.get(p)
            if e:  # fold: an edited voxel under a byte other than PASTE_SKIP whose type is in the mask now holds that byte
                idx = np.fromiter(e.keys(), dtype=np.int64, count=len(e))
                types_now = np.fromiter(e.values(), dtype=np.int64, count=len(e))
                tv = np.stack([idx & 31, (idx >> 5) & 31, idx >> 10], axis=1) + np.array(p, dtype=np.int64) * CHUNK_SIZE - origin
                inside = ((tv >= 0) & (tv < dims)).all(axis=1)
                tv = np.where(inside[:, None], tv, 0)
                b = t[tv[:, 2], tv[:, 1], tv[:, 0]].astype(np.int64)
                hit = inside & (b != PASTE_SKIP) & (((int(op["replace_mask"]) >> types_now) & 1) == 1)
                for i, v in zip(idx[hit].tolist(), b[hit].tolist()):
                    e[i] = v
        return sorted(dirty)

    def chunk_voxels(self, pos) -> Tuple[int, np.ndarray]:
        """(Uniform flag, voxels) of a loaded chunk read back from the device (vx_world_batch_read_voxels): flag 0 Varied, else
        1 + block type; voxels (32, 32, 32) uint8 indexed [z, y, x] -- a Uniform chunk's are all its type."""
        voxels, flags = self.device.read_voxels(np.array([self.chunks[tuple(pos)]], dtype=np.int32))
        v = voxels[0].reshape(CHUNK_SIZE, CHUNK_SIZE, CHUNK_SIZE)
        if flags[0]:
            v[:] = flags[0] - 1
        return int(flags[0]), v

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

    # ---- collision (vx_world_move_boxes) -----------------------------------------------------------------------------
    def move_boxes(self, pos, size, delta) -> Dict[str, np.ndarray]:
        """Move boxes with min corner pos (n, 3) and extent size by delta through the loaded voxels, stopping at solid ones
        and at unloaded space (vx_world_move_boxes; semantics in include/vx_b200.h: Y, then X, then Z).  size and delta
        broadcast to (n, 3).  Gravity, jumping and stepping up are the caller's.  The caller's arrays are not modified.
        Returns arrays per box: pos (the new min corner), slot (of the chunk holding floor(pos), -1 if not loaded), flags,
        blocked ((n, 6) bool: the move along that FaceDir was cut short), on_ground (blocked moving -Y), touched_unloaded and
        invalid (the box was left where it was)."""
        p = np.array(pos, dtype=np.float32).reshape(-1, 3)
        n = p.shape[0]
        s = np.ascontiguousarray(np.broadcast_to(np.asarray(size, dtype=np.float32), (n, 3)))
        d = np.ascontiguousarray(np.broadcast_to(np.asarray(delta, dtype=np.float32), (n, 3)))
        slots = self.start_slots(p)
        flags = self.device.move_boxes(p, s, d, slots)
        blocked = ((flags[:, None] >> np.arange(6, dtype=np.uint32)) & 1).astype(bool)
        return {"pos": p, "slot": slots, "flags": flags, "blocked": blocked, "on_ground": blocked[:, 3].copy(),
                "touched_unloaded": (flags & _lib.MOVE_TOUCHED_UNLOADED) != 0, "invalid": (flags & _lib.MOVE_INVALID) != 0}

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
