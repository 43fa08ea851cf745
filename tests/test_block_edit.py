"""Picking and block edits without a GPU: the ray cast's exact semantics (include/vx_b200.h, vx_world_raycast) pinned on the
CPU oracle (tests/ray_oracle.c) with answers worked out by hand, World's edit bookkeeping (set_blocks, re-applied edits, the chunks an edit
dirties) against a recording fake device, the pixel rays, and the ABI of VxRayHit."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import vx_ray_oracle
from differential_projection_voxel_renderer_b200 import _lib, api, camera, world as vxw, worldgen
from test_world_stream import CAMERA_WALK, FakeDevice as FakeDeviceWithoutEdits

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HIT, MISS, LEFT, INVALID = _lib.RAY_HIT, _lib.RAY_MISS, _lib.RAY_LEFT_WORLD, _lib.RAY_INVALID
STONE, UNIFORM_AIR, UNIFORM_STONE = 3, 1, 4


# ---- oracle DDA known answers -----------------------------------------------------------------------------------------

class Slots:
    """A hand-built world batch: slot-indexed positions, voxels, Uniform flags and neighbour rows."""

    def __init__(self, chunks):
        """chunks: list of (position, flag); neighbour rows link the listed positions."""
        self.pos = np.array([p for p, _ in chunks], dtype=np.int32).reshape(-1, 3)
        self.flags = np.array([f for _, f in chunks], dtype=np.uint8)
        self.vox = np.zeros((len(chunks), 32768), dtype=np.uint8)
        at = {tuple(p): s for s, p in enumerate(self.pos.tolist())}
        self.nbr = np.array([[at.get((p[0] + o[0], p[1] + o[1], p[2] + o[2]), -1) for o in vxw.FACE_OFFSETS]
                             for p in self.pos.tolist()], dtype=np.int32).reshape(-1, 6)

    def set(self, xyz, t=STONE):
        x, y, z = xyz
        s = int(np.flatnonzero((self.pos == [x >> 5, y >> 5, z >> 5]).all(axis=1))[0])
        self.vox[s, (z & 31) * 1024 + (y & 31) * 32 + (x & 31)] = t
        return s

    def cast(self, o, d, slot=0, max_t=100.0):
        hits, steps = vx_ray_oracle.raycast(self.pos, self.vox, self.flags, self.nbr, np.array([o], np.float32), np.array([d], np.float32),
                                 np.array([slot], np.int32), max_t, want_steps=True)
        return hits[0], int(steps[0])


def _hit(h, voxel, face, t, slot, block_type=STONE):
    assert h["status"] == HIT, h
    assert tuple(h["voxel"].tolist()) == tuple(voxel) and h["face"] == face and h["slot"] == slot and h["block_type"] == block_type, h
    assert np.float32(h["t"]).view(np.uint32) == np.float32(t).view(np.uint32), (h["t"], t)


def _not_hit(h, status):
    assert h["status"] == status, h
    assert h["slot"] == -1 and tuple(h["voxel"].tolist()) == (0, 0, 0) and h["face"] == -1 and h["t"] == 0 and h["block_type"] == 0, h


def test_axis_ray_hits_the_stone_through_its_negative_x_face():
    w = Slots([((0, 0, 0), 0)])
    w.set((5, 0, 0))
    h, steps = w.cast((0.5, 0.5, 0.5), (1, 0, 0))
    _hit(h, (5, 0, 0), 1, 4.5, 0)  # planes x = 1..5 at t = 0.5 .. 4.5; entering x = 5 through its -X face
    assert steps == 5


def test_ray_along_minus_z_crosses_into_the_neighbour_slot():
    w = Slots([((0, 0, 0), 0), ((0, 0, -1), 0)])
    s = w.set((3, 2, -3))
    assert s == 1
    h, steps = w.cast((3.5, 2.5, 1.5), (0, 0, -1))
    _hit(h, (3, 2, -3), 4, 3.5, 1)  # plane z = -2 at t = (-2 - 1.5) / -1; stepping -z enters through +Z
    assert steps == 4  # planes z = 1, 0, -1, -2


def test_diagonal_ray_through_a_voxel_edge_steps_x_before_y():
    w = Slots([((0, 0, 0), 0)])
    w.set((1, 0, 0))
    w.set((0, 1, 0))  # on the other side of the edge: never entered
    h, _ = w.cast((0.5, 0.5, 0.5), (1, 1, 0))
    _hit(h, (1, 0, 0), 1, 0.5, 0)
    w.vox[:] = 0
    w.set((0, 1, 0))
    w.set((1, 1, 0))
    h, steps = w.cast((0.5, 0.5, 0.5), (1, 1, 0))
    _hit(h, (1, 1, 0), 3, 0.5, 0)  # x then y at the same t: (1,0,0), then (1,1,0) entered through -Y
    assert steps == 2


def test_origin_inside_stone_is_a_hit_at_t_zero_without_a_face():
    w = Slots([((0, 0, 0), 0)])
    w.set((7, 8, 9), 2)
    h, steps = w.cast((7.25, 8.5, 9.75), (0, -1, 0))
    _hit(h, (7, 8, 9), -1, 0.0, 0, block_type=2)
    assert steps == 0


def test_uniform_solid_chunk_is_hit_at_its_face_and_uniform_air_is_walked_without_its_rows():
    w = Slots([((0, 0, 0), 0), ((1, 0, 0), UNIFORM_STONE)])
    h, _ = w.cast((30.5, 3.5, 3.5), (1, 0, 0))
    _hit(h, (32, 3, 3), 1, 1.5, 1, block_type=3)
    # a Uniform air chunk between: its voxel rows hold garbage that must not be read
    w = Slots([((0, 0, 0), 0), ((1, 0, 0), UNIFORM_AIR), ((2, 0, 0), 0)])
    w.vox[1] = 3
    w.set((70, 3, 3), 1)
    h, steps = w.cast((30.5, 3.5, 3.5), (1, 0, 0))
    _hit(h, (70, 3, 3), 1, 39.5, 2, block_type=1)
    assert steps == 40
    # starting inside a Uniform stone chunk
    w2 = Slots([((0, 0, 0), UNIFORM_STONE)])
    h, _ = w2.cast((1.5, 2.5, 3.5), (0, 1, 0))
    _hit(h, (1, 2, 3), -1, 0.0, 0, block_type=3)


def test_leaving_into_no_chunk_is_left_world_and_negative_coordinates_walk():
    w = Slots([((0, 0, 0), 0)])
    h, steps = w.cast((30.5, 3.5, 3.5), (1, 0, 0))
    _not_hit(h, LEFT)
    assert steps == 2  # x = 31, then the step out of the chunk
    w = Slots([((-1, -1, -1), 0), ((0, -1, -1), 0)])
    w.set((-5, -2, -3))  # on the line, but the walk passes beside it
    w.set((-5, -3, -4))
    h, steps = w.cast((2.0, -1.5, -2.5), (-1, -0.125, -0.25), slot=1)
    # x planes 2, 1, 0, ... at t = -0 (the origin lies on the face), 1, 2, ...; z plane -3 at t = 2 and -4 at 6; y plane -2 at
    # t = 4.  Ties go to x: x -> 1, 0, -1 (into slot 0), z -> -4, x -> -2, -3, y -> -3, x -> -4, -5 at t = 6
    _hit(h, (-5, -3, -4), 0, 6.0, 0)  # stepping -x enters through +X
    assert steps == 9


def test_max_t_just_below_and_at_the_hit():
    w = Slots([((0, 0, 0), 0)])
    w.set((5, 0, 0))
    below = np.nextafter(np.float32(4.5), np.float32(0))
    _not_hit(w.cast((0.5, 0.5, 0.5), (1, 0, 0), max_t=float(below))[0], MISS)
    _hit(w.cast((0.5, 0.5, 0.5), (1, 0, 0), max_t=4.5)[0], (5, 0, 0), 1, 4.5, 0)
    _not_hit(w.cast((0.5, 0.5, 0.5), (1, 0, 0), max_t=0.0)[0], MISS)


@pytest.mark.parametrize("o,d,slot,max_t", [
    ((0.5, 0.5, 0.5), (0, 0, 0), 0, 10.0),             # zero direction
    ((np.nan, 0.5, 0.5), (1, 0, 0), 0, 10.0),          # NaN origin
    ((0.5, 0.5, 0.5), (1, np.nan, 0), 0, 10.0),        # NaN direction
    ((0.5, 0.5, 0.5), (np.inf, 0, 0), 0, 10.0),        # infinite direction
    ((0.5, 0.5, 0.5), (1, 0, 0), 1, 10.0),             # start slot of another chunk
    ((0.5, 0.5, 0.5), (1, 0, 0), -1, 10.0),            # not loaded
    ((0.5, 0.5, 0.5), (1, 0, 0), 2, 10.0),             # beyond the batch
    ((0.5, 0.5, 0.5), (1, 0, 0), 0, -1.0),             # max_t < 0
    ((0.5, 0.5, 0.5), (1, 0, 0), 0, 10001.0),          # max_t > 1e4
    ((0.5, 0.5, 0.5), (1, 0, 0), 0, np.nan),           # max_t NaN
    ((16777216.0, 0.5, 0.5), (1, 0, 0), 0, 10.0),      # |o| >= 2^24
])
def test_invalid_rays(o, d, slot, max_t):
    w = Slots([((0, 0, 0), 0), ((1, 0, 0), 0)])
    w.set((5, 0, 0))
    _not_hit(w.cast(o, d, slot=slot, max_t=max_t)[0], INVALID)


# ---- World bookkeeping with a recording fake device ------------------------------------------------------------------

class FakeDevice(FakeDeviceWithoutEdits):
    """test_world_stream's recorder plus the two calls of this feature: edits land in the slot's voxels in list order (the
    last one wins), ray casts go to the ray-cast oracle over the slot arrays."""

    def set_blocks(self, slots, voxel_index, block_types):
        for s, i, t in zip(slots.tolist(), voxel_index.tolist(), block_types.tolist()):
            if self.flag[s] != 0:
                self.vox[s][:] = self.flag[s] - 1
                self.flag[s] = 0
            self.vox[s][i] = t
        self.calls.append(("set_blocks", slots.tolist(), voxel_index.tolist(), block_types.tolist()))

    def raycast(self, origins, dirs, start_slots, max_t):
        pos = np.zeros((self.capacity, 3), np.int32)
        vox = np.zeros((self.capacity, 32768), np.uint8)
        flags = np.ones(self.capacity, np.uint8)
        for s in self.pos:
            pos[s], vox[s], flags[s] = self.pos[s], self.vox[s], self.flag[s]
        nbr = np.array([self.nbr[s] for s in range(self.capacity)], dtype=np.int32)
        self.calls.append(("raycast", int(start_slots.size)))
        return vx_ray_oracle.raycast(pos, vox, flags, nbr, origins, dirs, start_slots, max_t)


def _world(ob, vd=1, center=(0.0, 0.0, 0.0)):
    dev = FakeDevice(ob, vxw.sphere_capacity(vd))
    w = vxw.World(vxw.WorldConfig(view_distance=vd, max_chunks_per_frame=1000), device=dev)
    w.update(center)
    return w, dev


def _index(x, y, z):
    return (z & 31) * 1024 + (y & 31) * 32 + (x & 31)


def test_edits_dirty_the_chunk_and_the_loaded_neighbours_across_border_faces(ob):
    w, dev = _world(ob)  # the chunk at the origin and its six face neighbours
    assert w.chunk_count() == 7
    assert w.set_blocks([(5, 6, 7)], [STONE]) == [(0, 0, 0)]
    assert w.set_blocks([(0, 0, 0)], [STONE]) == [(-1, 0, 0), (0, -1, 0), (0, 0, -1), (0, 0, 0)]
    assert w.set_blocks([(31, 31, 31)], [STONE]) == [(0, 0, 0), (0, 0, 1), (0, 1, 0), (1, 0, 0)]
    # chunk (1,0,0), local (31, 0, 5): its +X and -Y neighbours are not loaded
    assert w.set_blocks([(63, 0, 5)], [STONE]) == [(1, 0, 0)]
    # local x = 0 of chunk (1,0,0) borders the loaded (0,0,0)
    assert w.set_blocks([(32, 4, 4)], [STONE]) == [(0, 0, 0), (1, 0, 0)]
    slot = w.chunks[(1, 0, 0)]
    assert dev.vox[slot][_index(32, 4, 4)] == STONE and w.uniform_flags[(1, 0, 0)] == 0
    assert w.edits[(0, 0, 0)] == {_index(5, 6, 7): STONE, _index(0, 0, 0): STONE, _index(31, 31, 31): STONE}


def test_last_edit_of_a_voxel_wins_and_unloaded_chunks_raise(ob):
    w, dev = _world(ob)
    assert w.set_blocks([(1, 2, 3), (1, 2, 3), (4, 4, 4)], [STONE, 0, 2]) == [(0, 0, 0)]
    assert w.edits[(0, 0, 0)] == {_index(1, 2, 3): 0, _index(4, 4, 4): 2}
    assert dev.calls[-1] == ("set_blocks", [w.chunks[(0, 0, 0)]] * 3, [_index(1, 2, 3), _index(1, 2, 3), _index(4, 4, 4)], [STONE, 0, 2])
    assert dev.vox[w.chunks[(0, 0, 0)]][_index(1, 2, 3)] == 0
    n_calls = len(dev.calls)
    with pytest.raises(KeyError):
        w.set_blocks([(1, 1, 1), (64, 0, 0)], [STONE, STONE])  # (2,0,0) is not loaded: nothing is edited
    with pytest.raises(ValueError):
        w.set_blocks([(1, 1, 1)], [4])
    assert len(dev.calls) == n_calls and _index(1, 1, 1) not in w.edits[(0, 0, 0)]
    assert w.set_blocks(np.zeros((0, 3)), []) == [] and len(dev.calls) == n_calls


def test_uniform_chunk_becomes_varied_on_its_first_edit(ob):
    w, dev = _world(ob, center=(0.0, 200.0, 0.0))  # high above the terrain: Uniform air chunks
    p = (0, 6, 0)
    assert w.uniform_flags[p] == UNIFORM_AIR
    w.set_blocks([(3, 6 * 32 + 3, 3)], STONE)
    assert w.uniform_flags[p] == 0 and dev.flag[w.chunks[p]] == 0
    assert int(dev.vox[w.chunks[p]].sum()) == STONE


def test_edits_come_back_after_the_chunk_is_unloaded_and_generated_again(ob):
    w, dev = _world(ob, vd=1)
    w.set_blocks([(40, 5, 5), (33, 1, 2)], [STONE, 0])
    edits = dict(w.edits[(1, 0, 0)])
    far = (32.0 * 20, 0.0, 0.0)
    w.update(far)
    assert (1, 0, 0) not in w.chunks and w.edits[(1, 0, 0)] == edits  # kept while unloaded
    del dev.calls[:]
    w.update((0.0, 0.0, 0.0))
    assert (1, 0, 0) in w.chunks and w.uniform_flags[(1, 0, 0)] == 0
    names = [c[0] for c in dev.calls]
    g = names.index("generate")
    assert names[g + 1] == "set_blocks", names  # right after generate, before the neighbour rows
    slot = w.chunks[(1, 0, 0)]
    assert dev.calls[g + 1] == ("set_blocks", [slot, slot], list(edits), list(edits.values()))
    assert dev.vox[slot][_index(40, 5, 5)] == STONE and dev.vox[slot][_index(33, 1, 2)] == 0
    assert sum(n == "set_blocks" for n in names) == 1  # only the chunk with edits


def test_without_edits_a_camera_walk_makes_the_same_device_calls(ob):
    """The device of test_world_stream has no set_blocks: a World without edits never needs it."""
    runs = []
    for dev in (FakeDevice(ob, vxw.sphere_capacity(2)), FakeDeviceWithoutEdits(ob, vxw.sphere_capacity(2))):
        w = vxw.World(vxw.WorldConfig(view_distance=2, max_chunks_per_frame=6), device=dev)
        cache = vxw.MeshCache(w)
        for step, pos in enumerate(CAMERA_WALK):
            cam = camera.Camera(pos, 16 / 9, yaw=0.3 * step)
            w.update(cam.position)
            cache.update(w.get_visible_chunks(cam.position))
        runs.append(dev.calls)
    assert runs[0] == runs[1] and len(runs[0]) > 10


def test_refresh_remeshes_only_cached_chunks_in_one_call(ob):
    w, dev = _world(ob)
    cache = vxw.MeshCache(w)
    cache.update([(0, 0, 0), (1, 0, 0)])
    del dev.calls[:]
    dirty = w.set_blocks([(0, 5, 5)], STONE)  # local x = 0: (-1,0,0) is dirty too, but has no cache entry
    assert dirty == [(-1, 0, 0), (0, 0, 0)]
    assert cache.refresh(dirty + [(9, 9, 9)]) == [(0, 0, 0)]
    assert [c[0] for c in dev.calls] == ["set_blocks", "remesh"] and dev.calls[-1] == ("remesh", [w.chunks[(0, 0, 0)]])
    assert cache.refresh([]) == [] and len(dev.calls) == 2


def test_world_raycast_and_pick_on_the_fake_device(ob):
    w, dev = _world(ob, vd=1, center=(0.0, 10.0, 0.0))
    # straight down from above the terrain onto the surface of column (3, 3)
    r = w.raycast([(3.5, 31.5, 3.5), (3.5, 31.5, 3.5), (1e9, 0, 0)], [(0, -1, 0), (0, 1, 0), (1, 0, 0)], 100.0)
    h = worldgen.terrain_heights(3, 3, 1, 1)[0, 0]
    assert r["status"].tolist() == [HIT, LEFT, INVALID]
    assert r["voxel"][0].tolist() == [3, int(h), 3] and r["face"][0] == 2 and r["block_type"][0] == 1  # grass, entered through +Y
    assert r["chunk"][0].tolist() == [0, int(h) >> 5, 0] and r["local"][0].tolist() == [3, int(h) & 31, 3]
    assert r["distance"][0] == pytest.approx(31.5 - (h + 1)) and np.isinf(r["distance"][1])
    # break the block and cast again: the ray goes one voxel further
    w.set_blocks([r["voxel"][0]], 0)
    r2 = w.raycast([(3.5, 31.5, 3.5)], [(0, -1, 0)], 100.0)
    assert r2["voxel"][0].tolist() == [3, int(h) - 1, 3] and r2["block_type"][0] == 2
    cam = camera.Camera((0.0, 20.0, 20.0), 16 / 9, pitch=-0.6)
    p = w.pick(cam.position, cam.view_projection(), [(80, 45)], 160, 90, 200.0)
    assert p["status"][0] == HIT and p["t"][0] > 0


# ---- pixel rays ------------------------------------------------------------------------------------------------------

def test_pixel_rays_go_through_the_pixel_centres():
    cam = camera.Camera((1.0, 10.0, 20.0), 320 / 180, yaw=0.4, pitch=-0.2)
    vp = cam.view_projection()
    px = np.array([(0, 0), (159, 90), (319, 179), (17, 123)])
    o, d = api.pixel_rays(vp, cam.position, px, 320, 180)
    assert o.dtype == np.float32 and d.dtype == np.float32 and o.shape == d.shape == (4, 3)
    assert np.array_equal(o, np.repeat(cam.position.reshape(1, 3), 4, axis=0))
    assert np.allclose(np.linalg.norm(d.astype(np.float64), axis=1), 1.0, atol=1e-6)
    m = vp.reshape(4, 4).T.astype(np.float64)
    for (x, y), dd in zip(px.tolist(), d.astype(np.float64)):
        clip = m @ np.append(cam.position.astype(np.float64) + 50.0 * dd, 1.0)
        sx = (clip[0] / clip[3] + 1) * 0.5 * 320
        sy = (1 - clip[1] / clip[3]) * 0.5 * 180
        assert sx == pytest.approx(x + 0.5, abs=1e-3) and sy == pytest.approx(y + 0.5, abs=1e-3)


# ---- ABI -------------------------------------------------------------------------------------------------------------

def test_ray_hit_layout_constants_and_symbols(tmp_path):
    fields = [f for f, _ in _lib.VxRayHit._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "vx_b200.h"', "int main(void) {",
             '    printf("%zu", sizeof(VxRayHit));']
    lines += [f'    printf(" %zu", offsetof(VxRayHit, {f}));' for f in fields]
    lines += ['    printf(" %d %d %d %d\\n", VX_RAY_HIT, VX_RAY_MISS, VX_RAY_LEFT_WORLD, VX_RAY_INVALID);', "    return 0;", "}"]
    src = tmp_path / "ray_abi.c"
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "ray_abi"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, timeout=60, check=True).stdout.split()]
    assert out[0] == ctypes.sizeof(_lib.VxRayHit) == api.RAY_HIT_DTYPE.itemsize == 32
    assert out[1:1 + len(fields)] == [getattr(_lib.VxRayHit, f).offset for f in fields]
    assert out[1:1 + len(fields)] == [api.RAY_HIT_DTYPE.fields[f][1] for f in fields]
    assert out[1 + len(fields):] == [HIT, MISS, LEFT, INVALID] == [0, 1, 2, 3]
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for sym in ("vx_world_batch_set_blocks", "vx_world_raycast", "vx_world_raycast_device"):
        assert hasattr(lib, sym) and sym in _lib.PROTOTYPES
