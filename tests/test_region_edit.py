"""Region edits without a GPU: the exact semantics of vx_world_batch_fill_regions (include/vx_b200.h) pinned on the CPU oracle
(tests/region_oracle.c) with answers worked out by hand, the ABI of VxRegionOp, and World's fill bookkeeping (the chunks a
fill needs, folding into `edits`, replay after unloading, the chunks it dirties) against a fake device backed by the oracle."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import vx_region_oracle as vro
from differential_projection_voxel_renderer_b200 import _lib, api, camera, world as vxw
from test_block_edit import FakeDevice as FakeDeviceWithEdits, _index
from test_world_stream import CAMERA_WALK, FakeDevice as FakeDeviceWithoutEdits

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOX, BALL = _lib.REGION_BOX, _lib.REGION_BALL
AIR, GRASS, DIRT, STONE = 0, 1, 2, 3
UNIFORM_AIR, UNIFORM_STONE = 1, 4
PX, NX, PY, NY, PZ, NZ, CHANGED = 1, 2, 4, 8, 16, 32, 64


# ---- oracle known answers -----------------------------------------------------------------------------------------------

class Slots:
    """A hand-built world batch: slot-indexed positions, voxels and Uniform flags."""

    def __init__(self, chunks):
        self.pos = np.array([p for p, _ in chunks], dtype=np.int32).reshape(-1, 3)
        self.flags = np.array([f for _, f in chunks], dtype=np.uint8)
        self.vox = np.zeros((len(chunks), 32768), dtype=np.uint8)

    def slot(self, p):
        return int(np.flatnonzero((self.pos == p).all(axis=1))[0])

    def at(self, xyz):
        x, y, z = xyz
        s = self.slot((x >> 5, y >> 5, z >> 5))
        return int(self.flags[s] - 1) if self.flags[s] else int(self.vox[s, _index(x, y, z)])

    def set(self, xyz, t):
        x, y, z = xyz
        self.vox[self.slot((x >> 5, y >> 5, z >> 5)), _index(x, y, z)] = t

    def fill(self, ops, slots=None):
        slots = list(range(self.pos.shape[0])) if slots is None else slots
        rc, changed = vro.fill_regions(self.pos, self.vox, self.flags, np.array(ops), slots)
        assert rc == 0
        return changed.tolist()


def _solid(s, slot):
    """Local (x, y, z) of the non-air voxels of a Varied slot, sorted."""
    i = np.flatnonzero(s.vox[slot])
    return sorted(zip((i & 31).tolist(), ((i >> 5) & 31).tolist(), (i >> 10).tolist()))


def test_box_across_a_chunk_corner_with_negative_coordinates():
    corner = [((x, y, z), 0) for x in (-1, 0) for y in (-1, 0) for z in (-1, 0)]
    s = Slots(corner)
    changed = s.fill([vro.op(BOX, (-2, -2, -2), (1, 1, 1), block_type=STONE)])
    for (p, _), c in zip(corner, changed):
        lo = [30 if q < 0 else 0 for q in p]  # voxel -1 is chunk -1, local 31
        want = sorted((x, y, z) for x in (lo[0], lo[0] + 1) for y in (lo[1], lo[1] + 1) for z in (lo[2], lo[2] + 1))
        assert _solid(s, s.slot(p)) == want
        faces = sum((PX, PY, PZ)[e] if p[e] < 0 else (NX, NY, NZ)[e] for e in range(3))
        assert c == CHANGED | faces, (p, c)
    assert s.at((-2, -2, -2)) == STONE and s.at((-3, -2, -2)) == AIR and s.at((1, 1, 1)) == STONE and s.at((2, 1, 1)) == AIR


def test_ball_boundaries():
    s = Slots([((0, 0, 0), 0)])
    s.fill([vro.op(BALL, (5, 6, 7), radius_sq=0, block_type=STONE)])
    assert _solid(s, 0) == [(5, 6, 7)]
    s.vox[:] = 0
    s.fill([vro.op(BALL, (5, 5, 5), (99, -99, 12345), radius_sq=2, block_type=STONE)])  # b is ignored for a ball
    got = _solid(s, 0)
    assert len(got) == 1 + 6 + 12 and (6, 6, 5) in got and (6, 6, 6) not in got and (7, 5, 5) not in got
    s.vox[:] = 0
    s.fill([vro.op(BALL, (10, 10, 10), radius_sq=9, block_type=STONE)])  # r = 3 on the axes, (2, 2, 1) inside, (2, 2, 2) not
    got = set(_solid(s, 0))
    assert (13, 10, 10) in got and (14, 10, 10) not in got and (12, 12, 11) in got and (12, 12, 12) not in got
    assert len(got) == sum(1 for d in np.ndindex(7, 7, 7) if sum((c - 3) ** 2 for c in d) <= 9)


@pytest.mark.parametrize("mask", range(16))
def test_every_replace_mask(mask):
    s = Slots([((0, 0, 0), 0)])
    s.vox[0] = np.arange(32768) % 4  # every type in each row
    changed = s.fill([vro.op(BOX, (0, 0, 0), (31, 31, 31), block_type=DIRT, replace=mask)])
    t = np.arange(32768) % 4
    want = np.where((mask >> t) & 1 == 1, DIRT, t)
    assert np.array_equal(s.vox[0], want)
    d = (want != t).reshape(32, 32, 32)  # z, y, x
    planes = [d[:, :, 31], d[:, :, 0], d[:, 31, :], d[:, 0, :], d[31], d[0]]
    assert changed == [(CHANGED if d.any() else 0) | sum(1 << f for f, pl in enumerate(planes) if pl.any())]
    assert bool(changed[0] & NX) == bool(mask & 1 << AIR) and bool(changed[0] & PX) == bool(mask & 1 << STONE)  # x = 0 air, x = 31 stone


def test_air_only_places_without_overwriting_and_solid_only_carves():
    s = Slots([((0, 0, 0), 0)])
    s.set((4, 4, 4), GRASS)
    s.fill([vro.op(BOX, (3, 3, 3), (5, 5, 5), block_type=STONE, replace=1 << AIR)])
    assert s.at((4, 4, 4)) == GRASS and s.at((3, 3, 3)) == STONE and len(_solid(s, 0)) == 27
    s.fill([vro.op(BALL, (4, 4, 4), radius_sq=1, block_type=AIR, replace=0b1110)])
    assert s.at((4, 4, 4)) == AIR and s.at((5, 4, 4)) == AIR and s.at((5, 5, 4)) == STONE and len(_solid(s, 0)) == 20


def test_uniform_chunk_the_op_leaves_alone_stays_uniform_and_its_rows_are_not_written():
    s = Slots([((0, 0, 0), UNIFORM_STONE), ((1, 0, 0), UNIFORM_AIR)])
    s.vox[:] = 7  # rows of a Uniform slot are not its voxels: never read, never written
    assert s.fill([vro.op(BOX, (0, 0, 0), (40, 9, 9), block_type=DIRT, replace=1 << AIR)], [0]) == [0]  # mask excludes stone
    assert s.fill([vro.op(BOX, (0, 0, 0), (9, 9, 9), block_type=STONE)], [0]) == [0]                     # the type is equal
    assert s.fill([vro.op(BALL, (40, 5, 5), radius_sq=16, block_type=AIR)], [1]) == [0]
    assert s.flags.tolist() == [UNIFORM_STONE, UNIFORM_AIR] and (s.vox == 7).all()


def test_a_uniform_chunk_turned_varied_stays_varied_when_a_later_op_restores_it():
    s = Slots([((0, 0, 0), UNIFORM_AIR), ((1, 0, 0), 0)])
    s.vox[:] = 7
    s.vox[1] = 0
    ops = [vro.op(BOX, (31, 2, 2), (33, 4, 4), block_type=STONE), vro.op(BOX, (0, 0, 0), (40, 31, 31), block_type=AIR)]
    assert s.fill(ops) == [CHANGED, 0]  # no voxel differs in the end: no face bit; the Varied slot reports nothing
    assert s.flags.tolist() == [0, 0] and (s.vox == 0).all()  # the rows were filled with air, then the ops landed


@pytest.mark.parametrize("local,bits", [((31, 5, 6), PX), ((0, 5, 6), NX), ((5, 31, 6), PY), ((5, 0, 6), NY), ((5, 6, 31), PZ),
                                        ((5, 6, 0), NZ), ((0, 0, 0), NX | NY | NZ), ((31, 31, 31), PX | PY | PZ), ((5, 6, 7), 0)])
def test_border_face_bits(local, bits):
    s = Slots([((2, -3, 1), 0)])
    v = np.array(local) + np.array([64, -96, 32])
    assert s.fill([vro.op(BOX, v, v, block_type=STONE)]) == [CHANGED | bits]
    assert s.fill([vro.op(BOX, v, v, block_type=STONE)]) == [0]  # already stone: nothing differs


def test_an_op_that_only_reaches_other_chunks_changes_nothing():
    s = Slots([((0, 0, 0), 0), ((5, 0, 0), UNIFORM_AIR)])
    assert s.fill([vro.op(BALL, (100, 5, 5), radius_sq=400, block_type=STONE)]) == [0, 0]
    assert (s.vox == 0).all() and s.flags.tolist() == [0, UNIFORM_AIR]
    assert s.fill([vro.op(BOX, (0, 0, 0), (5, 5, 5), block_type=STONE)], []) == []


C29, R56 = 1 << 29, 1 << 56


@pytest.mark.parametrize("ops,slots", [
    ([vro.op(BOX, (0, 0, 0), (1, 1, 1), block_type=STONE)], [-1]),         # slot below the batch
    ([vro.op(BOX, (0, 0, 0), (1, 1, 1), block_type=STONE)], [2]),          # slot beyond the batch
    ([vro.op(BOX, (0, 0, 0), (1, 1, 1), block_type=STONE)], [1, 0, 1]),    # slot listed twice
    ([vro.op(2, (0, 0, 0), (1, 1, 1), block_type=STONE)], [0]),            # bad shape
    ([vro.op(-1, (0, 0, 0), (1, 1, 1), block_type=STONE)], [0]),           # bad shape
    ([vro.op(BOX, (0, 0, 0), (1, 1, 1), block_type=4)], [0]),              # block type above 3
    ([vro.op(BOX, (0, 0, 0), (1, 1, 1), block_type=STONE, replace=16)], [0]),  # replace mask above 15
    ([vro.op(BOX, (C29 + 1, 0, 0), (C29 + 1, 1, 1), block_type=STONE)], [0]),  # corner beyond 2^29
    ([vro.op(BOX, (0, 0, 0), (1, 1, C29 + 1), block_type=STONE)], [0]),
    ([vro.op(BOX, (0, -C29 - 1, 0), (1, 1, 1), block_type=STONE)], [0]),
    ([vro.op(BALL, (0, 0, -C29 - 1), radius_sq=4, block_type=STONE)], [0]),    # centre beyond 2^29
    ([vro.op(BALL, (0, 0, 0), radius_sq=-1, block_type=STONE)], [0]),          # radius_sq below 0
    ([vro.op(BALL, (0, 0, 0), radius_sq=R56 + 1, block_type=STONE)], [0]),     # radius_sq above 2^56
    ([vro.op(BOX, (0, 0, 0), (1, 1, 1), block_type=STONE), vro.op(BOX, (0, 0, 0), (1, 1, 1), block_type=5)], [0]),  # a later op
])
def test_invalid_calls_change_nothing(ops, slots):
    s = Slots([((0, 0, 0), 0), ((1, 0, 0), UNIFORM_AIR)])
    rc, changed = vro.fill_regions(s.pos, s.vox, s.flags, np.array(ops), slots)
    assert rc == -1 and not s.vox.any() and s.flags.tolist() == [0, UNIFORM_AIR]


def test_the_bounds_themselves_are_valid():
    s = Slots([((0, 0, 0), 0)])
    ops = [vro.op(BOX, (-C29, -C29, -C29), (C29, C29, C29), block_type=STONE, replace=1 << GRASS),
           vro.op(BALL, (C29, -C29, 0), (-C29 - 5, 0, 0), radius_sq=R56, block_type=DIRT),  # reaches x = 2^29 - 2^28 at the least
           vro.op(BALL, (16, 16, 16), radius_sq=R56, block_type=GRASS, replace=1 << AIR)]
    assert s.fill(ops) == [CHANGED | 63] and (s.vox == GRASS).all()


# ---- ABI -------------------------------------------------------------------------------------------------------------------

def test_region_op_layout_constants_and_symbols(tmp_path):
    fields = [f for f, _ in _lib.VxRegionOp._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "vx_b200.h"', "int main(void) {",
             '    printf("%zu", sizeof(VxRegionOp));']
    lines += [f'    printf(" %zu", offsetof(VxRegionOp, {f}));' for f in fields]
    lines += ['    printf(" %d %d\\n", VX_REGION_BOX, VX_REGION_BALL);', "    return 0;", "}"]
    src = tmp_path / "region_abi.c"
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "region_abi"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, timeout=60, check=True).stdout.split()]
    assert out[0] == ctypes.sizeof(_lib.VxRegionOp) == api.REGION_OP_DTYPE.itemsize == 40
    assert out[1:1 + len(fields)] == [getattr(_lib.VxRegionOp, f).offset for f in fields]
    assert out[1:1 + len(fields)] == [api.REGION_OP_DTYPE.fields[f][1] for f in fields]
    assert out[1 + len(fields):] == [BOX, BALL] == [0, 1]
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for sym in ("vx_world_batch_fill_regions", "vx_world_batch_read_voxels"):
        assert hasattr(lib, sym) and sym in _lib.PROTOTYPES


# ---- World bookkeeping on a fake device backed by the oracle -----------------------------------------------------------

class FakeDevice(FakeDeviceWithEdits):
    """test_block_edit's recorder plus the two calls of this feature: fills go to the region oracle over the listed slots,
    read_voxels returns the slots' rows and flags."""

    def fill_regions(self, ops, slots):
        sl = slots.tolist()
        pos = np.array([self.pos[s] for s in sl], dtype=np.int32).reshape(-1, 3)
        vox = np.stack([self.vox[s] for s in sl]) if sl else np.zeros((0, 32768), np.uint8)
        flags = np.array([self.flag[s] for s in sl], dtype=np.uint8)
        rc, changed = vro.fill_regions(pos, vox, flags, ops, np.arange(len(sl), dtype=np.int32))
        assert rc == 0
        for i, s in enumerate(sl):
            self.vox[s], self.flag[s] = vox[i], int(flags[i])
        self.calls.append(("fill_regions", ops.tobytes(), sl))
        return changed

    def read_voxels(self, slots):
        self.calls.append(("read_voxels", slots.tolist()))
        return np.stack([self.vox[s].copy() for s in slots.tolist()]), np.array([self.flag[s] for s in slots.tolist()], dtype=np.uint8)


def _world(ob, vd=1, center=(0.0, 0.0, 0.0)):
    dev = FakeDevice(ob, vxw.sphere_capacity(vd))
    w = vxw.World(vxw.WorldConfig(view_distance=vd, max_chunks_per_frame=1000), device=dev)
    w.update(center)
    return w, dev


def _state(w, dev, p):
    s = w.chunks[p]
    return dev.flag[s], dev.vox[s].tobytes()


def test_unloaded_chunks_raise_before_anything_changes(ob):
    w, dev = _world(ob)  # the chunk at the origin and its six face neighbours
    n_calls, before = len(dev.calls), {p: _state(w, dev, p) for p in w.chunks}
    with pytest.raises(KeyError):
        w.fill_box((0, 0, 0), (64, 1, 1), STONE)           # reaches (2, 0, 0)
    with pytest.raises(KeyError):
        w.fill_box((31, 31, 0), (32, 32, 0), STONE)        # (1, 1, 0), inside the loaded range on every axis
    with pytest.raises(KeyError):
        w.fill_ball((31, 31, 16), 2, STONE)                # (32, 32, 16) is in (1, 1, 0)
    assert len(dev.calls) == n_calls and not w.fills and {p: _state(w, dev, p) for p in w.chunks} == before
    # the bounding box of this ball reaches (1, 1, 0), none of its voxels do
    assert w.fill_ball((31, 31, 16), 1, STONE) == [(0, 0, 0), (0, 1, 0), (1, 0, 0)]
    assert dev.calls[-1][0] == "fill_regions" and sorted(dev.calls[-1][2]) == sorted(w.chunks[p] for p in [(0, 0, 0), (0, 1, 0), (1, 0, 0)])


def test_empty_regions_and_bad_arguments(ob):
    w, dev = _world(ob)
    n_calls = len(dev.calls)
    assert w.fill_box((5, 5, 5), (4, 9, 9), STONE) == [] and w.fill_ball((5, 5, 5), -1, STONE) == []
    assert w.fill_box((1000, 5, 5), (4, 9, 9), STONE) == []  # empty, so no chunk is needed
    for bad in (lambda: w.fill_box((0, 0, 0), (1, 1, 1), 4), lambda: w.fill_ball((0, 0, 0), 4, STONE, replace=[0, 4]),
                lambda: w.fill_ball((0, 0, 1 << 30), 4, STONE), lambda: w.fill_ball((0, 0, 0), (1 << 56) + 1, STONE)):
        with pytest.raises(ValueError):
            bad()
    assert len(dev.calls) == n_calls and not w.fills


def test_dirty_list_is_the_changed_chunks_and_their_neighbours_across_changed_faces(ob):
    w, dev = _world(ob, center=(0.0, 200.0, 0.0))  # Uniform air chunks around (0, 6, 0)
    y0 = 6 * 32
    assert w.fill_box((4, y0 + 4, 4), (6, y0 + 6, 6), STONE) == [(0, 6, 0)]  # bit 6 without a face bit
    assert w.uniform_flags[(0, 6, 0)] == 0 and w.uniform_flags[(1, 6, 0)] == UNIFORM_AIR
    assert w.fill_box((0, y0 + 4, 4), (0, y0 + 4, 4), STONE) == [(-1, 6, 0), (0, 6, 0)]
    assert w.fill_box((31, y0 + 31, 31), (32, y0 + 31, 31), STONE) == [(0, 6, 0), (0, 6, 1), (0, 7, 0), (1, 6, 0)]
    assert w.fill_ball((5, y0 + 5, 5), 4, STONE, replace=[AIR]) == [(0, 6, 0)]  # reaches (7, 5, 5), beyond the box
    assert w.fill_ball((5, y0 + 5, 5), 3, STONE) == []  # nothing differs
    assert w.fill_ball((16, y0 + 16, 16), 100, AIR, replace=[GRASS, DIRT]) == []
    assert w.uniform_flags[(1, 6, 0)] == 0 and dev.flag[w.chunks[(1, 6, 0)]] == 0


def test_fills_fold_into_edits(ob):
    w, dev = _world(ob)
    w.set_blocks([(5, 5, 5), (6, 5, 5), (20, 20, 20), (33, 5, 5)], [STONE, AIR, STONE, GRASS])
    w.fill_ball((5, 5, 5), 1, DIRT, replace=[STONE])  # (6,5,5) is air: not in the mask; (20,20,20) is outside
    assert w.edits[(0, 0, 0)] == {_index(5, 5, 5): DIRT, _index(6, 5, 5): AIR, _index(20, 20, 20): STONE}
    w.fill_box((6, 5, 5), (40, 5, 5), STONE)  # every type
    assert w.edits[(0, 0, 0)] == {_index(5, 5, 5): DIRT, _index(6, 5, 5): STONE, _index(20, 20, 20): STONE}
    assert w.edits[(1, 0, 0)] == {_index(33, 5, 5): STONE}
    s = w.chunks[(0, 0, 0)]
    for i, t in w.edits[(0, 0, 0)].items():  # `edits` holds the current type of each edited voxel
        assert dev.vox[s][i] == t


def test_fills_and_edits_come_back_after_the_chunks_are_unloaded_and_generated_again(ob):
    w, dev = _world(ob, vd=1, center=(0.0, 20.0, 0.0))
    w.fill_ball((40, 7, 10), 49, AIR, replace=[GRASS, DIRT, STONE])  # carve the terrain surface (heights 1..3) in (1, 0, 0)
    w.set_blocks([(40, 7, 10), (33, 1, 12)], [STONE, AIR])
    w.fill_box((34, 0, 0), (50, 6, 3), DIRT, replace=[AIR])          # fill the air above it
    w.fill_box((0, 40, 0), (3, 43, 3), STONE)                        # (0, 1, 0): Uniform air made Varied by a fill alone
    w.fill_box((10, 50, 10), (10, 50, 10), STONE)
    w.fill_box((10, 50, 10), (10, 50, 10), AIR)                      # (0, 1, 0) keeps a restored voxel
    w.fill_box((33, 0, 0), (40, 20, 3), STONE, replace=[])           # changes nothing: not replayed
    gone = [(1, 0, 0), (0, 1, 0)]
    before = {p: _state(w, dev, p) for p in gone}
    assert all(f == 0 for f, _ in before.values())
    w.update((32.0 * 20, 20.0, 0.0))
    assert not any(p in w.chunks for p in gone)
    del dev.calls[:]
    w.update((0.0, 20.0, 0.0))
    assert {p: _state(w, dev, p) for p in gone} == before and all(w.uniform_flags[p] == 0 for p in gone)
    names = [c[0] for c in dev.calls]
    g = names.index("generate")
    assert names[g + 1:g + 3] == ["fill_regions", "set_blocks"], names
    ops = np.frombuffer(dev.calls[g + 1][1], dtype=api.REGION_OP_DTYPE)
    assert ops.tobytes() == np.stack(w.fills[:-1]).tobytes()  # the fills that changed one of the two chunks, in issue order
    assert sorted(dev.calls[g + 1][2]) == sorted(w.chunks[p] for p in gone)
    assert names.count("fill_regions") == 1


def test_chunk_voxels_reads_flags_and_voxels(ob):
    w, dev = _world(ob, center=(0.0, 200.0, 0.0))
    flag, v = w.chunk_voxels((0, 6, 0))
    assert flag == UNIFORM_AIR and v.shape == (32, 32, 32) and not v.any()
    w.fill_box((1, 6 * 32 + 2, 3), (1, 6 * 32 + 2, 3), DIRT)
    flag, v = w.chunk_voxels((0, 6, 0))
    assert flag == 0 and v[3, 2, 1] == DIRT and int(v.sum()) == DIRT
    with pytest.raises(KeyError):
        w.chunk_voxels((50, 0, 0))


def test_without_fills_a_camera_walk_makes_the_same_device_calls(ob):
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


def test_region_contains_agrees_with_the_oracle():
    rng = np.random.default_rng(3)
    s = Slots([((x, y, z), 0) for x in (-1, 0) for y in (-1, 0) for z in (-1, 0)])
    for _ in range(20):
        shape = int(rng.integers(0, 2))
        a = rng.integers(-40, 40, 3)
        op = vro.op(shape, a, a + rng.integers(-3, 30, 3), radius_sq=int(rng.integers(0, 900)), block_type=STONE)
        s.vox[:] = 0
        s.fill([op])
        v = np.stack(np.meshgrid(np.arange(-32, 32), np.arange(-32, 32), np.arange(-32, 32), indexing="ij"), -1).reshape(-1, 3)
        inside = vxw.region_contains(op, v)
        assert [s.at(tuple(p)) == STONE for p in v[::97].tolist()] == inside[::97].tolist()
