"""Swept-box collision without a GPU: the exact semantics of vx_world_move_boxes (include/vx_b200.h) pinned on the CPU
oracle (tests/move_oracle.c, vxo_move_boxes) with answers worked out by hand, World.move_boxes against a recording fake
device, and the ABI of the move flags."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import vx_move_oracle
from differential_projection_voxel_renderer_b200 import _lib, camera, world as vxw, worldgen
from test_block_edit import STONE, UNIFORM_AIR, UNIFORM_STONE, FakeDevice as FakeDeviceWithoutMoves, Slots
from test_world_stream import CAMERA_WALK

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNLOADED, INVALID = _lib.MOVE_TOUCHED_UNLOADED, _lib.MOVE_INVALID
PX, NX, PY, NY, PZ, NZ = (1 << f for f in range(6))  # blocked-move bits in FaceDir order
F32 = np.float32


def move(w, p, s, d, slot=0):
    """One box through the oracle over a Slots world: (pos, slot, flags, voxel bytes read)."""
    pos, slots, flags, reads = vx_move_oracle.move_boxes(w.pos, w.vox, w.flags, w.nbr, np.array([p], F32), np.array([s], F32),
                                                       np.array([d], F32), np.array([slot], np.int32), want_reads=True)
    return pos[0], int(slots[0]), int(flags[0]), int(reads[0])


def same_bits(got, want):
    assert np.array_equal(np.asarray(got, F32).view(np.uint32), np.asarray(want, F32).view(np.uint32)), (got, want)


def slot_of(w, chunk):
    return int(np.flatnonzero((w.pos == chunk).all(axis=1))[0])


def _key(f):
    b = int(F32(f).view(np.uint32))
    return b if b < 1 << 31 else -(b & 0x7FFFFFFF) - 1


def _from_key(k):
    return np.array(k if k >= 0 else (-(k + 1)) | 0x80000000, np.uint32).view(F32)[()]


def largest_fitting(top, s):
    """The largest f32 m with fl(m + s) <= top, found independently of the kernel: f32 + f32 rounded in f64 and then to
    f32 is the f32 sum (53 >= 2 * 24 + 2 bits: double rounding is innocuous), bisected over all finite f32."""
    fits = lambda m: F32(np.float64(m) + np.float64(s)) <= F32(top)
    lo, hi = _key(-np.finfo(F32).max), _key(np.finfo(F32).max)
    assert fits(_from_key(lo)) and not fits(_from_key(hi))
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if fits(_from_key(mid)) else (lo, mid)
    return _from_key(lo)


# ---- oracle known answers ----------------------------------------------------------------------------------------------

def test_a_falling_player_box_lands_on_flat_ground_at_an_exact_integer():
    w = Slots([((0, 0, 0), 0)])
    for x in range(32):
        for z in range(32):
            w.set((x, 4, z))
    p, slot, flags, reads = move(w, (3.2, 7.3, 5.1), (0.6, 1.8, 0.6), (0, -5, 0))
    same_bits(p, (3.2, 5.0, 5.1))  # layers 6, 5 are air, 4 is stone: the box rests on y = 5
    assert (slot, flags, reads) == (0, NY, 3)
    p, _, flags, _ = move(w, (3.2, 7.3, 5.1), (0.6, 1.8, 0.6), (0, -1, 0))
    same_bits(p, (3.2, F32(7.3) - F32(1), 5.1))
    assert flags == 0
    # resting on the ground: blocked at once, still on the ground
    p, _, flags, reads = move(w, (3.2, 5.0, 5.1), (0.6, 1.8, 0.6), (0.25, -0.08, 0))
    same_bits(p, (F32(3.2) + F32(0.25), 5.0, 5.1))
    assert flags == NY and reads == 1 + 2  # the stone layer below, then layer x = 4 (y = 5, 6) of the X move


@pytest.mark.parametrize("face", range(6))
def test_a_wall_in_each_direction_stops_the_box_flush_against_it(face):
    a, sign = face // 2, (1 if face % 2 == 0 else -1)
    w = Slots([((0, 0, 0), 0)])
    wall = [16, 16, 16]
    wall[a] += 3 * sign
    w.set(tuple(wall))
    d = [0.0, 0.0, 0.0]
    d[a] = 5.0 * sign
    p, slot, flags, reads = move(w, (16, 16, 16), (1, 1, 1), d)
    want = [16.0, 16.0, 16.0]
    want[a] = 18.0 if sign > 0 else 14.0  # flush against the wall's face, never into it
    same_bits(p, want)
    assert (slot, flags, reads) == (0, 1 << face, 3)  # layers 17, 18, 19 (or 15, 14, 13)
    # beyond the swept layers (17 .. 21 or 15 .. 11): no block, the whole delta
    w.vox[:] = 0
    wall[a] += 3 * sign
    w.set(tuple(wall))
    p, _, flags, _ = move(w, (16, 16, 16), (1, 1, 1), d)
    want[a] = 16.0 + d[a]
    same_bits(p, want)
    assert flags == 0


def _snap_cases():
    """(L, s) pairs for which the blocked + move needs each correction of its first guess m = fl(L - s): one where
    fl(m + s) > L (one ulp down), one where the next f32 above m still fits (one ulp up).  Searched over seeded random
    inputs; each turns up about once in 10^4 to 10^5."""
    rng = np.random.default_rng(11)
    L = rng.integers(-(1 << 19), 1 << 19, 4_000_000).astype(F32)
    s = (rng.random(4_000_000) * 16.0).astype(F32)
    s[s == 0] = F32(0.5)
    m = L - s
    down = np.flatnonzero(m + s > L)
    up = np.flatnonzero(np.nextafter(m, F32(np.inf)) + s <= L)
    assert down.size and up.size
    return [("down", int(L[down[0]]), s[down[0]]), ("up", int(L[up[0]]), s[up[0]])]


@pytest.mark.parametrize("which,L,s", _snap_cases())
def test_the_plus_snap_corrects_its_first_guess_both_ways(which, L, s):
    m0 = F32(L) - s
    if which == "down":
        assert m0 + s > F32(L)
    else:
        assert np.nextafter(m0, F32(np.inf)) + s <= F32(L)
    # a box whose top lies half a voxel below layer L, moving +X by 1: layer L is the only layer scanned, and it is stone
    x0 = F32(m0 - F32(0.5))
    chunks = sorted({(int(np.floor(x0)) >> 5, 0, 0), (L >> 5, 0, 0)})
    w = Slots([(c, 0) for c in chunks])
    w.set((L, 0, 0))
    p, slot, flags, reads = move(w, (x0, 0.5, 0.5), (s, s, s), (1, 0, 0), slot=slot_of(w, (int(np.floor(x0)) >> 5, 0, 0)))
    assert flags == PX and reads == 1
    want = largest_fitting(L, s)
    assert want != m0  # the correction was needed
    same_bits(p[0], want)
    assert slot == slot_of(w, (int(np.floor(want)) >> 5, 0, 0))


def test_the_plus_snap_of_a_box_whose_top_guess_is_near_zero_is_bounded():
    """Blocked at L = 16 with s = 16, the first guess fl(L - s) is 0, where the f32 are 2^19 times denser than at 16: the
    answer (2^-20: 16 + 2^-20 is a tie that rounds to the even 16) lies some 2^30 ulps above the guess."""
    w = Slots([((-1, 0, 0), 0), ((0, 0, 0), 0)])
    w.set((16, 1, 0))
    p, slot, flags, reads = move(w, (-0.0935135, 0.5, 0.5), (16, 1.25, 0.5), (0.867, 0, 0), slot=0)
    same_bits(p[0], largest_fitting(16, 16))
    assert p[0] == F32(2.0 ** -20) and (slot, flags) == (1, PX)


def test_a_box_inside_a_block_moves_out_and_is_not_blocked_by_what_it_overlaps():
    w = Slots([((0, 0, 0), 0)])
    w.set((5, 5, 5))
    for d, want in (((0, 1, 0), (5.25, 6.25, 5.25)), ((0, -1, 0), (5.25, 4.25, 5.25)), ((1, 0, 0), (6.25, 5.25, 5.25)),
                    ((0, 0, -1), (5.25, 5.25, 4.25))):
        p, _, flags, _ = move(w, (5.25, 5.25, 5.25), (0.5, 0.5, 0.5), d)
        same_bits(p, want)
        assert flags == 0
    # a box overlapping stone on its bottom row walks sideways through air above the stone... and is stopped by new stone
    w.set((7, 5, 5))
    p, _, flags, _ = move(w, (5.0, 5.5, 5.0), (1.0, 1.0, 1.0), (3, 0, 0))
    same_bits(p, (6.0, 5.5, 5.0))
    assert flags == PX


def test_zero_delta_moves_nothing_and_reads_nothing():
    w = Slots([((0, 0, 0), 0)])
    w.set((5, 5, 5))
    for d in ((0, 0, 0), (-0.0, 0.0, -0.0)):
        p, slot, flags, reads = move(w, (5.25, 5.25, 5.25), (0.5, 0.5, 0.5), d)
        same_bits(p, (5.25, 5.25, 5.25))
        assert (slot, flags, reads) == (0, 0, 0)


def test_a_delta_of_exactly_sixteen_crosses_into_the_next_chunk():
    w = Slots([((0, 0, 0), 0), ((1, 0, 0), 0), ((2, 0, 0), 0)])
    p, slot, flags, reads = move(w, (63.5, 0.5, 0.5), (16, 16, 16), (16, 0, 0), slot=1)
    same_bits(p, (79.5, 0.5, 0.5))  # layers 80 .. 95, all in chunk 2
    assert (slot, flags, reads) == (2, 0, 16 * 17 * 17)
    w.set((20, 3, 3))
    p, slot, flags, _ = move(w, (32.0, 0.5, 0.5), (16, 16, 16), (-16, 0, 0), slot=1)
    same_bits(p, (21.0, 0.5, 0.5))  # layers 31 down to 16: stone at 20
    assert (slot, flags) == (0, NX)
    p, slot, flags, _ = move(w, (63.96875, 31.5, 0.5), (16, 0.5, 0.5), (16, 0, 0), slot=1)  # the farthest layer: 95
    same_bits(p, (79.96875, 31.5, 0.5))
    assert (slot, flags) == (2, 0)


def test_uniform_solid_and_uniform_air_chunks_need_no_voxel_rows():
    w = Slots([((0, 0, 0), 0), ((0, -1, 0), UNIFORM_STONE)])
    w.vox[1] = 0  # a Uniform chunk's rows are never read: air rows under a Uniform stone flag
    p, slot, flags, reads = move(w, (3.5, 3.5, 3.5), (0.5, 0.5, 0.5), (0, -8, 0))
    same_bits(p, (3.5, 0.0, 3.5))
    assert (slot, flags, reads) == (0, NY, 3)  # layers 2, 1, 0 read; -1 judged by its flag
    w = Slots([((0, 0, 0), 0), ((0, -1, 0), UNIFORM_AIR)])
    w.vox[1] = STONE  # stone rows under a Uniform air flag
    p, slot, flags, reads = move(w, (3.5, 3.5, 3.5), (0.5, 0.5, 0.5), (0, -8, 0))
    same_bits(p, (3.5, -4.5, 3.5))
    assert (slot, flags, reads) == (1, 0, 3)


def test_an_unloaded_neighbour_is_a_wall_and_sets_bit_six():
    w = Slots([((0, 0, 0), 0)])
    p, slot, flags, reads = move(w, (30.5, 5, 5), (1, 1, 1), (3, 0, 0))
    # flush against x = 32: fl(31 + 2^-19 + 1) is a tie that rounds to the even 32, so the box ends one ulp beyond 31
    same_bits(p, (largest_fitting(32, 1), 5.0, 5.0))
    assert p[0] == np.nextafter(F32(31), F32(32))
    assert (slot, flags, reads) == (0, PX | UNLOADED, 0)
    p, _, flags, _ = move(w, (5, 0.5, 5), (1, 1, 1), (0, -2, 0))
    same_bits(p, (5.0, 0.0, 5.0))
    assert flags == NY | UNLOADED
    # a box already reaching into the unloaded chunk is stopped by its next layer; its corner now lies there: slot -1
    p, slot, flags, _ = move(w, (31.5, 5, 5), (1, 1, 1), (0.75, 0, 0))
    same_bits(p, (32.0, 5.0, 5.0))
    assert (slot, flags) == (-1, PX | UNLOADED)
    assert move(w, p, (1, 1, 1), (0.75, 0, 0), slot=slot)[2] == INVALID
    # stone blocks before the unloaded chunk: bit 6 stays clear
    w.set((31, 5, 5))
    assert move(w, (29.0, 5, 5), (1, 1, 1), (10, 0, 0))[2] == PX


def test_a_loaded_chunk_off_the_x_y_z_hop_path_counts_as_not_loaded():
    w = Slots([((0, 0, 0), 0), ((0, 1, 0), 0), ((1, 1, 0), 0)])  # (1, 0, 0) is not loaded
    p, slot, flags, _ = move(w, (31.0, 31.5, 5.0), (0.5, 0.25, 0.5), (1, 1, 0))
    # Y first: into chunk (0, 1, 0); then X: layer 32 is in (1, 1, 0), reached from slot (0, 0, 0) through (1, 0, 0)
    same_bits(p, (largest_fitting(32, 0.5), 32.5, 5.0))
    assert (slot, flags) == (slot_of(w, (0, 1, 0)), PX | UNLOADED)
    # from the new slot the X hop reaches (1, 1, 0) directly
    x = p[0]
    p, slot, flags, _ = move(w, p, (0.5, 0.25, 0.5), (1, 0, 0), slot=slot)
    same_bits(p, (x + F32(1), 32.5, 5.0))
    assert (slot, flags) == (slot_of(w, (1, 1, 0)), 0)


@pytest.mark.parametrize("p,s,d,slot", [
    ((np.nan, 1, 1), (1, 1, 1), (0, 0, 0), 0),              # NaN position
    ((1, 1, 1), (1, np.inf, 1), (0, 0, 0), 0),              # infinite size
    ((1, 1, 1), (1, 1, 1), (0, 0, np.nan), 0),              # NaN delta
    ((1, 1, 1), (1, 1, 1), (-np.inf, 0, 0), 0),             # infinite delta
    ((1, 1, 1), (0, 1, 1), (1, 0, 0), 0),                   # empty extent
    ((1, 1, 1), (1, -1, 1), (1, 0, 0), 0),                  # negative extent
    ((1, 1, 1), (1, 1, np.nextafter(F32(16), F32(99))), (1, 0, 0), 0),  # extent above 16
    ((1, 1, 1), (1, 1, 1), (np.nextafter(F32(16), F32(99)), 0, 0), 0),   # delta above 16
    ((1, 1, 1), (1, 1, 1), (0, -np.nextafter(F32(16), F32(99)), 0), 0),  # delta below -16
    ((1048576.0, 1, 1), (1, 1, 1), (1, 0, 0), 2),           # |p| = 2^20 (slot 2 is the chunk at x = 2^20 / 32)
    ((-1048576.0, 1, 1), (1, 1, 1), (1, 0, 0), 3),          # |p| = 2^20, negative
    ((1000000.0, 1, 1), (0.01, 1, 1), (1, 0, 0), 4),        # fl(p + s) == p: a degenerate box
    ((1, 1, 1), (1, 1, 1), (1, 0, 0), -1),                  # not loaded
    ((1, 1, 1), (1, 1, 1), (1, 0, 0), 1),                   # the slot of another chunk
    ((1, 1, 1), (1, 1, 1), (1, 0, 0), 5),                   # beyond the batch
])
def test_invalid_boxes_are_left_where_they_are(p, s, d, slot):
    w = Slots([((0, 0, 0), 0), ((1, 0, 0), 0), ((32768, 0, 0), 0), ((-32768, 0, 0), 0), ((31250, 0, 0), 0)])
    got, got_slot, flags, reads = move(w, p, s, d, slot=slot)
    same_bits(got, p)
    assert (got_slot, flags, reads) == (slot, INVALID, 0)


def test_sixteen_is_a_valid_extent_and_delta_and_fl_p_plus_s_decides_degeneracy():
    w = Slots([((0, 0, 0), 0), ((31250, 0, 0), 0)])
    assert move(w, (1, 1, 1), (16, 16, 16), (-16, 16, 0))[2] & INVALID == 0
    ulp = F32(0.0625)  # the spacing of f32 at 10^6
    p, _, flags, _ = move(w, (1000000.0, 1, 1), (ulp, 1, 1), (0, 0, 1), slot=1)
    same_bits(p, (1000000.0, 1, 2))
    assert flags == 0


# ---- World with a recording fake device ---------------------------------------------------------------------------------

class FakeDevice(FakeDeviceWithoutMoves):
    """test_block_edit's recorder plus vx_world_move_boxes through the oracle over the slot arrays, in place like the C call."""

    def move_boxes(self, pos, size, delta, slots):
        assert pos.dtype == size.dtype == delta.dtype == np.float32 and slots.dtype == np.int32
        assert pos.flags.c_contiguous and size.shape == delta.shape == pos.shape and slots.shape == (pos.shape[0],)
        P = np.zeros((self.capacity, 3), np.int32)
        vox = np.zeros((self.capacity, 32768), np.uint8)
        flags = np.ones(self.capacity, np.uint8)
        for s in self.pos:
            P[s], vox[s], flags[s] = self.pos[s], self.vox[s], self.flag[s]
        nbr = np.array([self.nbr[s] for s in range(self.capacity)], dtype=np.int32)
        self.calls.append(("move_boxes", slots.tolist()))
        new_pos, new_slots, out = vx_move_oracle.move_boxes(P, vox, flags, nbr, pos, size, delta, slots)
        pos[:] = new_pos
        slots[:] = new_slots
        return out


def _world(ob, vd=1, center=(0.0, 10.0, 0.0)):
    dev = FakeDevice(ob, vxw.sphere_capacity(vd))
    w = vxw.World(vxw.WorldConfig(view_distance=vd, max_chunks_per_frame=1000), device=dev)
    w.update(center)
    return w, dev


def test_world_move_boxes_lands_on_the_terrain_and_decodes_the_flags(ob):
    w, dev = _world(ob)
    h = int(worldgen.terrain_heights(3, 3, 1, 1)[0, 0])  # the column's top solid voxel
    start = np.array([(3.2, h + 6.5, 3.2), (np.nan, 0, 0), (5.0 * 32, 0.0, 0.0), (10.1, h + 40.0, 10.1)], F32)
    keep = start.copy()
    r = w.move_boxes(start, (0.6, 1.8, 0.6), [(0, -8, 0), (0, -1, 0), (0, -1, 0), (0, 0, 0)])
    assert np.array_equal(start, keep, equal_nan=True)  # the caller's array is not modified
    assert dev.calls[-1] == ("move_boxes", w.start_slots(keep).tolist())
    same_bits(r["pos"][0], (3.2, h + 1, 3.2))
    assert r["on_ground"].tolist() == [True, False, False, False]
    assert r["invalid"].tolist() == [False, True, True, False]  # NaN; a chunk that is not loaded (slot -1)
    assert r["flags"].tolist() == [NY, INVALID, INVALID, 0] and not r["touched_unloaded"].any()
    assert r["blocked"].shape == (4, 6) and r["blocked"].tolist()[0] == [False, False, False, True, False, False]
    assert r["slot"].tolist() == [w.chunks[(0, (h + 1) >> 5, 0)], -1, -1, w.start_slots(keep[3:])[0]]
    same_bits(r["pos"][1:], keep[1:])
    # into the top of the loaded world: unloaded space stops the box
    top = max(p[1] for p in w.chunks if p[0] == 0 and p[2] == 0) * 32 + 31
    r = w.move_boxes([(3.2, top - 2.0, 3.2)], (0.6, 1.8, 0.6), (0, 5, 0))
    same_bits(r["pos"][0], (3.2, largest_fitting(top + 1, F32(1.8)), 3.2))
    assert r["blocked"][0, 2] and r["touched_unloaded"][0] and r["flags"][0] == PY | UNLOADED


def test_without_moves_a_camera_walk_makes_the_same_device_calls(ob):
    """World never calls move_boxes by itself: a world without moves drives the device exactly as before."""
    runs = []
    for dev in (FakeDevice(ob, vxw.sphere_capacity(2)), FakeDeviceWithoutMoves(ob, vxw.sphere_capacity(2))):
        w = vxw.World(vxw.WorldConfig(view_distance=2, max_chunks_per_frame=6), device=dev)
        cache = vxw.MeshCache(w)
        for step, pos in enumerate(CAMERA_WALK):
            cam = camera.Camera(pos, 16 / 9, yaw=0.3 * step)
            w.update(cam.position)
            cache.update(w.get_visible_chunks(cam.position))
        runs.append(dev.calls)
    assert runs[0] == runs[1] and len(runs[0]) > 10


# ---- ABI ---------------------------------------------------------------------------------------------------------------

def test_move_flag_constants_and_symbols(tmp_path):
    src = tmp_path / "move_abi.c"
    src.write_text('#include <stdio.h>\n#include "vx_b200.h"\n'
                   'int main(void) { printf("%d %d\\n", VX_MOVE_TOUCHED_UNLOADED, VX_MOVE_INVALID); return 0; }\n')
    exe = tmp_path / "move_abi"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60, check=True).stdout.split()
    assert [int(v) for v in out] == [_lib.MOVE_TOUCHED_UNLOADED, _lib.MOVE_INVALID] == [64, 128]
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for sym in ("vx_world_move_boxes", "vx_world_move_boxes_device"):
        assert hasattr(lib, sym) and sym in _lib.PROTOTYPES
