"""Copy and paste without a GPU: the exact semantics of vx_world_batch_copy_region and vx_world_batch_paste
(include/vx_b200.h) pinned on the CPU oracle (tests/paste_oracle.c) with answers worked out by hand, the ABI of VxPasteOp,
and World's copy / paste bookkeeping (the chunks a paste needs, folding into `edits`, replay with the fills after
unloading, the chunks it dirties) against a fake device backed by the oracles."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import vx_paste_oracle as vpo
from differential_projection_voxel_renderer_b200 import _lib, api, camera, world as vxw
from test_block_edit import _index
from test_region_edit import FakeDevice as FakeDeviceWithFills, Slots, _solid
from test_world_stream import CAMERA_WALK

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SKIP = api.PASTE_SKIP
AIR, GRASS, DIRT, STONE = 0, 1, 2, 3
UNIFORM_AIR, UNIFORM_STONE = 1, 4
PX, NX, PY, NY, PZ, NZ, CHANGED = 1, 2, 4, 8, 16, 32, 64
C29 = 1 << 29


def _paste(s, items, slots=None, replace=0xF):
    """Paste [(origin, template)] into the hand-built world s (test_region_edit.Slots) in one call; returns the change bytes."""
    ops, blob = vpo.pack(items, replace)
    slots = list(range(s.pos.shape[0])) if slots is None else slots
    rc, changed = vpo.paste(s.pos, s.vox, s.flags, ops, blob, slots)
    assert rc == 0
    return changed.tolist()


def _copy(s, lo, dims):
    rc, box = vpo.copy_region(s.pos, s.vox, s.flags, lo, dims, vpo.chunk_table(s.pos, lo, dims))
    assert rc == 0
    return box


# ---- oracle known answers -----------------------------------------------------------------------------------------------

def test_template_straddling_a_chunk_corner_with_negative_origin():
    corner = [((x, y, z), 0) for x in (-1, 0) for y in (-1, 0) for z in (-1, 0)]
    s = Slots(corner)
    t = (np.arange(64).reshape(4, 4, 4) % 3 + 1).astype(np.uint8)  # [z, y, x], types 1..3
    changed = _paste(s, [((-2, -2, -2), t)])
    for x in range(-2, 2):
        for y in range(-2, 2):
            for z in range(-2, 2):
                assert s.at((x, y, z)) == t[z + 2, y + 2, x + 2]
    assert s.at((-3, -2, -2)) == AIR and s.at((2, 1, 1)) == AIR and s.at((-2, -3, 0)) == AIR
    for (p, _), c in zip(corner, changed):
        assert len(_solid(s, s.slot(p))) == 8
        assert c == CHANGED | sum((PX, PY, PZ)[e] if p[e] < 0 else (NX, NY, NZ)[e] for e in range(3)), (p, c)
    assert np.array_equal(_copy(s, (-2, -2, -2), (4, 4, 4)), t)


def test_skip_bytes_leave_their_voxels_alone():
    s = Slots([((0, 0, 0), 0)])
    s.set((1, 1, 1), DIRT)
    t = np.full((3, 3, 3), SKIP, np.uint8)
    t[1, 1, 1], t[0, 0, 0], t[2, 2, 2] = STONE, AIR, GRASS  # (1,1,1) <- stone, (0,0,0) <- air (already), (2,2,2) <- grass
    assert _paste(s, [((0, 0, 0), t)]) == [CHANGED]
    assert _solid(s, 0) == [(1, 1, 1), (2, 2, 2)] and s.at((1, 1, 1)) == STONE and s.at((2, 2, 2)) == GRASS
    assert _paste(s, [((0, 0, 0), np.full((3, 3, 3), SKIP, np.uint8))]) == [0]
    assert _solid(s, 0) == [(1, 1, 1), (2, 2, 2)]


@pytest.mark.parametrize("mask", range(16))
def test_every_replace_mask(mask):
    s = Slots([((0, 0, 0), 0)])
    s.vox[0] = np.arange(32768) % 4  # every type in each row
    t = ((np.arange(32768) // 4) % 4).astype(np.uint8).reshape(32, 32, 32)  # every (old, new) pair
    changed = _paste(s, [((0, 0, 0), t)], replace=mask)
    old = np.arange(32768) % 4
    want = np.where((mask >> old) & 1 == 1, t.reshape(-1), old)
    assert np.array_equal(s.vox[0], want)
    d = (want != old).reshape(32, 32, 32)
    planes = [d[:, :, 31], d[:, :, 0], d[:, 31, :], d[:, 0, :], d[31], d[0]]
    assert changed == [(CHANGED if d.any() else 0) | sum(1 << f for f, pl in enumerate(planes) if pl.any())]


def test_uniform_chunk_no_op_changes_stays_uniform_and_its_rows_are_not_written():
    s = Slots([((0, 0, 0), UNIFORM_STONE), ((1, 0, 0), UNIFORM_AIR)])
    s.vox[:] = 7  # rows of a Uniform slot are not its voxels: never read, never written
    stone = np.full((4, 4, 40), STONE, np.uint8)
    assert _paste(s, [((0, 0, 0), stone)], [0]) == [0]                                    # the type is equal
    assert _paste(s, [((0, 0, 0), np.full((4, 4, 4), DIRT, np.uint8))], [0], replace=1 << AIR) == [0]  # mask excludes stone
    assert _paste(s, [((32, 0, 0), np.full((4, 4, 4), SKIP, np.uint8))], [1]) == [0]      # all SKIP
    assert _paste(s, [((100, 0, 0), np.full((4, 4, 4), DIRT, np.uint8))]) == [0, 0]       # reaches neither chunk
    assert s.flags.tolist() == [UNIFORM_STONE, UNIFORM_AIR] and (s.vox == 7).all()


def test_a_uniform_chunk_turned_varied_stays_varied_when_a_later_op_restores_it():
    s = Slots([((0, 0, 0), UNIFORM_AIR), ((1, 0, 0), 0)])
    s.vox[:] = 7
    s.vox[1] = 0
    a = np.full((3, 3, 3), STONE, np.uint8)
    b = np.full((32, 32, 41), AIR, np.uint8)
    assert _paste(s, [((31, 2, 2), a), ((0, 0, 0), b)]) == [CHANGED, 0]  # no voxel differs in the end
    assert s.flags.tolist() == [0, 0] and (s.vox == 0).all()


@pytest.mark.parametrize("local,bits", [((31, 5, 6), PX), ((0, 5, 6), NX), ((5, 31, 6), PY), ((5, 0, 6), NY), ((5, 6, 31), PZ),
                                        ((5, 6, 0), NZ), ((0, 0, 0), NX | NY | NZ), ((31, 31, 31), PX | PY | PZ), ((5, 6, 7), 0)])
def test_border_face_bits(local, bits):
    s = Slots([((2, -3, 1), 0)])
    v = np.array(local) + np.array([64, -96, 32])
    one = np.full((1, 1, 1), STONE, np.uint8)
    assert _paste(s, [(v, one)]) == [CHANGED | bits]
    assert _paste(s, [(v, one)]) == [0]


def test_overlapping_ops_the_later_one_wins():
    s = Slots([((0, 0, 0), 0), ((0, 0, -1), UNIFORM_AIR)])
    a = np.full((4, 4, 4), DIRT, np.uint8)
    b = np.full((2, 2, 2), STONE, np.uint8)
    b[0, 0, 0] = SKIP
    assert _paste(s, [((0, 0, -2), a), ((1, 1, 1), b)]) == [CHANGED | NX | NY | NZ, CHANGED | NX | NY | PZ]
    assert s.at((1, 1, 1)) == DIRT and s.at((2, 1, 1)) == STONE and s.at((2, 2, 2)) == STONE and s.at((3, 3, 1)) == DIRT
    assert s.at((0, 0, -1)) == DIRT and s.at((0, 0, -2)) == DIRT and s.at((0, 0, -3)) == AIR
    _paste(s, [((1, 1, 1), b), ((0, 0, 0), a)])  # the other order: a covers b
    assert s.at((2, 2, 2)) == DIRT


def test_copy_reads_rows_flags_and_unloaded_space():
    s = Slots([((0, 0, 0), 0), ((1, 0, 0), UNIFORM_STONE), ((0, 0, 1), UNIFORM_AIR)])
    s.vox[1] = 7  # a Uniform slot's rows are not read
    s.set((30, 2, 31), GRASS)
    box = _copy(s, (30, 2, 30), (4, 1, 4))  # x 30..33, z 30..33: chunks (0,0,0) (1,0,0) (0,0,1) and unloaded (1,0,1)
    want = np.array([[[AIR, AIR, STONE, STONE]], [[GRASS, AIR, STONE, STONE]], [[AIR, AIR, SKIP, SKIP]], [[AIR, AIR, SKIP, SKIP]]],
                    np.uint8)
    assert box.shape == (4, 1, 4) and np.array_equal(box, want)
    assert np.array_equal(_copy(s, (-3, 0, 0), (2, 1, 1)), [[[SKIP, SKIP]]])
    # the copy pastes back: SKIP bytes leave unloaded space alone and are never needed
    s.vox[0] = 0
    assert _paste(s, [((30, 2, 30), box)], [0, 1, 2]) == [CHANGED | PZ, 0, 0]
    assert s.at((30, 2, 31)) == GRASS and s.flags.tolist() == [0, UNIFORM_STONE, UNIFORM_AIR]


def _paste_rc(ops, blob, slots=(0,), n_template_bytes=None):
    s = Slots([((0, 0, 0), 0), ((1, 0, 0), UNIFORM_AIR)])
    rc, _ = vpo.paste(s.pos, s.vox, s.flags, ops, blob, list(slots), n_template_bytes)
    return rc, s


ONE = np.array([STONE], np.uint8)


@pytest.mark.parametrize("ops,blob,slots,nbytes", [
    ([vpo.op((0, 0, 0), (1, 1, 1))], ONE, [-1], None),                          # slot below the batch
    ([vpo.op((0, 0, 0), (1, 1, 1))], ONE, [2], None),                           # slot beyond the batch
    ([vpo.op((0, 0, 0), (1, 1, 1))], ONE, [1, 0, 1], None),                     # slot listed twice
    ([vpo.op((0, 0, 0), (1, 1, 1), replace=16)], ONE, [0], None),               # replace mask above 15
    ([vpo.op((0, 0, 0), (0, 1, 1))], ONE, [0], None),                           # a dimension of 0
    ([vpo.op((0, 0, 0), (1, -1, 1))], ONE, [0], None),                          # a negative dimension
    ([vpo.op((0, 0, 0), (1, 1, 1025))], np.full(1025, STONE, np.uint8), [0], None),  # a dimension above 1024
    ([vpo.op((C29 + 1, 0, 0), (1, 1, 1))], ONE, [0], None),                     # origin beyond 2^29
    ([vpo.op((0, -C29 - 1, 0), (1, 1, 1))], ONE, [0], None),                    # origin below -2^29
    ([vpo.op((0, 0, C29 - 1), (1, 1, 3))], np.full(3, STONE, np.uint8), [0], None),  # far corner beyond 2^29
    ([vpo.op((0, 0, 0), (1, 1, 1), offset=-1)], ONE, [0], None),                # offset below 0
    ([vpo.op((0, 0, 0), (2, 1, 1))], ONE, [0], None),                           # template beyond the buffer
    ([vpo.op((0, 0, 0), (1, 1, 1), offset=1)], ONE, [0], None),
    ([vpo.op((0, 0, 0), (1, 1, 1))], np.array([STONE, STONE], np.uint8), [0], 0),   # n_template_bytes counts, not the array
    ([vpo.op((0, 0, 0), (1, 1, 1))], np.array([4], np.uint8), [0], None),       # template byte 4
    ([vpo.op((0, 0, 0), (1, 1, 2))], np.array([STONE, 0xFE], np.uint8), [0], None),  # template byte 0xFE
    ([vpo.op((0, 0, 0), (1, 1, 1)), vpo.op((0, 0, 0), (1, 1, 1), offset=1)], np.array([STONE, 9], np.uint8), [0], None),  # a later op
])
def test_invalid_pastes_change_nothing(ops, blob, slots, nbytes):
    rc, s = _paste_rc(np.array(ops), blob, slots, nbytes)
    assert rc == -1 and not s.vox.any() and s.flags.tolist() == [0, UNIFORM_AIR]


def test_template_bytes_no_op_covers_are_not_checked():
    rc, s = _paste_rc(np.array([vpo.op((0, 0, 0), (1, 1, 1), offset=1)]), np.array([9, STONE, 200], np.uint8))
    assert rc == 0 and s.at((0, 0, 0)) == STONE


@pytest.mark.parametrize("lo,dims,table", [
    ((0, 0, 0), (0, 1, 1), None),               # a dimension of 0
    ((0, 0, 0), (1, 1025, 1), None),            # a dimension above 1024
    ((-C29 - 1, 0, 0), (1, 1, 1), None),        # lo below -2^29
    ((0, 0, C29 + 1), (1, 1, 1), None),         # lo beyond 2^29
    ((0, C29 - 1, 0), (1, 3, 1), None),         # far corner beyond 2^29
    ((0, 0, 0), (1, 1, 1), [2]),                # slot beyond the batch
    ((0, 0, 0), (1, 1, 1), [-2]),               # slot below -1
    ((0, 0, 0), (1, 1, 1), [1]),                # slot 1 holds chunk (1, 0, 0), not (0, 0, 0): a stale table
    ((0, 0, 0), (40, 1, 1), [1, 0]),
])
def test_invalid_copies_write_nothing(lo, dims, table):
    s = Slots([((0, 0, 0), 0), ((1, 0, 0), UNIFORM_AIR)])
    t = np.zeros(1, np.int32) if table is None else np.array(table, np.int32)
    rc, box = vpo.copy_region(s.pos, s.vox, s.flags, lo, dims, t)
    assert rc == -1 and box is None


def test_the_bounds_themselves_are_valid():
    s = Slots([((0, 0, 0), 0)])
    lo, hi = -C29, C29 - 1023
    line = np.full((1, 1, 1024), STONE, np.uint8)
    ops, blob = vpo.pack([((lo, lo, lo), line), ((hi, C29, C29), line), ((0, 0, 0), np.full((1, 1, 1), DIRT, np.uint8))], replace=15)
    rc, changed = vpo.paste(s.pos, s.vox, s.flags, ops, blob, [0])
    assert rc == 0 and changed.tolist() == [CHANGED | NX | NY | NZ] and s.at((0, 0, 0)) == DIRT
    for lo3, dims in (((lo, lo, lo), (1024, 1, 1)), ((hi, C29, C29), (1024, 1, 1)), ((0, 0, 0), (1024, 1024, 1))):
        rc, box = vpo.copy_region(s.pos, s.vox, s.flags, lo3, dims, vpo.chunk_table(s.pos, lo3, dims))
        assert rc == 0 and box.shape == tuple(dims[::-1])
    assert box[0, 0, 0] == DIRT and box[0, 0, 1] == AIR and box[0, 0, 32] == SKIP


# ---- ABI -------------------------------------------------------------------------------------------------------------------

def test_paste_op_layout_constants_and_symbols(tmp_path):
    fields = [f for f, _ in _lib.VxPasteOp._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "vx_b200.h"', "int main(void) {",
             '    printf("%zu", sizeof(VxPasteOp));']
    lines += [f'    printf(" %zu", offsetof(VxPasteOp, {f}));' for f in fields]
    lines += ['    printf(" %d\\n", (int)VX_PASTE_SKIP);', "    return 0;", "}"]
    src = tmp_path / "paste_abi.c"
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "paste_abi"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, timeout=60, check=True).stdout.split()]
    assert out[0] == ctypes.sizeof(_lib.VxPasteOp) == api.PASTE_OP_DTYPE.itemsize == 40
    assert out[1:1 + len(fields)] == [getattr(_lib.VxPasteOp, f).offset for f in fields]
    assert out[1:1 + len(fields)] == [api.PASTE_OP_DTYPE.fields[f][1] for f in fields]
    assert out[1 + len(fields):] == [SKIP] == [_lib.PASTE_SKIP] == [0xFF]
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for sym in ("vx_world_batch_copy_region", "vx_world_batch_paste"):
        assert hasattr(lib, sym) and sym in _lib.PROTOTYPES


# ---- World bookkeeping on a fake device backed by the oracles ----------------------------------------------------------

class FakeDevice(FakeDeviceWithFills):
    """test_region_edit's recorder plus the two calls of this feature, both on the paste oracle over the slot arrays."""

    def _arrays(self):
        pos = np.zeros((self.capacity, 3), np.int32)
        vox = np.zeros((self.capacity, 32768), np.uint8)
        flags = np.ones(self.capacity, np.uint8)
        for s in self.pos:
            pos[s], vox[s], flags[s] = self.pos[s], self.vox[s], self.flag[s]
        return pos, vox, flags

    def copy_region(self, lo, dims, chunk_slots):
        rc, box = vpo.copy_region(*self._arrays(), lo, dims, chunk_slots)
        assert rc == 0
        self.calls.append(("copy_region", tuple(lo.tolist()), tuple(dims.tolist()), chunk_slots.tobytes()))
        return box

    def paste(self, ops, templates, slots):
        sl = slots.tolist()
        pos = np.array([self.pos[s] for s in sl], dtype=np.int32).reshape(-1, 3)
        vox = np.stack([self.vox[s] for s in sl]) if sl else np.zeros((0, 32768), np.uint8)
        flags = np.array([self.flag[s] for s in sl], dtype=np.uint8)
        rc, changed = vpo.paste(pos, vox, flags, ops, templates, np.arange(len(sl), dtype=np.int32))
        assert rc == 0
        for i, s in enumerate(sl):
            self.vox[s], self.flag[s] = vox[i], int(flags[i])
        self.calls.append(("paste", ops.tobytes(), templates.tobytes(), sl))
        return changed


def _world(ob, vd=1, center=(0.0, 0.0, 0.0), dev_class=FakeDevice):
    dev = dev_class(ob, vxw.sphere_capacity(vd))
    w = vxw.World(vxw.WorldConfig(view_distance=vd, max_chunks_per_frame=1000), device=dev)
    w.update(center)
    return w, dev


def _state(w, dev, p):
    s = w.chunks[p]
    return dev.flag[s], (dev.vox[s] if dev.flag[s] == 0 else np.full(32768, dev.flag[s] - 1, np.uint8)).tobytes()


def test_unloaded_chunks_raise_before_anything_changes_and_skip_only_chunks_are_not_needed(ob):
    w, dev = _world(ob)  # the chunk at the origin and its six face neighbours
    n_calls, before = len(dev.calls), {p: _state(w, dev, p) for p in w.chunks}
    t = np.full((2, 2, 2), STONE, np.uint8)
    with pytest.raises(KeyError):
        w.paste(t, (31, 31, 0))                            # reaches (1, 1, 0)
    with pytest.raises(KeyError):
        w.paste(np.full((1, 1, 40), DIRT, np.uint8), (30, 0, 0))  # reaches (2, 0, 0)
    for bad in (lambda: w.paste(np.full((2, 2, 2), 4, np.uint8), (0, 0, 0)), lambda: w.paste(np.zeros((0, 2, 2), np.uint8), (0, 0, 0)),
                lambda: w.paste(np.zeros((2, 2), np.uint8), (0, 0, 0)), lambda: w.paste(t, (0, 0, C29)),
                lambda: w.paste(t, (0, 0, 0), replace=[5]), lambda: w.copy_region((0, 0, 0), (-1, 0, 0)),
                lambda: w.copy_region((0, 0, 0), (1024, 0, 0))):
        with pytest.raises(ValueError):
            bad()
    assert len(dev.calls) == n_calls and not w.pastes and {p: _state(w, dev, p) for p in w.chunks} == before
    assert w.paste(np.full((2, 2, 2), SKIP, np.uint8), (31, 31, 0)) == [] and len(dev.calls) == n_calls
    # the same footprint with SKIP over (1, 1, 0): only the three loaded chunks are listed
    t[:, 1, 1] = SKIP
    assert w.paste(t, (31, 31, 0), replace=[AIR]) == [(0, 0, -1), (0, 0, 0), (0, 1, 0), (1, 0, 0)]
    assert dev.calls[-1][0] == "paste" and sorted(dev.calls[-1][3]) == sorted(w.chunks[p] for p in [(0, 0, 0), (0, 1, 0), (1, 0, 0)])


def test_dirty_list_is_the_changed_chunks_and_their_neighbours_across_changed_faces(ob):
    w, dev = _world(ob, center=(0.0, 200.0, 0.0))  # Uniform air chunks around (0, 6, 0)
    y0 = 6 * 32
    one = np.full((1, 1, 1), STONE, np.uint8)
    assert w.paste(np.full((3, 3, 3), STONE, np.uint8), (4, y0 + 4, 4)) == [(0, 6, 0)]
    assert w.uniform_flags[(0, 6, 0)] == 0 and w.uniform_flags[(1, 6, 0)] == UNIFORM_AIR
    assert w.paste(one, (0, y0 + 4, 4)) == [(-1, 6, 0), (0, 6, 0)]
    assert w.paste(np.full((1, 1, 2), STONE, np.uint8), (31, y0 + 31, 31)) == [(0, 6, 0), (0, 6, 1), (0, 7, 0), (1, 6, 0)]
    assert w.paste(one, (0, y0 + 4, 4)) == []  # nothing differs
    assert w.paste(np.full((1, 1, 1), AIR, np.uint8), (33, y0 + 5, 5), replace=[GRASS]) == []
    assert w.uniform_flags[(1, 6, 0)] == 0 and dev.flag[w.chunks[(1, 6, 0)]] == 0
    assert len(w.pastes) == 5 and sorted(w._pastes_at) == [(0, 6, 0), (1, 6, 0)]


def test_pastes_fold_into_edits(ob):
    w, dev = _world(ob)
    w.set_blocks([(5, 5, 5), (6, 5, 5), (20, 20, 20), (33, 5, 5), (7, 5, 5)], [STONE, AIR, STONE, GRASS, DIRT])
    t = np.array([[[DIRT, DIRT, SKIP]]], np.uint8)  # x 5..7
    w.paste(t, (5, 5, 5), replace=[STONE, GRASS])  # (6,5,5) is air: not in the mask; (7,5,5) under SKIP; (20,20,20) outside
    assert w.edits[(0, 0, 0)] == {_index(5, 5, 5): DIRT, _index(6, 5, 5): AIR, _index(20, 20, 20): STONE, _index(7, 5, 5): DIRT}
    w.paste(np.array([[[STONE] * 36]], np.uint8), (6, 5, 5))  # every type, across into (1, 0, 0)
    assert w.edits[(0, 0, 0)] == {_index(5, 5, 5): DIRT, _index(6, 5, 5): STONE, _index(20, 20, 20): STONE, _index(7, 5, 5): STONE}
    assert w.edits[(1, 0, 0)] == {_index(33, 5, 5): STONE}
    for p in ((0, 0, 0), (1, 0, 0)):
        s = w.chunks[p]
        for i, v in w.edits[p].items():  # `edits` holds the current type of each edited voxel
            assert dev.vox[s][i] == v


def _edit_script(w):
    """Interleaved set_blocks, fills and pastes around the chunks (1, 0, 0) and (0, 1, 0)."""
    rng = np.random.default_rng(7)
    w.fill_ball((40, 7, 10), 49, AIR, replace=[GRASS, DIRT, STONE])
    w.paste(rng.choice(np.array([AIR, DIRT, STONE, SKIP], np.uint8), (6, 5, 9)), (36, 2, 8))
    w.set_blocks([(40, 7, 10), (33, 1, 12)], [STONE, AIR])
    w.paste(np.where(rng.random((4, 4, 4)) < 0.5, SKIP, GRASS).astype(np.uint8), (38, 3, 9), replace=[AIR])
    w.paste(np.full((2, 2, 2), STONE, np.uint8), (38, 3, 9), replace=[AIR])
    w.fill_box((34, 0, 0), (50, 6, 3), DIRT, replace=[AIR])
    w.paste(np.full((3, 3, 3), STONE, np.uint8), (1, 40, 1))     # (0, 1, 0): Uniform air made Varied by a paste alone
    w.set_blocks([(2, 41, 2)], [GRASS])
    w.fill_box((1, 40, 1), (1, 40, 1), AIR)
    w.paste(np.full((1, 1, 1), DIRT, np.uint8), (2, 41, 2), replace=[GRASS])
    w.paste(np.full((5, 5, 5), DIRT, np.uint8), (33, 0, 0), replace=[])  # changes nothing: not replayed


def test_interleaved_edits_fills_and_pastes_come_back_after_unloading(ob):
    w, dev = _world(ob, vd=1, center=(0.0, 20.0, 0.0))
    ref, ref_dev = _world(ob, vd=1, center=(0.0, 20.0, 0.0))
    _edit_script(w)
    _edit_script(ref)
    gone = [(1, 0, 0), (0, 1, 0)]
    want = {p: _state(ref, ref_dev, p) for p in gone}
    assert {p: _state(w, dev, p) for p in gone} == want and all(f == 0 for f, _ in want.values())
    w.update((32.0 * 20, 20.0, 0.0))
    assert not any(p in w.chunks for p in gone)
    del dev.calls[:]
    w.update((0.0, 20.0, 0.0))
    assert {p: _state(w, dev, p) for p in gone} == want and all(w.uniform_flags[p] == 0 for p in gone)
    names = [c[0] for c in dev.calls]
    g = names.index("generate")
    # issue order: fill 0, pastes 0..2, fill 1, paste 3, fill 2, paste 4, then `edits`; paste 5 changed nothing
    assert names[g + 1:g + 7] == ["fill_regions", "paste", "fill_regions", "paste", "fill_regions", "paste"], names
    assert names[g + 7] == "set_blocks" and names.count("paste") == 3 and "copy_region" not in names
    assert np.frombuffer(dev.calls[g + 2][1], api.PASTE_OP_DTYPE)["offset"].tolist() == [0, 270, 334]  # one call, packed templates


def test_copy_region_makes_one_call_and_pastes_back(ob):
    w, dev = _world(ob, center=(0.0, 200.0, 0.0))
    y0 = 6 * 32
    t = (np.arange(8, dtype=np.uint8).reshape(2, 2, 2) % 3) + 1
    w.paste(t, (30, y0 + 30, 30))
    n = len(dev.calls)
    box = w.copy_region((30, y0 + 30, 30), (33, y0 + 32, 32))  # reaches the unloaded (1, 7, 0), (1, 6, 1), ...
    assert len(dev.calls) == n + 1 and dev.calls[-1][0] == "copy_region" and box.shape == (3, 3, 4)
    assert np.array_equal(box[:2, :2, :2], t) and not box[2, :2, :2].any() and (box[2, :2, 2:] == SKIP).all()
    assert box[2, 2, 3] == SKIP and box[0, 0, 3] == AIR  # (33, y0+32, 32) is in the unloaded (1, 7, 1); (33, y0+30, 30) in (1, 6, 0)
    before = {p: _state(w, dev, p) for p in w.chunks}
    assert w.paste(box, (30, y0 + 30, 30)) == []  # pasting the copy back changes nothing and needs no unloaded chunk
    assert {p: _state(w, dev, p) for p in w.chunks} == before


def test_without_pastes_a_camera_walk_with_fills_makes_the_same_device_calls(ob):
    runs = []
    for dev_class in (FakeDevice, FakeDeviceWithFills):
        w, dev = _world(ob, vd=2, dev_class=dev_class)
        w.config.max_chunks_per_frame = 6
        cache = vxw.MeshCache(w)
        w.fill_ball((5, 5, 5), 30, AIR, replace=[1, 2, 3])
        w.fill_box((30, 0, 0), (40, 3, 40), STONE, replace=[AIR])
        w.set_blocks([(6, 6, 6)], [STONE])
        for step, pos in enumerate(CAMERA_WALK + [(400.0, 10.0, 0.0)] * 8 + [(0.0, 10.0, 20.0)] * 8):  # away and back: replays
            cam = camera.Camera(pos, 16 / 9, yaw=0.3 * step)
            w.update(cam.position)
            cache.update(w.get_visible_chunks(cam.position))
        runs.append((dev.calls, len(w.fills), {p: list(v) for p, v in w._fills_at.items()}))
        assert not w.pastes and not w._pastes_at
    assert runs[0] == runs[1] and len(runs[0][0]) > 10
    names = [c[0] for c in runs[0][0]]
    assert names.count("fill_regions") > 2 and "paste" not in names
