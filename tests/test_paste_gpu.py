"""Copy and paste on the device: World.copy_region / World.paste (vx_world_batch_copy_region, vx_world_batch_paste) mixed with
fills and set_blocks, checked against an independent host mirror that applies each call's history in order -- the paste
oracle (tests/paste_oracle.c) for pastes, the region oracle for fills, plain assignment for set_blocks -- voxel for voxel,
change byte for change byte, dirty list, meshes and frame; copies of random boxes against the mirror; the undo recipe; a
clone; a multi-op call over Uniform and Varied chunks; pastes surviving unload and reload; a 256 x 64 x 256 copy and paste."""
import numpy as np
import pytest

import vx_paste_oracle as vpo
from differential_projection_voxel_renderer_b200 import api, camera, world as vxw
from test_block_edit_gpu import _mesh_arrays, _world
from test_region_edit_gpu import Mirror, _check_state, _dirty, _fill, _oracle_meshes, _random_round, _record_fills
from test_world_gpu import WALK

pytestmark = pytest.mark.gpu

SKIP = api.PASTE_SKIP
AIR, STONE = 0, 3
W, H = 320, 180


class PasteMirror(Mirror):
    """test_region_edit_gpu's mirror plus pastes (through the paste oracle) and copies."""

    def _chunks(self, lo, hi):
        lo, hi = np.asarray(lo, np.int64) >> 5, np.asarray(hi, np.int64) >> 5
        return [p for p in ((int(x), int(y), int(z)) for x in range(lo[0], hi[0] + 1) for y in range(lo[1], hi[1] + 1)
                            for z in range(lo[2], hi[2] + 1)) if p in self.flag]

    def paste(self, op, template):
        """Apply one op to every loaded chunk its box reaches; returns {position: change byte} and those chunks before."""
        origin = op["origin"].astype(np.int64)
        ps = self._chunks(origin, origin + op["dims"] - 1)
        before = {p: (self.flag[p], self.vox[p].copy()) for p in ps}
        vox = np.stack([self.vox[p] for p in ps]) if ps else np.zeros((0, 32768), np.uint8)
        flags = np.array([self.flag[p] for p in ps], dtype=np.uint8)
        o = op.copy()
        o["offset"] = 0
        rc, changed = vpo.paste(np.array(ps, np.int32).reshape(-1, 3), vox, flags, o.reshape(1), template.reshape(-1),
                                np.arange(len(ps), dtype=np.int32))
        assert rc == 0
        for i, p in enumerate(ps):
            self.flag[p] = int(flags[i])
            if flags[i] == 0:
                self.vox[p] = vox[i]
        return dict(zip(ps, changed.tolist())), before

    def copy(self, lo, hi):
        lo, hi = np.asarray(lo, np.int64), np.asarray(hi, np.int64)
        out = np.full(tuple((hi - lo + 1)[::-1]), SKIP, np.uint8)
        for p in self._chunks(lo, hi):
            c = np.array(p, np.int64) * 32
            a, b = np.maximum(lo, c), np.minimum(hi, c + 31)
            v = self.vox[p].reshape(32, 32, 32)
            out[a[2] - lo[2]:b[2] - lo[2] + 1, a[1] - lo[1]:b[1] - lo[1] + 1, a[0] - lo[0]:b[0] - lo[0] + 1] = \
                v[a[2] - c[2]:b[2] - c[2] + 1, a[1] - c[1]:b[1] - c[1] + 1, a[0] - c[0]:b[0] - c[0] + 1]
        return out


def _record_pastes(w):
    calls = []
    orig = w.device.paste

    def rec(ops, templates, slots):
        changed = orig(ops, templates, slots)
        calls.append((ops.copy(), templates.copy(), slots.copy(), changed.copy()))
        return changed
    w.device.paste = rec
    return calls


def _paste(w, m, calls, template, origin, replace=None):
    """One World.paste, checked against the mirror: its change bytes and the dirty list.  None if World refused it."""
    n = len(calls)
    try:
        got = w.paste(template, origin, replace=replace)
    except KeyError:
        return None
    if len(calls) == n:  # all SKIP: no call
        assert got == [] and (np.asarray(template) == SKIP).all()
        return got
    ops, _, slots, changed = calls[-1]
    want, before = m.paste(ops[0], np.ascontiguousarray(template, np.uint8))
    at = {s: p for p, s in w.chunks.items()}
    sent = {at[s]: c for s, c in zip(slots.tolist(), changed.tolist())}
    assert all(want[p] == c for p, c in sent.items()), "paste: change bytes differ from the oracle"
    assert all(c == 0 for p, c in want.items() if p not in sent), "paste: a chunk the op changes was not sent"
    assert set(got) == _dirty(w, m, before) and got == sorted(got)
    return got


def _setup(ctx, ob, vd):
    cam = camera.Camera(WALK[0], W / H, pitch=-0.35)
    w = _world(ctx, vd, cam.position)
    cache = vxw.MeshCache(w)
    cache.update(sorted(w.chunks))
    return cam, cam.view_projection(), w, cache, PasteMirror(w), _record_fills(w), _record_pastes(w)


def _structure(rng, size):
    """A seeded structure: random solid types in a random blob, transparent air elsewhere."""
    t = rng.integers(1, 4, (size, size, size)).astype(np.uint8)
    g = np.indices((size, size, size)) - (size - 1) / 2
    keep = (g ** 2).sum(axis=0) <= (size / 2) ** 2 * rng.uniform(0.4, 1.0)
    return np.where(keep & (rng.random(t.shape) < 0.8), t, SKIP).astype(np.uint8)


@pytest.mark.parametrize("vd", [3, 12])
def test_paste_rounds_match_the_mirror_meshes_and_frames(ctx, ob, vd):
    cam, vp, w, cache, m, fills, pastes = _setup(ctx, ob, vd)
    cfg, ocfg, atlas = api.default_frame_config(W, H), ob.default_frame_config(W, H, n_threads=2), ob.default_atlas()
    prev, om_prev = w.batch.download(), _oracle_meshes(ob, w, m)
    rng = np.random.default_rng(200 + vd)
    done = 0
    for r in range(4):
        round_fills, (xyz, types) = _random_round(rng, w, cam.position)
        dirty = set()
        for i, (kind, args) in enumerate(round_fills):
            if i % 2 == 0:
                got = _fill(w, m, fills, kind, args)
                dirty.update(got or [])
            c = np.array(args[0])
            size = int(rng.choice([3, 8, 16, 24]))
            if rng.random() < 0.5:
                t = _structure(rng, size)
            else:  # a copy of the ground somewhere near, pasted here
                src = c + rng.integers(-40, 40, 3)
                t = w.copy_region(src, src + [size - 1, size // 2, size - 1])
                assert np.array_equal(t, m.copy(src, src + [size - 1, size // 2, size - 1])), "copy differs from the mirror"
            replace = [None, [AIR], [1, 2, 3]][int(rng.integers(0, 3))]
            got = _paste(w, m, pastes, t, c - np.array(t.shape[::-1]) // 2, replace)
            done += got is not None
            dirty.update(got or [])
        try:
            dirty.update(w.set_blocks(xyz, types))
            m.set_blocks(xyz, types)
        except KeyError:
            pass
        prev, om_prev, _ = _check_state(w, m, cache, prev, dirty, om_prev, ob, cam, vp, cfg, ocfg, atlas, ctx, f"vd {vd} round {r}")
    assert done >= 16
    w.batch.release()


def test_copies_of_random_boxes_match_the_mirror(ctx, ob):
    _, _, w, _, m, _, _ = _setup(ctx, ob, 3)
    rng = np.random.default_rng(5)
    allp = np.array(sorted(w.chunks))
    lo_w, hi_w = allp.min(axis=0) * 32 - 40, allp.max(axis=0) * 32 + 72  # reaching beyond the loaded world on every side
    uniform = skip = 0
    for i in range(40):
        dims = rng.integers(1, [200, 80, 200] if i % 4 else [4, 4, 4])
        lo = rng.integers(lo_w, hi_w - dims)
        box = w.copy_region(lo, lo + dims - 1)
        assert box.shape == tuple(dims[::-1]) and np.array_equal(box, m.copy(lo, lo + dims - 1)), f"copy {lo} {dims}"
        skip += bool((box == SKIP).any())
        uniform += any(m.flag[p] != 0 for p in m._chunks(lo, lo + dims - 1))
    assert skip >= 5 and uniform >= 5
    w.batch.release()


def test_undo_recipe_and_clone(ctx, ob):
    cam, vp, w, cache, m, _, pastes = _setup(ctx, ob, 3)
    cfg = api.default_frame_config(W, H)
    color0, depth0, _ = vxw.frame(w, cache, cam.position, vp, cfg, ctx)
    c = np.array(cam.position, np.int64) + [0, -20, -30]
    t = _structure(np.random.default_rng(1), 24)
    lo, hi = c, c + np.array(t.shape[::-1]) - 1
    snapshot = w.copy_region(lo, hi)
    before = {p: w.chunk_voxels(p)[1].copy() for p in m._chunks(lo, hi)}
    dirty = set(_paste(w, m, pastes, t, lo))
    assert dirty
    dirty |= set(_paste(w, m, pastes, snapshot, lo))
    for p, v in before.items():
        assert np.array_equal(w.chunk_voxels(p)[1], v), f"undo: voxels of {p} differ from before the paste"
    cache.refresh(dirty)
    color1, depth1, _ = vxw.frame(w, cache, cam.position, vp, cfg, ctx)
    assert np.array_equal(color0, color1) and np.array_equal(depth0.view(np.uint32), depth1.view(np.uint32)), "undo: frame differs"
    # clone: copy a region with terrain in it and paste it elsewhere; the destination then reads back as the source
    src = c + [-40, -10, 10]
    region = w.copy_region(src, src + [47, 23, 47])
    assert (region != SKIP).all() and len(np.unique(region)) > 1
    dst = src + [60, 5, -20]
    assert _paste(w, m, pastes, region, dst) is not None
    assert np.array_equal(w.copy_region(dst, dst + [47, 23, 47]), region)
    w.batch.release()


def test_multi_op_call_over_uniform_and_varied_chunks(ctx, ob):
    _, _, w, _, m, _, _ = _setup(ctx, ob, 3)
    air = next(p for p in sorted(w.chunks) if w.uniform_flags[p] == 1)
    stone = next(p for p in sorted(w.chunks) if w.uniform_flags[p] == 4)
    varied = [p for p in sorted(w.chunks) if w.uniform_flags[p] == 0][:3]
    ps = [air, stone] + varied
    c = lambda p, o: np.array(p) * 32 + o
    rng = np.random.default_rng(9)
    items = [(c(air, 0), np.full((32, 32, 32), STONE, np.uint8), 1 << 1),          # mask excludes air: stays Uniform
             (c(stone, 8), np.full((9, 9, 9), AIR, np.uint8), 1 << 3),             # carves Uniform stone
             (c(stone, 8), np.full((9, 9, 9), STONE, np.uint8), 0xF),              # ... and restores it: stays Varied
             (c(varied[0], -4), _structure(rng, 40), 1 << AIR),
             (c(varied[1], -10), rng.integers(0, 4, (20, 30, 40)).astype(np.uint8), 0xF),
             (c(varied[2], 5), np.where(rng.random((30, 30, 30)) < 0.5, SKIP, 2).astype(np.uint8), 0b1100)]
    ops, blob = vpo.pack([(o, t) for o, t, _ in items])
    ops["replace_mask"] = [r for _, _, r in items]
    slots = np.array([w.chunks[p] for p in ps], np.int32)
    vox = np.stack([m.vox[p] for p in ps])
    flags = np.array([m.flag[p] for p in ps], np.uint8)
    rc, want = vpo.paste(np.array(ps, np.int32), vox, flags, ops, blob, np.arange(len(ps), dtype=np.int32))
    assert rc == 0
    got = w.device.paste(ops, blob, slots)
    assert got.tolist() == want.tolist()
    assert want[0] == 0 and flags[0] == 1 and want[1] & 64 and flags[1] == 0
    for i, p in enumerate(ps):
        f, v = w.chunk_voxels(p)
        assert f == flags[i] and v.tobytes() == vox[i].tobytes()
    # refused at the C boundary before anything changes or is written
    raw = w.device.read_voxels(slots)
    bad_blob = blob.copy()
    bad_blob[int(ops[4]["offset"]) + 17] = 4
    for bad_ops, bad_t, bad_slots in ((ops, blob, np.array([slots[0], slots[0]], np.int32)), (ops, blob, np.array([w.capacity], np.int32)),
                                      (ops, bad_blob, slots), (ops, blob[:-1], slots),
                                      (vpo.op((0, 0, 0), (1, 1, 1), replace=16).reshape(1), blob, slots),
                                      (vpo.op((0, 0, 0), (1, 1, 1025)).reshape(1), np.zeros(1025, np.uint8), slots),
                                      (vpo.op((0, 0, (1 << 29) - 1), (1, 1, 3)).reshape(1), blob, slots)):
        with pytest.raises(api.VxError):
            w.device.paste(bad_ops, bad_t, bad_slots)
    again = w.device.read_voxels(slots)
    assert again[0].tobytes() == raw[0].tobytes() and again[1].tobytes() == raw[1].tobytes()
    lo = np.array(air, np.int64) * 32
    for bad_lo, dims, table in ((lo, [1, 1, 1], [w.chunks[stone]]), (lo, [1, 1, 1], [w.capacity]), (lo, [0, 1, 1], [w.chunks[air]]),
                                (lo, [1025, 1, 1], [w.chunks[air]] * 33)):
        out = np.full(tuple(max(d, 1) for d in dims[::-1]), 0xAB, np.uint8)
        with pytest.raises(api.VxError):
            w.device.ctx.check(w.device.ctx.lib.vx_world_batch_copy_region(
                w.device.ctx.handle, w.batch.handle, api._p(bad_lo.astype(np.int32)), api._p(np.array(dims, np.int32)),
                api._p(np.array(table, np.int32)), api._p(out)))
        assert (out == 0xAB).all()
    w.batch.release()


def test_pastes_survive_unloading(ctx, ob):
    cam, vp, w, cache, m, fills, pastes = _setup(ctx, ob, 3)
    cfg = api.default_frame_config(W, H)
    rng = np.random.default_rng(11)
    c = np.array(cam.position, np.int64) + [0, -25, -40]
    dirty = set(_paste(w, m, pastes, _structure(rng, 16), c))
    dirty |= set(_fill(w, m, fills, "fill_ball", (tuple(c + 8), 30, AIR, None)))
    w.set_blocks([tuple(c + 8)], [STONE])
    m.set_blocks([tuple(c + 8)], [STONE])
    dirty |= set(_paste(w, m, pastes, _structure(rng, 24), c + [4, 4, 4], [AIR]))
    cache.refresh(dirty)
    keep = {p: w.chunk_voxels(p)[1].copy() for p in dirty}
    meshes = {p: _mesh_arrays(w.batch.download(), w.chunks[p]) for p in dirty if p in cache.cached}
    color0, depth0, _ = vxw.frame(w, cache, cam.position, vp, cfg, ctx)
    far = cam.position + np.array([32.0 * 12, 0, 0], np.float32)
    vxw.frame(w, cache, far, camera.Camera(far, W / H).view_projection(), cfg, ctx)
    assert not any(p in w.chunks for p in dirty)
    color1, depth1, _ = vxw.frame(w, cache, cam.position, vp, cfg, ctx)
    for p in dirty:
        assert np.array_equal(w.chunk_voxels(p)[1], keep[p]), f"voxels of {p} differ after reloading"
    got = w.batch.download()
    assert all(_mesh_arrays(got, w.chunks[p]) == q for p, q in meshes.items())
    assert np.array_equal(color0, color1) and np.array_equal(depth0.view(np.uint32), depth1.view(np.uint32))
    w.batch.release()


def test_large_copy_and_paste_at_view_distance_12(ctx, ob):
    w = _world(ctx, 12, (0.0, 10.0, 20.0))
    m = PasteMirror(w)
    calls = _record_pastes(w)
    lo, hi = np.array([-128, 0, -128]), np.array([127, 63, 127])
    box = w.copy_region(lo, hi)
    assert box.shape == (256, 64, 256) and np.array_equal(box, m.copy(lo, hi))
    dst = lo + [0, 64, 0]
    got = _paste(w, m, calls, box, dst)
    assert got and len(calls[-1][2]) == 128
    assert np.array_equal(w.copy_region(dst, dst + (hi - lo)), box)
    for p in m._chunks(dst, dst + (hi - lo)):
        f, v = w.chunk_voxels(p)
        assert f == m.flag[p] and v.tobytes() == m.vox[p].tobytes()
    w.batch.release()
