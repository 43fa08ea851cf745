"""Region edits on the device: World.fill_box / fill_ball (vx_world_batch_fill_regions) mixed with set_blocks, checked against
an independent host mirror that applies each call's history in order -- the region oracle (tests/region_oracle.c) for fills,
plain assignment for set_blocks -- voxel for voxel, change byte for change byte, dirty list, meshes and frame; an explosion at
a picked voxel; fills surviving unload and reload; a multi-op call over Uniform and Varied chunks."""
import math

import numpy as np
import pytest

import vx_region_oracle as vro
from differential_projection_voxel_renderer_b200 import _lib, api, camera, world as vxw, worldgen
from test_block_edit_gpu import _mesh_arrays, _oracle_mesh, _world
from test_world_gpu import WALK

pytestmark = pytest.mark.gpu

BOX, BALL = _lib.REGION_BOX, _lib.REGION_BALL
AIR, STONE = 0, 3
W, H = 320, 180


class Mirror:
    """Per loaded chunk position: Uniform flag and voxel row (all its type for a Uniform chunk), from the host generator."""

    def __init__(self, w):
        allp = sorted(w.chunks)
        g = worldgen.generate_world(np.array(allp, dtype=np.int32).reshape(-1, 3))
        self.flag = {p: int(g.uniform_flags[i]) for i, p in enumerate(allp)}
        self.vox = {p: g.voxels[i].copy() if g.uniform_flags[i] == 0 else np.full(32768, g.uniform_flags[i] - 1, np.uint8)
                    for i, p in enumerate(allp)}

    def fill(self, op):
        """Apply op to every loaded chunk its bounding box reaches; returns {position: change byte} and the state of those
        chunks before."""
        a = op["a"].astype(np.int64)
        r = math.isqrt(int(op["radius_sq"])) if int(op["shape"]) == BALL else 0
        lo, hi = (a - r, a + r) if int(op["shape"]) == BALL else (a, op["b"].astype(np.int64))
        ps = [p for p in np.ndindex(*(hi // 32 - lo // 32 + 1))]
        ps = [q for q in (tuple(int(c) for c in np.array(p) + lo // 32) for p in ps) if q in self.flag]
        before = {p: (self.flag[p], self.vox[p].copy()) for p in ps}
        pos = np.array(ps, dtype=np.int32).reshape(-1, 3)
        vox = np.stack([self.vox[p] for p in ps])
        flags = np.array([self.flag[p] for p in ps], dtype=np.uint8)
        rc, changed = vro.fill_regions(pos, vox, flags, op.reshape(1), np.arange(len(ps), dtype=np.int32))
        assert rc == 0
        for i, p in enumerate(ps):
            self.flag[p] = int(flags[i])
            if flags[i] == 0:
                self.vox[p] = vox[i]
        return dict(zip(ps, changed.tolist())), before

    def set_blocks(self, xyz, types):
        for v, t in zip(np.asarray(xyz, np.int64).reshape(-1, 3).tolist(), np.broadcast_to(types, (len(xyz),)).tolist()):
            p = (v[0] >> 5, v[1] >> 5, v[2] >> 5)
            self.flag[p] = 0
            self.vox[p][(v[2] & 31) * 1024 + (v[1] & 31) * 32 + (v[0] & 31)] = t

    def slots(self, w):
        """Slot-indexed positions, voxels, flags and neighbour rows for the oracle mesher."""
        cap = w.capacity
        pos, flags = np.zeros((cap, 3), np.int32), np.ones(cap, np.uint8)
        nbr, vox = np.full((cap, 6), -1, np.int32), np.zeros((cap, 32768), np.uint8)
        for p, s in w.chunks.items():
            pos[s], flags[s], nbr[s], vox[s] = p, self.flag[p], w._neighbor_row(p), self.vox[p]
        return pos, vox, flags, nbr


def _dirty(w, m, before):
    """The chunks whose meshes can change, from the mirror's state before and now: a changed flag or voxel row, plus the loaded
    neighbour across each border plane with a changed voxel."""
    out = set()
    for p, (f0, v0) in before.items():
        f1, v1 = m.flag[p], m.vox[p]
        d = (v0 != v1).reshape(32, 32, 32)
        if f0 == f1 and not d.any():
            continue
        out.add(p)
        for plane, o in zip((d[:, :, 31], d[:, :, 0], d[:, 31], d[:, 0], d[31], d[0]), vxw.FACE_OFFSETS):
            q = (p[0] + o[0], p[1] + o[1], p[2] + o[2])
            if plane.any() and q in w.chunks:
                out.add(q)
    return out


def _record_fills(w):
    calls = []
    orig = w.device.fill_regions

    def rec(ops, slots):
        changed = orig(ops, slots)
        calls.append((ops.copy(), slots.copy(), changed.copy()))
        return changed
    w.device.fill_regions = rec
    return calls


def _fill(w, m, calls, kind, args):
    """One World fill, checked against the mirror: its change bytes, and the dirty list.  None if World refused it."""
    try:
        got = getattr(w, kind)(*args[:3], replace=args[3])
    except KeyError:
        return None
    ops, slots, changed = calls[-1]
    want, before = m.fill(ops[0])
    at = {s: p for p, s in w.chunks.items()}
    sent = {at[s]: c for s, c in zip(slots.tolist(), changed.tolist())}
    assert all(want[p] == c for p, c in sent.items()), f"{kind}{args}: change bytes differ from the oracle"
    assert all(c == 0 for p, c in want.items() if p not in sent), f"{kind}{args}: a chunk the op changes was not sent"
    assert set(got) == _dirty(w, m, before) and got == sorted(got)
    return got


def _random_round(rng, w, centre):
    """Seeded boxes and balls around the surface near the camera column, and a few set_blocks edits."""
    h = worldgen.terrain_heights(int(centre[0]) - 64, int(centre[2]) - 64, 128, 128)
    out = []
    for _ in range(8):
        dx, dz = rng.integers(0, 128, 2)
        c = (int(centre[0]) - 64 + int(dx), int(h[dz, dx]) + int(rng.integers(-4, 3)), int(centre[2]) - 64 + int(dz))
        block = int(rng.integers(0, 4))
        replace = [None, [AIR], [1, 2, 3], list(rng.choice(4, int(rng.integers(0, 4)), replace=False))][int(rng.integers(0, 4))]
        if rng.random() < 0.5:
            out.append(("fill_ball", (c, int(rng.choice([0, 2, 9, 64, int(rng.integers(0, 577))])), block, replace)))
        else:
            ext = rng.integers(0, [40, 12, 40])
            out.append(("fill_box", (c, tuple(np.array(c) + ext), block, replace)))
    xyz = [np.array(out[i][1][0]) + rng.integers(-3, 4, 3) for i in range(4)]
    return out, (xyz, rng.integers(0, 4, len(xyz)))


def _check_state(w, m, cache, prev, dirty, om_prev, ob, cam, vp, cfg, ocfg, atlas, ctx, tag):
    """Voxels and flags of every loaded chunk, meshes after refresh, and the frame, against the mirror and the oracle."""
    for p in w.chunks:
        flag, v = w.chunk_voxels(p)
        assert flag == m.flag[p] and v.tobytes() == m.vox[p].tobytes(), f"{tag}: voxels of {p} differ from the mirror"
    refreshed = cache.refresh(dirty)
    got = w.batch.download()
    om = _oracle_meshes(ob, w, m)
    rs = {w.chunks[p] for p in refreshed}
    for p, s in w.chunks.items():
        assert _mesh_arrays(got, s) == _oracle_mesh(om, s), f"{tag}: mesh of {p} differs from the oracle"
        if s not in rs:
            assert _mesh_arrays(got, s) == _mesh_arrays(prev, s), f"{tag}: mesh of {p} changed without a refresh"
        if _oracle_mesh(om, s) != _oracle_mesh(om_prev, s):
            assert p in dirty, f"{tag}: the oracle mesh of {p} changed but it is not in the dirty list"
    color, depth, surv = vxw.frame(w, cache, cam.position, vp, cfg, ctx)
    ids = np.array([s for s in cache.visible_mesh_slots(w.get_visible_chunks_frustum(cam.position, vp)).tolist() if om.has_mesh[s]],
                   dtype=np.int32)
    oc, od, osurv = ob.render_frame(om, ids, vp, cam.position, ocfg, atlas)
    assert surv.tolist() == osurv.tolist()
    assert np.array_equal(depth.view(np.uint32), od.view(np.uint32)) and np.array_equal(color, oc), f"{tag}: frame differs"
    return got, om, (color, depth)


def _setup(ctx, ob, vd):
    cam = camera.Camera(WALK[0], W / H, pitch=-0.35)
    w = _world(ctx, vd, cam.position)
    cache = vxw.MeshCache(w)
    cache.update(sorted(w.chunks))
    return cam, cam.view_projection(), w, cache, Mirror(w), _record_fills(w)


def _oracle_meshes(ob, w, m):
    pos, vox, flags, nbr = m.slots(w)
    return ob.mesh_chunks(vox, nbr, flags, pos)


@pytest.mark.parametrize("vd", [3, 12])
def test_fill_rounds_match_the_mirror_meshes_and_frames(ctx, ob, vd):
    cam, vp, w, cache, m, calls = _setup(ctx, ob, vd)
    cfg, ocfg, atlas = api.default_frame_config(W, H), ob.default_frame_config(W, H, n_threads=2), ob.default_atlas()
    prev, om_prev = w.batch.download(), _oracle_meshes(ob, w, m)
    rng = np.random.default_rng(100 + vd)
    done = 0
    for r in range(4):
        fills, (xyz, types) = _random_round(rng, w, cam.position)
        dirty = set()
        for kind, args in fills:
            got = _fill(w, m, calls, kind, args)
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


def test_explosion_at_a_picked_voxel_and_fills_survive_unloading(ctx, ob):
    cam, vp, w, cache, m, calls = _setup(ctx, ob, 3)
    cfg, ocfg, atlas = api.default_frame_config(W, H), ob.default_frame_config(W, H, n_threads=2), ob.default_atlas()
    prev, om_prev = w.batch.download(), _oracle_meshes(ob, w, m)
    vxw.frame(w, cache, cam.position, vp, cfg, ctx)
    first = w.pick(cam.position, vp, [(W // 2, H // 2)], W, H, 384.0)
    assert first["status"][0] == _lib.RAY_HIT
    v0 = first["voxel"][0]
    dirty = _fill(w, m, calls, "fill_ball", (v0, 36, AIR, [1, 2, 3]))
    assert dirty and tuple(int(c) for c in v0 >> 5) in dirty
    roof = _fill(w, m, calls, "fill_box", (v0 + [-4, 3, -4], v0 + [4, 4, 4], STONE, [AIR]))  # over the crater, air only
    assert roof is not None
    dirty += roof
    prev, om_prev, _ = _check_state(w, m, cache, prev, set(dirty), om_prev, ob, cam, vp, cfg, ocfg, atlas, ctx, "explosion")
    after = w.pick(cam.position, vp, [(W // 2, H // 2)], W, H, 384.0)
    assert after["status"][0] == _lib.RAY_HIT and after["voxel"][0].tolist() != v0.tolist()
    # walk away until the edited chunks unload, then back: voxels, flags, meshes and the frame come back
    edited = sorted({p for p in m.flag if m.flag[p] == 0 and p in w.chunks})
    keep = {p: w.chunk_voxels(p) for p in edited}
    meshes = {p: _mesh_arrays(prev, w.chunks[p]) for p in w.chunks}
    color0, depth0, _ = vxw.frame(w, cache, cam.position, vp, cfg, ctx)
    far = cam.position + np.array([32.0 * 12, 0, 0], np.float32)
    vxw.frame(w, cache, far, camera.Camera(far, W / H).view_projection(), cfg, ctx)
    assert not any(p in w.chunks for p in dirty)
    color1, depth1, _ = vxw.frame(w, cache, cam.position, vp, cfg, ctx)
    for p in edited:
        f, v = w.chunk_voxels(p)
        assert f == keep[p][0] and v.tobytes() == keep[p][1].tobytes(), f"voxels of {p} differ after reloading"
    got = w.batch.download()
    assert sorted(w.chunks) == sorted(meshes)
    again = {p: _mesh_arrays(got, w.chunks[p]) for p in cache.cached}
    assert again == {p: meshes[p] for p in cache.cached} and set(dirty) <= cache.cached
    assert np.array_equal(color0, color1) and np.array_equal(depth0.view(np.uint32), depth1.view(np.uint32))
    w.batch.release()


def test_multi_op_call_over_uniform_and_varied_chunks(ctx, ob):
    _, _, w, _, m, _ = _setup(ctx, ob, 3)
    air = next(p for p in sorted(w.chunks) if w.uniform_flags[p] == 1)
    stone = next(p for p in sorted(w.chunks) if w.uniform_flags[p] == 4)
    varied = [p for p in sorted(w.chunks) if w.uniform_flags[p] == 0][:3]
    ps = [air, stone] + varied
    c = lambda p, o: tuple(int(v) for v in np.array(p) * 32 + o)
    ops = np.stack([vro.op(BOX, c(air, 0), c(air, 31), block_type=STONE, replace=1 << 1),     # mask excludes air: stays Uniform
                    vro.op(BALL, c(stone, 16), radius_sq=64, block_type=AIR, replace=1 << 3),  # carves Uniform stone
                    vro.op(BALL, c(stone, 16), radius_sq=64, block_type=STONE),                # ... and restores it: stays Varied
                    vro.op(BOX, c(varied[0], -4), c(varied[0], 35), block_type=2, replace=1 << AIR),
                    vro.op(BALL, c(varied[1], 0), radius_sq=200, block_type=AIR),
                    vro.op(BOX, c(varied[2], 0), c(varied[2], 31), block_type=1, replace=0b1100)])
    slots = np.array([w.chunks[p] for p in ps], np.int32)
    pos = np.array(ps, np.int32)
    vox = np.stack([m.vox[p] for p in ps])
    flags = np.array([m.flag[p] for p in ps], np.uint8)
    rc, want = vro.fill_regions(pos, vox, flags, ops, np.arange(len(ps), dtype=np.int32))
    assert rc == 0
    got = w.device.fill_regions(ops, slots)
    assert got.tolist() == want.tolist()
    assert want[0] == 0 and flags[0] == 1 and want[1] & 64 and flags[1] == 0  # every op is applied to every listed slot
    for i, p in enumerate(ps):
        f, v = w.chunk_voxels(p)
        assert f == flags[i] and v.tobytes() == vox[i].tobytes()
    # refused at the C boundary before anything changes
    raw = w.device.read_voxels(slots)
    for bad_ops, bad_slots in ((ops, np.array([slots[0], slots[0]], np.int32)), (ops, np.array([w.capacity], np.int32)),
                               (np.stack([ops[0], vro.op(BOX, (0, 0, 0), (1, 1, 1), block_type=4)]), slots),
                               (vro.op(BALL, (0, 0, 0), radius_sq=-1).reshape(1), slots),
                               (vro.op(BOX, (0, 0, 0), (1, 1, (1 << 29) + 1)).reshape(1), slots)):
        with pytest.raises(api.VxError):
            w.device.fill_regions(bad_ops, bad_slots)
    again = w.device.read_voxels(slots)
    assert again[0].tobytes() == raw[0].tobytes() and again[1].tobytes() == raw[1].tobytes()
    w.batch.release()
