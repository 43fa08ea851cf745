"""Picking and block edits on the device: vx_world_raycast against its CPU oracle (tests/ray_oracle.c) bit for bit, block edits
(vx_world_batch_set_blocks + MeshCache.refresh) against the oracle mesher and renderer over the edited host world, the
break / place loop through World.pick, and a cross-check of picking against the rendered depth buffer."""
import numpy as np
import pytest

import vx_ray_oracle
from differential_projection_voxel_renderer_b200 import _lib, api, camera, world as vxw, worldgen
from test_world_gpu import WALK

pytestmark = pytest.mark.gpu

HIT = _lib.RAY_HIT
MAX_T = 384.0


def _world(ctx, vd, center):
    w = vxw.World(vxw.WorldConfig(view_distance=vd, max_chunks_per_frame=1 << 20), ctx=ctx)
    w.update(center)
    return w


def _host_slots(w):
    """The world batch as the oracle sees it: slot-indexed positions, voxels, flags and neighbour rows of the generated
    world with World.edits applied the way vx_world_batch_set_blocks applies them."""
    cap = w.capacity
    pos = np.zeros((cap, 3), np.int32)
    flags = np.ones(cap, np.uint8)
    nbr = np.full((cap, 6), -1, np.int32)
    vox = np.zeros((cap, 32768), np.uint8)
    allp = sorted(w.chunks)
    g = worldgen.generate_world(np.array(allp, dtype=np.int32).reshape(-1, 3))
    for i, p in enumerate(allp):
        s = w.chunks[p]
        pos[s], flags[s], nbr[s] = p, g.uniform_flags[i], w._neighbor_row(p)
        if flags[s] == 0:
            vox[s] = g.voxels[i]
    for p, edits in w.edits.items():
        if p in w.chunks:
            s = w.chunks[p]
            if flags[s]:
                vox[s] = flags[s] - 1
                flags[s] = 0
            for i, t in edits.items():
                vox[s, i] = t
    return pos, vox, flags, nbr


def _random_rays(rng, w, n):
    """Origins inside the loaded world (the first half on the voxel lattice or half-way between), directions random unit
    vectors (every other ray) or axis-aligned / lattice diagonals with components in {-1, 0, 1}, not normalised."""
    c = np.array(sorted(w.chunks), dtype=np.float64)
    o = (c[rng.integers(0, c.shape[0], n)] + rng.random((n, 3))) * 32.0
    o[:n // 2] = np.floor(o[:n // 2] * 2.0) / 2.0
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    lattice = rng.integers(-1, 2, size=(n, 3)).astype(np.float64)
    lattice[~lattice.any(axis=1)] = (0, 1, 0)
    d[1::2] = lattice[1::2]
    return o.astype(np.float32), d.astype(np.float32)


def _device_raycast(ctx, w, o, d, max_t):
    """The same rays through vx_world_raycast_device on device arrays."""
    import torch
    dev = torch.device("cuda", ctx.device)
    to = torch.from_numpy(o).to(dev)
    td = torch.from_numpy(d).to(dev)
    ts = torch.from_numpy(w.start_slots(o)).to(dev)
    th = torch.zeros((o.shape[0], 32), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)
    ctx.check(ctx.lib.vx_world_raycast_device(ctx.handle, w.batch.handle, to.data_ptr(), td.data_ptr(), ts.data_ptr(), o.shape[0],
                                              float(max_t), th.data_ptr()))
    ctx.synchronize()
    return th.cpu().numpy().reshape(-1).view(api.RAY_HIT_DTYPE)


@pytest.mark.parametrize("vd", [3, 12])
def test_raycast_matches_the_oracle_bit_for_bit(ctx, ob, vd):
    w = _world(ctx, vd, WALK[0])
    host = _host_slots(w)
    W, H = 320, 180
    px = np.stack(np.meshgrid(np.arange(W), np.arange(H)), axis=-1).reshape(-1, 2)
    origins, dirs = [], []
    for step in (0, 2, 3):
        cam = camera.Camera(WALK[step], W / H, yaw=0.4 * step, pitch=-0.2)
        o, d = api.pixel_rays(cam.view_projection(), cam.position, px, W, H)
        origins.append(o)
        dirs.append(d)
    o, d = _random_rays(np.random.default_rng(vd), w, 100_000)
    o = np.concatenate(origins + [o])
    d = np.concatenate(dirs + [d])
    got = w.raycast(o, d, MAX_T)
    want = vx_ray_oracle.raycast(*host, o, d, w.start_slots(o), MAX_T)
    assert got["hits"].tobytes() == want.tobytes(), f"{int((got['hits'] != want).sum())} of {o.shape[0]} rays differ"
    assert _device_raycast(ctx, w, o, d, MAX_T).tobytes() == want.tobytes()
    status = np.bincount(want["status"], minlength=4)
    assert status[HIT] > o.shape[0] // 4 and status[_lib.RAY_MISS] + status[_lib.RAY_LEFT_WORLD] > 0, status
    with pytest.raises(api.VxError):  # a start slot outside [-1, capacity)
        w.device.raycast(o[:1], d[:1], np.array([w.capacity], np.int32), MAX_T)
    w.batch.release()


def _mesh_arrays(got, s):
    b, c = int(got["quad_base"][s]), int(got["quad_count"][s])
    return bool(got["has_mesh"][s]), got["quads"][b:b + c].tobytes(), got["slice_offsets"][s].tobytes(), got["face_aabb"][s].tobytes()


def _oracle_mesh(om, s):
    if not om.has_mesh[s]:
        return False, b"", om.slice_offsets[s].tobytes(), om.face_aabb[s].tobytes()
    return True, om.chunk_quads(s).tobytes(), om.slice_offsets[s].tobytes(), om.face_aabb[s].tobytes()


def _edit_rounds(rng, w):
    """Seeded rounds of edits: interior voxels, border and corner voxels, a Uniform-air and a Uniform-stone chunk made
    Varied, a chunk emptied; repeated voxels with different types inside a round."""
    varied = [p for p in sorted(w.chunks) if w.uniform_flags[p] == 0]
    air = [p for p in sorted(w.chunks) if w.uniform_flags[p] == 1 and (p[0], p[1] - 1, p[2]) in w.chunks]
    stone = [p for p in sorted(w.chunks) if w.uniform_flags[p] == 4]
    assert varied and air and stone
    base = lambda p: np.array(p, np.int64) * 32
    rounds = []
    xyz = [base(varied[i]) + rng.integers(1, 31, 3) for i in rng.integers(0, len(varied), 40)]
    rounds.append((xyz + xyz[:5], list(rng.integers(0, 4, 40)) + list(rng.integers(0, 4, 5))))
    border = []
    for i in rng.integers(0, len(varied), 30):
        loc = rng.integers(0, 32, 3)
        loc[rng.integers(0, 3)] = rng.choice([0, 31])
        border.append(base(varied[i]) + loc)
    border += [base(varied[0]), base(varied[-1]) + 31]
    rounds.append((border, list(rng.integers(0, 4, len(border)))))
    made = [base(air[0]) + [5, 0, 7], base(air[0]) + [6, 1, 7], base(stone[0]) + [3, 31, 3], base(stone[0]) + [0, 0, 0]]
    rounds.append((made, [3, 2, 0, 0]))
    g = np.stack(np.meshgrid(np.arange(32), np.arange(32), np.arange(32), indexing="ij"), axis=-1).reshape(-1, 3)
    emptied = varied[len(varied) // 2]
    rounds.append((list(base(emptied) + g), [0] * g.shape[0]))
    return rounds, emptied


@pytest.mark.parametrize("mesh_all", [True, False])
def test_edits_remesh_exactly_what_changes(ctx, ob, mesh_all):
    """mesh_all: every chunk is meshed once, so every mesh equals the oracle's after every round; else only the chunks in
    view are, and the others must stay without a mesh.  In both, the refreshed meshes equal the oracle's over the edited
    host world and every other mesh is byte-identical to the previous round; the frame equals the oracle renderer's."""
    W, H = 320, 180
    cam = camera.Camera(WALK[0], W / H, pitch=-0.2)
    vp = cam.view_projection()
    w = _world(ctx, 3, cam.position)
    cache = vxw.MeshCache(w)
    visible = w.get_visible_chunks_frustum(cam.position, vp)
    cache.update(sorted(w.chunks) if mesh_all else visible)
    prev = w.batch.download()
    cfg, ocfg, atlas = api.default_frame_config(W, H), ob.default_frame_config(W, H, n_threads=2), ob.default_atlas()
    rounds, emptied = _edit_rounds(np.random.default_rng(7), w)
    for r, (xyz, types) in enumerate(rounds):
        dirty = w.set_blocks(xyz, types)
        refreshed = cache.refresh(dirty)
        assert refreshed == [p for p in dirty if p in cache.cached]
        got = w.batch.download()
        pos, vox, flags, nbr = _host_slots(w)
        om = ob.mesh_chunks(vox, nbr, flags, pos)
        refreshed_slots = {w.chunks[p] for p in refreshed}
        for p, s in w.chunks.items():
            if s in refreshed_slots or (mesh_all and p in cache.cached):
                assert _mesh_arrays(got, s) == _oracle_mesh(om, s), f"round {r}: mesh of {p} differs from the oracle"
            if s not in refreshed_slots:
                assert _mesh_arrays(got, s) == _mesh_arrays(prev, s), f"round {r}: mesh of {p} changed without a refresh"
            if p not in cache.cached:
                assert not got["has_mesh"][s]
        prev = got
        color, depth, surv = vxw.frame(w, cache, cam.position, vp, cfg, ctx)
        ids = np.array([s for s in cache.visible_mesh_slots(w.get_visible_chunks_frustum(cam.position, vp)).tolist() if om.has_mesh[s]],
                       dtype=np.int32)
        oc, od, osurv = ob.render_frame(om, ids, vp, cam.position, ocfg, atlas)
        assert surv.tolist() == osurv.tolist()
        assert np.array_equal(depth.view(np.uint32), od.view(np.uint32)) and np.array_equal(color, oc), f"round {r}: frame differs"
    assert w.uniform_flags[emptied] == 0 and not prev["has_mesh"][w.chunks[emptied]]
    with pytest.raises(api.VxError):  # block type out of range at the C boundary
        w.device.set_blocks(np.array([0], np.int32), np.array([0], np.int32), np.array([4], np.uint8))
    w.batch.release()


def test_break_and_place_through_pick_and_edits_survive_unloading(ctx, ob):
    W, H = 320, 180
    cam = camera.Camera(WALK[0], W / H, pitch=-0.35)
    vp = cam.view_projection()
    w = _world(ctx, 3, cam.position)
    cache = vxw.MeshCache(w)
    cfg = api.default_frame_config(W, H)
    vxw.frame(w, cache, cam.position, vp, cfg, ctx)
    centre = [(W // 2, H // 2)]
    first = w.pick(cam.position, vp, centre, W, H, MAX_T)
    assert first["status"][0] == HIT and first["face"][0] >= 0
    v0, t0 = first["voxel"][0].copy(), float(first["t"][0])
    # break: the ray goes on to a voxel behind
    cache.refresh(w.set_blocks([v0], 0))
    second = w.pick(cam.position, vp, centre, W, H, MAX_T)
    assert second["status"][0] == HIT and second["voxel"][0].tolist() != v0.tolist() and float(second["t"][0]) >= t0
    # place stone in the voxel the ray came from before entering the new hit: the ray now stops there, nearer
    f = int(second["face"][0])
    placed = second["voxel"][0] + np.array(vxw.FACE_OFFSETS[f])
    cache.refresh(w.set_blocks([placed], 3))
    third = w.pick(cam.position, vp, centre, W, H, MAX_T)
    assert third["status"][0] == HIT and third["voxel"][0].tolist() == placed.tolist() and third["block_type"][0] == 3
    assert float(third["t"][0]) <= float(second["t"][0])
    fields = ("status", "voxel", "face", "t", "block_type")  # the slot may change when the chunk comes back
    before = {k: third["hits"][k].tobytes() for k in fields}
    color0, depth0, _ = vxw.frame(w, cache, cam.position, vp, cfg, ctx)
    # walk away until the edited chunk unloads, then back
    cp = tuple(int(c) for c in placed >> 5)
    far = cam.position + np.array([32.0 * 12, 0, 0], np.float32)
    vxw.frame(w, cache, far, camera.Camera(far, W / H).view_projection(), cfg, ctx)
    assert cp not in w.chunks and cp in w.edits
    color1, depth1, _ = vxw.frame(w, cache, cam.position, vp, cfg, ctx)
    assert cp in w.chunks
    again = w.pick(cam.position, vp, centre, W, H, MAX_T)["hits"]
    assert {k: again[k].tobytes() for k in fields} == before
    assert np.array_equal(color0, color1) and np.array_equal(depth0.view(np.uint32), depth1.view(np.uint32))
    pos, vox, flags, nbr = _host_slots(w)
    om = ob.mesh_chunks(vox, nbr, flags, pos)
    got = w.batch.download()
    assert _mesh_arrays(got, w.chunks[cp]) == _oracle_mesh(om, w.chunks[cp])
    w.batch.release()


def test_pick_agrees_with_the_rendered_depth(ctx):
    """Tolerance, not bit parity: picking walks voxels, the frame rasterizes quads.  For the bench camera at 1280x720 over
    the view-distance-12 world, at least 99 % of the covered pixels (finite depth) are hits whose entry point projects to
    the depth buffer's z/w within 1e-3; pixels on quad edges may see the neighbouring surface.  At least 99 % of the sky
    pixels hit nothing that the frame drew (a ray may still hit a loaded chunk the frame did not draw)."""
    W, H = 1280, 720
    cam = camera.Camera((0.0, 10.0, 20.0), W / H)
    vp = cam.view_projection()
    w = _world(ctx, 12, cam.position)
    cache = vxw.MeshCache(w)
    _, depth, surv = vxw.frame(w, cache, cam.position, vp, api.default_frame_config(W, H), ctx)
    px = np.stack(np.meshgrid(np.arange(W), np.arange(H)), axis=-1).reshape(-1, 2)
    r = w.pick(cam.position, vp, px, W, H, 1e4)
    depth = depth.reshape(-1)
    covered = np.isfinite(depth)
    hit = r["status"] == HIT
    o, d = api.pixel_rays(vp, cam.position, px, W, H)
    p = o.astype(np.float64) + r["t"].astype(np.float64)[:, None] * d.astype(np.float64)
    m = vp.reshape(4, 4).T.astype(np.float64)
    clip = np.concatenate([p, np.ones((p.shape[0], 1))], axis=1) @ m.T
    zw = clip[:, 2] / clip[:, 3]
    agree = covered & hit & (np.abs(zw - depth) <= 1e-3)
    assert covered.sum() > W * H // 4
    assert agree.sum() >= 0.99 * covered.sum(), f"{int(agree.sum())} of {int(covered.sum())} covered pixels agree"
    drawn = set(surv.tolist())
    sky = ~covered
    sky_ok = sky & ~(hit & np.isin(r["hits"]["slot"], list(drawn)))
    assert sky_ok.sum() >= 0.99 * sky.sum(), f"{int(sky_ok.sum())} of {int(sky.sum())} sky pixels"
    w.batch.release()
