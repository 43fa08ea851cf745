"""Texturing and shading on the GPU with a non-default atlas, lights and clear colours, bit for bit against the oracle.

Every colour the frame kernels write is a 9-bit payload (face, block type, texel nibble) looked up in a 512-entry table
that the host builds from the atlas and the shading config.  With the default atlas and light most mistakes in that path
are invisible (tests/vx_shading.py); here every frame uses the discriminating atlas (or a seeded permutation of it) and
the light set LIGHTS, and colour, depth bits and draw order must equal the oracle fed the same atlas and config.  The
tests run on contexts of their own, so no other test sees their atlas.
"""
import ctypes as C

import numpy as np
import pytest

import vx_kat as kat
import vx_scenes
import vx_shading as vs

from differential_projection_voxel_renderer_b200 import api, camera

pytestmark = pytest.mark.gpu

BIN_CAP0 = 2048  # bin entries per tile of a new context (the default build)
ATLASES = {"discriminating": None, "seed1": 1, "seed2": 2}


@pytest.fixture(scope="module")
def actx():
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture
def fresh():
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def scene5(actx, ob):
    pos, world, p, v, nb = vx_scenes.terrain_scene(5)
    batch = api.BinaryGreedyMesher.mesh_batch(v, p, nb, None, actx)
    ref = ob.mesh_chunks(v, nb, None, p)
    yield p, batch, ref
    batch.release()


@pytest.fixture(scope="module")
def terr(actx, ob):
    vox, pos = vs.terraces()
    batch = api.BinaryGreedyMesher.mesh_batch(vox, pos, None, None, actx)
    ref = ob.mesh_chunks(vox, None, None, pos)
    yield pos, batch, ref
    batch.release()


def visible(ob, p, ref, vp, eye, vd):
    return np.flatnonzero((ob.cull_chunks(p, vp, eye, vd) != 0) & (ref.has_mesh != 0)).astype(np.int32)


def cfgs(ob, w, h, light=None, clear=None, threads=4):
    a, o = api.default_frame_config(w, h), ob.default_frame_config(w, h, n_threads=threads)
    for c in (a, o):
        if light is not None:
            vs.apply_light(c, light)
        if clear is not None:
            c.clear_color = clear
    return a, o


def assert_same(got, want, what=""):
    if len(got) > 2 and len(want) > 2 and got[2] is not None:
        assert np.array_equal(got[2], want[2]), f"{what}: draw order differs"
    if got[1] is not None:
        assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32)), f"{what}: depth not bit-identical"
    bad = got[0] != want[0]
    assert not bad.any(), f"{what}: {int(bad.sum())} pixels differ in colour, first at {np.argwhere(bad)[:4].tolist()}"


def counters(ctx):
    cnt = (C.c_uint32 * 32)()
    ctx.check(ctx.lib.vx_frame_counters(ctx.handle, cnt))
    return np.frombuffer(cnt, dtype=np.uint32).copy()


def device_frame(ctx, h, w):
    import torch
    from differential_projection_voxel_renderer_b200 import multigpu
    dc, dd, rows, width = api.framebuffer_device(ctx)
    assert (rows, width) == (h, w)
    dev = torch.device("cuda", ctx.device)
    c = multigpu.device_bytes_as_tensor(dc, w * h * 4, dev).cpu().numpy().view(np.uint32).reshape(h, w)
    d = multigpu.device_bytes_as_tensor(dd, w * h * 4, dev).cpu().numpy().view(np.float32).reshape(h, w)
    return c, d


# ---- 1. the frame path: every light, three atlases, every camera of the path, and the terraces --------------------------
@pytest.mark.parametrize("atlas_name", list(ATLASES))
def test_frame_path_lights_and_atlases(actx, ob, scene5, terr, atlas_name):
    p, batch, ref = scene5
    tp, tb, tref = terr
    atlas, oatlas = vs.discriminating_atlas(ATLASES[atlas_name])
    actx.set_atlas(atlas)
    w, h = 640, 360
    for lname, light in vs.LIGHTS.items():
        cfg, ocfg = cfgs(ob, w, h, light)
        for cam_i in range(len(vx_scenes.CAMERA_PATH)):  # camera 5 sits inside the terrain: near-clipped texel interpolation
            cam = vx_scenes.path_camera(cam_i, w, h)
            vp = cam.view_projection()
            ids = visible(ob, p, ref, vp, cam.position, 5)
            want = ob.render_frame(ref, ids, vp, cam.position, ocfg, oatlas)
            assert_same(api.render_frame(batch, vp, cam.position, cfg, mesh_ids=ids, ctx=actx), want, f"{lname}, camera {cam_i}")
        for k in range(3):
            vp, eye = vs.terraces_view(w, h, k)
            ids = np.arange(len(tp), dtype=np.int32)
            want = ob.render_frame(tref, ids, vp, eye, ocfg, oatlas)
            assert_same(api.render_frame(tb, vp, eye, cfg, mesh_ids=ids, ctx=actx), want, f"{lname}, terraces view {k}")


def test_full_frame_1280x720_vd12_and_texel_coverage(actx, ob, terr):
    pos, world, p, v, nb = vx_scenes.terrain_scene(12)
    batch = api.BinaryGreedyMesher.mesh_batch(v, p, nb, None, actx)
    ref = ob.mesh_chunks(v, nb, None, p)
    atlas, oatlas = vs.discriminating_atlas()
    actx.set_atlas(atlas)
    w, h = 1280, 720
    cam = vx_scenes.main_camera(w, h)
    vp = cam.view_projection()
    cfg, ocfg = cfgs(ob, w, h, vs.LIGHTS["L"], threads=8)
    want = ob.render_frame(ref, visible(ob, p, ref, vp, cam.position, 12), vp, cam.position, ocfg, oatlas)
    assert_same(api.render_frame(batch, vp, cam.position, cfg, mesh_ids=None, view_distance=12, ctx=actx), want, "1280x720 vd12, L")
    # shading off: every covered pixel decodes to a (type, nibble) of the atlas.  The terrain is grass where this camera
    # looks, so the terraces (all three block types) have to show every (type, nibble) pair.
    cfg, ocfg = cfgs(ob, w, h, vs.LIGHTS["shading_off"], threads=8)
    c, d, s = api.render_frame(batch, vp, cam.position, cfg, mesh_ids=None, view_distance=12, ctx=actx)
    assert_same((c, d, s), ob.render_frame(ref, visible(ob, p, ref, vp, cam.position, 12), vp, cam.position, ocfg, oatlas), "vd12 unshaded")
    seen = {tuple(x) for x in vs.decode(c, np.isfinite(d), atlas)}
    assert {t for t, _ in seen} >= {1}
    batch.release()
    tp, tb, tref = terr
    for k in range(3):
        tvp, eye = vs.terraces_view(w, h, k)
        ids = np.arange(len(tp), dtype=np.int32)
        c, d, s = api.render_frame(tb, tvp, eye, cfg, mesh_ids=ids, ctx=actx)
        assert_same((c, d, s), ob.render_frame(tref, ids, tvp, eye, ocfg, oatlas), f"terraces view {k} unshaded")
        seen |= {tuple(x) for x in vs.decode(c, np.isfinite(d), atlas)}
    assert seen == {(t, n) for t in vs.TYPES for n in range(16)}, sorted({(t, n) for t in vs.TYPES for n in range(16)} - seen)
    # the faces: with L and with -L every face of the terraces has a light of its own, so each shaded frame matches only
    # if every face bit and face normal is right
    for lname in ("L", "minus_L"):
        cfg, ocfg = cfgs(ob, w, h, vs.LIGHTS[lname], threads=8)
        tvp, eye = vs.terraces_view(w, h, 1)
        ids = np.arange(len(tp), dtype=np.int32)
        assert_same(api.render_frame(tb, tvp, eye, cfg, mesh_ids=ids, ctx=actx), ob.render_frame(tref, ids, tvp, eye, ocfg, oatlas), lname)


# ---- 2. other frame configurations --------------------------------------------------------------------------------------
@pytest.mark.parametrize("lname", ["L", "minus_L"])
def test_other_frame_configurations(actx, ob, scene5, terr, lname):
    p, batch, ref = scene5
    atlas, oatlas = vs.discriminating_atlas(1)
    actx.set_atlas(atlas)
    light = vs.LIGHTS[lname]
    w, h = 640, 360
    tp, tb, tref = terr
    cam = vx_scenes.path_camera(1, w, h)
    for what, b, r, pp, vp, eye in (("terrain", batch, ref, p, cam.view_projection(), cam.position),
                                     ("terraces", tb, tref, tp, *vs.terraces_view(w, h, 0))):
        ids = visible(ob, pp, r, vp, eye, 5)
        cfg, ocfg = cfgs(ob, w, h, light)
        want = ob.render_frame(r, ids, vp, eye, ocfg, oatlas)
        # stripes of 2 and 4
        for n in (2, 4):
            rows = (h + n - 1) // n
            parts = []
            for g in range(n):
                c = api.VxFrameConfig.from_buffer_copy(cfg)
                c.stripe_y0, c.stripe_rows = g * rows, min(rows, h - g * rows)
                parts.append(api.render_frame(b, vp, eye, c, mesh_ids=ids, ctx=actx))
            assert_same((np.concatenate([x[0] for x in parts]), np.concatenate([x[1] for x in parts]), parts[0][2]), want, f"{what}, {n} stripes")
        # device filter A
        assert_same(api.render_frame(b, vp, eye, cfg, mesh_ids=None, view_distance=5, ctx=actx), want, f"{what}, filter A")
        # macrotile
        mw = ob.render_frame_macrotile(r, ids, vp, ocfg, oatlas)
        got = api.render_frame_macrotile(b, ids, vp, cfg, ctx=actx)
        assert_same(got, mw[:2], f"{what}, macrotile")  # its projected-mesh order is tested in test_frame_gpu.py
        cm = api.VxFrameConfig.from_buffer_copy(cfg)
        cm.macrotile = 1
        assert_same(api.render_frame(b, vp, eye, cm, mesh_ids=ids, ctx=actx)[:2], mw[:2], f"{what}, cfg.macrotile")
        # occlusion pass
        co = api.VxFrameConfig.from_buffer_copy(cfg)
        co.occlusion_culling = 1
        oco = ob.FrameConfig.from_buffer_copy(ocfg)
        oco.occlusion_culling = 1
        assert_same(api.render_frame(b, vp, eye, co, mesh_ids=ids, ctx=actx), ob.render_frame(r, ids, vp, eye, oco, oatlas), f"{what}, occlusion")
    # the random view-projection generator of test_random_cameras_bit_exact (and its rolled / sheared matrices)
    w, h = 320, 180
    cfg, ocfg = cfgs(ob, w, h, light, threads=3)
    rng = np.random.default_rng(2026)
    mats = []
    for i in range(20):
        cam = camera.Camera(rng.uniform([-150, -30, -150], [150, 80, 150]), w / h, yaw=float(rng.uniform(-np.pi, np.pi)),
                            pitch=float(rng.uniform(-1.5, 1.5)), fov_deg=float(rng.choice([20.0, 45.0, 70.0, 110.0, 150.0])),
                            near=float(rng.choice([0.1, 0.01, 5.0])))
        mats.append((cam.view_projection(), cam.position))
    for i in range(6):
        cam = camera.Camera(rng.uniform([-80, 5, -80], [80, 40, 80]), w / h, yaw=float(rng.uniform(-3, 3)), pitch=float(rng.uniform(-0.6, 0.6)))
        m = cam.view_projection().reshape(4, 4).T.astype(np.float64)
        a = float(rng.uniform(-np.pi, np.pi))
        roll = np.array([[np.cos(a), -np.sin(a), 0, 0], [np.sin(a), np.cos(a), 0, 0], [0, 0, 1, 0], [0, 0, 0, 1]])
        shear = np.eye(4)
        shear[0, 1] = rng.uniform(-0.3, 0.3)
        mats.append((np.ascontiguousarray((shear @ roll @ m).astype(np.float32).T.reshape(16)), cam.position))
    covered = 0
    for k, (vp, eye) in enumerate(mats):
        ids = visible(ob, p, ref, vp, eye, 5)
        want = ob.render_frame(ref, ids, vp, eye, ocfg, oatlas)
        assert_same(api.render_frame(batch, vp, eye, cfg, mesh_ids=ids, ctx=actx), want, f"random matrix {k}")
        covered += int(np.isfinite(want[1]).sum())
    assert covered > 100000


# ---- 3. clear colours and frame sizes -----------------------------------------------------------------------------------
@pytest.mark.parametrize("clear", vs.CLEARS, ids=[f"{c:08x}" for c in vs.CLEARS])
def test_clear_colours_and_sizes(actx, ob, scene5, clear):
    """The fused clear writes four pixels at a time with a scalar tail; widths 1, 127 and 641 leave a tail, the heights
    partial tiles.  An all-sky camera and an empty draw list leave nothing but the clear colour."""
    p, batch, ref = scene5
    atlas, oatlas = vs.discriminating_atlas()
    actx.set_atlas(atlas)
    for w, h in ((1, 1), (127, 33), (641, 359)):
        cfg, ocfg = cfgs(ob, w, h, vs.LIGHTS["shading_off"], clear=clear, threads=2)
        cam = camera.Camera((0.0, 10.0, 20.0), w / h, yaw=0.2, pitch=-0.1)
        vp = cam.view_projection()
        ids = visible(ob, p, ref, vp, cam.position, 5)
        want = ob.render_frame(ref, ids, vp, cam.position, ocfg, oatlas)
        assert_same(api.render_frame(batch, vp, cam.position, cfg, mesh_ids=ids, ctx=actx), want, f"{w}x{h}")
        if w > 1:
            assert (want[0] == clear).any() and np.isfinite(want[1]).any()
        sky = camera.Camera((0.0, 100.0, 0.0), w / h, pitch=1.5)  # looking up: nothing in view
        ids = visible(ob, p, ref, sky.view_projection(), sky.position, 5)
        want = ob.render_frame(ref, ids, sky.view_projection(), sky.position, ocfg, oatlas)
        assert (want[0] == clear).all()
        assert_same(api.render_frame(batch, sky.view_projection(), sky.position, cfg, mesh_ids=ids, ctx=actx), want, f"{w}x{h}, sky")
        got = api.render_frame(batch, vp, cam.position, cfg, mesh_ids=np.zeros(0, np.int32), ctx=actx)
        assert got[2].size == 0 and (got[0] == clear).all() and np.isinf(got[1]).all(), f"{w}x{h}, empty list"
        assert_same(api.render_frame(batch, vp, cam.position, cfg, mesh_ids=None, view_distance=5, ctx=actx),
                    ob.render_frame(ref, visible(ob, p, ref, vp, cam.position, 5), vp, cam.position, ocfg, oatlas), f"{w}x{h}, filter A")


# ---- 4. read-modify-write and barycentric paths (vx_render_mesh, vx_bary.cu) --------------------------------------------
@pytest.mark.parametrize("lname", ["L", "minus_L", "negative_ambient_clamps_to_0", "shading_off"])
def test_mesh_paths_with_rasterizer_shading(actx, ob, terr, lname):
    tp, tb, tref = terr
    atlas, oatlas = vs.discriminating_atlas(2)
    light = vs.LIGHTS[lname]
    w, h = 320, 200
    r = api.Rasterizer(actx, atlas)
    r.shading = api.ShadingConfig(*light[:3])
    r.enable_shading = bool(light[3])
    ocfg = vs.apply_light(ob.default_frame_config(w, h), light)

    def start():
        fb = api.Framebuffer(w, h)
        fb.clear(0x00FF00FF)
        fb.depth_buffer[40:60, 50:150] = 0.9  # existing contents take part in the depth test
        fb.color_buffer[40:60, 50:150] = 0x80010203
        return fb, fb.color_buffer.copy(), fb.depth_buffer.copy()

    for k in range(3):
        vp, eye = vs.terraces_view(w, h, k)
        for rect in ((0, 0, w, h), (0, 48, w, 51), (17, 9, 200, 150)):
            fb, oc, od = start()
            for mid in range(len(tp)):
                ob.render_mesh(tref, mid, vp, ocfg, oatlas, rect, oc, od)
                if rect == (0, 0, w, h):
                    r.render_mesh(tb, mid, vp, fb)
                elif rect[0] == 0 and rect[2] == w:
                    r.render_mesh_into_slice(tb, mid, vp, fb, rect[1], rect[3])
                else:
                    r.render_mesh_into_tile(tb, mid, vp, fb, *rect)
            assert_same((fb.color_buffer, fb.depth_buffer), (oc, od), f"render_mesh view {k} rect {rect}")
            fb, oc, od = start()
            for mid in range(len(tp)):
                ob.render_mesh_tiny_quads(tref, mid, vp, ocfg, oatlas, rect, False, oc, od)
                r.render_mesh_tiny_quads(tb, mid, vp, fb, rect, False)
            assert_same((fb.color_buffer, fb.depth_buffer), (oc, od), f"tiny quads (barycentric) view {k} rect {rect}")
        assert int(np.isfinite(od).sum()) > 5000
    # render_mesh_with_up: a rolled camera takes the barycentric rasterizer, a level one the span renderer
    for eye, center, up in (((70.0, 30.0, 60.0), (30.0, 6.0, 30.0), (0.5, 0.8, 0.2)), ((66.0, 30.0, 70.0), (30.0, 8.0, 30.0), (0.0, 1.0, 0.0))):
        proj = camera.perspective_rh(np.radians(np.float32(70.0)), w / h, 0.1, 1000.0)
        vp = np.ascontiguousarray(camera.mat4_mul(proj, camera.look_at_rh(eye, center, up)).reshape(16), dtype=np.float32)
        fb, oc, od = start()
        for mid in range(len(tp)):
            ob.render_mesh_with_up(tref, mid, vp, ocfg, oatlas, up, oc, od)
            r.render_mesh_with_up(tb, mid, vp, fb, up)
        assert_same((fb.color_buffer, fb.depth_buffer), (oc, od), f"render_mesh_with_up {up}")
        assert int(np.isfinite(od).sum()) > 5000


# ---- 5. the table cache: one input changes per frame ---------------------------------------------------------------------
def _frame_inputs(step, w, h, ob):
    (atlas, oatlas), light, clear = step
    cfg, ocfg = cfgs(ob, w, h, light, clear=clear)
    return atlas, oatlas, cfg, ocfg


def test_table_cache_synchronous(fresh, ob, scene5, terr):
    tp, tb, tref = terr
    w, h = 320, 200
    vp, eye = vs.terraces_view(w, h, 1)
    ids = np.arange(len(tp), dtype=np.int32)
    for i, step in enumerate(vs.cache_sequence()):
        atlas, oatlas, cfg, ocfg = _frame_inputs(step, w, h, ob)
        fresh.set_atlas(atlas)
        want = ob.render_frame(tref, ids, vp, eye, ocfg, oatlas)
        assert_same(api.render_frame(tb, vp, eye, cfg, mesh_ids=ids, ctx=fresh), want, f"frame {i}")
        # the read-modify-write path shares the table
        fb = api.Framebuffer(w, h)
        fb.clear(0)
        oc, od = fb.color_buffer.copy(), fb.depth_buffer.copy()
        ob.render_mesh(tref, 1, vp, ocfg, oatlas, (0, 0, w, h), oc, od)
        fresh.check(fresh.lib.vx_render_mesh(fresh.handle, tb.handle, 1, vp.ctypes.data, C.byref(cfg),
                                             np.array([0, 0, w, h], np.int32).ctypes.data, fb.color_buffer.ctypes.data,
                                             fb.depth_buffer.ctypes.data))
        assert_same((fb.color_buffer, fb.depth_buffer), (oc, od), f"frame {i}, render_mesh")


def test_table_cache_async_lanes_graph_replay(ob, terr):
    tp, tb, tref = terr
    w, h = 320, 200
    vp, eye = vs.terraces_view(w, h, 1)
    vp_t, eye_t = tuple(vp.tolist()), tuple(eye.tolist())
    ids = visible(ob, tp, tref, vp, eye, 5)
    lanes = api.FrameLanes(0, 3)
    try:
        prev_atlas = None
        for i, step in enumerate(vs.cache_sequence()):
            atlas, oatlas, cfg, ocfg = _frame_inputs(step, w, h, ob)
            if prev_atlas is None or bytes(atlas) != prev_atlas:
                lanes.set_atlas(atlas)
                prev_atlas = bytes(atlas)
            want = ob.render_frame(tref, ids, vp, eye, ocfg, oatlas)
            if i == 0:  # a synchronous frame per lane sizes its scratch
                for c in lanes.ctxs:
                    api.render_frame_device(tb, vp_t, eye_t, cfg, 5, c)
            cfga = api.VxFrameConfig.from_buffer_copy(cfg)
            cfga.async_submit = 1
            for _ in range(2 * len(lanes)):  # two per lane: the second replays the lane's captured graph
                api.render_frame_device(tb, vp_t, eye_t, cfga, 5, lanes.next())
            lanes.synchronize()
            for li, c in enumerate(lanes.ctxs):
                api.frame_stats(c)  # raises if the frame overflowed
                assert_same(device_frame(c, h, w), want[:2], f"frame {i}, lane {li}")
    finally:
        lanes.close()


@pytest.mark.parametrize("n_lanes", [1, 3])
def test_table_cache_pipelined(fresh, ob, terr, n_lanes):
    """FrameLoop.submit / wait: the atlas or the light changes between two submits while the earlier frame is in flight."""
    tp, tb, tref = terr
    w, h = 320, 200
    vp, eye = vs.terraces_view(w, h, 1)
    ids = visible(ob, tp, tref, vp, eye, 5)
    seq = vs.cache_sequence()
    cfg0 = cfgs(ob, w, h)[0]
    loop = api.FrameLoop(tb, cfg0, view_distance=5, want_depth=True, ctx=fresh, lanes=n_lanes)
    try:
        loop.render(vp, eye)  # sizes the first lane's scratch
        pend = []
        for i, step in enumerate(seq + seq):
            atlas, oatlas, cfg, ocfg = _frame_inputs(step, w, h, ob)
            loop.lanes.set_atlas(atlas)
            C.memmove(C.byref(loop.cfg), C.byref(cfg), C.sizeof(api.VxFrameConfig))
            pend.append((i, loop.submit(vp, eye), ob.render_frame(tref, ids, vp, eye, ocfg, oatlas)))
            if len(pend) == 2:
                j, t, want = pend.pop(0)
                assert_same(loop.wait(t), want, f"frame {j}")
        for j, t, want in pend:
            assert_same(loop.wait(t), want, f"frame {j}")
    finally:
        loop.close()


# ---- 6. an overflowed in-flight frame keeps the atlas and light it was submitted with -------------------------------------
@pytest.fixture(scope="module")
def stack(actx, ob):
    """1152 one-layer plates at one position (tests/test_frame_capacity_gpu.py): 2 x 1152 triangles in every tile at
    128 x 64, so the first frame of a new context overflows its 2048-entry bins."""
    n = 1152
    vox = np.stack([kat.chunk_plate(1 + k % 3) for k in range(n)])
    pos = np.zeros((n, 3), dtype=np.int32)
    batch = api.BinaryGreedyMesher.mesh_batch(vox, pos, None, None, actx)
    ref = ob.mesh_chunks(vox, None, None, pos)
    yield batch, ref, pos
    batch.release()


@pytest.mark.parametrize("change", ["atlas", "light"])
def test_overflowed_inflight_frame_keeps_its_inputs(fresh, ob, stack, change):
    batch, ref, pos = stack
    w, h = 128, 64
    proj = camera.perspective_rh(np.radians(np.float32(70.0)), w / h, 0.1, 1000.0)
    eye = np.asarray((16.0, 10.0, 16.0), dtype=np.float32)
    vp = np.ascontiguousarray(camera.mat4_mul(proj, camera.look_at_rh(eye, (16.0, 0.0, 16.0), (0.0, 0.0, -1.0))).reshape(16), dtype=np.float32)
    ids = np.flatnonzero(ob.cull_chunks(pos, vp, eye, 2)).astype(np.int32)
    a, b = vs.discriminating_atlas(), vs.discriminating_atlas(1)
    la, lb = vs.LIGHTS["L"], vs.LIGHTS["minus_L"]  # the plates' tops (+Y) get 0.3 and 0.3 + 0.7 * 0.53
    if change == "light":
        b = a
    else:
        lb = la
    cfg_a, ocfg_a = cfgs(ob, w, h, la)
    cfg_b, ocfg_b = cfgs(ob, w, h, lb)
    want_a = ob.render_frame(ref, ids, vp, eye, ocfg_a, a[1])
    want_b = ob.render_frame(ref, ids, vp, eye, ocfg_b, b[1])
    assert np.isfinite(want_a[1]).all() and not np.array_equal(want_a[0], want_b[0])
    loop = api.FrameLoop(batch, cfg_a, view_distance=2, want_depth=True, ctx=fresh, lanes=1)
    try:
        fresh.set_atlas(a[0])
        k = loop.submit(vp, eye)
        fresh.set_atlas(b[0])
        C.memmove(C.byref(loop.cfg), C.byref(cfg_b), C.sizeof(api.VxFrameConfig))
        k1 = loop.submit(vp, eye)
        assert_same(loop.wait(k), want_a, f"frame k ({change} A)")
        cnt = counters(fresh)
        assert cnt[4] == 0 and cnt[5] > BIN_CAP0, cnt[:8]  # frame k needed more than the new context's bins: it overflowed
        assert_same(loop.wait(k1), want_b, f"frame k + 1 ({change} B)")
        # and the context still holds B for the next frame
        assert_same(api.render_frame(batch, vp, eye, cfg_b, mesh_ids=ids, ctx=fresh), want_b, "synchronous frame after")
    finally:
        loop.close()


# ---- 7. api.Rasterizer: an atlas per Rasterizer, shading on every mesh entry point ----------------------------------------
def test_two_rasterizers_share_a_context(fresh, ob, terr):
    tp, tb, tref = terr
    w, h = 320, 200
    vp, eye = vs.terraces_view(w, h, 0)
    a, oa = vs.discriminating_atlas(1)
    od_atlas = vs.default_atlas_pair()[1]
    ra = api.Rasterizer(fresh, a)
    rd = api.Rasterizer(fresh)  # the default atlas, although the context last loaded A
    assert rd.atlas is None and ra.atlas is a
    ocfg = ob.default_frame_config(w, h)
    fb = api.Framebuffer(w, h)
    fb.clear(0xFF87CEEB)
    oc, od = fb.color_buffer.copy(), fb.depth_buffer.copy()
    for mid in range(len(tp)):  # alternate: each draw equals the oracle with its own atlas
        r, atl = (ra, oa) if mid % 2 == 0 else (rd, od_atlas)
        ob.render_mesh(tref, mid, vp, ocfg, atl, (0, 0, w, h), oc, od)
        r.render_mesh(tb, mid, vp, fb)
        assert_same((fb.color_buffer, fb.depth_buffer), (oc, od), f"mesh {mid}")
    # Rasterizer.shading reaches render_mesh, render_mesh_tiny_quads and render_mesh_with_up
    light = vs.LIGHTS["minus_L"]
    ra.shading = api.ShadingConfig(light[0], light[1], light[2])
    sc = vs.apply_light(ob.default_frame_config(w, h), light)
    up = (0.3, 0.9, 0.1)
    proj = camera.perspective_rh(np.radians(np.float32(70.0)), w / h, 0.1, 1000.0)
    rolled = np.ascontiguousarray(camera.mat4_mul(proj, camera.look_at_rh(eye, (30.0, 8.0, 30.0), up)).reshape(16), dtype=np.float32)
    for name in ("render_mesh", "tiny_quads", "with_up"):
        fb = api.Framebuffer(w, h)
        fb.clear(0)
        oc, od = fb.color_buffer.copy(), fb.depth_buffer.copy()
        plain = api.Framebuffer(w, h)
        plain.clear(0)
        for mid in range(len(tp)):
            if name == "render_mesh":
                ob.render_mesh(tref, mid, vp, sc, oa, (0, 0, w, h), oc, od)
                ra.render_mesh(tb, mid, vp, fb)
            elif name == "tiny_quads":
                ob.render_mesh_tiny_quads(tref, mid, vp, sc, oa, (0, 0, w, h), False, oc, od)
                ra.render_mesh_tiny_quads(tb, mid, vp, fb, (0, 0, w, h), False)
            else:
                ob.render_mesh_with_up(tref, mid, rolled, sc, oa, up, oc, od)
                ra.render_mesh_with_up(tb, mid, rolled, fb, up)
        assert_same((fb.color_buffer, fb.depth_buffer), (oc, od), name)
        assert int(np.isfinite(od).sum()) > 5000
