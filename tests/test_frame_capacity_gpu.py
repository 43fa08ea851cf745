"""Frames that do not fit the scratch a context starts with, bit for bit against the CPU oracle.

A frame context starts with 2048 entries per tile bin, two triangle slots per quad of the batch (+ 1024) and one setup
unit per mesh id + one per 128 quads of the batch.  A frame that needs more sets an overflow bit; the synchronous paths
grow the scratch and render the frame again, the pipelined path re-renders inside vx_render_frame_end, an async frame
reports VX_ERR_CAPACITY through vx_frame_stats and grows the scratch for the lane's next frame.  Capacities only grow,
so every overflow test runs on a context of its own (`fresh`), and every test also shows from the frame counters that
the path it is about was taken.
"""
import ctypes as C

import numpy as np
import pytest

import vx_kat as kat
import vx_scenes

from differential_projection_voxel_renderer_b200 import api, camera

pytestmark = pytest.mark.gpu

BIN_CAP0 = 2048          # bin entries per tile of a new context (the default build's VX_BIN_CAP0; stress builds use less)
SEQ_QUAD_LIMIT = 1 << 21  # quads one frame can draw: the draw sequence is 23 bits = quad rank * 4 + sub-triangle
CHECKER_QUADS = 98304     # kat.chunk_checker3d_typed


@pytest.fixture
def fresh():
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def scene5(ctx, ob):
    pos, world, p, v, nb = vx_scenes.terrain_scene(5)
    batch = api.BinaryGreedyMesher.mesh_batch(v, p, nb, None, ctx)
    ref = ob.mesh_chunks(v, nb, None, p)
    yield p, batch, ref
    batch.release()


def _batch(ctx, ob, vox, pos):
    vox = np.ascontiguousarray(vox, dtype=np.uint8).reshape(len(pos), -1)
    pos = np.asarray(pos, dtype=np.int32).reshape(-1, 3)
    return api.BinaryGreedyMesher.mesh_batch(vox, pos, None, None, ctx), ob.mesh_chunks(vox, None, None, pos), pos


@pytest.fixture(scope="module")
def stack(ctx, ob):
    """1152 one-layer plates at the same position, block types cycling: 2 x 1152 triangles in every tile at 128 x 64,
    none of them big, every fragment of a pixel at the same depth (the first plate in the list wins)."""
    n = 1152
    vox = np.stack([kat.chunk_plate(1 + k % 3) for k in range(n)])
    batch, ref, pos = _batch(ctx, ob, vox, [(0, 0, 0)] * n)
    yield batch, ref, pos
    batch.release()


def _look(eye, center, up, w, h):
    proj = camera.perspective_rh(np.radians(np.float32(70.0)), w / h, 0.1, 1000.0)
    return camera.mat4_mul(proj, camera.look_at_rh(eye, center, up)).reshape(16), np.asarray(eye, dtype=np.float32)


def _down_view(w, h, height=10.0):
    """Straight down onto the middle of chunk (0, 0, 0): a plate at y = 0 fills the screen."""
    return _look((16.0, height, 16.0), (16.0, 0.0, 16.0), (0.0, 0.0, -1.0), w, h)


def counters(ctx):
    cnt = (C.c_uint32 * 32)()
    ctx.check(ctx.lib.vx_frame_counters(ctx.handle, cnt))
    return np.frombuffer(cnt, dtype=np.uint32).copy()


def assert_same(got, want, what=""):
    c, d = got[0], got[1]
    oc, od = want[0], want[1]
    if len(got) > 2 and len(want) > 2:
        assert np.array_equal(got[2], want[2]), f"{what}: draw order differs"
    assert np.array_equal(d.view(np.uint32), od.view(np.uint32)), f"{what}: depth not bit-identical"
    assert np.array_equal(c, oc), f"{what}: colour not bit-identical"


def oracle(ob, ref, ids, vp, eye, w, h):
    return ob.render_frame(ref, np.asarray(ids, np.int32), vp, eye, ob.default_frame_config(w, h, n_threads=4), ob.default_atlas())


def device_frame(ctx, h, w):
    import torch
    from differential_projection_voxel_renderer_b200 import multigpu
    dc, dd, rows, width = api.framebuffer_device(ctx)
    assert (rows, width) == (h, w)
    dev = torch.device("cuda", ctx.device)
    c = multigpu.device_bytes_as_tensor(dc, w * h * 4, dev).cpu().numpy().view(np.uint32).reshape(h, w)
    d = multigpu.device_bytes_as_tensor(dd, w * h * 4, dev).cpu().numpy().view(np.float32).reshape(h, w)
    return c, d


# ---- 1. bin overflow, synchronous frames --------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["full", "stripes", "macrotile", "filter_a"])
def test_bin_overflow_sync_frame(fresh, ob, stack, scene5, mode):
    batch, ref, pos = stack
    w, h = 128, 64
    vp, eye = _down_view(w, h)
    ids = np.arange(len(pos), dtype=np.int32)
    cfg = api.default_frame_config(w, h)
    if mode == "macrotile":
        want = ob.render_frame_macrotile(ref, ids, vp, ob.default_frame_config(w, h, n_threads=4), ob.default_atlas())
        cfg.macrotile = 1
    else:
        want = oracle(ob, ref, ids, vp, eye, w, h)
    assert np.isfinite(want[1]).all()  # the plates cover every pixel

    def frame():
        if mode == "stripes":
            parts = []
            for y0, y1 in ((0, 24), (24, 64)):
                c = api.VxFrameConfig.from_buffer_copy(cfg)
                c.stripe_y0, c.stripe_rows = y0, y1 - y0
                parts.append(api.render_frame(batch, vp, eye, c, mesh_ids=ids, ctx=fresh))
                if y0 == 0:
                    assert counters(fresh)[5] > BIN_CAP0  # the first stripe overflowed the new context's bins
            assert all(np.array_equal(p[2], parts[0][2]) for p in parts)
            return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]), parts[0][2]
        if mode == "filter_a":
            vis = ob.cull_chunks(pos, vp, eye, 2)
            assert vis.all()
            return api.render_frame(batch, vp, eye, cfg, mesh_ids=None, view_distance=2, ctx=fresh)
        return api.render_frame(batch, vp, eye, cfg, mesh_ids=ids, ctx=fresh)

    assert_same(frame(), want, f"{mode}, first frame")
    cnt = counters(fresh)
    assert cnt[4] == 0 and cnt[5] > BIN_CAP0 and cnt[6] == 0, cnt[:8]  # fullest bin above the starting capacity, no big list
    assert_same(frame(), want, f"{mode}, grown context")
    # a terrain frame whose work-item plan reads the stack's oversized tile counters (another tile grid)
    p, tb, tref = scene5
    tw, th = 640, 360
    cam = vx_scenes.path_camera(0, tw, th)
    tvp = cam.view_projection()
    tids = np.flatnonzero((ob.cull_chunks(p, tvp, cam.position, 5) != 0) & (tref.has_mesh != 0)).astype(np.int32)
    got = api.render_frame(tb, tvp, cam.position, api.default_frame_config(tw, th), mesh_ids=tids, ctx=fresh)
    assert_same(got, oracle(ob, tref, tids, tvp, cam.position, tw, th), f"{mode}, terrain after the stack")


# ---- 2. bin overflow on the read-modify-write path (vx_render_mesh) -----------------------------------------------------
def _flat_vp(w, h):
    """Orthographic, chunk (0, 0, 0)'s x / y square onto the w x h screen, every point at depth 0.5: all the z layers of
    a mesh tie, so the earliest-drawn fragment of a pixel wins (and an existing depth of 0.5 beats them all)."""
    m = np.zeros((4, 4), dtype=np.float64)
    m[0, 0], m[0, 3] = 2.0 / 32.0, -1.0
    m[1, 1], m[1, 3] = 2.0 / 32.0, -1.0
    m[2, 3] = 0.5
    m[3, 3] = 1.0
    return np.ascontiguousarray(m.T.reshape(16).astype(np.float32))


@pytest.mark.parametrize("target", [(0, 0, 128, 32), (0, 8, 128, 17), (3, 5, 120, 26)])
def test_bin_overflow_read_modify_write(fresh, ob, target):
    vox = kat.chunk_z_plates(16).reshape(1, -1)
    batch, ref, _ = _batch(fresh, ob, vox, [(0, 0, 0)])
    w, h = 128, 32
    vp = _flat_vp(w, h)
    fb = api.Framebuffer(w, h)
    fb.clear(0xFF87CEEB)
    fb.depth_buffer[4:12, 20:60] = 0.5   # equal depth: the existing contents keep these pixels
    fb.color_buffer[4:12, 20:60] = 0xFF112233
    fb.depth_buffer[14:30, 70:110] = 0.75  # farther: the mesh replaces them
    fb.color_buffer[14:30, 70:110] = 0xFF445566
    oc, od = fb.color_buffer.copy(), fb.depth_buffer.copy()
    ob.render_mesh(ref, 0, vp, ob.default_frame_config(w, h), ob.default_atlas(), target, oc, od)
    r = api.Rasterizer(fresh)
    if target == (0, 0, w, h):
        r.render_mesh(batch, 0, vp, fb)
    elif target[0] == 0 and target[2] == w:
        r.render_mesh_into_slice(batch, 0, vp, fb, target[1], target[3])
    else:
        r.render_mesh_into_tile(batch, 0, vp, fb, *target)
    cnt = counters(fresh)
    assert cnt[4] == 0 and cnt[5] > BIN_CAP0, cnt[:8]  # the first attempt's bins overflowed
    assert np.array_equal(fb.depth_buffer.view(np.uint32), od.view(np.uint32)), target
    assert np.array_equal(fb.color_buffer, oc), target
    x0, y0, tw, th = target
    inside = oc[y0:y0 + th, x0:x0 + tw]
    assert len(np.unique(inside)) > 3 and (inside[max(0, 4 - y0):12 - y0, 20 - x0:60 - x0] == 0xFF112233).all()
    batch.release()


# ---- 3. pipelined frames ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lanes", [1, 3])
def test_bin_overflow_pipelined(fresh, ob, stack, lanes):
    batch, ref, pos = stack
    w, h = 128, 64
    vp, eye = _down_view(w, h)
    want = oracle(ob, ref, np.flatnonzero(ob.cull_chunks(pos, vp, eye, 2)), vp, eye, w, h)
    loop = api.FrameLoop(batch, api.default_frame_config(w, h), view_distance=2, want_depth=True, ctx=fresh, lanes=lanes)
    try:
        for rnd in range(2):  # two frames in flight on every lane: the second was enqueued with the lane's first scratch
            ts = [loop.submit(vp, eye) for _ in range(2 * lanes)]
            for t in ts:
                assert_same(loop.wait(t), want, f"round {rnd}, frame {t}")
        for lane in loop.lanes.ctxs:
            cnt = counters(lane)
            assert cnt[4] == 0 and cnt[5] > BIN_CAP0  # every lane started small and overflowed
    finally:
        loop.close()


# ---- 4. asynchronous device frames --------------------------------------------------------------------------------------
def _async_until_ok(submit, c, max_frames=3):
    """After an async frame that overflowed: vx_frame_stats grew the scratch, so the lane's next async frames settle
    (one more per capacity that the overflowed frame could not size, e.g. work items planned from its counters) --
    returns the stats of the first clean frame, fails if the lane stays stuck."""
    for k in range(max_frames):
        submit()
        try:
            return api.frame_stats(c), k + 1
        except api.VxError as e:
            assert e.code == -4 and int(counters(c)[4]) & ~0x123 == 0  # only grown capacities (1, 2, 32, 256)
    pytest.fail("the lane did not recover from the overflow")


def _async_then_recover(c, ob, batch, want, vp, eye, w, h, sync_first):
    cfg = api.default_frame_config(w, h)
    cfga = api.VxFrameConfig.from_buffer_copy(cfg)
    cfga.async_submit = 1
    api.render_frame_device(batch, vp, eye, cfga, 2, c)
    with pytest.raises(api.VxError) as e:
        api.frame_stats(c)
    assert e.value.code == -4  # VX_ERR_CAPACITY
    if sync_first:
        assert_same(api.render_frame(batch, vp, eye, cfg, mesh_ids=None, view_distance=2, ctx=c), want, "synchronous re-render")
    st, _ = _async_until_ok(lambda: api.render_frame_device(batch, vp, eye, cfga, 2, c), c)
    assert st.reserved[0] > BIN_CAP0
    assert_same(device_frame(c, h, w), want, "next async frame")


def test_bin_overflow_async_frames(fresh, ob, stack):
    batch, ref, pos = stack
    w, h = 128, 64
    vp, eye = _down_view(w, h)
    want = oracle(ob, ref, np.flatnonzero(ob.cull_chunks(pos, vp, eye, 2)), vp, eye, w, h)
    _async_then_recover(fresh, ob, batch, want, vp, eye, w, h, sync_first=True)
    lanes = api.FrameLanes(0, 3)
    try:
        for i, c in enumerate(lanes.ctxs):
            _async_then_recover(c, ob, batch, want, vp, eye, w, h, sync_first=(i == 0))
    finally:
        lanes.close()


# ---- 5. near-clip second pieces and the big-triangle list ---------------------------------------------------------------
def test_near_clip_pieces_and_big_list(fresh, ob, scene5):
    p, tb, tref = scene5
    w, h = 640, 360
    cam = vx_scenes.path_camera(5, w, h)  # inside the terrain: triangles cut by the near plane
    vp = cam.view_projection()
    ids = np.flatnonzero((ob.cull_chunks(p, vp, cam.position, 5) != 0) & (tref.has_mesh != 0)).astype(np.int32)
    got = api.render_frame(tb, vp, cam.position, api.default_frame_config(w, h), mesh_ids=ids, ctx=fresh)
    assert_same(got, oracle(ob, tref, ids, vp, cam.position, w, h), "terrain, camera inside")

    n = 40
    vox = np.stack([kat.chunk_plate(1 + k % 3) for k in range(n)])
    batch, ref, pos = _batch(fresh, ob, vox, [(0, 0, 0)] * n)
    # just above a plate, looking along it: both top triangles have corners behind the near plane and are cut into two
    vp, eye = _look((16.0, 1.5, 16.0), (16.0, 1.2, 0.0), (0.0, 1.0, 0.0), w, h)
    ids = np.arange(3, dtype=np.int32)
    got = api.render_frame(batch, vp, eye, api.default_frame_config(w, h), mesh_ids=ids, ctx=fresh)
    assert_same(got, oracle(ob, ref, ids, vp, eye, w, h), "near clip")
    assert counters(fresh)[13] > 0  # second pieces of near-clipped triangles
    near, eye_n = _down_view(w, h)                                             # each plate's top: 2 screen-filling triangles
    far, eye_f = _look((16.0, 60.0, 200.0), (16.0, 0.0, 16.0), (0.0, 1.0, 0.0), w, h)  # a few tiles wide: nothing big
    seen = []
    # the work-item plan of a frame reads the previous frame's big-triangle boxes: big -> none -> few -> many -> few
    for kind, k in (("big", n), ("none", n), ("big", 1), ("big", n), ("big", 1), ("none", 1)):
        vp, eye = (near, eye_n) if kind == "big" else (far, eye_f)
        ids = np.arange(k, dtype=np.int32)
        got = api.render_frame(batch, vp, eye, api.default_frame_config(w, h), mesh_ids=ids, ctx=fresh)
        assert_same(got, oracle(ob, ref, ids, vp, eye, w, h), f"{kind} x {k}")
        n_big = int(counters(fresh)[6])
        seen.append(n_big)
        if kind == "none":
            assert n_big == 0 and (got[0] != api.default_frame_config(w, h).clear_color).sum() > 0
        elif k == 1:
            assert 1 <= n_big <= 64, n_big    # tiles test the boxes themselves
        else:
            assert n_big > 64, n_big          # every tile goes through a work item
    print("big triangles per frame:", seen)
    batch.release()


# ---- 6. the 2^21-quad draw-sequence limit -------------------------------------------------------------------------------
def test_draw_sequence_edge(fresh, ob):
    """21 checkerboard chunks = 2,064,384 quads, just under 2^21: quad ranks >= 2^20 fill bit 31 of the key's low word.
    Twenty copies sit at one near position (ties: the first copy keeps every pixel, copies 11.. rank above 2^20 and
    lose), one chunk beside and behind them is drawn last and wins where it shows.  A 22nd chunk is refused."""
    n_pad = 21
    vox = [kat.chunk_checker3d_typed(1 + k % 3) for k in range(n_pad)] + [kat.chunk_checker3d_typed(kat.STONE)]
    pos = [(0, 0, 0)] * n_pad + [(1, 0, -2)]
    batch, ref, pos = _batch(fresh, ob, np.stack(vox), pos)
    far = n_pad
    assert (batch.download()["quad_count"] == CHECKER_QUADS).all()
    w, h = 256, 128
    vp, eye = _look((32.0, 16.0, 70.0), (32.0, 16.0, 0.0), (0.0, 1.0, 0.0), w, h)
    ids = np.array(list(range(20)) + [far], dtype=np.int32)
    assert ids.size * CHECKER_QUADS < SEQ_QUAD_LIMIT <= (ids.size + 1) * CHECKER_QUADS
    want = oracle(ob, ref, ids, vp, eye, w, h)
    got = api.render_frame(batch, vp, eye, api.default_frame_config(w, h), mesh_ids=ids, ctx=fresh)
    assert_same(got, want, "21 chunks")
    cnt = counters(fresh)
    assert cnt[4] == 0 and cnt[1] == ids.size * CHECKER_QUADS
    assert got[2][-1] == far  # drawn last: its quad ranks start at 20 * 98304 >= 2^20
    c, d = got[0], got[1]
    only_far = oracle(ob, ref, [far], vp, eye, w, h)
    only_first = oracle(ob, ref, [0], vp, eye, w, h)
    won_by_far = np.isinf(only_first[1]) & np.isfinite(only_far[1]) & (c == only_far[0])
    kept_by_first = np.isfinite(only_first[1]) & (d.view(np.uint32) == only_first[1].view(np.uint32)) & (c == only_first[0])
    assert won_by_far.sum() > 100 and kept_by_first.sum() > 100, (won_by_far.sum(), kept_by_first.sum())
    # copy 11 (quad ranks from 11 * 98304 > 2^20) has another block type than copy 0: a lost tie would show
    assert not np.array_equal(oracle(ob, ref, [11], vp, eye, w, h)[0][kept_by_first], c[kept_by_first])

    ids22 = np.array(list(range(n_pad)) + [far], dtype=np.int32)
    sentinel = np.full((h, w), 0x12345678, dtype=np.uint32)
    with pytest.raises(api.VxError) as e:
        api.render_frame(batch, vp, eye, api.default_frame_config(w, h), mesh_ids=ids22, color_out=sentinel, ctx=fresh)
    assert e.value.code == -4 and "2^21" in str(e.value)
    assert (sentinel == 0x12345678).all()  # nothing of the refused frame reached the caller
    assert_same(api.render_frame(batch, vp, eye, api.default_frame_config(w, h), mesh_ids=ids, ctx=fresh), want, "after the refusal")
    batch.release()


# ---- 7. duplicate mesh ids ----------------------------------------------------------------------------------------------
def _checker_one(ctx, ob):
    return _batch(ctx, ob, kat.chunk_checker3d_typed(kat.STONE).reshape(1, -1), [(0, 0, 0)])


def _checker_view(w, h):
    return _look((16.0, 40.0, 60.0), (16.0, 16.0, 16.0), (0.0, 1.0, 0.0), w, h)


def _assert_grew_past_the_estimates(cnt, n_ids, batch_quads):
    # a new context sizes setup units as n_ids + batch quads / 128 + 1 and triangle slots as 2 x batch quads + 1024
    assert cnt[7] > n_ids + batch_quads // 128 + 1, cnt[:8]
    assert 2 * int(cnt[1]) > 2 * batch_quads + 1024, cnt[:8]


@pytest.mark.parametrize("ids", [[0, 0], [0, 0, 0]])
def test_duplicate_ids_one_chunk_sync(fresh, ob, ids):
    batch, ref, _ = _checker_one(fresh, ob)
    w, h = 256, 128
    vp, eye = _checker_view(w, h)
    want = oracle(ob, ref, ids, vp, eye, w, h)
    assert want[2].tolist() == ids  # the oracle draws every repeat
    got = api.render_frame(batch, vp, eye, api.default_frame_config(w, h), mesh_ids=np.array(ids, np.int32), ctx=fresh)
    assert_same(got, want, f"ids {ids}")
    cnt = counters(fresh)
    assert cnt[4] == 0 and cnt[1] == len(ids) * CHECKER_QUADS
    _assert_grew_past_the_estimates(cnt, len(ids), CHECKER_QUADS)
    assert_same(api.render_frame(batch, vp, eye, api.default_frame_config(w, h), mesh_ids=np.array(ids, np.int32), ctx=fresh), want, "again")
    batch.release()


def test_duplicate_ids_terrain_sync(fresh, ob, scene5):
    p, tb, tref = scene5
    w, h = 640, 360
    for cam_i in (0, 3):
        cam = vx_scenes.path_camera(cam_i, w, h)
        vp = cam.view_projection()
        vis = np.flatnonzero((ob.cull_chunks(p, vp, cam.position, 5) != 0) & (tref.has_mesh != 0)).astype(np.int32)
        ids = np.concatenate([vis, vis[::2], vis[::-3]]).astype(np.int32)  # repeats after, and in reverse
        want = oracle(ob, tref, ids, vp, cam.position, w, h)
        assert want[2].size > vis.size
        got = api.render_frame(tb, vp, cam.position, api.default_frame_config(w, h), mesh_ids=ids, ctx=fresh)
        assert_same(got, want, f"camera {cam_i}")


def test_duplicate_ids_pipelined(fresh, ob):
    batch, ref, _ = _checker_one(fresh, ob)
    w, h = 256, 128
    vp, eye = _checker_view(w, h)
    cfg = api.default_frame_config(w, h)
    lists = [np.array([0, 0], np.int32), np.array([0, 0, 0], np.int32)]
    wants = [oracle(ob, ref, ids, vp, eye, w, h) for ids in lists]
    bufs = [(fresh.host_array((h, w), np.uint32), fresh.host_array((h, w), np.float32), np.empty(4, np.int32)) for _ in lists]
    vpa, eyea = np.ascontiguousarray(vp, np.float32), np.ascontiguousarray(eye, np.float32)
    for rnd in range(2):
        tickets = []
        for ids, (c, d, _) in zip(lists, bufs):  # both enqueued before either is waited for
            t = C.c_int32(0)
            fresh.check(fresh.lib.vx_render_frame_begin(fresh.handle, batch.handle, ids.ctypes.data, int(ids.size), vpa.ctypes.data,
                                                        eyea.ctypes.data, 0, C.byref(cfg), c.ctypes.data, d.ctypes.data, C.byref(t)))
            tickets.append(t.value)
        for t, (c, d, s), want in zip(tickets, bufs, wants):
            ns = C.c_int32(0)
            fresh.check(fresh.lib.vx_render_frame_end(fresh.handle, t, s.ctypes.data, C.byref(ns)))
            assert_same((c, d, s[:ns.value]), want, f"round {rnd}, ticket {t}")
    _assert_grew_past_the_estimates(counters(fresh), 3, CHECKER_QUADS)
    batch.release()


def test_duplicate_ids_async_stats(fresh, ob):
    """An async frame whose repeated ids overflow the setup units and triangle slots reports VX_ERR_CAPACITY; the stats
    call grows the scratch, so the lane's next async frame (no synchronous frame in between) is exact."""
    import torch
    batch, ref, _ = _checker_one(fresh, ob)
    w, h = 256, 128
    vp, eye = _checker_view(w, h)
    ids = np.array([0, 0], np.int32)
    want = oracle(ob, ref, ids, vp, eye, w, h)
    d_ids = torch.tensor(ids, dtype=torch.int32, device=torch.device("cuda", fresh.device))
    cfga = api.default_frame_config(w, h)
    cfga.async_submit = 1
    vpa, eyea = np.ascontiguousarray(vp, np.float32), np.ascontiguousarray(eye, np.float32)

    def submit():
        torch.cuda.synchronize(fresh.device)
        fresh.check(fresh.lib.vx_render_frame_device(fresh.handle, batch.handle, C.c_void_p(d_ids.data_ptr()), int(ids.size),
                                                     vpa.ctypes.data, eyea.ctypes.data, 0, C.byref(cfga)))

    submit()
    with pytest.raises(api.VxError) as e:
        api.frame_stats(fresh)
    assert e.value.code == -4
    assert int(counters(fresh)[4]) & 0x100  # setup units overflowed (triangle slots, value 1, overflow once there are units for every quad)
    # the first frame set up only the units it had room for, so it undercounts triangles and bin entries
    st, n = _async_until_ok(submit, fresh)
    print("async frames until the lane recovered:", n)
    assert st.n_quads == 2 * CHECKER_QUADS and st.n_survivors == 2
    assert_same(device_frame(fresh, h, w), want, "async frame after the stats call")
    # and a synchronous frame on the grown lane
    assert_same(api.render_frame(batch, vp, eye, api.default_frame_config(w, h), mesh_ids=ids, ctx=fresh), want, "sync")
    batch.release()
