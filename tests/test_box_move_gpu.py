"""Swept-box collision on the device: vx_world_move_boxes against its CPU oracle (tests/move_oracle.c, vxo_move_boxes) bit
for bit through both entry points, before and after block edits; a gravity loop chained on the device through the in-place
arrays; a placed and broken pillar; and the no-new-overlap invariant checked without the oracle."""
import numpy as np
import pytest

import vx_move_oracle
from differential_projection_voxel_renderer_b200 import _lib, api, world as vxw, worldgen
from test_block_edit_gpu import _host_slots, _world
from test_box_move import largest_fitting
from test_world_gpu import WALK

pytestmark = pytest.mark.gpu

F32 = np.float32
PX, NY = 1 << 0, 1 << 3
PLAYER = (0.6, 1.8, 0.6)


def _surface(w):
    """terrain_heights over the loaded world's columns and their origin: heights[z - z0, x - x0]."""
    c = np.array(sorted(w.chunks), dtype=np.int64)
    x0, z0 = int(c[:, 0].min()) * 32, int(c[:, 2].min()) * 32
    nx, nz = (int(c[:, 0].max()) + 1) * 32 - x0, (int(c[:, 2].max()) + 1) * 32 - z0
    return worldgen.terrain_heights(x0, z0, nx, nz), x0, z0


def _random_boxes(rng, w, n):
    """Seeded boxes in the loaded world: half dropped near the terrain surface, half anywhere; a third of the corners on the
    voxel lattice, a third on half-lattice points, a third random; player-sized boxes, boxes up to 2 and up to 16 on a
    side; deltas tiny, up to 1, up to 16 and exactly +-16 on one axis, a fifth of the components zero."""
    c = np.array(sorted(w.chunks), dtype=np.float64)
    p = (c[rng.integers(0, c.shape[0], n)] + rng.random((n, 3))) * 32.0
    heights, x0, z0 = _surface(w)
    near = rng.random(n) < 0.5
    xi, zi = np.floor(p[near, 0]).astype(np.int64) - x0, np.floor(p[near, 2]).astype(np.int64) - z0
    p[near, 1] = heights[zi, xi] + 1.0 + rng.uniform(-3.0, 4.0, int(near.sum()))
    grid = rng.integers(0, 3, n)
    p[grid == 0] = np.floor(p[grid == 0])
    p[grid == 1] = np.floor(p[grid == 1] * 2.0) / 2.0
    kind = rng.integers(0, 3, n)
    size = np.where((kind == 0)[:, None], np.array(PLAYER), np.where((kind == 1)[:, None], 2.0, 16.0) * (1.0 - rng.random((n, 3))))
    size[rng.random((n, 3)) < 0.02] = 16.0
    kind = rng.integers(0, 4, n)
    delta = np.where((kind == 0)[:, None], rng.normal(size=(n, 3)) * 1e-3,
                     np.where((kind == 3)[:, None], rng.uniform(-16.0, 16.0, (n, 3)), rng.uniform(-1.0, 1.0, (n, 3))))
    sixteen = np.flatnonzero(kind == 2)
    delta[sixteen, rng.integers(0, 3, sixteen.size)] = rng.choice([-16.0, 16.0], sixteen.size)
    delta[rng.random((n, 3)) < 0.2] = 0.0
    return p.astype(F32), size.astype(F32), delta.astype(F32)


def _device_move(ctx, w, pos, size, delta, slots):
    """The same boxes through vx_world_move_boxes_device on device arrays."""
    import torch
    dev = torch.device("cuda", ctx.device)
    tp, ts = torch.from_numpy(pos.copy()).to(dev), torch.from_numpy(slots.copy()).to(dev)
    tsz, td = torch.from_numpy(size).to(dev), torch.from_numpy(delta).to(dev)
    tf = torch.zeros(pos.shape[0], dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)
    ctx.check(ctx.lib.vx_world_move_boxes_device(ctx.handle, w.batch.handle, tp.data_ptr(), tsz.data_ptr(), td.data_ptr(), ts.data_ptr(),
                                                 pos.shape[0], tf.data_ptr()))
    ctx.synchronize()
    return tp.cpu().numpy(), ts.cpu().numpy(), tf.cpu().numpy().view(np.uint32)


def _solid_counter(w, host):
    """Counts the voxels of a voxel box that are solid or in a chunk that is not loaded (by position), from a summed-volume
    table over the loaded world plus one chunk all round -- independent of the oracle and of the neighbour hops."""
    pos, vox, flags, _ = host
    c = np.array(sorted(w.chunks), dtype=np.int64)
    lo = c.min(axis=0) - 1
    dims = (c.max(axis=0) + 2 - lo) * 32
    g = np.ones(dims, dtype=np.uint8)
    for p, s in w.chunks.items():
        q = (np.array(p) - lo) * 32
        block = vox[s].reshape(32, 32, 32).transpose(2, 1, 0) != 0 if flags[s] == 0 else np.full((32, 32, 32), flags[s] != 1)
        g[q[0]:q[0] + 32, q[1]:q[1] + 32, q[2]:q[2] + 32] = block
    sat = np.zeros(dims + 1, dtype=np.int32)
    sat[1:, 1:, 1:] = g.cumsum(0, dtype=np.int32).cumsum(1, dtype=np.int32).cumsum(2, dtype=np.int32)
    base = lo * 32

    def count(a, b):  # voxels a .. b inclusive, (n, 3) world coordinates; empty boxes count 0
        a, b1 = a - base, b - base + 1
        assert (a >= 0).all() and (b1 <= dims).all()
        t = 0
        for m in range(8):
            ix = [b1[:, k] if (m >> k) & 1 else a[:, k] for k in range(3)]
            sign = (-1) ** (3 - bin(m).count("1"))
            t = t + sign * sat[ix[0], ix[1], ix[2]].astype(np.int64)
        return np.where((b1 > a).all(axis=1), t, 0)
    return count


def _voxel_range(p, s):
    return np.floor(p).astype(np.int64), np.ceil(p + s).astype(np.int64) - 1  # p + s in f32, as the kernel


def _edit_near(rng, w, pos, n):
    """n seeded edits around the boxes (stone-heavy, some air): voxels within two of a box corner in loaded chunks."""
    v = np.floor(pos[rng.integers(0, pos.shape[0], 4 * n)]).astype(np.int64) + rng.integers(-2, 3, (4 * n, 3))
    v = v[[tuple(c) in w.chunks for c in (v >> 5).tolist()]][:n]
    w.set_blocks(v, rng.choice([0, 1, 3, 3], v.shape[0]))


@pytest.mark.parametrize("vd", [3, 12])
def test_moves_match_the_oracle_bit_for_bit_before_and_after_edits(ctx, ob, vd):
    w = _world(ctx, vd, WALK[0])
    rng = np.random.default_rng(100 + vd)
    pos, size, delta = _random_boxes(rng, w, 200_000)
    pos[-1, 0], size[-2, 1], delta[-3, 2] = np.nan, 0.0, 17.0  # invalid for certain
    slots = w.start_slots(pos)
    for rnd in range(2):
        host = _host_slots(w)
        want_pos, want_slots, want_flags = vx_move_oracle.move_boxes(*host, pos, size, delta, slots)
        got = w.move_boxes(pos, size, delta)
        assert np.array_equal(got["pos"].view(np.uint32), want_pos.view(np.uint32)), \
            f"round {rnd}: {int((got['pos'].view(np.uint32) != want_pos.view(np.uint32)).any(axis=1).sum())} boxes differ"
        assert np.array_equal(got["slot"], want_slots) and np.array_equal(got["flags"], want_flags)
        dp, ds, dfl = _device_move(ctx, w, pos, size, delta, slots)
        assert np.array_equal(dp.view(np.uint32), want_pos.view(np.uint32)) and np.array_equal(ds, want_slots)
        assert np.array_equal(dfl, want_flags)
        bits = [(want_flags >> b & 1).sum() for b in range(8)]
        assert min(bits[:6]) > 100 and bits[3] > 10_000 and bits[6] > 0, bits  # every direction blocked; walls at the edge
        assert 3 <= bits[7] < 20_000, bits
        valid = (want_flags & _lib.MOVE_INVALID) == 0
        assert (want_slots[valid] >= 0).mean() > 0.99
        if vd == 3:  # nothing solid or unloaded is newly overlapped
            count = _solid_counter(w, host)
            a0, b0 = _voxel_range(pos[valid], size[valid])
            a1, b1 = _voxel_range(want_pos[valid], size[valid])
            new = count(a1, b1) - count(np.maximum(a0, a1), np.minimum(b0, b1))
            assert (new == 0).all(), f"{int((new != 0).sum())} boxes moved into solid voxels"
        _edit_near(rng, w, pos, 5000)
    with pytest.raises(api.VxError):  # a slot outside [-1, capacity) at the host entry point
        w.device.move_boxes(pos[:1].copy(), size[:1], delta[:1], np.array([w.capacity], np.int32))
    w.batch.release()


def test_a_gravity_loop_chained_on_the_device_equals_the_oracle_tick_by_tick(ctx, ob):
    """200 ticks of v_y <- max(v_y - 0.08, -3.9), delta = v, v_y <- 0 when the move was blocked vertically; the loop runs
    on the context's stream through the arrays the kernel updates in place, and the history is read back at the end."""
    import torch
    w = _world(ctx, 3, WALK[0])
    rng = np.random.default_rng(5)
    n, ticks = 4096, 200
    pos, size, _ = _random_boxes(rng, w, n)
    pos[0], size[0] = (0.2, 40.0, 20.2), PLAYER  # the player, dropped from above the terrain
    vel = np.zeros((n, 3), F32)
    vel[1:, 0::2] = rng.uniform(-0.3, 0.3, (n - 1, 2))
    slots = w.start_slots(pos)
    g, vmin = F32(0.08), F32(-3.9)
    dev = torch.device("cuda", ctx.device)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    hist_pos = torch.empty((ticks, n, 3), dtype=torch.float32, device=dev)
    hist_slot = torch.empty((ticks, n), dtype=torch.int32, device=dev)
    hist_flags = torch.empty((ticks, n), dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)
    with torch.cuda.stream(stream):
        tp, tsz, ts = (torch.from_numpy(a.copy()).to(dev) for a in (pos, size, slots))
        tv, delta = torch.from_numpy(vel.copy()).to(dev), torch.empty((n, 3), dtype=torch.float32, device=dev)
        tg, tvmin = torch.tensor(g, device=dev), torch.tensor(vmin, device=dev)
        for t in range(ticks):
            tv[:, 1] = torch.maximum(tv[:, 1] - tg, tvmin)
            delta.copy_(tv)
            ctx.check(ctx.lib.vx_world_move_boxes_device(ctx.handle, w.batch.handle, tp.data_ptr(), tsz.data_ptr(), delta.data_ptr(),
                                                         ts.data_ptr(), n, hist_flags[t].data_ptr()))
            tv[:, 1] = torch.where((hist_flags[t] & 12) != 0, torch.zeros_like(tv[:, 1]), tv[:, 1])
            hist_pos[t].copy_(tp)
            hist_slot[t].copy_(ts)
    stream.synchronize()
    got_pos, got_slot, got_flags = hist_pos.cpu().numpy(), hist_slot.cpu().numpy(), hist_flags.cpu().numpy().view(np.uint32)
    host = _host_slots(w)
    for t in range(ticks):
        vel[:, 1] = np.maximum(vel[:, 1] - g, vmin)
        pos, slots, flags = vx_move_oracle.move_boxes(*host, pos, size, vel, slots)
        vel[:, 1] = np.where((flags & 12) != 0, F32(0), vel[:, 1])
        assert np.array_equal(got_pos[t].view(np.uint32), pos.view(np.uint32)), f"tick {t}: positions differ"
        assert np.array_equal(got_slot[t], slots) and np.array_equal(got_flags[t], flags), f"tick {t}"
    # the player came to rest on the terrain: on the ground, at an integer height, unmoved for the last ticks
    h = int(worldgen.terrain_heights(0, 20, 1, 1)[0, 0])
    assert got_flags[-1, 0] & NY and got_pos[-1, 0, 1] == h + 1
    assert (got_pos[-20:, 0] == got_pos[-1, 0]).all()
    assert (got_flags[-1] & NY).sum() > n // 2
    w.batch.release()


def test_a_placed_pillar_stops_a_walk_flush_and_breaking_it_lets_the_walk_go_on(ctx):
    w = _world(ctx, 3, WALK[0])
    # a stone platform at y = 12 with air above it, x 2..15, z 19..22 (chunk (0, 0, 0)), and a pillar at x = 10
    xs, ys, zs = np.meshgrid(np.arange(2, 16), np.arange(12, 18), np.arange(19, 23), indexing="ij")
    xyz = np.stack([xs, ys, zs], axis=-1).reshape(-1, 3)
    w.set_blocks(xyz, np.where(xyz[:, 1] == 12, 3, 0))
    pillar = [(10, 13, 20), (10, 14, 20)]
    w.set_blocks(pillar, 3)
    p = np.array([(4.2, 13.0, 20.2)], F32)
    step = (0.3, -0.1, 0.0)
    stop = largest_fitting(10, F32(0.6))
    for _ in range(30):
        r = w.move_boxes(p, PLAYER, step)
        assert r["on_ground"][0] and r["pos"][0, 1] == 13.0
        p = r["pos"]
    assert p[0, 0].view(np.uint32) == stop.view(np.uint32) and r["flags"][0] == PX | NY  # flush against the pillar
    assert F32(p[0, 0] + F32(0.6)) <= 10 < F32(np.nextafter(p[0, 0], F32(99)) + F32(0.6))
    w.set_blocks(pillar, 0)
    for _ in range(8):
        r = w.move_boxes(p, PLAYER, step)
        assert r["flags"][0] == NY
        p = r["pos"]
    assert p[0, 0] > 11.0
    w.batch.release()
