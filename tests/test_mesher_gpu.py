"""Parity of the CUDA mesher with the CPU oracle: quad lists bit-exact per chunk (through the C ABI)."""
import numpy as np
import pytest

import vx_kat as kat
import vx_scenes

from differential_projection_voxel_renderer_b200 import api, worldgen

pytestmark = pytest.mark.gpu


def assert_batches_equal(got: dict, batch, ref):
    n = ref.n_chunks
    assert got["quad_count"].tolist() == ref.quad_count.tolist()
    assert got["has_mesh"].tolist() == ref.has_mesh.tolist()
    assert np.array_equal(got["slice_offsets"], ref.slice_offsets)
    assert np.array_equal(got["face_aabb"], ref.face_aabb)
    for i in range(n):  # chunk ranges are allocated in completion order on the GPU: compare per chunk
        assert np.array_equal(batch.chunk_quads(i).reshape(-1), ref.chunk_quads(i).reshape(-1)), f"chunk {i}"
    assert got["quads"].shape[0] == ref.quads.size // 3


def run_both(ctx, ob, vox, nb=None, uf=None, pos=None):
    vox = np.ascontiguousarray(vox, dtype=np.uint8).reshape(-1, 32768)
    batch = api.BinaryGreedyMesher.mesh_batch(vox, pos, nb, uf, ctx)
    got = batch.download()
    ref = ob.mesh_chunks(vox, nb, uf, pos)
    assert_batches_equal(got, batch, ref)
    batch.release()
    return ref


def test_greedy_slice_kats(ctx, ob):
    masks = kat.slice_masks()
    m1 = np.zeros(32, np.uint32); m1[0] = 1
    m2 = np.zeros(32, np.uint32); m2[0] = 0b1111
    m3 = np.zeros(32, np.uint32); m3[:3] = 0b1111
    all_masks = [m1, m2, m3] + list(masks.values())
    rng = np.random.default_rng(11)
    for dens in (1, 2, 3):
        for _ in range(40):
            m = rng.integers(0, 2 ** 32, size=32, dtype=np.uint64).astype(np.uint32)
            for _ in range(dens - 1):
                m &= rng.integers(0, 2 ** 32, size=32, dtype=np.uint64).astype(np.uint32)
            all_masks.append(m)
    got = api.BinaryGreedyMesher.greedy_mesh_slices(np.stack(all_masks), ctx)
    for m, g in zip(all_masks, got):
        assert np.array_equal(g, ob.greedy_mesh_slice(m))
    assert got[0].tolist() == [[0, 0, 1, 1]] and got[2].tolist() == [[0, 0, 3, 4]]  # binary_greedy.rs:822-855
    assert api.BinaryGreedyMesher.greedy_mesh_slice(np.zeros(32, np.uint32), ctx).shape[0] == 0


def test_chunk_kats(ctx, ob):
    chunks = [kat.chunk_single_voxel(), kat.chunk_single_voxel(0, 0, 0), kat.chunk_single_voxel(31, 31, 31),
              kat.chunk_two_adjacent(), kat.chunk_2x2_plane(), kat.chunk_two_types(), kat.chunk_dense_solid(),
              kat.chunk_slab(), np.zeros(32768, np.uint8)]
    ref = run_both(ctx, ob, np.stack(chunks))
    assert ref.quad_count[:7].tolist() == [6, 6, 6, 6, 6, 10, 6]
    assert ref.has_mesh[8] == 0  # all-air Varied chunk -> None (binary_greedy.rs:116-120)


def test_mesh_chunk_api_matches_reference_kats(ctx):
    m = api.BinaryGreedyMesher.mesh_chunk(kat.chunk_single_voxel(), ctx=ctx)  # tests/meshing_tests.rs:55
    assert m.quad_count() == 6
    for f in range(6):
        q = api.unpack_quads(m.quads[int(m.slice_offsets[f, 0]):int(m.slice_offsets[f, 32])])
        assert q.tolist() == [[16, 16, 1, 1, kat.STONE]]
    assert api.BinaryGreedyMesher.mesh_chunk(np.zeros(32768, np.uint8), ctx=ctx) is None


def test_uniform_flags_and_neighbour_codes(ctx, ob):
    a = kat.empty_chunk(); kat.set_block(a, 31, 5, 5, kat.STONE); kat.set_block(a, 5, 31, 5, kat.GRASS)
    b = kat.empty_chunk(); kat.set_block(b, 0, 5, 5, kat.STONE)
    vox = np.stack([a.reshape(-1), b.reshape(-1), np.full(32768, 3, np.uint8), np.zeros(32768, np.uint8)])
    uf = np.array([0, 0, 1 + 3, 1 + 0], dtype=np.uint8)  # chunk 2 Uniform(Stone), chunk 3 Uniform(Air)
    nb = np.full((4, 6), -1, dtype=np.int32)
    nb[0, 0] = 1; nb[1, 1] = 0
    nb[0, 2] = 2      # +Y neighbour is the Uniform(Stone) chunk (by index)
    nb[0, 4] = 3      # +Z neighbour is Uniform(Air)
    nb[1, 0] = -3     # code: uniform solid
    nb[1, 2] = -2     # code: uniform air
    ref = run_both(ctx, ob, vox, nb, uf)
    assert ref.has_mesh.tolist() == [1, 1, 0, 0]


def test_terrain_world_with_neighbours(ctx, ob):
    _, world, p, v, nb = vx_scenes.terrain_scene(5)
    ref = run_both(ctx, ob, v, nb, None, p)
    assert ref.has_mesh.sum() > 50
    # same world through the uniform-flag path (indices into the full chunk list)
    ref2 = run_both(ctx, ob, world.voxels, world.neighbor_table(), world.uniform_flags, world.positions)
    varied = np.flatnonzero(world.uniform_flags == 0)
    assert ref2.quad_count[varied].tolist() == ref.quad_count.tolist()


def test_random_chunks_and_regrow(ctx, ob):
    rng = np.random.default_rng(5)
    chunks = [worldgen.random_chunk(rng, d, t) for d, t in ((0.5, 3), (0.05, 3), (0.95, 2), (0.3, 1))]
    chunks.append(kat.chunk_checker3d())  # 98,304 quads: forces the quad-stream regrow path
    vox = np.stack(chunks)
    nb = np.full((5, 6), -1, dtype=np.int32)
    nb[0] = [1, 2, 3, 1, 2, 3]  # arbitrary Varied neighbours on all six sides
    nb[4] = [0, 0, 0, 0, 0, 0]
    ref = run_both(ctx, ob, vox, nb)
    assert ref.quad_count[4] > 49152


def test_shared_memory_pool_boundaries(ctx, ob):
    """The mesher keeps a chunk's quads in a 2112-entry shared-memory pool (128 per (face, slice) unit while staging)
    and falls back to a second emitting pass beyond that: exactly full, one past full, one unit of 128 / 129 / 512
    quads."""
    def isolated(cells):
        c = kat.empty_chunk().reshape(32, 32, 32)  # [z][y][x]
        for (x, y, z) in cells:
            c[z, y, x] = 1 + (x + y + z) % 3
        return c.reshape(-1)
    grid = [(2 * i, 2 * j, 2 * k) for i in range(8) for j in range(11) for k in range(4)]
    assert len(grid) == 352
    exactly_full = isolated(grid)                    # 352 voxels x 6 faces = 2112 quads, <= 88 per unit
    one_more = isolated(grid + [(16, 0, 8)])          # 2118 quads: second pass
    row128 = isolated([(2 * i, 0, 2 * k) for i in range(16) for k in range(8)])    # +-Y units of slice 0: 128 quads each
    row129 = isolated([(2 * i, 0, 2 * k) for i in range(16) for k in range(8)] + [(1, 0, 17)])
    plane512 = isolated([(x, 0, z) for x in range(32) for z in range(32) if (x + z) % 2 == 0])  # 512 per +-Y unit
    vox = np.stack([exactly_full, one_more, row128, row129, plane512])
    ref = run_both(ctx, ob, vox, None)
    assert ref.quad_count.tolist()[:2] == [2112, 2118]


def test_full_size_properties(ctx, ob):
    """BASELINE size (cfg 3: every Varied chunk of the vd-12 world): size-independent checks on the whole batch
    + bit-exact comparison of a sample of chunks (the oracle meshes ~1.3k chunks/s)."""
    _, world, p, v, nb = vx_scenes.terrain_scene(12)
    batch = api.BinaryGreedyMesher.mesh_batch(v, p, nb, None, ctx)
    got = batch.download()
    n = p.shape[0]
    assert got["quad_count"].sum() == got["quads"].shape[0]
    # chunk ranges tile the quad stream exactly
    order = np.argsort(got["quad_base"], kind="stable")
    nz = order[got["quad_count"][order] > 0]
    ends = got["quad_base"][nz] + got["quad_count"][nz]
    assert got["quad_base"][nz][0] == 0 and np.array_equal(ends[:-1], got["quad_base"][nz][1:])
    # slice offsets monotone and closed by the count
    so = got["slice_offsets"].reshape(n, 198).astype(np.int64)
    lists = so.reshape(n, 6, 33)
    assert (np.diff(lists, axis=2) >= 0).all()
    assert np.array_equal(lists[:, 5, 32], got["quad_count"].astype(np.int64))
    assert np.array_equal(lists[:, 1:, 0], lists[:, :-1, 32])
    # every quad's area sums to the number of exposed voxel faces (counted with numpy on the voxel grid)
    sample = np.random.default_rng(1).choice(n, size=24, replace=False)
    for i in sample.tolist():
        uq = api.unpack_quads(batch.chunk_quads(i))
        area = int((uq[:, 2] * uq[:, 3]).sum())
        vol = v[i].reshape(32, 32, 32) != 0  # [z,y,x]
        exposed = 0
        for axis, (fp, fn) in zip((2, 1, 0), ((0, 1), (2, 3), (4, 5))):  # array axis for x, y, z
            for f, sign in ((fp, 1), (fn, -1)):
                shifted = np.zeros_like(vol)
                src = [slice(None)] * 3; dst = [slice(None)] * 3
                if sign == 1: src[axis] = slice(1, None); dst[axis] = slice(0, -1)
                else: src[axis] = slice(0, -1); dst[axis] = slice(1, None)
                shifted[tuple(dst)] = vol[tuple(src)]
                j = nb[i, f]
                if j >= 0:  # border plane from the neighbour chunk
                    nvol = v[j].reshape(32, 32, 32) != 0
                    edge = [slice(None)] * 3; nedge = [slice(None)] * 3
                    edge[axis] = -1 if sign == 1 else 0
                    nedge[axis] = 0 if sign == 1 else -1
                    shifted[tuple(edge)] = nvol[tuple(nedge)]
                elif j == -3:
                    edge = [slice(None)] * 3; edge[axis] = -1 if sign == 1 else 0
                    shifted[tuple(edge)] = True
                exposed += int((vol & ~shifted).sum())
        assert area == exposed, f"chunk {i}"
    # the vd-12 world is small enough for the oracle (~1.3k chunks/s): compare every chunk bit for bit
    full = ob.mesh_chunks(v, nb, None, p)
    for i in range(n):
        assert np.array_equal(batch.chunk_quads(i).reshape(-1), full.chunk_quads(i).reshape(-1)), f"chunk {i}"
    batch.release()


def test_remesh_into_existing_batch_is_idempotent(ctx):
    import ctypes as C
    _, world, p, v, nb = vx_scenes.terrain_scene(4)
    b1 = api.BinaryGreedyMesher.mesh_batch(v, p, nb, None, ctx)
    first = {k: a.copy() for k, a in b1.download().items()}
    # remesh in place from host-uploaded copies held by a second batch's staging: use the device entry point
    import torch
    dv = torch.from_numpy(v).cuda(); dn = torch.from_numpy(nb).cuda()
    ctx.check(ctx.lib.vx_remesh_chunks_device(ctx.handle, C.c_void_p(dv.data_ptr()), C.c_void_p(dn.data_ptr()), None, b1.handle))
    b1._host = None
    second = b1.download()
    assert first["quad_count"].tolist() == second["quad_count"].tolist()
    for i in range(p.shape[0]):
        fb, fc = int(first["quad_base"][i]), int(first["quad_count"][i])
        assert np.array_equal(first["quads"][fb:fb + fc], b1.chunk_quads(i))
    b1.release()


def test_invalid_arguments_fail_loudly(ctx):
    with pytest.raises(api.VxError):
        api.BinaryGreedyMesher.mesh_batch(np.full((1, 32768), 7, np.uint8), ctx=ctx)
    import ctypes as C
    h = C.c_void_p()
    assert ctx.lib.vx_mesh_chunks(ctx.handle, None, None, None, None, 3, C.byref(h)) == -1


def test_chunk_subset_meshing_matches_the_full_batch(ctx, ob):
    """vx_mesh_chunk_subset_device (one rank of a chunk-sharded remesh): the shard's meshes equal the same chunks of
    the full batch, with neighbour halos taken from chunks that are NOT in the shard."""
    import torch
    import vx_scenes
    from differential_projection_voxel_renderer_b200 import sharding
    pos, world, p, v, nb = vx_scenes.terrain_scene(4)
    n = p.shape[0]
    ref = ob.mesh_chunks(v, nb, None, p)
    dev = torch.device("cuda", 0)
    dv, dn, dp = torch.from_numpy(v).to(dev), torch.from_numpy(nb).to(dev), torch.from_numpy(p).to(dev)
    shards = []
    for world_size in (3,):
        for r in range(world_size):
            ids = sharding.chunk_shard(n, r, world_size)
            dids = torch.from_numpy(ids).to(dev)
            b = api.BinaryGreedyMesher.mesh_batch_subset(dv.data_ptr(), dp.data_ptr(), dn.data_ptr(), 0, n, dids.data_ptr(), ids.size, ctx)
            got = b.download()
            for j, cid in enumerate(ids.tolist()):
                assert np.array_equal(b.chunk_quads(j).reshape(-1), ref.chunk_quads(cid).reshape(-1)), (r, cid)
            assert np.array_equal(got["slice_offsets"], ref.slice_offsets[ids])
            assert np.array_equal(got["face_aabb"], ref.face_aabb[ids])
            # steady-state re-mesh into the same batch gives the same result
            api.BinaryGreedyMesher.mesh_batch_subset(dv.data_ptr(), dp.data_ptr(), dn.data_ptr(), 0, n, dids.data_ptr(), ids.size, ctx, batch=b)
            again = b.download()
            assert np.array_equal(again["quad_count"], got["quad_count"])
            for j, cid in enumerate(ids.tolist()):
                assert np.array_equal(b.chunk_quads(j).reshape(-1), ref.chunk_quads(cid).reshape(-1)), ("remesh", r, cid)
            shards.append(got)
            b.release()
        merged = sharding.merge_mesh_shards(shards, n, world_size)
        assert np.array_equal(merged["quads"].reshape(-1), ref.quads.reshape(-1)[:merged["quads"].size])
        assert np.array_equal(merged["quad_base"], ref.quad_base) and np.array_equal(merged["has_mesh"], ref.has_mesh)


def test_incremental_update_matches_a_full_remesh(ctx, ob):
    """vx_mesh_batch_update (edit -> re-mesh the chunk and its six neighbours, main.rs:225-280): after every round of
    edits each chunk's mesh equals the oracle's mesh of the edited world, including the rounds where the quad stream
    runs out of room and its live quads are compacted."""
    import vx_scenes
    pos, world, p, v, nb = vx_scenes.terrain_scene(3)
    v = v.copy()
    n = p.shape[0]
    batch = api.BinaryGreedyMesher.mesh_batch(v, p, nb, None, ctx)
    rng = np.random.default_rng(11)
    fell_back = False
    for rnd in range(12):
        k = int(rng.integers(1, 9))
        ids = rng.choice(n, size=k, replace=False).astype(np.int32)
        for cid in ids.tolist():
            vol = v[cid].reshape(32, 32, 32)  # [z][y][x]
            mode = rnd % 4
            if mode == 0:    # dig a shaft down to y = 0 at a border column (changes the neighbour's border faces)
                vol[0:3, :, 29:32] = 0
            elif mode == 1:  # stone pillar on the +X border
                vol[10:14, :, 31] = 3
            elif mode == 2:  # noisy block of mixed types: many small quads
                vol[4:20, 8:24, 4:20] = rng.integers(0, 4, size=(16, 16, 16), dtype=np.uint8)
            else:            # clear the whole chunk (mesh disappears)
                vol[...] = 0
        before = batch.info().total_quads
        nre = batch.update(ids, v[ids])
        assert ids.size <= nre <= 7 * ids.size
        info = batch.info()
        if info.total_quads < before:
            fell_back = True  # the stream was compacted
        ref = ob.mesh_chunks(v, nb, None, p)
        got = batch.download()
        assert np.array_equal(got["quad_count"], ref.quad_count), rnd
        assert np.array_equal(got["has_mesh"], ref.has_mesh) and info.n_meshes == int(ref.has_mesh.sum())
        assert np.array_equal(got["slice_offsets"], ref.slice_offsets) and np.array_equal(got["face_aabb"], ref.face_aabb)
        for i in range(n):
            assert np.array_equal(batch.chunk_quads(i).reshape(-1), ref.chunk_quads(i).reshape(-1)), (rnd, i)
    # the updated cache renders like a freshly meshed world
    cam = vx_scenes.path_camera(1, 320, 180)
    vp = cam.view_projection()
    cfg = api.default_frame_config(320, 180)
    c1, d1, s1 = api.render_frame(batch, vp, cam.position, cfg, view_distance=3, ctx=ctx)
    fresh = api.BinaryGreedyMesher.mesh_batch(v, p, nb, None, ctx)
    c2, d2, s2 = api.render_frame(fresh, vp, cam.position, cfg, view_distance=3, ctx=ctx)
    assert np.array_equal(c1, c2) and np.array_equal(d1.view(np.uint32), d2.view(np.uint32)) and np.array_equal(s1, s2)
    print("compacted the quad stream at least once:", fell_back)
    fresh.release()
    batch.release()
    # a batch that does not own its world refuses the update
    import torch
    dv = torch.from_numpy(v).cuda()
    import ctypes as C
    h = C.c_void_p()
    ctx.check(ctx.lib.vx_mesh_chunks_device(ctx.handle, C.c_void_p(dv.data_ptr()), None, None, None, n, C.byref(h)))
    b2 = api.MeshBatch(ctx, h)
    with pytest.raises(api.VxError):
        b2.update(np.array([0], np.int32), v[:1])
    b2.release()


def test_update_leaves_chunks_outside_its_list_untouched(ctx, ob):
    """vx_mesh_batch_update re-meshes only the edited chunks and the neighbours listed for them, also when the quad stream
    is full.  C lists E as its +X neighbour, E lists no neighbours: an edit of E's x = 0 plane changes the faces C would
    get, but C is not in the list, so its mesh stays bit-identical (stale, like the reference's mesh cache)."""
    C, E = 0, 1
    c = kat.empty_chunk().reshape(32, 32, 32)  # [z][y][x]
    c[4:20, 2:30, 31] = kat.STONE              # a wall on C's +X border
    e = kat.empty_chunk().reshape(32, 32, 32)
    e[10:12, 10:12, 10:12] = kat.DIRT
    vox = np.stack([c.reshape(-1), e.reshape(-1), kat.chunk_single_voxel()])  # the third chunk is filler
    nb = np.full((3, 6), -1, dtype=np.int32)
    nb[C, 0] = E
    batch = api.BinaryGreedyMesher.mesh_batch(vox, None, nb, None, ctx)
    before = batch.download()
    c_quads = batch.chunk_quads(C).copy()
    new_e = e.copy()
    new_e[:, :, 0] = kat.GRASS                 # E's x = 0 plane now hides C's wall
    vox[E] = new_e.reshape(-1)
    assert batch.update(np.array([E], np.int32), vox[E:E + 1]) == 1
    ref = ob.mesh_chunks(vox, nb, None, None)
    assert not np.array_equal(ref.chunk_quads(C).reshape(-1), c_quads.reshape(-1))  # a re-mesh of C would change it
    got = batch.download()
    assert np.array_equal(batch.chunk_quads(C), c_quads)
    for k in ("quad_count", "slice_offsets", "face_aabb", "has_mesh"):
        assert np.array_equal(got[k][C], before[k][C]), k
    assert np.array_equal(batch.chunk_quads(E).reshape(-1), ref.chunk_quads(E).reshape(-1))
    assert got["quad_count"][E] == ref.quad_count[E] and got["has_mesh"][E] == ref.has_mesh[E]
    assert np.array_equal(got["slice_offsets"][E], ref.slice_offsets[E]) and np.array_equal(got["face_aabb"][E], ref.face_aabb[E])
    batch.release()


def test_device_terrain_generation_matches_the_oracle(ctx, ob):
    """vx_generate_terrain (SURVEY 8f N1): voxels and Uniform flags equal the ORACLE's Chunk::generate_terrain (chunk.rs:114-207
    over the restated noise 0.9.0 Perlin, oracle/vx_oracle.c) chunk by chunk, bit for bit; the device-generated world meshes
    to the same quads without ever being uploaded."""
    import ctypes as C
    import torch
    pos = worldgen.lattice_sphere((1, 0, -2), 6)
    dev = torch.device("cuda", 0)
    d_vox = torch.empty((pos.shape[0], 32768), dtype=torch.uint8, device=dev)
    flags = api.generate_terrain(pos, d_vox.data_ptr(), ctx)
    got = d_vox.cpu().numpy()
    assert (flags == 0).sum() > 50 and (flags == 1).sum() > 50 and (flags == 4).sum() > 50
    for i, p in enumerate(pos.tolist()):
        oflag, ovox = ob.generate_terrain(p)
        assert int(flags[i]) == oflag, p
        if oflag == 0:
            assert np.array_equal(got[i], ovox), p
    world = worldgen.generate_world(pos)  # the host generator (pinned to the oracle by tests/test_oracle_kat.py) for the neighbour table
    assert np.array_equal(flags, world.uniform_flags) and np.array_equal(got, world.voxels)
    # far from the origin (large coordinates, negative cells) and another seed
    far = np.array([[4000, 0, -3999], [-1234, -1, 777], [-1, 0, -1], [255, 0, 256], [-70000, 0, 65536]], dtype=np.int32)
    d2 = torch.empty((far.shape[0], 32768), dtype=torch.uint8, device=dev)
    f2 = api.generate_terrain(far, d2.data_ptr(), ctx, api.terrain_params(777))
    g2 = d2.cpu().numpy()
    for i, p in enumerate(far.tolist()):
        oflag, ovox = ob.generate_terrain(p, seed=777)
        assert int(f2[i]) == oflag and (oflag != 0 or np.array_equal(g2[i], ovox)), p
    # mesh straight from the device-resident world
    nb = world.neighbor_table()
    d_nb = torch.from_numpy(nb).to(dev)
    d_fl = torch.from_numpy(flags).to(dev)
    d_pos = torch.from_numpy(pos).to(dev)
    h = C.c_void_p()
    ctx.check(ctx.lib.vx_mesh_chunks_device(ctx.handle, C.c_void_p(d_vox.data_ptr()), C.c_void_p(d_pos.data_ptr()), C.c_void_p(d_nb.data_ptr()),
                                            C.c_void_p(d_fl.data_ptr()), pos.shape[0], C.byref(h)))
    batch = api.MeshBatch(ctx, h)
    ref = ob.mesh_chunks(world.voxels, nb, world.uniform_flags, pos)
    g = batch.download()
    assert np.array_equal(g["quad_count"], ref.quad_count) and np.array_equal(g["has_mesh"], ref.has_mesh)
    for i in np.flatnonzero(ref.has_mesh).tolist():
        assert np.array_equal(batch.chunk_quads(i).reshape(-1), ref.chunk_quads(i).reshape(-1))
    batch.release()
