"""Texturing and shading on the CPU: the oracle's face light, shade and texel sample against a plain float32 restatement;
the properties of the discriminating atlas and of the light set (tests/vx_shading.py); and a sensitivity control that
shows, on oracle frames, that the discriminating atlas exposes simulated kernel mistakes the default atlas hides."""
import ctypes as C

import numpy as np
import pytest

import vx_scenes
import vx_shading as vs

SEEDS = (None, 1, 2)
FACES = range(6)


# ---- plain restatements (float32, left-to-right, as the reference crate evaluates them) ----------------------------------
def face_light_np(light_dir, ambient, diffuse, face):
    """compute_face_lighting rasterizer.rs:1204-1216: clamp(ambient + diffuse * max(n . l, 0), 0, 1) in f32.
    f32::max returns the other operand for NaN; f32::clamp keeps NaN."""
    n = np.zeros(3, dtype=np.float32)
    n[face >> 1] = -1.0 if face & 1 else 1.0
    ld = np.asarray(light_dir, dtype=np.float32)
    with np.errstate(all="ignore"):
        dot = n[0] * ld[0] + n[1] * ld[1]
        dot = dot + n[2] * ld[2]
        lam = dot if dot > 0 else np.float32(0.0)
        light = np.float32(ambient) + np.float32(diffuse) * lam
    if light < 0:
        light = np.float32(0.0)
    if light > 1:
        light = np.float32(1.0)
    return np.float32(light)


def shade_np(base, light):
    """shade_color_u32 shading.rs:90-110: 8.8 fixed-point light (saturating `as u32`), channels clamped to 255, alpha 0xFF."""
    with np.errstate(all="ignore"):
        lf = np.float32(light) * np.float32(256.0)
    if lf != lf or lf <= 0:
        fp = 0
    elif lf >= 4294967296.0:
        fp = 0xFFFFFFFF
    else:
        fp = int(lf)
    ch = [(int(base) >> s) & 0xFF for s in (16, 8, 0)]
    r, g, b = (min(((c * fp) & 0xFFFFFFFF) >> 8, 255) for c in ch)
    return 0xFF000000 | (r << 16) | (g << 8) | b


def sample_np(palette_bytes, index_bytes, tex, u, v):
    """MicroTexture::sample texture.rs:19-38 from the raw atlas bytes."""
    x, y = u & 7, v & 7
    pixel = (y << 3) | x
    byte = index_bytes[tex * 32 + (pixel >> 1)]
    nib = (byte >> 4) & 15 if pixel & 1 == 0 else byte & 15
    return int(np.frombuffer(palette_bytes, dtype=np.uint32)[tex * 16 + nib])


def _ocfg(ob, light):
    return vs.apply_light(ob.default_frame_config(8, 8), light)


def _same_f32(a, b):
    a, b = np.float32(a), np.float32(b)
    return (np.isnan(a) and np.isnan(b)) or a.view(np.uint32) == b.view(np.uint32)


# ---- the oracle's primitives against the restatement --------------------------------------------------------------------
EXTRA_LIGHTS = [0.0, -0.0, 1.0, 0.3, 0.35, 0.999, 1e-8, 0.5 / 256, 1.0 / 256, 2.0, -1.0, 1e12, float("inf"), float("-inf"),
                float("nan")]


@pytest.mark.parametrize("name", list(vs.LIGHTS))
def test_oracle_face_light_matches_restatement(ob, name):
    light = vs.LIGHTS[name]
    cfg = _ocfg(ob, light)
    for face in FACES:
        got = ob.lib().vxo_face_light(C.byref(cfg), C.c_int(face))
        want = face_light_np(light[0], light[1], light[2], face)
        assert _same_f32(got, want), (name, face, got, want)


def test_oracle_shade_matches_restatement(ob):
    rng = np.random.default_rng(7)
    ext = np.array([0, 1, 254, 255], dtype=np.uint32)
    bases = [int((a << 24) | (r << 16) | (g << 8) | b) for a in (0, 0x7F, 0xFF) for r in ext for g in ext for b in ext]
    bases += [int(x) for x in rng.integers(0, 1 << 32, 500, dtype=np.uint64)]
    lights = list(EXTRA_LIGHTS)
    for light in vs.LIGHTS.values():
        lights += [float(face_light_np(light[0], light[1], light[2], f)) for f in FACES]
    lights += [float(x) for x in rng.uniform(0.0, 1.0, 50).astype(np.float32)]
    f = ob.lib().vxo_shade_color_u32
    for light in lights:
        for base in bases:
            assert f(base, light) == shade_np(base, light), (hex(base), light)


@pytest.mark.parametrize("seed", SEEDS + ("random", "default"))
def test_oracle_texture_sample_matches_restatement(ob, seed):
    if seed == "default":
        atlas = ob.default_atlas()
    elif seed == "random":
        raw = np.random.default_rng(11).integers(0, 256, 384, dtype=np.uint8).tobytes()
        atlas = ob.Atlas.from_buffer_copy(raw)
    else:
        atlas = vs.discriminating_atlas(seed)[1]
    pal, ind = bytes(atlas.palette), bytes(atlas.indices)
    f = ob.lib().vxo_texture_sample
    for tex in range(4):
        for u in range(16):      # u, v >= 8 wrap (u & 7)
            for v in range(16):
                assert f(C.byref(atlas), C.c_int(tex), C.c_uint8(u), C.c_uint8(v)) == sample_np(pal, ind, tex, u, v)


# ---- properties of the inputs -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", SEEDS)
def test_discriminating_atlas_properties(seed):
    a, o = vs.discriminating_atlas(seed)
    assert bytes(a) == bytes(o)
    nib = vs.atlas_nibbles(a)[1:]
    # every texel differs from its four neighbours, across the 7 -> 0 wrap too
    for axis in (1, 2):
        for shift in (1, -1):
            assert (nib != np.roll(nib, shift, axis=axis)).all()
    # the two nibbles of every index byte differ (a high / low swap is visible)
    assert (nib[:, :, 0::2] != nib[:, :, 1::2]).all()
    # not symmetric under transposition or mirroring, for every type
    for t in range(3):
        assert not np.array_equal(nib[t], nib[t].T)
        assert not np.array_equal(nib[t], nib[t][:, ::-1])
        assert not np.array_equal(nib[t], nib[t][::-1, :])
    # the index tables of types 1, 2, 3 are pairwise different
    ind = np.frombuffer(bytes(a.indices), dtype=np.uint8).reshape(4, 32)
    for i in range(1, 4):
        for j in range(i + 1, 4):
            assert not np.array_equal(ind[i], ind[j])
    # 48 distinct palette entries, some with alpha != 0xFF, still distinct after shading at any light >= 0.3
    pal = vs.atlas_palette(a)[1:].reshape(-1)
    assert len(set(pal.tolist())) == 48
    assert ((pal >> 24) != 0xFF).sum() >= 16 and ((pal >> 24) == 0xFF).any()
    for fp in range(int(np.float32(0.3) * np.float32(256.0)), 257):
        shaded = {shade_np(int(c), fp / 256.0) for c in pal}
        assert len(shaded) == 48, fp
    # the palette's colours are no clear colour of the default config
    assert 0xFF87CEEB not in pal.tolist()


def test_seeded_atlases_differ():
    atl = [bytes(vs.discriminating_atlas(s)[0]) for s in SEEDS]
    assert len(set(atl)) == len(atl)
    assert bytes(vs.discriminating_atlas(1)[0]) == bytes(vs.discriminating_atlas(1)[1])


def test_light_set_properties(ob):
    lights = {name: [float(ob.lib().vxo_face_light(C.byref(_ocfg(ob, l)), C.c_int(f))) for f in FACES] for name, l in vs.LIGHTS.items()}
    # L and -L: every pair of faces gets a different light in at least one of the two
    for f in FACES:
        for g in range(f + 1, 6):
            assert lights["L"][f] != lights["L"][g] or lights["minus_L"][f] != lights["minus_L"][g], (f, g)
    # the default light does not separate the three negative faces; L / -L do
    d = ob.default_frame_config(8, 8)
    dl = [ob.lib().vxo_face_light(C.byref(d), C.c_int(f)) for f in FACES]
    assert dl[1] == dl[3] == dl[5]
    assert abs(float(np.linalg.norm(np.asarray(vs.L, np.float32))) - 1.0) < 1e-6
    # unnormalised light: +Y is clamped to 1.0, a fixed-point factor of 256 (the palette colour, alpha forced to 0xFF)
    assert lights["unnormalised_clamps_to_1"][2] == 1.0 and shade_np(0x12345678, 1.0) == 0xFF345678
    # negative ambient: some faces clamp to 0 (black), others stay lit
    neg = lights["negative_ambient_clamps_to_0"]
    assert min(neg) == 0.0 and max(neg) > 0.0 and shade_np(0xFFFFFFFF, 0.0) == 0xFF000000
    # no diffuse, ambient exactly 1: every face 1.0
    assert lights["no_diffuse_ambient_1"] == [1.0] * 6
    # +inf component: +X clamps to 1, -X gets the ambient term; 0 * inf is NaN on the faces without an x component, and
    # max(NaN, 0) = 0 leaves them the ambient term too
    inf = lights["inf_light"]
    assert inf[0] == 1.0 and inf[1:] == [np.float32(0.3)] * 5
    # NaN ambient: NaN light on every face, which shades to black
    assert all(np.isnan(x) for x in lights["nan_ambient"]) and shade_np(0xFFFFFFFF, float("nan")) == 0xFF000000
    assert vs.LIGHTS["shading_off"][3] == 0 and all(l[3] == 1 for n, l in vs.LIGHTS.items() if n != "shading_off")


def test_clear_colours():
    pal = vs.atlas_palette(vs.discriminating_atlas()[0])[1:].reshape(-1).tolist()
    assert vs.CLEARS[:3] == [0x00000000, 0xFFFFFFFF, 0x00FF00FF]
    assert vs.CLEARS[3] in pal and vs.CLEARS[3] >> 24 == 0xFF


def test_cache_sequence_changes_one_input_at_a_time():
    seq = vs.cache_sequence()
    bits = lambda xs: [np.float32(x).tobytes() for x in xs]
    for i, ((a, l, c), (b, m, d)) in enumerate(zip(seq, seq[1:])):
        changed = [not np.array_equal(vs.atlas_palette(a[0]), vs.atlas_palette(b[0])),
                   not np.array_equal(vs.atlas_nibbles(a[0]), vs.atlas_nibbles(b[0])), c != d]
        changed += [x != y for x, y in zip(bits(l[0]) + bits(l[1:3]) + [l[3]], bits(m[0]) + bits(m[1:3]) + [m[3]])]
        if i < len(seq) - 2:
            assert sum(changed) == 1, (i, changed)
    assert seq[-1] == seq[0] and len(seq) >= 13


def test_apply_light_writes_both_config_structs(ob):
    from differential_projection_voxel_renderer_b200 import _lib
    for light in vs.LIGHTS.values():
        o = vs.apply_light(ob.default_frame_config(4, 4), light)
        a = vs.apply_light(_lib.VxFrameConfig(), light)
        for c in (o, a):
            assert all(_same_f32(c.light_dir[i], light[0][i]) for i in range(3))
            assert _same_f32(c.ambient, light[1]) and _same_f32(c.diffuse, light[2]) and c.enable_shading == light[3]


# ---- sensitivity control: simulated kernel mistakes change oracle frames --------------------------------------------------
def _mistakes(palette, nib):
    """name -> (palette, nibbles) of the atlas a kernel with that mistake would effectively draw with."""
    out = {}
    for a, b in ((1, 2), (2, 3)):  # reads another block type's index table
        n = nib.copy()
        n[[a, b]] = n[[b, a]]
        out[f"type_table_{a}_{b}"] = (palette, n)
    for k in (1, 2, 4, 8):  # wrong nibble bits
        p = palette.copy()
        p[1:] = palette[1:, np.arange(16) ^ k]
        out[f"palette_xor_{k}"] = (p, nib)
    out["nibble_swap"] = (palette, nib[:, :, np.arange(8) ^ 1])
    out["transpose"] = (palette, nib.transpose(0, 2, 1).copy())
    out["shift_u"] = (palette, np.roll(nib, -1, axis=2))
    out["shift_v"] = (palette, np.roll(nib, -1, axis=1))
    return out


@pytest.fixture(scope="module")
def frames(ob):
    """320 x 180 oracle renderers, atlas -> frame: the seeded terrain (scene 5, camera 0) and the terraces (view 0).  The
    terrain shows only grass there, so the mistakes that involve dirt and stone alone are measured on the terraces."""
    pos, world, p, v, nb = vx_scenes.terrain_scene(5)
    ref = ob.mesh_chunks(v, nb, None, p)
    w, h = 320, 180
    cam = vx_scenes.path_camera(0, w, h)
    vp = cam.view_projection()
    ids = np.flatnonzero((ob.cull_chunks(p, vp, cam.position, 5) != 0) & (ref.has_mesh != 0)).astype(np.int32)
    tvox, tpos = vs.terraces()
    tref = ob.mesh_chunks(tvox, None, None, tpos)
    tvp, teye = vs.terraces_view(w, h)
    tids = np.arange(len(tpos), dtype=np.int32)
    cfg = ob.default_frame_config(w, h, n_threads=4)
    return {"terrain": lambda atlas: ob.render_frame(ref, ids, vp, cam.position, cfg, atlas),
            "terraces": lambda atlas: ob.render_frame(tref, tids, tvp, teye, cfg, atlas)}


def sensitivity(render, atlas_pair):
    """Fraction of covered pixels each simulated mistake changes."""
    base_c, base_d, _ = render(atlas_pair[1])
    covered = np.isfinite(base_d)
    assert covered.sum() > 10000
    pal, nib = vs.atlas_palette(atlas_pair[1]), vs.atlas_nibbles(atlas_pair[1])
    out = {}
    for name, (p, n) in _mistakes(pal, nib).items():
        c, d, _ = render(vs.make_atlas(p, n)[1])
        assert np.array_equal(d.view(np.uint32), base_d.view(np.uint32))  # texturing never changes depth
        out[name] = float((c != base_c)[covered].mean())
    return out


GRASS_FREE = {"type_table_2_3"}  # mistakes that change no grass pixel


@pytest.mark.parametrize("scene", ["terrain", "terraces"])
def test_sensitivity_control_on_the_oracle(frames, scene):
    frac = sensitivity(frames[scene], vs.discriminating_atlas())
    print(scene, "changed fraction of covered pixels per mistake:", {k: round(v, 3) for k, v in frac.items()})
    weak = {k: v for k, v in frac.items() if v < 0.01 and not (scene == "terrain" and k in GRASS_FREE)}
    assert not weak, f"mistakes the discriminating atlas does not expose: {weak}"
    # the default atlas is blind to a wrong block type's index table and to wrong nibble bits 1-3
    frac_default = sensitivity(frames[scene], vs.default_atlas_pair())
    print(scene, "same with the default atlas:", {k: round(v, 3) for k, v in frac_default.items()})
    for name in ("type_table_1_2", "type_table_2_3", "palette_xor_2", "palette_xor_4", "palette_xor_8"):
        assert frac_default[name] == 0.0, (name, frac_default[name])
