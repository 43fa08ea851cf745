"""Atlases, shading configs and clear colours that tell texturing and shading mistakes apart.

The default atlas hides most of them: its noise palettes hold two colours chosen by nibble % 2 and block types 1-3 share
one index table, and the default light gives the three negative faces the same light.  `discriminating_atlas` is built
so that a wrong texel, nibble, block type or palette entry always changes the colour; `LIGHTS` gives every face pair a
different light in at least one config and reaches every clamp of the face lighting.  Both product (api) and oracle
structs are produced from the same bytes.
"""
import numpy as np

from differential_projection_voxel_renderer_b200 import api

TYPES = (1, 2, 3)  # the block types that are drawn (0 is air)


def atlas_nibbles(atlas) -> np.ndarray:
    """(4, 8, 8) u8 texel nibbles [type, v, u] of an atlas struct (either kind): texel (u, v) is pixel v * 8 + u, the high
    nibble of index byte pixel / 2 for even u, the low one for odd u (MicroTexture::sample texture.rs:19-38)."""
    ind = np.frombuffer(bytes(atlas.indices), dtype=np.uint8).reshape(4, 8, 4)
    out = np.empty((4, 8, 8), dtype=np.uint8)
    out[:, :, 0::2] = ind >> 4
    out[:, :, 1::2] = ind & 15
    return out


def atlas_palette(atlas) -> np.ndarray:
    return np.frombuffer(bytes(atlas.palette), dtype=np.uint32).reshape(4, 16).copy()


def make_atlas(palette, nibbles):
    """(api.VxAtlas, ob.Atlas) with the same bytes, from a (4, 16) u32 palette and (4, 8, 8) [type, v, u] nibbles."""
    from oracle import binding as ob
    nib = np.asarray(nibbles, dtype=np.uint8).reshape(4, 8, 8)
    assert int(nib.max()) < 16
    ind = ((nib[:, :, 0::2] << 4) | nib[:, :, 1::2]).astype(np.uint8)
    raw = np.ascontiguousarray(palette, dtype=np.uint32).reshape(4, 16).tobytes() + ind.tobytes()
    return api.VxAtlas.from_buffer_copy(raw), ob.Atlas.from_buffer_copy(raw)


def _palette(rng) -> np.ndarray:
    """48 entries for types 1-3 whose red channels are 8 + 5 k for k = 0..47 in shuffled order: at any light >= 0.3
    (a fixed-point factor >= 76 / 256) channels 5 apart stay apart after shading.  Alpha bytes cycle through
    0x00, 0x40, 0x80, 0xC0, 0xFF, so shading (which writes 0xFF) and the unshaded path (which keeps them) differ."""
    red = 8 + 5 * rng.permutation(48)
    green = rng.integers(0, 256, 48)
    blue = rng.integers(0, 256, 48)
    alpha = np.array([0x00, 0x40, 0x80, 0xC0, 0xFF])[np.arange(48) % 5]
    pal = np.zeros((4, 16), dtype=np.uint32)
    pal[0] = 0xFF00FF00 | np.arange(16, dtype=np.uint32)  # type 0 is never drawn
    pal[1:] = ((alpha << 24) | (red << 16) | (green << 8) | blue).astype(np.uint32).reshape(3, 16)
    return pal


def discriminating_atlas(seed=None):
    """nibble(t, u, v) = (u + 3 v + 5 t) mod 16, passed through a seeded permutation of 0..15 when a seed is given:
    u-neighbours differ by 1 (7 across the wrap), v-neighbours by 3 (5 across the wrap), so both nibbles of every index
    byte and the four neighbours of every texel differ; the pattern is not symmetric under transposition or mirroring;
    the tables of types 1, 2 and 3 are offset by 5 from each other.  Returns (api.VxAtlas, ob.Atlas)."""
    rng = np.random.default_rng(20261020 if seed is None else seed)
    t = np.arange(4)[:, None, None]
    v = np.arange(8)[None, :, None]
    u = np.arange(8)[None, None, :]
    nib = (u + 3 * v + 5 * t) % 16
    if seed is not None:
        nib = rng.permutation(16)[nib]
    return make_atlas(_palette(rng), nib)


def default_atlas_pair():
    """TextureAtlas::default as (api.VxAtlas, ob.Atlas), built by the oracle (no device library needed)."""
    from oracle import binding as ob
    o = ob.default_atlas()
    return api.VxAtlas.from_buffer_copy(bytes(o)), o


def terraces():
    """2 x 2 chunks of 4 x 4-block columns, 4..19 blocks tall, block types 1, 2, 3 mixed column by column.  The seeded
    terrain is grass wherever a camera of the path looks (dirt and stone show on a fraction of a percent of its pixels),
    so this scene is what puts every block type, and all six faces, on many pixels.  Returns (voxels (4, 32768),
    positions (4, 3)); borders between the chunks are meshed as air."""
    pos = np.array([(cx, 0, cz) for cz in range(2) for cx in range(2)], dtype=np.int32)
    z, y, x = np.meshgrid(np.arange(32), np.arange(32), np.arange(32), indexing="ij")
    vox = []
    for cx, _, cz in pos:
        bx, bz = (cx * 32 + x) // 4, (cz * 32 + z) // 4
        height = 4 + 3 * ((bx * 5 + bz * 3) % 6)
        vox.append(np.where(y < height, 1 + (bx + 2 * bz) % 3, 0).astype(np.uint8).reshape(-1))
    return np.stack(vox), pos


def terraces_view(w, h, k=0):
    """(view-projection, eye) of three views over the terraces: k = 0 from the +x +z corner, 1 from the -x -z corner
    (the other three faces), 2 low and close (large texels, steep perspective)."""
    from differential_projection_voxel_renderer_b200 import camera
    eye, center = [((66.0, 30.0, 70.0), (30.0, 8.0, 30.0)), ((-4.0, 32.0, 0.0), (34.0, 6.0, 34.0)),
                   ((40.0, 14.0, 70.0), (30.0, 6.0, 30.0))][k]
    proj = camera.perspective_rh(np.radians(np.float32(70.0)), w / h, 0.1, 1000.0)
    vp = camera.mat4_mul(proj, camera.look_at_rh(eye, center, (0.0, 1.0, 0.0))).reshape(16)
    return np.ascontiguousarray(vp, dtype=np.float32), np.asarray(eye, dtype=np.float32)


def decode(color, covered, atlas):
    """(type, nibble) of every covered pixel of an unshaded frame drawn with a discriminating atlas (its 48 palette
    entries are distinct), as an (n, 2) array; fails on a colour that is no palette entry of types 1-3."""
    pal = atlas_palette(atlas)
    lut = {int(pal[t, i]): (t, i) for t in TYPES for i in range(16)}
    assert len(lut) == 48
    vals, inv = np.unique(color[covered], return_inverse=True)
    missing = [hex(int(c)) for c in vals if int(c) not in lut]
    assert not missing, f"covered pixels with no palette colour: {missing[:8]}"
    return np.array([lut[int(c)] for c in vals], dtype=np.int32).reshape(-1, 2)[inv]


def _normalise(v):
    v = np.asarray(v, dtype=np.float32)
    return tuple(float(x) for x in (v / np.float32(np.sqrt(np.float32((v * v).sum())))).astype(np.float32))


L = _normalise((1.0, -2.0, 3.0))
NEG_L = tuple(-x for x in L)

# name -> (light_dir, ambient, diffuse, enable_shading)
LIGHTS = {
    "L": (L, 0.3, 0.7, 1),
    "minus_L": (NEG_L, 0.3, 0.7, 1),
    "unnormalised_clamps_to_1": ((0.0, 3.0, 0.0), 0.6, 0.9, 1),
    "negative_ambient_clamps_to_0": (L, -0.2, 0.5, 1),
    "no_diffuse_ambient_1": (L, 1.0, 0.0, 1),
    "inf_light": ((float("inf"), 0.5, 0.25), 0.3, 0.7, 1),
    "nan_ambient": (L, float("nan"), 0.7, 1),
    "shading_off": (L, 0.3, 0.7, 0),
}


def apply_light(cfg, light):
    """Writes (light_dir, ambient, diffuse, enable_shading) into an api.VxFrameConfig or an ob.FrameConfig."""
    d, amb, dif, on = light
    cfg.light_dir[0], cfg.light_dir[1], cfg.light_dir[2] = d
    cfg.ambient, cfg.diffuse, cfg.enable_shading = amb, dif, on
    return cfg


def cache_sequence():
    """(atlas pair, light, clear colour) per frame for the colour-table cache: each frame changes exactly one input of the
    one before -- atlas palette, atlas indices, enable_shading, ambient, diffuse, each light_dir component (the last one
    +0.0 -> -0.0), clear colour --, and the last frame returns to the first one's inputs."""
    a0 = discriminating_atlas()
    pal, nib = atlas_palette(a0[0]), atlas_nibbles(a0[0])
    a_pal = make_atlas(pal[:, np.arange(16) ^ 5], nib)
    a_ind = make_atlas(pal[:, np.arange(16) ^ 5], np.roll(nib, 3, axis=2))
    sky = 0xFF87CEEB
    d, amb, dif, _ = LIGHTS["L"]
    seq = [(a0, LIGHTS["L"], sky), (a_pal, LIGHTS["L"], sky)]
    lights = [LIGHTS["L"], (d, amb, dif, 0), (d, amb, dif, 1), (d, 0.45, dif, 1), (d, 0.45, 0.2, 1)]
    cur = list(d)
    for i, x in enumerate((0.5, -0.25, 0.0)):
        cur[i] = x
        lights.append((tuple(cur), 0.45, 0.2, 1))
    lights.append(((cur[0], cur[1], -0.0), 0.45, 0.2, 1))
    seq += [(a_ind, light, sky) for light in lights]
    seq += [(a_ind, lights[-1], 0x00FF00FF), seq[0]]
    return seq


def clears():
    """Clear colours: transparent black, opaque white, alpha 0 magenta, and a palette entry of discriminating_atlas()."""
    return [0x00000000, 0xFFFFFFFF, 0x00FF00FF, int(atlas_palette(discriminating_atlas()[0])[1, 4])]


CLEARS = clears()
