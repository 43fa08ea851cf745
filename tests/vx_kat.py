"""Known-answer cases restated from the reference's own tests (data only; cited per case)."""
import numpy as np

AIR, GRASS, DIRT, STONE = 0, 1, 2, 3


def empty_chunk():
    return np.zeros((32, 32, 32), dtype=np.uint8)  # [z, y, x]


def set_block(c, x, y, z, t):
    c[z, y, x] = t


def chunk_single_voxel(x=16, y=16, z=16, t=STONE):
    c = empty_chunk()
    set_block(c, x, y, z, t)
    return c.reshape(-1)


def chunk_two_adjacent():  # tests/meshing_tests.rs:193-220
    c = empty_chunk()
    set_block(c, 10, 10, 10, STONE)
    set_block(c, 11, 10, 10, STONE)
    return c.reshape(-1)


def chunk_2x2_plane():  # tests/meshing_tests.rs:257-281
    c = empty_chunk()
    for x in range(2):
        for z in range(2):
            set_block(c, x, 0, z, STONE)
    return c.reshape(-1)


def chunk_two_types():  # tests/meshing_tests.rs:418-470 (different block types are not merged)
    c = empty_chunk()
    set_block(c, 5, 5, 5, STONE)
    set_block(c, 6, 5, 5, GRASS)
    return c.reshape(-1)


def chunk_dense_solid():  # benches/meshing.rs:28-41 (Varied chunk that is all Stone)
    return np.full(32768, STONE, dtype=np.uint8)


def chunk_slab(height=8):  # benches/differential_projection.rs:8-24: y < 8 + ((x + z) % 4) Stone
    c = empty_chunk()
    z, y, x = np.meshgrid(np.arange(32), np.arange(32), np.arange(32), indexing="ij")
    c[y < height + ((x + z) % 4)] = STONE
    return c.reshape(-1)


def chunk_checker3d():  # worst case for the quad count: 16384 isolated voxels -> 98304 quads
    z, y, x = np.meshgrid(np.arange(32), np.arange(32), np.arange(32), indexing="ij")
    return np.where((x + y + z) % 2 == 0, STONE, AIR).astype(np.uint8).reshape(-1)


# benches/microbench.rs:21-38 slice masks
def slice_masks():
    full = np.full(32, 0xFFFFFFFF, dtype=np.uint32)
    checker = np.array([0xFFFFFFFF if r % 2 == 0 else 0 for r in range(32)], dtype=np.uint32)
    sparse = np.full(32, 0x80000001, dtype=np.uint32)
    alt_bits = np.array([0xAAAAAAAA if r % 2 == 0 else 0x55555555 for r in range(32)], dtype=np.uint32)
    return {"empty": np.zeros(32, np.uint32), "full": full, "checker_rows": checker, "sparse": sparse, "alt_bits": alt_bits}


def quads_of_face(unpacked, slice_offsets, face):
    a, b = int(slice_offsets[face, 0]), int(slice_offsets[face, 32])
    return unpacked[a:b]


def slice_of_quad(slice_offsets, face, k):
    """slice index of the k-th quad of a face."""
    so = slice_offsets[face]
    q = int(so[0]) + k
    return int(np.searchsorted(so[:33], q, side="right") - 1)


# ---- scenes that outgrow the frame scratch a context starts with (tests/test_frame_capacity_gpu.py) ---------------------
def chunk_plate(t=STONE, y=0):
    """One full 32 x 32 layer of block type t: six greedy quads, the top one a single 32 x 32 face."""
    c = empty_chunk()
    c[:, y, :] = t
    return c.reshape(-1)


def chunk_checker3d_typed(t=STONE):
    """chunk_checker3d with block type t: 98304 quads of one voxel face each."""
    z, y, x = np.meshgrid(np.arange(32), np.arange(32), np.arange(32), indexing="ij")
    return np.where((x + y + z) % 2 == 0, t, AIR).astype(np.uint8).reshape(-1)


def chunk_z_plates(n=16):
    """n layers at z = 0, 2, 4, ..., each a full 32 x 32 layer whose block type cycles with x + y + layer: no two
    neighbouring voxels of a layer share a type, so every voxel face of a layer is a quad of its own (1024 per side)."""
    c = empty_chunk()
    y, x = np.meshgrid(np.arange(32), np.arange(32), indexing="ij")
    for k in range(n):
        c[2 * k] = (1 + (x + y + k) % 3).astype(np.uint8)
    return c.reshape(-1)
