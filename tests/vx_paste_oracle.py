"""ctypes binding of tests/paste_oracle.c, the CPU oracle of vx_world_batch_copy_region and vx_world_batch_paste (test
infrastructure).  The shared library is built with gcc into a temporary directory on first use, so the tree is never
written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from differential_projection_voxel_renderer_b200 import api

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "paste_oracle.c")
_lib = None
SKIP = api.PASTE_SKIP


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        out = os.path.join(tempfile.gettempdir(), f"vx_paste_oracle_{os.getuid()}_{hashlib.sha1(src).hexdigest()[:12]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", tmp, _SRC])
            os.replace(tmp, out)
        _lib = C.CDLL(out)
        _lib.vxo_copy_region.restype = C.c_int
        _lib.vxo_paste.restype = C.c_int
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def op(origin, dims, offset=0, replace=0xF):
    """One VxPasteOp record (api.PASTE_OP_DTYPE)."""
    r = np.zeros((), dtype=api.PASTE_OP_DTYPE)
    r["origin"], r["dims"], r["offset"], r["replace_mask"] = origin, dims, offset, replace
    return r


def pack(origins_templates, replace=0xF):
    """Ops and one template buffer from [(origin, template (sz, sy, sx))], templates back to back in list order."""
    ops, blobs, at = [], [], 0
    for origin, t in origins_templates:
        t = np.ascontiguousarray(t, dtype=np.uint8)
        ops.append(op(origin, t.shape[::-1], at, replace))
        blobs.append(t.reshape(-1))
        at += t.size
    return np.stack(ops), (np.concatenate(blobs) if blobs else np.zeros(0, np.uint8))


def chunk_table(positions, lo, dims):
    """The chunk_slots table of vx_world_batch_copy_region for slot-indexed positions (S, 3): -1 where no slot holds the chunk."""
    lo, dims = np.asarray(lo, np.int64), np.asarray(dims, np.int64)
    c0, c1 = lo >> 5, (lo + dims - 1) >> 5
    at = {tuple(p): s for s, p in enumerate(np.asarray(positions).reshape(-1, 3).tolist())}
    return np.array([[[at.get((x, y, z), -1) for x in range(c0[0], c1[0] + 1)] for y in range(c0[1], c1[1] + 1)]
                     for z in range(c0[2], c1[2] + 1)], dtype=np.int32)


def copy_region(positions, voxels, uniform_flags, lo, dims, chunk_slots):
    """vxo_copy_region: returns (status, box (dims[2], dims[1], dims[0]) or None) with status 0 or -1 (VX_ERR_INVALID)."""
    positions = np.ascontiguousarray(positions, dtype=np.int32).reshape(-1, 3)
    voxels = np.ascontiguousarray(voxels, dtype=np.uint8)
    uniform_flags = np.ascontiguousarray(uniform_flags, dtype=np.uint8)
    lo, dims = np.ascontiguousarray(lo, dtype=np.int32).reshape(3), np.ascontiguousarray(dims, dtype=np.int32).reshape(3)
    chunk_slots = np.ascontiguousarray(chunk_slots, dtype=np.int32).reshape(-1)
    size = int(np.prod(np.clip(dims.astype(np.int64), 0, 1024)))
    out = np.full(max(size, 1), 0xAB, dtype=np.uint8)
    rc = lib().vxo_copy_region(_p(positions), _p(voxels), _p(uniform_flags), C.c_int32(positions.shape[0]), _p(lo), _p(dims), _p(chunk_slots),
                               _p(out))
    return int(rc), (out[:size].reshape(dims[::-1]) if rc == 0 else None)


def paste(positions, voxels, uniform_flags, ops, templates, slots, n_template_bytes=None):
    """vxo_paste over slot-indexed world arrays (positions (S,3), voxels (S,32768), flags (S,)); voxels and flags are updated
    in place, so they must be contiguous arrays of the right dtype.  Returns (status, changed) with status 0 or -1
    (VX_ERR_INVALID, nothing changed)."""
    positions = np.ascontiguousarray(positions, dtype=np.int32).reshape(-1, 3)
    s = positions.shape[0]
    assert voxels.dtype == np.uint8 and voxels.flags.c_contiguous and voxels.size == s * 32768
    assert uniform_flags.dtype == np.uint8 and uniform_flags.flags.c_contiguous and uniform_flags.size == s
    ops = np.ascontiguousarray(ops, dtype=api.PASTE_OP_DTYPE).reshape(-1)
    templates = np.ascontiguousarray(templates, dtype=np.uint8).reshape(-1)
    n_bytes = templates.size if n_template_bytes is None else int(n_template_bytes)
    slots = np.ascontiguousarray(slots, dtype=np.int32).reshape(-1)
    changed = np.zeros(slots.size, dtype=np.uint8)
    rc = lib().vxo_paste(_p(positions), _p(voxels), _p(uniform_flags), C.c_int32(s), _p(ops), C.c_int32(ops.size), _p(templates),
                         C.c_int64(n_bytes), _p(slots), C.c_int32(slots.size), _p(changed))
    return int(rc), changed
