"""ctypes binding of tests/region_oracle.c, the CPU oracle of vx_world_batch_fill_regions (test infrastructure).  The shared
library is built with gcc into a temporary directory on first use, so the tree is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from differential_projection_voxel_renderer_b200 import api

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "region_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        out = os.path.join(tempfile.gettempdir(), f"vx_region_oracle_{os.getuid()}_{hashlib.sha1(src).hexdigest()[:12]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", tmp, _SRC])
            os.replace(tmp, out)
        _lib = C.CDLL(out)
        _lib.vxo_fill_regions.restype = C.c_int
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def op(shape, a, b=(0, 0, 0), radius_sq=0, block_type=0, replace=0xF):
    """One VxRegionOp record (api.REGION_OP_DTYPE)."""
    r = np.zeros((), dtype=api.REGION_OP_DTYPE)
    r["shape"], r["a"], r["b"], r["radius_sq"], r["block_type"], r["replace_mask"] = shape, a, b, radius_sq, block_type, replace
    return r


def fill_regions(positions, voxels, uniform_flags, ops, slots):
    """vxo_fill_regions over slot-indexed world arrays (positions (S,3), voxels (S,32768), flags (S,)); voxels and flags are
    updated in place, so they must be contiguous arrays of the right dtype.  Returns (status, changed) with status 0 or -1
    (VX_ERR_INVALID, nothing changed)."""
    positions = np.ascontiguousarray(positions, dtype=np.int32).reshape(-1, 3)
    s = positions.shape[0]
    assert voxels.dtype == np.uint8 and voxels.flags.c_contiguous and voxels.size == s * 32768
    assert uniform_flags.dtype == np.uint8 and uniform_flags.flags.c_contiguous and uniform_flags.size == s
    ops = np.ascontiguousarray(ops, dtype=api.REGION_OP_DTYPE).reshape(-1)
    slots = np.ascontiguousarray(slots, dtype=np.int32).reshape(-1)
    changed = np.zeros(slots.size, dtype=np.uint8)
    rc = lib().vxo_fill_regions(_p(positions), _p(voxels), _p(uniform_flags), C.c_int32(s), _p(ops), C.c_int32(ops.size), _p(slots),
                                C.c_int32(slots.size), _p(changed))
    return int(rc), changed
