"""ctypes binding of tests/ray_oracle.c, the CPU oracle of vx_world_raycast (test infrastructure).  The shared library is
built with gcc into a temporary directory on first use, so the tree is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ray_oracle.c")
_lib = None

RAY_HIT_DTYPE = np.dtype([("status", "<i4"), ("slot", "<i4"), ("voxel", "<i4", (3,)), ("face", "<i4"), ("t", "<f4"),
                          ("block_type", "u1"), ("pad", "u1", (3,))])  # vxo_ray_hit = VxRayHit, 32 bytes


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        out = os.path.join(tempfile.gettempdir(), f"vx_ray_oracle_{os.getuid()}_{hashlib.sha1(src).hexdigest()[:12]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                                   "-Wextra", "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, out)
        _lib = C.CDLL(out)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def raycast(positions, voxels, uniform_flags, neighbors, origins, dirs, start_slots, max_t, want_steps=False):
    """vxo_raycast over slot-indexed world arrays (positions (S,3), voxels (S,32768), flags (S,), neighbours (S,6)).
    Returns the hits as a RAY_HIT_DTYPE array (and the face crossings per ray with want_steps)."""
    positions = np.ascontiguousarray(positions, dtype=np.int32).reshape(-1, 3)
    s = positions.shape[0]
    voxels = np.ascontiguousarray(voxels, dtype=np.uint8).reshape(s, 32768)
    flags = np.ascontiguousarray(uniform_flags, dtype=np.uint8).reshape(s)
    neighbors = np.ascontiguousarray(neighbors, dtype=np.int32).reshape(s, 6)
    origins = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
    n = origins.shape[0]
    dirs = np.ascontiguousarray(dirs, dtype=np.float32).reshape(n, 3)
    slots = np.ascontiguousarray(start_slots, dtype=np.int32).reshape(n)
    hits = np.zeros(n, dtype=RAY_HIT_DTYPE)
    steps = np.zeros(n, dtype=np.int32)
    lib().vxo_raycast(_p(positions), _p(voxels), _p(flags), _p(neighbors), C.c_int32(s), _p(origins), _p(dirs), _p(slots),
                      C.c_int32(n), C.c_float(max_t), _p(hits), _p(steps))
    return (hits, steps) if want_steps else hits
