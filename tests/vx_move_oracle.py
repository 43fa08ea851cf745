"""ctypes binding of tests/move_oracle.c, the CPU oracle of vx_world_move_boxes (test infrastructure).  The shared library
is built with gcc into a temporary directory on first use, so the tree is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "move_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        out = os.path.join(tempfile.gettempdir(), f"vx_move_oracle_{os.getuid()}_{hashlib.sha1(src).hexdigest()[:12]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                                   "-Wextra", "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, out)
        _lib = C.CDLL(out)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def move_boxes(positions, voxels, uniform_flags, neighbors, pos, size, delta, slots, want_reads=False):
    """vxo_move_boxes over slot-indexed world arrays (positions (S,3), voxels (S,32768), flags (S,), neighbours (S,6), as
    vx_ray_oracle.raycast takes them).  pos / size / delta (n, 3) f32 (size and delta broadcast), slots (n,).  Returns new
    arrays (pos, slots, flags) -- and the voxel bytes each move read with want_reads."""
    positions = np.ascontiguousarray(positions, dtype=np.int32).reshape(-1, 3)
    s = positions.shape[0]
    voxels = np.ascontiguousarray(voxels, dtype=np.uint8).reshape(s, 32768)
    flags = np.ascontiguousarray(uniform_flags, dtype=np.uint8).reshape(s)
    neighbors = np.ascontiguousarray(neighbors, dtype=np.int32).reshape(s, 6)
    pos = np.array(pos, dtype=np.float32).reshape(-1, 3)
    n = pos.shape[0]
    size = np.ascontiguousarray(np.broadcast_to(np.asarray(size, dtype=np.float32), (n, 3)))
    delta = np.ascontiguousarray(np.broadcast_to(np.asarray(delta, dtype=np.float32), (n, 3)))
    slots = np.array(slots, dtype=np.int32).reshape(n)
    out = np.zeros(n, dtype=np.uint32)
    reads = np.zeros(n, dtype=np.int64)
    lib().vxo_move_boxes(_p(positions), _p(voxels), _p(flags), _p(neighbors), C.c_int32(s), _p(pos), _p(size), _p(delta), _p(slots),
                         C.c_int32(n), _p(out), _p(reads))
    return (pos, slots, out, reads) if want_reads else (pos, slots, out)
