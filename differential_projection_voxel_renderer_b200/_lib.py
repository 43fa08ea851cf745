"""ctypes loader for libvx_b200.so (the C ABI in include/vx_b200.h).

There is no CPU fallback: if the shared library is missing the import of the
product API raises, and without a CUDA device `Context()` raises VxError
(VX_ERR_NO_DEVICE).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# VX_B200_LIB: development override (kernel tuning variants); the product always loads the in-tree library
LIB_PATH = os.environ.get("VX_B200_LIB") or os.path.join(_HERE, "libvx_b200.so")

VX_OK = 0
VX_ERR_INVALID = -1
VX_ERR_NO_DEVICE = -2
VX_ERR_CUDA = -3
VX_ERR_CAPACITY = -4
VX_ERR_OOM = -5

NBR_NONE = -1
NBR_UNIFORM_AIR = -2
NBR_UNIFORM_SOLID = -3

RAY_HIT = 0
RAY_MISS = 1
RAY_LEFT_WORLD = 2
RAY_INVALID = 3


class VxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libvx_b200: {msg} (code {code})")
        self.code = code


class VxAtlas(C.Structure):
    _fields_ = [("palette", (C.c_uint32 * 16) * 4), ("indices", (C.c_uint8 * 32) * 4)]


class VxFrameConfig(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("clear_color", C.c_uint32),
                ("backface_culling", C.c_int32), ("enable_shading", C.c_int32),
                ("light_dir", C.c_float * 3), ("ambient", C.c_float), ("diffuse", C.c_float),
                ("stripe_y0", C.c_int32), ("stripe_rows", C.c_int32),
                ("differential_projection", C.c_int32), ("async_submit", C.c_int32),
                ("profile_kernels", C.c_int32), ("macrotile", C.c_int32),
                ("occlusion_culling", C.c_int32), ("occlusion_grid_w", C.c_int32), ("occlusion_grid_h", C.c_int32),
                ("frames_in_flight", C.c_int32)]


class VxTerrainParams(C.Structure):
    _fields_ = [("perm", C.c_int32 * 512), ("grad", (C.c_double * 2) * 8), ("scale", C.c_double), ("amplitude", C.c_double)]


class VxFacePacket32(C.Structure):
    _fields_ = [("len", C.c_uint8), ("u_min", C.c_uint8 * 32), ("v_min", C.c_uint8 * 32), ("u_len", C.c_uint8 * 32),
                ("v_len", C.c_uint8 * 32), ("axis_pos", C.c_uint8 * 32), ("block_type", C.c_uint8 * 32), ("pad", C.c_uint8 * 31)]


class VxMeshBatchInfo(C.Structure):
    _fields_ = [("n_chunks", C.c_int32), ("n_meshes", C.c_int32), ("total_quads", C.c_int64)]


class VxMeshBatchDevice(C.Structure):
    _fields_ = [("d_quads", C.c_void_p), ("d_quad_base", C.c_void_p), ("d_quad_count", C.c_void_p),
                ("d_slice_offsets", C.c_void_p), ("d_face_aabb", C.c_void_p), ("d_has_mesh", C.c_void_p),
                ("d_positions", C.c_void_p)]


class VxStripeSync(C.Structure):
    _fields_ = [("d_wait_flag", C.c_void_p), ("wait_value", C.c_uint32), ("d_signal_flag", C.c_void_p), ("signal_value", C.c_uint32),
                ("timeout_us", C.c_int32), ("n_arrive", C.c_int32), ("arrive_stride_words", C.c_int32), ("d_arrive_flags", C.c_void_p),
                ("arrive_value", C.c_uint32), ("release_value", C.c_uint32), ("n_release", C.c_int32), ("signal_after", C.c_int32),
                ("release_flags", C.c_void_p)]


class VxShardLayout(C.Structure):
    _fields_ = [("rank_stride", C.c_int64), ("off_quad_base", C.c_int64), ("off_quad_count", C.c_int64),
                ("off_slice_offsets", C.c_int64), ("off_face_aabb", C.c_int64), ("off_has_mesh", C.c_int64),
                ("off_quads", C.c_int64), ("quads_capacity", C.c_int64), ("rows_per_rank", C.c_int32), ("reserved", C.c_int32)]


class VxRayHit(C.Structure):
    _fields_ = [("status", C.c_int32), ("slot", C.c_int32), ("voxel", C.c_int32 * 3), ("face", C.c_int32), ("t", C.c_float),
                ("block_type", C.c_uint8), ("pad", C.c_uint8 * 3)]


class VxFrameStats(C.Structure):
    _fields_ = [("n_input", C.c_int32), ("n_survivors", C.c_int32), ("n_quads", C.c_int32),
                ("n_triangles", C.c_int32), ("n_bin_entries", C.c_int32), ("n_kernel_launches", C.c_int32),
                ("reserved", C.c_int32 * 2)]


# every symbol include/vx_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_I = C.c_int32
PROTOTYPES = {
    "vx_context_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "vx_context_destroy": (None, [_P]),
    "vx_error_string": (C.c_char_p, [C.c_int]),
    "vx_last_error": (C.c_char_p, [_P]),
    "vx_device_synchronize": (C.c_int, [_P]),
    "vx_context_stream": (_P, [_P]),
    "vx_context_launch_count": (C.c_int64, [_P]),
    "vx_host_alloc": (C.c_int, [_P, C.c_size_t, C.POINTER(_P)]),
    "vx_host_free": (None, [_P, _P]),
    "vx_device_alloc": (C.c_int, [_P, C.c_size_t, C.POINTER(_P)]),
    "vx_device_free": (C.c_int, [_P, _P]),
    "vx_ipc_export": (C.c_int, [_P, _P, _P]),
    "vx_ipc_open": (C.c_int, [_P, _P, C.POINTER(_P)]),
    "vx_ipc_close": (C.c_int, [_P, _P]),
    "vx_signal_flags": (C.c_int, [_P, _P, _I, C.c_uint32]),
    "vx_wait_flags": (C.c_int, [_P, _P, _I, _I, C.c_uint32, _I]),
    "vx_wait_then_signal": (C.c_int, [_P, _P, _I, _I, C.c_uint32, _P, _I, C.c_uint32, _I]),
    "vx_wait_status": (C.c_int, [_P, C.POINTER(_I)]),
    "vx_shard_layout": (C.c_int, [_I, C.c_int64, C.POINTER(VxShardLayout)]),
    "vx_mesh_shard_pack": (C.c_int, [_P, _P, C.POINTER(VxShardLayout), _P]),
    "vx_mesh_shard_pack_async": (C.c_int, [_P, _P, C.POINTER(VxShardLayout), _P]),
    "vx_mesh_batch_assemble_shards": (C.c_int, [_P, _I, _I, _P, C.POINTER(VxShardLayout), _P, _P, C.POINTER(_P)]),
    "vx_mesh_batch_assemble_shards_async": (C.c_int, [_P, _I, _I, _P, C.POINTER(VxShardLayout), _P, C.POINTER(_P)]),
    "vx_generate_terrain": (C.c_int, [_P, _P, _I, C.POINTER(VxTerrainParams), _P, _P]),
    "vx_mesh_chunks": (C.c_int, [_P, _P, _P, _P, _P, _I, C.POINTER(_P)]),
    "vx_mesh_batch_update": (C.c_int, [_P, _P, _P, _I, _P, _P, C.POINTER(_I)]),
    "vx_mesh_chunks_device": (C.c_int, [_P, _P, _P, _P, _P, _I, C.POINTER(_P)]),
    "vx_mesh_chunk_subset_device": (C.c_int, [_P, _P, _P, _P, _P, _I, _P, _I, C.POINTER(_P)]),
    "vx_remesh_chunks_device": (C.c_int, [_P, _P, _P, _P, _P]),
    "vx_mesh_batch_info": (C.c_int, [_P, _P, C.POINTER(VxMeshBatchInfo)]),
    "vx_mesh_batch_device": (C.c_int, [_P, C.POINTER(VxMeshBatchDevice)]),
    "vx_mesh_batch_download": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "vx_mesh_batch_upload": (C.c_int, [_P, _P, C.c_int64, _P, _P, _P, _P, _P, _P, _I, C.POINTER(_P)]),
    "vx_mesh_batch_release": (None, [_P, _P]),
    "vx_greedy_mesh_slices": (C.c_int, [_P, _P, _I, _P, _P]),
    "vx_cull_chunks": (C.c_int, [_P, _P, _I, _P, _P, _I, _I, _P]),
    "vx_horizon_cull": (C.c_int, [_P, _P, _P, _I, _P, _I, _I, C.c_float, C.c_float, C.c_float, C.POINTER(_I)]),
    "vx_default_frame_config": (None, [C.POINTER(VxFrameConfig), _I, _I]),
    "vx_default_atlas": (None, [C.POINTER(VxAtlas)]),
    "vx_set_atlas": (C.c_int, [_P, C.POINTER(VxAtlas)]),
    "vx_render_frame": (C.c_int, [_P, _P, _P, _I, _P, _P, _I, C.POINTER(VxFrameConfig), _P, _P, _P, C.POINTER(_I)]),
    "vx_world_batch_create": (C.c_int, [_P, _I, C.POINTER(_P)]),
    "vx_world_batch_grow": (C.c_int, [_P, _P, _I]),
    "vx_world_batch_assign": (C.c_int, [_P, _P, _P, _I, _P, _P]),
    "vx_world_batch_generate": (C.c_int, [_P, _P, _P, _I, _P, C.POINTER(VxTerrainParams), _P]),
    "vx_world_batch_unload": (C.c_int, [_P, _P, _P, _I]),
    "vx_world_batch_remesh": (C.c_int, [_P, _P, _P, _I]),
    "vx_world_batch_set_blocks": (C.c_int, [_P, _P, _P, _P, _P, _I]),
    "vx_world_raycast": (C.c_int, [_P, _P, _P, _P, _P, _I, C.c_float, _P]),
    "vx_world_raycast_device": (C.c_int, [_P, _P, _P, _P, _P, _I, C.c_float, _P]),
    "vx_render_mesh_tiny_quads": (C.c_int, [_P, _P, _I, _P, C.POINTER(VxFrameConfig), _P, _I, _P, _P]),
    "vx_render_mesh_with_up": (C.c_int, [_P, _P, _I, _P, C.POINTER(VxFrameConfig), _P, _P, _P]),
    "vx_render_frame_macrotile": (C.c_int, [_P, _P, _P, _I, _P, C.POINTER(VxFrameConfig), _P, _P, _P, C.POINTER(_I)]),
    "vx_span_walk_quads": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P]),
    "vx_span_walk_quads_device": (C.c_int, [_P, _P, _P, _I, _I, _I, _P, _P]),
    "vx_fill_spans": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P]),
    "vx_hyper_pipeline_render": (C.c_int, [_P, _P, _P, _I, _P, _I, _I, _P, _P, C.POINTER(_I)]),
    "vx_render_frame_begin": (C.c_int, [_P, _P, _P, _I, _P, _P, _I, C.POINTER(VxFrameConfig), _P, _P, C.POINTER(_I)]),
    "vx_render_frame_end": (C.c_int, [_P, _I, _P, C.POINTER(_I)]),
    "vx_render_frame_stripe": (C.c_int, [_P, _P, _P, _I, _P, _P, _I, C.POINTER(VxFrameConfig), _P, _P, C.POINTER(VxStripeSync)]),
    "vx_render_frame_device": (C.c_int, [_P, _P, _P, _I, _P, _P, _I, C.POINTER(VxFrameConfig)]),
    "vx_render_frame_into": (C.c_int, [_P, _P, _P, _I, _P, _P, _I, C.POINTER(VxFrameConfig), _P, _P]),
    "vx_framebuffer_device": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_I), C.POINTER(_I)]),
    "vx_frame_stats": (C.c_int, [_P, C.POINTER(VxFrameStats)]),
    "vx_frame_counters": (C.c_int, [_P, _P]),
    "vx_frame_kernel_times": (C.c_int, [_P, _P]),
    "vx_frame_trace": (C.c_int, [_P, _P, _I, C.POINTER(_I)]),
    "vx_frame_setup_trace": (C.c_int, [_P, _P, _I, C.POINTER(_I)]),
    "vx_frame_bin_counts": (C.c_int, [_P, _P, _I, C.POINTER(_I), C.POINTER(_I)]),
    "vx_frame_bin_tasks": (C.c_int, [_P, _P, _I, C.POINTER(_I), C.POINTER(_I)]),
    "vx_render_mesh": (C.c_int, [_P, _P, _I, _P, C.POINTER(VxFrameConfig), _P, _P, _P]),
    "vx_face_packets": (C.c_int, [_P, _P, _I, _P, _I, _P]),
    "vx_face_basis": (C.c_int, [_P, _P, _P, _P, _I, _P, _P]),
    "vx_project_packet": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P]),
    "vx_transform_vertices": (C.c_int, [_P, _P, _I, _P, _P, _P]),
    "vx_selftest_division": (C.c_int, [_P, C.c_uint64, C.c_uint64, _I, _P]),
    "vx_project_mesh_vertices": (C.c_int, [_P, _P, _I, _P, _I, _P, C.c_int64]),
}

_lib = None


def load():
    """Load libvx_b200.so and bind every prototype.  Raises if the library or a symbol is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build the CUDA library first (python -c 'import __graft_entry__ as g; g.build()'"
            " or make -C differential_projection_voxel_renderer_b200/csrc).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
