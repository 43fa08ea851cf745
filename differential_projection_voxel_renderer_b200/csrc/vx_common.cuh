// vx_common.cuh -- shared host-side plumbing for libvx_b200.so (context, device buffers, error handling).
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/vx_b200.h"

#define VX_NUM_SMS_B200 148

struct VxDeviceBuffer {
    void *ptr = nullptr;
    size_t bytes = 0;
    // grow-only device allocation; contents are NOT preserved on growth
    cudaError_t reserve(size_t need) {
        if (need <= bytes) return cudaSuccess;
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
        size_t want = need + need / 4 + 256;
        cudaError_t e = cudaMalloc(&ptr, want);
        if (e == cudaSuccess) bytes = want;
        return e;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
    }
    template <typename T> T *as() const { return reinterpret_cast<T *>(ptr); }
};

struct VxPinnedBuffer {
    void *ptr = nullptr;
    size_t bytes = 0;
    cudaError_t reserve(size_t need) {
        if (need <= bytes) return cudaSuccess;
        if (ptr) cudaFreeHost(ptr);
        ptr = nullptr;
        bytes = 0;
        cudaError_t e = cudaMallocHost(&ptr, need + need / 4 + 256);
        if (e == cudaSuccess) bytes = need + need / 4 + 256;
        return e;
    }
    void release() {
        if (ptr) cudaFreeHost(ptr);
        ptr = nullptr;
        bytes = 0;
    }
    template <typename T> T *as() const { return reinterpret_cast<T *>(ptr); }
};

struct VxMeshBatch {
    int32_t n_chunks = 0;
    int64_t cap_quads = 0;   // capacity of d_quads in quads
    // read back from the cursor on demand (vx_mesh_batch_info, which takes a const batch)
    mutable int64_t total_quads = -1; // -1 until read back
    mutable int32_t n_meshes = -1;
    VxDeviceBuffer quads, quad_base, quad_count, slice_offsets, face_aabb, has_mesh, positions;
    VxDeviceBuffer cursor; // MeshCursor (vx_mesh.cu): quad cursor, mesh counter, overflow flag, work counter
    // world copy owned by the batch (vx_mesh_chunks, vx_world_batch_create): lets vx_mesh_batch_update and
    // vx_world_batch_remesh re-mesh chunks and their neighbours without re-uploading the world
    VxDeviceBuffer world_voxels, world_neighbors, world_flags, update_ids;
    bool owns_world = false, has_neighbors = false;
    std::vector<int32_t> host_neighbors; // [n][6] host copy for the neighbour invalidation list
};

struct VxFrameScratch;

struct VxContext {
    int device = 0;
    int num_sms = VX_NUM_SMS_B200;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr; // device -> host frame transfers of the pipelined frame path (created on first use)
    int64_t launches = 0;
    std::string last_error;
    VxAtlas atlas;
    bool atlas_dirty = true;
    VxFrameScratch *frame = nullptr; // owned by vx_frame.cu
    // small reusable staging buffers
    VxDeviceBuffer tmp_a, tmp_b, tmp_c, tmp_d;
    VxPinnedBuffer pinned;
    // vx_multi.cu: device copy of the last flag-pointer table, status word of the wait kernel
    VxDeviceBuffer multi_ptrs, multi_status;
    uint32_t *multi_ptrs_host[32] = {};
    int multi_ptrs_n = 0;
};

inline int vx_fail(VxContext *ctx, int code, const char *msg) {
    if (ctx) ctx->last_error = msg ? msg : "";
    return code;
}

inline int vx_cuda_fail(VxContext *ctx, cudaError_t e, const char *what, const char *file, int line) {
    char buf[512];
    snprintf(buf, sizeof(buf), "%s: %s (%s:%d)", what, cudaGetErrorString(e), file, line);
    if (ctx) ctx->last_error = buf;
    return e == cudaErrorMemoryAllocation ? VX_ERR_OOM : VX_ERR_CUDA;
}

#define VX_CUDA(ctx, expr)                                                        \
    do {                                                                          \
        cudaError_t _e = (expr);                                                  \
        if (_e != cudaSuccess) return vx_cuda_fail((ctx), _e, #expr, __FILE__, __LINE__); \
    } while (0)

#define VX_CHECK_LAUNCH(ctx)                                                      \
    do {                                                                          \
        (ctx)->launches++;                                                        \
        cudaError_t _e = cudaGetLastError();                                      \
        if (_e != cudaSuccess) return vx_cuda_fail((ctx), _e, "kernel launch", __FILE__, __LINE__); \
    } while (0)

// frame scratch lifetime hooks implemented in vx_frame.cu
void vx_frame_scratch_destroy(VxContext *ctx);

// vx_multi.cu: copy a table of n <= 32 device flag pointers to ctx->multi_ptrs (again only when it differs from the last one)
int vx_stage_flag_table(VxContext *ctx, uint32_t *const *flags, int n);

// cross-GPU waits give up after timeout_us (<= 0: VX_HANDOFF_TIMEOUT_US) so that a lost peer cannot hang the device
constexpr int32_t VX_HANDOFF_TIMEOUT_US = 2000000;
inline unsigned long long vx_timeout_ns(int32_t timeout_us) {
    return (unsigned long long)(timeout_us > 0 ? timeout_us : VX_HANDOFF_TIMEOUT_US) * 1000ull;
}
