// vx_ray.cu -- ray casting through the voxels of a world batch (picking): one thread per ray, an Amanatides-Woo walk from
// voxel to voxel that crosses chunk borders through the batch's neighbour table (no position -> slot lookup).  The exact
// semantics are written down in include/vx_b200.h; the CPU oracle (vxo_raycast) restates them statement for statement.
// Every face crossing is computed in closed form, ((float)plane - o) / d, one correctly rounded subtraction and division
// (compiled with -fmad=false like the other exact files), so the kernel and the oracle produce the same bits.  Nothing
// here touches the frame kernels or their buffers.
#include "vx_common.cuh"

namespace {

constexpr int RAY_THREADS = 128;
constexpr float RAY_MAX_T = 1e4f;
constexpr float RAY_MAX_ORIGIN = 16777216.0f; // 2^24: every start voxel coordinate is an exact float

#ifdef VX_DEBUG_CHECKS
// set when a walk takes more steps than its bound (see the header); read and cleared by vx_world_raycast
__device__ unsigned int g_ray_bound_exceeded;
#endif

struct RayWorld {
    const uint8_t *voxels;    // [slot][32768]
    const uint8_t *flags;     // [slot] 0 Varied, else 1 + block type
    const int32_t *neighbors; // [slot][6] FaceDir order
    const int32_t *positions; // [slot][3]
    int32_t n_slots;
};

__device__ __forceinline__ float face_t(int32_t plane, float o, float d) { return ((float)plane - o) / d; }

// parameter of the next face crossing on one axis: plane v + 1 stepping up, v stepping down, none without a step
__device__ __forceinline__ float next_t(int32_t v, int32_t step, float o, float d) {
    return step == 0 ? INFINITY : face_t(step > 0 ? v + 1 : v, o, d);
}

__device__ __forceinline__ int voxel_type(uint8_t flag, const uint8_t *chunk, int32_t lx, int32_t ly, int32_t lz) {
    if (flag != 0) return flag - 1; // Uniform: no voxel rows, no load
    return __ldg(chunk + lz * 1024 + ly * 32 + lx);
}

__global__ void __launch_bounds__(RAY_THREADS) raycast_kernel(RayWorld w, const float *__restrict__ origins, const float *__restrict__ dirs,
                                                              const int32_t *__restrict__ start_slots, int32_t n, float max_t,
                                                              VxRayHit *__restrict__ hits) {
    const int32_t i = blockIdx.x * RAY_THREADS + threadIdx.x;
    if (i >= n) return;
    VxRayHit h;
    h.status = VX_RAY_INVALID;
    h.slot = -1;
    h.voxel[0] = h.voxel[1] = h.voxel[2] = 0;
    h.face = -1;
    h.t = 0.0f;
    h.block_type = 0;
    h.pad[0] = h.pad[1] = h.pad[2] = 0;

    const float ox = origins[3 * (size_t)i], oy = origins[3 * (size_t)i + 1], oz = origins[3 * (size_t)i + 2];
    const float dx = dirs[3 * (size_t)i], dy = dirs[3 * (size_t)i + 1], dz = dirs[3 * (size_t)i + 2];
    int32_t slot = start_slots[i];
    bool ok = max_t >= 0.0f && max_t <= RAY_MAX_T;
    ok = ok && isfinite(ox) && isfinite(oy) && isfinite(oz) && isfinite(dx) && isfinite(dy) && isfinite(dz);
    ok = ok && fabsf(ox) < RAY_MAX_ORIGIN && fabsf(oy) < RAY_MAX_ORIGIN && fabsf(oz) < RAY_MAX_ORIGIN;
    ok = ok && (dx != 0.0f || dy != 0.0f || dz != 0.0f);
    ok = ok && slot >= 0 && slot < w.n_slots;
    int32_t vx = 0, vy = 0, vz = 0;
    if (ok) {
        vx = (int32_t)floorf(ox);
        vy = (int32_t)floorf(oy);
        vz = (int32_t)floorf(oz);
        const int32_t *p = w.positions + 3 * (size_t)slot;
        ok = p[0] == (vx >> 5) && p[1] == (vy >> 5) && p[2] == (vz >> 5);
    }
    if (!ok) {
        hits[i] = h;
        return;
    }

    const int32_t sx = dx > 0.0f ? 1 : (dx < 0.0f ? -1 : 0);
    const int32_t sy = dy > 0.0f ? 1 : (dy < 0.0f ? -1 : 0);
    const int32_t sz = dz > 0.0f ? 1 : (dz < 0.0f ? -1 : 0);
    int32_t lx = vx & 31, ly = vy & 31, lz = vz & 31;
    uint8_t flag = w.flags[slot];
    const uint8_t *chunk = w.voxels + (size_t)slot * VX_CHUNK_VOLUME;
    int type = voxel_type(flag, chunk, lx, ly, lz);
    int face = -1;
    float t = 0.0f;
    float tx = next_t(vx, sx, ox, dx), ty = next_t(vy, sy, oy, dy), tz = next_t(vz, sz, oz, dz);
#ifdef VX_DEBUG_CHECKS
    const double bound = (sx ? floor((double)fabsf(dx) * max_t) + 3.0 : 0.0) + (sy ? floor((double)fabsf(dy) * max_t) + 3.0 : 0.0) +
                         (sz ? floor((double)fabsf(dz) * max_t) + 3.0 : 0.0);
    double steps = 0.0;
#endif
    h.status = VX_RAY_MISS;
    while (type == 0) {
        // the axis with the smallest tnext, ties x before y before z
        const int axis = (tx <= ty && tx <= tz) ? 0 : (ty <= tz ? 1 : 2);
        t = axis == 0 ? tx : (axis == 1 ? ty : tz);
        if (t > max_t) break; // VX_RAY_MISS
#ifdef VX_DEBUG_CHECKS
        steps += 1.0;
        if (steps > bound) atomicOr(&g_ray_bound_exceeded, 1u);
#endif
        const int32_t s = axis == 0 ? sx : (axis == 1 ? sy : sz);
        int32_t l;
        if (axis == 0) {
            vx += s;
            l = lx += s;
            tx = next_t(vx, sx, ox, dx);
        } else if (axis == 1) {
            vy += s;
            l = ly += s;
            ty = next_t(vy, sy, oy, dy);
        } else {
            vz += s;
            l = lz += s;
            tz = next_t(vz, sz, oz, dz);
        }
        face = 2 * axis + (s > 0 ? 1 : 0); // a step up enters through the voxel's negative face
        if ((uint32_t)l > 31u) {            // into the neighbour chunk across FaceDir 2*axis (+) or 2*axis+1 (-)
            const int32_t nb = w.neighbors[6 * (size_t)slot + 2 * axis + (s > 0 ? 0 : 1)];
            if (nb < 0) {
                h.status = VX_RAY_LEFT_WORLD;
                break;
            }
            slot = nb;
            lx &= 31;
            ly &= 31;
            lz &= 31;
            flag = w.flags[slot];
            chunk = w.voxels + (size_t)slot * VX_CHUNK_VOLUME;
        }
        type = voxel_type(flag, chunk, lx, ly, lz);
    }
    if (type != 0) {
        h.status = VX_RAY_HIT;
        h.slot = slot;
        h.voxel[0] = vx;
        h.voxel[1] = vy;
        h.voxel[2] = vz;
        h.face = face;
        h.t = t;
        h.block_type = (uint8_t)type;
    }
    hits[i] = h;
}

int world_batch_ok(VxContext *ctx, const VxMeshBatch *b, const char *who) {
    if (!ctx || !b) return vx_fail(ctx, VX_ERR_INVALID, who);
    if (!b->owns_world || !b->has_neighbors) return vx_fail(ctx, VX_ERR_INVALID, "not a world batch (vx_world_batch_create)");
    return VX_OK;
}

int launch_raycast(VxContext *ctx, const VxMeshBatch *b, const float *d_origins, const float *d_dirs, const int32_t *d_slots, int32_t n,
                   float max_t, VxRayHit *d_hits) {
    const RayWorld w{b->world_voxels.as<uint8_t>(), b->world_flags.as<uint8_t>(), b->world_neighbors.as<int32_t>(), b->positions.as<int32_t>(),
                     b->n_chunks};
    raycast_kernel<<<(n + RAY_THREADS - 1) / RAY_THREADS, RAY_THREADS, 0, ctx->stream>>>(w, d_origins, d_dirs, d_slots, n, max_t, d_hits);
    VX_CHECK_LAUNCH(ctx);
    return VX_OK;
}

} // namespace

extern "C" {

int vx_world_raycast(VxContext *ctx, const VxMeshBatch *b, const float *origins, const float *dirs, const int32_t *start_slots,
                     int32_t n, float max_t, VxRayHit *hits_out) {
    int rc = world_batch_ok(ctx, b, "vx_world_raycast: bad argument");
    if (rc != VX_OK) return rc;
    if (n < 0 || (n > 0 && (!origins || !dirs || !start_slots || !hits_out))) return vx_fail(ctx, VX_ERR_INVALID, "vx_world_raycast: bad argument");
    for (int32_t i = 0; i < n; ++i)
        if (start_slots[i] < -1 || start_slots[i] >= b->n_chunks) return vx_fail(ctx, VX_ERR_INVALID, "vx_world_raycast: start slot out of range");
    if (n == 0) return VX_OK;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t nn = (size_t)n;
    // inputs staged back to back: origins, dirs (12 bytes a ray each), start slots
    VX_CUDA(ctx, ctx->tmp_a.reserve(28 * nn));
    VX_CUDA(ctx, ctx->tmp_b.reserve(sizeof(VxRayHit) * nn));
    uint8_t *in = ctx->tmp_a.as<uint8_t>();
    VX_CUDA(ctx, cudaMemcpyAsync(in, origins, 12 * nn, cudaMemcpyHostToDevice, ctx->stream));
    VX_CUDA(ctx, cudaMemcpyAsync(in + 12 * nn, dirs, 12 * nn, cudaMemcpyHostToDevice, ctx->stream));
    VX_CUDA(ctx, cudaMemcpyAsync(in + 24 * nn, start_slots, 4 * nn, cudaMemcpyHostToDevice, ctx->stream));
    rc = launch_raycast(ctx, b, reinterpret_cast<const float *>(in), reinterpret_cast<const float *>(in + 12 * nn),
                        reinterpret_cast<const int32_t *>(in + 24 * nn), n, max_t, ctx->tmp_b.as<VxRayHit>());
    if (rc != VX_OK) return rc;
    VX_CUDA(ctx, cudaMemcpyAsync(hits_out, ctx->tmp_b.ptr, sizeof(VxRayHit) * nn, cudaMemcpyDeviceToHost, ctx->stream));
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
#ifdef VX_DEBUG_CHECKS
    unsigned int exceeded = 0;
    VX_CUDA(ctx, cudaMemcpyFromSymbol(&exceeded, g_ray_bound_exceeded, sizeof(exceeded)));
    if (exceeded) {
        const unsigned int zero = 0;
        VX_CUDA(ctx, cudaMemcpyToSymbol(g_ray_bound_exceeded, &zero, sizeof(zero)));
        return vx_fail(ctx, VX_ERR_CUDA, "internal step bound exceeded in the ray cast kernel (VX_DEBUG_CHECKS build)");
    }
#endif
    return VX_OK;
}

int vx_world_raycast_device(VxContext *ctx, const VxMeshBatch *b, const float *d_origins, const float *d_dirs, const int32_t *d_start_slots,
                            int32_t n, float max_t, VxRayHit *d_hits_out) {
    int rc = world_batch_ok(ctx, b, "vx_world_raycast_device: bad argument");
    if (rc != VX_OK) return rc;
    if (n < 0 || (n > 0 && (!d_origins || !d_dirs || !d_start_slots || !d_hits_out)))
        return vx_fail(ctx, VX_ERR_INVALID, "vx_world_raycast_device: bad argument");
    if (n == 0) return VX_OK;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    return launch_raycast(ctx, b, d_origins, d_dirs, d_start_slots, n, max_t, d_hits_out);
}

} // extern "C"
