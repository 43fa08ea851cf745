// vx_ray.cu -- ray casting through the voxels of a world batch (picking): one thread per ray, an Amanatides-Woo walk from
// voxel to voxel that crosses chunk borders through the batch's neighbour table (no position -> slot lookup).  The exact
// semantics are written down in include/vx_b200.h; the CPU oracle (vxo_raycast) restates them statement for statement.
// Every face crossing is computed in closed form, ((float)plane - o) / d, one correctly rounded subtraction and division
// (compiled with -fmad=false like the other exact files), so the kernel and the oracle produce the same bits.  Nothing
// here touches the frame kernels or their buffers.  The swept-box moves (collision, vx_world_move_boxes) read the same
// arrays with the same neighbour-table hops and are exact in the same way.
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

// ---- swept boxes (vx_world_move_boxes) ------------------------------------------------------------------------------
// One thread per box; the axes are moved one after the other (Y, X, Z), each scanning the voxel layers the box's leading
// face sweeps, nearest first, across the box's cross-section on the other two axes.  Every voxel a move reads lies in the
// 3 x 3 x 3 chunks around the box's slot (the bounds checked on the inputs guarantee it; VX_DEBUG_CHECKS checks it).

constexpr int MOVE_THREADS = 128;
constexpr float MOVE_MAX_POS = 1048576.0f; // 2^20
constexpr float MOVE_MAX_SIZE = 16.0f;
constexpr float MOVE_MAX_DELTA = 16.0f;

#ifdef VX_DEBUG_CHECKS
// set when a move reaches a chunk outside the 3 x 3 x 3 neighbourhood of its slot; read and cleared by vx_world_move_boxes
__device__ unsigned int g_move_bound_exceeded;
#endif

// slot of the chunk at offset (ox, oy, oz) in {-1,0,1}^3 from `slot`: the X hop, then Y, then Z; -1 if a hop finds no chunk
__device__ __forceinline__ int32_t hop_slot(const int32_t *__restrict__ nbr, int32_t slot, int32_t ox, int32_t oy, int32_t oz) {
#ifdef VX_DEBUG_CHECKS
    if ((uint32_t)(ox + 1) > 2u || (uint32_t)(oy + 1) > 2u || (uint32_t)(oz + 1) > 2u) {
        atomicOr(&g_move_bound_exceeded, 1u);
        return -1;
    }
#endif
    if (ox != 0 && (slot = __ldg(nbr + 6 * (size_t)slot + (ox > 0 ? 0 : 1))) < 0) return -1;
    if (oy != 0 && (slot = __ldg(nbr + 6 * (size_t)slot + (oy > 0 ? 2 : 3))) < 0) return -1;
    if (oz != 0 && (slot = __ldg(nbr + 6 * (size_t)slot + (oz > 0 ? 4 : 5))) < 0) return -1;
    return slot;
}

// Layer L (world voxel coordinate on axis A) across voxels lo..hi on the other two axes (E1 < E2, E1 innermost).  Chunks are
// visited E2-major; each one is resolved (an unloaded one makes the layer solid and sets *unloaded), a Uniform one is
// judged by its flag, a Varied one is scanned byte by byte until its first solid voxel -- unless the layer is already
// known to be solid.
template <int A>
__device__ bool layer_solid(const RayWorld &w, int32_t slot, const int32_t (&c)[3], int32_t L, const int32_t (&lo)[3], const int32_t (&hi)[3],
                            bool *unloaded) {
    constexpr int E1 = A == 0 ? 1 : 0, E2 = A == 2 ? 1 : 2;
    constexpr int32_t STRIDE[3] = {1, 32, 1024};
    bool solid = false;
    for (int32_t c2 = lo[E2] >> 5; c2 <= (hi[E2] >> 5); ++c2) {
        for (int32_t c1 = lo[E1] >> 5; c1 <= (hi[E1] >> 5); ++c1) {
            int32_t o[3];
            o[A] = (L >> 5) - c[A];
            o[E1] = c1 - c[E1];
            o[E2] = c2 - c[E2];
            const int32_t s = hop_slot(w.neighbors, slot, o[0], o[1], o[2]);
            if (s < 0) {
                solid = *unloaded = true;
                continue;
            }
            const uint8_t flag = __ldg(w.flags + s);
            if (flag != 0) { // Uniform: no voxel rows, no load
                solid = solid || flag != 1;
                continue;
            }
            if (solid) continue;
            const uint8_t *row = w.voxels + (size_t)s * VX_CHUNK_VOLUME + (L & 31) * STRIDE[A];
            const int32_t a1 = max(lo[E1], c1 * 32), b1 = min(hi[E1], c1 * 32 + 31);
            const int32_t a2 = max(lo[E2], c2 * 32), b2 = min(hi[E2], c2 * 32 + 31);
            for (int32_t v2 = a2; v2 <= b2 && !solid; ++v2)
                for (int32_t v1 = a1; v1 <= b1; ++v1)
                    if (__ldg(row + (v2 & 31) * STRIDE[E2] + (v1 & 31) * STRIDE[E1]) != 0) {
                        solid = true;
                        break;
                    }
        }
    }
    return solid;
}

// f32 values in order as integers (-0 just below +0) and back: the f32 between two others are the keys between theirs
__device__ __forceinline__ int64_t f32_key(float f) {
    const int32_t b = __float_as_int(f);
    return b >= 0 ? (int64_t)b : -(int64_t)(b & 0x7fffffff) - 1;
}
__device__ __forceinline__ float key_f32(int64_t k) { return __int_as_float(k >= 0 ? (int32_t)k : (int32_t)((uint32_t)(-(k + 1)) | 0x80000000u)); }

// Moves the box along axis A by d (the header states the rule); returns the flag bits of this axis.
template <int A>
__device__ uint32_t move_axis(const RayWorld &w, int32_t slot, const int32_t (&c)[3], float (&p)[3], const float (&sz)[3], float d) {
    if (d == 0.0f) return 0;
    constexpr int E1 = A == 0 ? 1 : 0, E2 = A == 2 ? 1 : 2;
    int32_t lo[3], hi[3];
    lo[E1] = (int32_t)floorf(p[E1]);
    hi[E1] = (int32_t)ceilf(p[E1] + sz[E1]) - 1;
    lo[E2] = (int32_t)floorf(p[E2]);
    hi[E2] = (int32_t)ceilf(p[E2] + sz[E2]) - 1;
    const float cand = p[A] + d;
    bool unloaded = false;
    if (d > 0.0f) {
        const int32_t last = (int32_t)ceilf(cand + sz[A]) - 1;
        for (int32_t L = (int32_t)ceilf(p[A] + sz[A]); L <= last; ++L) {
            if (layer_solid<A>(w, slot, c, L, lo, hi, &unloaded)) {
                // the largest f32 m with fl(m + size) <= L, bisected between p_a (fits) and cand (does not): <= 32 steps
                const float top = (float)L;
                int64_t lo = f32_key(p[A]), hi = f32_key(cand);
                while (hi - lo > 1) {
                    const int64_t mid = lo + ((hi - lo) >> 1);
                    if (key_f32(mid) + sz[A] <= top) lo = mid;
                    else hi = mid;
                }
                p[A] = key_f32(lo);
                return (1u << (2 * A)) | (unloaded ? (uint32_t)VX_MOVE_TOUCHED_UNLOADED : 0u);
            }
        }
    } else {
        const int32_t last = (int32_t)floorf(cand);
        for (int32_t L = (int32_t)floorf(p[A]) - 1; L >= last; --L) {
            if (layer_solid<A>(w, slot, c, L, lo, hi, &unloaded)) {
                p[A] = (float)(L + 1);
                return (1u << (2 * A + 1)) | (unloaded ? (uint32_t)VX_MOVE_TOUCHED_UNLOADED : 0u);
            }
        }
    }
    p[A] = cand;
    return 0;
}

__global__ void __launch_bounds__(MOVE_THREADS) move_boxes_kernel(RayWorld w, float *pos, const float *__restrict__ size,
                                                                  const float *__restrict__ delta, int32_t *slots, int32_t n,
                                                                  uint32_t *__restrict__ flags_out) {
    const int32_t i = blockIdx.x * MOVE_THREADS + threadIdx.x;
    if (i >= n) return;
    float p[3], sz[3], d[3];
    for (int k = 0; k < 3; ++k) {
        p[k] = pos[3 * (size_t)i + k];
        sz[k] = size[3 * (size_t)i + k];
        d[k] = delta[3 * (size_t)i + k];
    }
    const int32_t slot = slots[i];
    bool ok = slot >= 0 && slot < w.n_slots;
    for (int k = 0; k < 3; ++k) {
        ok = ok && isfinite(p[k]) && isfinite(sz[k]) && isfinite(d[k]);
        ok = ok && fabsf(p[k]) < MOVE_MAX_POS && sz[k] > 0.0f && sz[k] <= MOVE_MAX_SIZE && fabsf(d[k]) <= MOVE_MAX_DELTA;
        ok = ok && p[k] + sz[k] > p[k];
    }
    int32_t c[3] = {0, 0, 0};
    if (ok) {
        const int32_t *q = w.positions + 3 * (size_t)slot;
        for (int k = 0; k < 3; ++k) {
            c[k] = q[k];
            ok = ok && c[k] == ((int32_t)floorf(p[k]) >> 5);
        }
    }
    if (!ok) {
        flags_out[i] = VX_MOVE_INVALID;
        return;
    }
    uint32_t f = move_axis<1>(w, slot, c, p, sz, d[1]);
    f |= move_axis<0>(w, slot, c, p, sz, d[0]);
    f |= move_axis<2>(w, slot, c, p, sz, d[2]);
    for (int k = 0; k < 3; ++k) pos[3 * (size_t)i + k] = p[k];
    slots[i] = hop_slot(w.neighbors, slot, ((int32_t)floorf(p[0]) >> 5) - c[0], ((int32_t)floorf(p[1]) >> 5) - c[1],
                        ((int32_t)floorf(p[2]) >> 5) - c[2]);
    flags_out[i] = f;
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

int launch_move_boxes(VxContext *ctx, const VxMeshBatch *b, float *d_pos, const float *d_size, const float *d_delta, int32_t *d_slots,
                      int32_t n, uint32_t *d_flags) {
    const RayWorld w{b->world_voxels.as<uint8_t>(), b->world_flags.as<uint8_t>(), b->world_neighbors.as<int32_t>(), b->positions.as<int32_t>(),
                     b->n_chunks};
    move_boxes_kernel<<<(n + MOVE_THREADS - 1) / MOVE_THREADS, MOVE_THREADS, 0, ctx->stream>>>(w, d_pos, d_size, d_delta, d_slots, n, d_flags);
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

int vx_world_move_boxes(VxContext *ctx, const VxMeshBatch *b, float *pos_inout, const float *size, const float *delta, int32_t *slots_inout,
                        int32_t n, uint32_t *flags_out) {
    int rc = world_batch_ok(ctx, b, "vx_world_move_boxes: bad argument");
    if (rc != VX_OK) return rc;
    if (n < 0 || (n > 0 && (!pos_inout || !size || !delta || !slots_inout || !flags_out)))
        return vx_fail(ctx, VX_ERR_INVALID, "vx_world_move_boxes: bad argument");
    for (int32_t i = 0; i < n; ++i)
        if (slots_inout[i] < -1 || slots_inout[i] >= b->n_chunks) return vx_fail(ctx, VX_ERR_INVALID, "vx_world_move_boxes: slot out of range");
    if (n == 0) return VX_OK;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t nn = (size_t)n;
    // inputs staged back to back: pos, size, delta (12 bytes a box each), slots
    VX_CUDA(ctx, ctx->tmp_a.reserve(40 * nn));
    VX_CUDA(ctx, ctx->tmp_b.reserve(4 * nn));
    uint8_t *in = ctx->tmp_a.as<uint8_t>();
    float *d_pos = reinterpret_cast<float *>(in);
    int32_t *d_slots = reinterpret_cast<int32_t *>(in + 36 * nn);
    VX_CUDA(ctx, cudaMemcpyAsync(d_pos, pos_inout, 12 * nn, cudaMemcpyHostToDevice, ctx->stream));
    VX_CUDA(ctx, cudaMemcpyAsync(in + 12 * nn, size, 12 * nn, cudaMemcpyHostToDevice, ctx->stream));
    VX_CUDA(ctx, cudaMemcpyAsync(in + 24 * nn, delta, 12 * nn, cudaMemcpyHostToDevice, ctx->stream));
    VX_CUDA(ctx, cudaMemcpyAsync(d_slots, slots_inout, 4 * nn, cudaMemcpyHostToDevice, ctx->stream));
    rc = launch_move_boxes(ctx, b, d_pos, reinterpret_cast<const float *>(in + 12 * nn), reinterpret_cast<const float *>(in + 24 * nn), d_slots, n,
                           ctx->tmp_b.as<uint32_t>());
    if (rc != VX_OK) return rc;
    VX_CUDA(ctx, cudaMemcpyAsync(pos_inout, d_pos, 12 * nn, cudaMemcpyDeviceToHost, ctx->stream));
    VX_CUDA(ctx, cudaMemcpyAsync(slots_inout, d_slots, 4 * nn, cudaMemcpyDeviceToHost, ctx->stream));
    VX_CUDA(ctx, cudaMemcpyAsync(flags_out, ctx->tmp_b.ptr, 4 * nn, cudaMemcpyDeviceToHost, ctx->stream));
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
#ifdef VX_DEBUG_CHECKS
    unsigned int exceeded = 0;
    VX_CUDA(ctx, cudaMemcpyFromSymbol(&exceeded, g_move_bound_exceeded, sizeof(exceeded)));
    if (exceeded) {
        const unsigned int zero = 0;
        VX_CUDA(ctx, cudaMemcpyToSymbol(g_move_bound_exceeded, &zero, sizeof(zero)));
        return vx_fail(ctx, VX_ERR_CUDA, "a move left the 3 x 3 x 3 chunks around its slot (VX_DEBUG_CHECKS build)");
    }
#endif
    return VX_OK;
}

int vx_world_move_boxes_device(VxContext *ctx, const VxMeshBatch *b, float *d_pos_inout, const float *d_size, const float *d_delta,
                               int32_t *d_slots_inout, int32_t n, uint32_t *d_flags_out) {
    int rc = world_batch_ok(ctx, b, "vx_world_move_boxes_device: bad argument");
    if (rc != VX_OK) return rc;
    if (n < 0 || (n > 0 && (!d_pos_inout || !d_size || !d_delta || !d_slots_inout || !d_flags_out)))
        return vx_fail(ctx, VX_ERR_INVALID, "vx_world_move_boxes_device: bad argument");
    if (n == 0) return VX_OK;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    return launch_move_boxes(ctx, b, d_pos_inout, d_size, d_delta, d_slots_inout, n, d_flags_out);
}

} // extern "C"
