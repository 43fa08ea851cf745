/* CPU oracle of vx_world_raycast (include/vx_b200.h states the semantics; csrc/vx_ray.cu is the kernel).  TEST
 * INFRASTRUCTURE: built and loaded by tests/vx_ray_oracle.py with gcc -ffp-contract=off, so every f32 subtraction and
 * division rounds once, as in the kernel (compiled with -fmad=false).  The product library never links it. */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define VXO_CHUNK_VOLUME 32768
#define VXO_RAY_HIT 0
#define VXO_RAY_MISS 1
#define VXO_RAY_LEFT_WORLD 2
#define VXO_RAY_INVALID 3
typedef struct {
    int32_t status, slot, voxel[3], face;
    float t;
    uint8_t block_type, pad[3];
} vxo_ray_hit; /* = VxRayHit */

/* The DDA of vx_world_raycast, statement for statement, over the arrays a world batch holds, indexed by slot:
 * positions [n_slots][3], voxels [n_slots][32768] (rows of Uniform slots are not read), flags [n_slots] (0 Varied, else
 * 1 + block type), neighbors [n_slots][6].  steps_out (n, may be NULL) receives the face crossings each ray took. */
static float ray_next_t(int32_t v, int32_t step, float o, float d) {
    return step == 0 ? INFINITY : ((float)(step > 0 ? v + 1 : v) - o) / d;
}

static int ray_voxel_type(uint8_t flag, const uint8_t *chunk, int32_t lx, int32_t ly, int32_t lz) {
    if (flag != 0) return flag - 1;
    return chunk[lz * 1024 + ly * 32 + lx];
}

void vxo_raycast(const int32_t *positions, const uint8_t *voxels, const uint8_t *flags, const int32_t *neighbors, int32_t n_slots,
                 const float *origins, const float *dirs, const int32_t *start_slots, int32_t n, float max_t, vxo_ray_hit *hits,
                 int32_t *steps_out) {
    for (int32_t i = 0; i < n; ++i) {
        vxo_ray_hit h;
        memset(&h, 0, sizeof(h));
        h.status = VXO_RAY_INVALID;
        h.slot = -1;
        h.face = -1;
        int32_t steps = 0;
        const float ox = origins[3 * i], oy = origins[3 * i + 1], oz = origins[3 * i + 2];
        const float dx = dirs[3 * i], dy = dirs[3 * i + 1], dz = dirs[3 * i + 2];
        int32_t slot = start_slots[i];
        int ok = max_t >= 0.0f && max_t <= 1e4f;
        ok = ok && isfinite(ox) && isfinite(oy) && isfinite(oz) && isfinite(dx) && isfinite(dy) && isfinite(dz);
        ok = ok && fabsf(ox) < 16777216.0f && fabsf(oy) < 16777216.0f && fabsf(oz) < 16777216.0f;
        ok = ok && (dx != 0.0f || dy != 0.0f || dz != 0.0f);
        ok = ok && slot >= 0 && slot < n_slots;
        int32_t vx = 0, vy = 0, vz = 0;
        if (ok) {
            vx = (int32_t)floorf(ox);
            vy = (int32_t)floorf(oy);
            vz = (int32_t)floorf(oz);
            const int32_t *p = positions + 3 * (size_t)slot;
            ok = p[0] == (vx >> 5) && p[1] == (vy >> 5) && p[2] == (vz >> 5);
        }
        if (ok) {
            const int32_t sx = dx > 0.0f ? 1 : (dx < 0.0f ? -1 : 0);
            const int32_t sy = dy > 0.0f ? 1 : (dy < 0.0f ? -1 : 0);
            const int32_t sz = dz > 0.0f ? 1 : (dz < 0.0f ? -1 : 0);
            int32_t lx = vx & 31, ly = vy & 31, lz = vz & 31;
            uint8_t flag = flags[slot];
            const uint8_t *chunk = voxels + (size_t)slot * VXO_CHUNK_VOLUME;
            int type = ray_voxel_type(flag, chunk, lx, ly, lz);
            int face = -1;
            float t = 0.0f;
            float tx = ray_next_t(vx, sx, ox, dx), ty = ray_next_t(vy, sy, oy, dy), tz = ray_next_t(vz, sz, oz, dz);
            h.status = VXO_RAY_MISS;
            while (type == 0) {
                const int axis = (tx <= ty && tx <= tz) ? 0 : (ty <= tz ? 1 : 2); /* smallest tnext, ties x, y, z */
                t = axis == 0 ? tx : (axis == 1 ? ty : tz);
                if (t > max_t) break;
                ++steps;
                const int32_t s = axis == 0 ? sx : (axis == 1 ? sy : sz);
                int32_t l;
                if (axis == 0) {
                    vx += s;
                    l = lx += s;
                    tx = ray_next_t(vx, sx, ox, dx);
                } else if (axis == 1) {
                    vy += s;
                    l = ly += s;
                    ty = ray_next_t(vy, sy, oy, dy);
                } else {
                    vz += s;
                    l = lz += s;
                    tz = ray_next_t(vz, sz, oz, dz);
                }
                face = 2 * axis + (s > 0 ? 1 : 0);
                if ((uint32_t)l > 31u) {
                    const int32_t nb = neighbors[6 * (size_t)slot + 2 * axis + (s > 0 ? 0 : 1)];
                    if (nb < 0) {
                        h.status = VXO_RAY_LEFT_WORLD;
                        break;
                    }
                    slot = nb;
                    lx &= 31;
                    ly &= 31;
                    lz &= 31;
                    flag = flags[slot];
                    chunk = voxels + (size_t)slot * VXO_CHUNK_VOLUME;
                }
                type = ray_voxel_type(flag, chunk, lx, ly, lz);
            }
            if (type != 0) {
                h.status = VXO_RAY_HIT;
                h.slot = slot;
                h.voxel[0] = vx;
                h.voxel[1] = vy;
                h.voxel[2] = vz;
                h.face = face;
                h.t = t;
                h.block_type = (uint8_t)type;
            }
        }
        hits[i] = h;
        if (steps_out) steps_out[i] = steps;
    }
}
