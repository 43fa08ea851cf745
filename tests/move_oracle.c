/* CPU oracle of vx_world_move_boxes (include/vx_b200.h states the semantics; csrc/vx_ray.cu is the kernel).  TEST
 * INFRASTRUCTURE: built and loaded by tests/vx_move_oracle.py with gcc -ffp-contract=off, so every f32 addition rounds
 * once, as in the kernel (compiled with -fmad=false).  The product library never links it.  It reads the same
 * slot-indexed world arrays as the ray-cast oracle (tests/ray_oracle.c): positions [n_slots][3], voxels [n_slots][32768]
 * (rows of Uniform slots are not read), flags [n_slots] (0 Varied, else 1 + block type), neighbors [n_slots][6]. */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define VXO_CHUNK_VOLUME 32768
/* vx_world_move_boxes, statement for statement over the same slot-indexed arrays (include/vx_b200.h states the rule):
 * pos and slots (n x 3, n) are updated in place, flags_out (n) receives the flag bits, reads_out (n, may be NULL) the voxel
 * bytes each move loaded (Uniform chunks and chunks that are not loaded cost none). */
#define VXO_MOVE_TOUCHED_UNLOADED (1u << 6)
#define VXO_MOVE_INVALID (1u << 7)

static int32_t move_hop_slot(const int32_t *nbr, int32_t slot, int32_t ox, int32_t oy, int32_t oz) {
    if (ox != 0 && (slot = nbr[6 * (size_t)slot + (ox > 0 ? 0 : 1)]) < 0) return -1;
    if (oy != 0 && (slot = nbr[6 * (size_t)slot + (oy > 0 ? 2 : 3)]) < 0) return -1;
    if (oz != 0 && (slot = nbr[6 * (size_t)slot + (oz > 0 ? 4 : 5)]) < 0) return -1;
    return slot;
}

typedef struct {
    const uint8_t *voxels, *flags;
    const int32_t *neighbors;
    int64_t reads;
} vxo_move_world;

static int move_layer_solid(vxo_move_world *w, int a, int32_t slot, const int32_t *c, int32_t L, const int32_t *lo, const int32_t *hi,
                            int *unloaded) {
    static const int32_t STRIDE[3] = {1, 32, 1024};
    const int e1 = a == 0 ? 1 : 0, e2 = a == 2 ? 1 : 2;
    int solid = 0;
    for (int32_t c2 = lo[e2] >> 5; c2 <= (hi[e2] >> 5); ++c2) {
        for (int32_t c1 = lo[e1] >> 5; c1 <= (hi[e1] >> 5); ++c1) {
            int32_t o[3];
            o[a] = (L >> 5) - c[a];
            o[e1] = c1 - c[e1];
            o[e2] = c2 - c[e2];
            const int32_t s = move_hop_slot(w->neighbors, slot, o[0], o[1], o[2]);
            if (s < 0) {
                solid = *unloaded = 1;
                continue;
            }
            const uint8_t flag = w->flags[s];
            if (flag != 0) {
                solid = solid || flag != 1;
                continue;
            }
            if (solid) continue;
            const uint8_t *row = w->voxels + (size_t)s * VXO_CHUNK_VOLUME + (L & 31) * STRIDE[a];
            const int32_t a1 = lo[e1] > c1 * 32 ? lo[e1] : c1 * 32, b1 = hi[e1] < c1 * 32 + 31 ? hi[e1] : c1 * 32 + 31;
            const int32_t a2 = lo[e2] > c2 * 32 ? lo[e2] : c2 * 32, b2 = hi[e2] < c2 * 32 + 31 ? hi[e2] : c2 * 32 + 31;
            for (int32_t v2 = a2; v2 <= b2 && !solid; ++v2)
                for (int32_t v1 = a1; v1 <= b1; ++v1) {
                    ++w->reads;
                    if (row[(v2 & 31) * STRIDE[e2] + (v1 & 31) * STRIDE[e1]] != 0) {
                        solid = 1;
                        break;
                    }
                }
        }
    }
    return solid;
}

static int64_t move_f32_key(float f) {
    int32_t b;
    memcpy(&b, &f, 4);
    return b >= 0 ? (int64_t)b : -(int64_t)(b & 0x7fffffff) - 1;
}

static float move_key_f32(int64_t k) {
    const uint32_t b = k >= 0 ? (uint32_t)k : ((uint32_t)(-(k + 1)) | 0x80000000u);
    float f;
    memcpy(&f, &b, 4);
    return f;
}

static uint32_t move_axis(vxo_move_world *w, int a, int32_t slot, const int32_t *c, float *p, const float *sz, float d) {
    if (d == 0.0f) return 0;
    const int e1 = a == 0 ? 1 : 0, e2 = a == 2 ? 1 : 2;
    int32_t lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
    lo[e1] = (int32_t)floorf(p[e1]);
    hi[e1] = (int32_t)ceilf(p[e1] + sz[e1]) - 1;
    lo[e2] = (int32_t)floorf(p[e2]);
    hi[e2] = (int32_t)ceilf(p[e2] + sz[e2]) - 1;
    const float cand = p[a] + d;
    int unloaded = 0;
    if (d > 0.0f) {
        const int32_t last = (int32_t)ceilf(cand + sz[a]) - 1;
        for (int32_t L = (int32_t)ceilf(p[a] + sz[a]); L <= last; ++L) {
            if (move_layer_solid(w, a, slot, c, L, lo, hi, &unloaded)) {
                const float top = (float)L;
                int64_t lo = move_f32_key(p[a]), hi = move_f32_key(cand);
                while (hi - lo > 1) {
                    const int64_t mid = lo + ((hi - lo) >> 1);
                    if (move_key_f32(mid) + sz[a] <= top) lo = mid;
                    else hi = mid;
                }
                p[a] = move_key_f32(lo);
                return (1u << (2 * a)) | (unloaded ? VXO_MOVE_TOUCHED_UNLOADED : 0u);
            }
        }
    } else {
        const int32_t last = (int32_t)floorf(cand);
        for (int32_t L = (int32_t)floorf(p[a]) - 1; L >= last; --L) {
            if (move_layer_solid(w, a, slot, c, L, lo, hi, &unloaded)) {
                p[a] = (float)(L + 1);
                return (1u << (2 * a + 1)) | (unloaded ? VXO_MOVE_TOUCHED_UNLOADED : 0u);
            }
        }
    }
    p[a] = cand;
    return 0;
}

void vxo_move_boxes(const int32_t *positions, const uint8_t *voxels, const uint8_t *flags, const int32_t *neighbors, int32_t n_slots,
                    float *pos, const float *size, const float *delta, int32_t *slots, int32_t n, uint32_t *flags_out, int64_t *reads_out) {
    for (int32_t i = 0; i < n; ++i) {
        vxo_move_world w = {voxels, flags, neighbors, 0};
        float p[3], sz[3], d[3];
        for (int k = 0; k < 3; ++k) {
            p[k] = pos[3 * (size_t)i + k];
            sz[k] = size[3 * (size_t)i + k];
            d[k] = delta[3 * (size_t)i + k];
        }
        const int32_t slot = slots[i];
        int ok = slot >= 0 && slot < n_slots;
        for (int k = 0; k < 3; ++k) {
            ok = ok && isfinite(p[k]) && isfinite(sz[k]) && isfinite(d[k]);
            ok = ok && fabsf(p[k]) < 1048576.0f && sz[k] > 0.0f && sz[k] <= 16.0f && fabsf(d[k]) <= 16.0f;
            ok = ok && p[k] + sz[k] > p[k];
        }
        int32_t c[3] = {0, 0, 0};
        if (ok) {
            const int32_t *q = positions + 3 * (size_t)slot;
            for (int k = 0; k < 3; ++k) {
                c[k] = q[k];
                ok = ok && c[k] == ((int32_t)floorf(p[k]) >> 5);
            }
        }
        if (!ok) {
            flags_out[i] = VXO_MOVE_INVALID;
        } else {
            uint32_t f = move_axis(&w, 1, slot, c, p, sz, d[1]);
            f |= move_axis(&w, 0, slot, c, p, sz, d[0]);
            f |= move_axis(&w, 2, slot, c, p, sz, d[2]);
            for (int k = 0; k < 3; ++k) pos[3 * (size_t)i + k] = p[k];
            slots[i] = move_hop_slot(neighbors, slot, ((int32_t)floorf(p[0]) >> 5) - c[0], ((int32_t)floorf(p[1]) >> 5) - c[1],
                                     ((int32_t)floorf(p[2]) >> 5) - c[2]);
            flags_out[i] = f;
        }
        if (reads_out) reads_out[i] = w.reads;
    }
}
