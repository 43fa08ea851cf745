/* CPU oracle of vx_world_batch_fill_regions (include/vx_b200.h states the semantics; csrc/vx_mesh.cu is the kernel).  TEST
 * INFRASTRUCTURE: built and loaded by tests/vx_region_oracle.py with gcc; the product library never links it.  It reads the
 * same slot-indexed world arrays as the ray-cast and move oracles: positions [n_slots][3], voxels [n_slots][32768] (rows of
 * Uniform slots are not read), flags [n_slots] (0 Varied, else 1 + block type). */
#include <stdint.h>
#include <string.h>

#define VXO_CHUNK_VOLUME 32768

typedef struct { /* VxRegionOp */
    int64_t radius_sq;
    int32_t shape;
    int32_t a[3], b[3];
    uint8_t block_type;
    uint8_t replace_mask;
    uint8_t pad[2];
} vxo_region_op;

#define VXO_REGION_BOX 0
#define VXO_REGION_BALL 1
#define VXO_COORD (1 << 29)
#define VXO_RADIUS_SQ ((int64_t)1 << 56)

static int64_t isqrt64(int64_t n) { /* floor(sqrt(n)) for 0 <= n <= 2^56, by bisection */
    int64_t lo = 0, hi = (int64_t)1 << 28;
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) / 2;
        if (mid * mid <= n) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

/* r = isqrt64(radius_sq) for a ball */
static int region_inside(const vxo_region_op *op, int64_t r, const int64_t v[3]) {
    if (op->shape == VXO_REGION_BOX) {
        for (int e = 0; e < 3; ++e)
            if (v[e] < op->a[e] || v[e] > op->b[e]) return 0;
        return 1;
    }
    int64_t sum = 0;
    for (int e = 0; e < 3; ++e) {
        const int64_t d = v[e] - op->a[e];
        if (d < -r || d > r) return 0;
        sum += d * d;
    }
    return sum <= op->radius_sq;
}

/* vx_world_batch_fill_regions over the slot-indexed arrays: returns 0, or -1 (VX_ERR_INVALID) before anything changes;
 * voxels and flags are updated in place, changed_out (n) receives the change bits of slots[i]. */
int vxo_fill_regions(const int32_t *positions, uint8_t *voxels, uint8_t *flags, int32_t n_slots_total, const vxo_region_op *ops, int32_t n_ops,
                     const int32_t *slots, int32_t n, uint8_t *changed_out) {
    /* invalid arguments */
    for (int32_t i = 0; i < n; ++i) {
        if (slots[i] < 0 || slots[i] >= n_slots_total) return -1;
        for (int32_t k = 0; k < i; ++k)
            if (slots[k] == slots[i]) return -1;
    }
    for (int32_t i = 0; i < n_ops; ++i) {
        const vxo_region_op *op = &ops[i];
        if (op->shape != VXO_REGION_BOX && op->shape != VXO_REGION_BALL) return -1;
        if (op->block_type > 3 || op->replace_mask > 15) return -1;
        for (int e = 0; e < 3; ++e) {
            if (op->a[e] < -VXO_COORD || op->a[e] > VXO_COORD) return -1;
            if (op->shape == VXO_REGION_BOX && (op->b[e] < -VXO_COORD || op->b[e] > VXO_COORD)) return -1;
        }
        if (op->shape == VXO_REGION_BALL && (op->radius_sq < 0 || op->radius_sq > VXO_RADIUS_SQ)) return -1;
    }
    static uint8_t before[VXO_CHUNK_VOLUME], cur[VXO_CHUNK_VOLUME];
    for (int32_t i = 0; i < n; ++i) {
        const int32_t s = slots[i];
        uint8_t *row = voxels + (size_t)s * VXO_CHUNK_VOLUME;
        const uint8_t flag = flags[s];
        /* the slot's voxels: its rows, or its Uniform type */
        if (flag != 0) memset(before, flag - 1, VXO_CHUNK_VOLUME);
        else memcpy(before, row, VXO_CHUNK_VOLUME);
        memcpy(cur, before, VXO_CHUNK_VOLUME);
        int varied = flag == 0;
        /* each op in order; a Uniform slot turns Varied at the first op that changes one of its voxels */
        for (int32_t k = 0; k < n_ops; ++k) {
            const vxo_region_op *op = &ops[k];
            const int64_t r = op->shape == VXO_REGION_BALL ? isqrt64(op->radius_sq) : 0;
            for (int32_t z = 0; z < 32; ++z)
                for (int32_t y = 0; y < 32; ++y)
                    for (int32_t x = 0; x < 32; ++x) {
                        const int64_t v[3] = {(int64_t)positions[3 * s] * 32 + x, (int64_t)positions[3 * s + 1] * 32 + y,
                                              (int64_t)positions[3 * s + 2] * 32 + z};
                        uint8_t *t = &cur[z * 1024 + y * 32 + x];
                        if (!region_inside(op, r, v) || !((op->replace_mask >> *t) & 1) || *t == op->block_type) continue;
                        *t = op->block_type;
                        varied = 1;
                    }
        }
        /* change bits: a border plane differs (FaceDir order), the voxels or the flag differ */
        uint8_t bits = 0;
        for (int32_t z = 0; z < 32; ++z)
            for (int32_t y = 0; y < 32; ++y)
                for (int32_t x = 0; x < 32; ++x) {
                    const int32_t j = z * 1024 + y * 32 + x;
                    if (cur[j] == before[j]) continue;
                    bits |= 64;
                    if (x == 31) bits |= 1;
                    if (x == 0) bits |= 2;
                    if (y == 31) bits |= 4;
                    if (y == 0) bits |= 8;
                    if (z == 31) bits |= 16;
                    if (z == 0) bits |= 32;
                }
        if (flag != 0 && varied) {
            bits |= 64;
            flags[s] = 0;
        }
        /* a slot whose flag stays Uniform keeps its rows */
        if (flags[s] == 0) memcpy(row, cur, VXO_CHUNK_VOLUME);
        changed_out[i] = bits;
    }
    return 0;
}
