/* CPU oracle of vx_world_batch_copy_region and vx_world_batch_paste (include/vx_b200.h states the semantics;
 * csrc/vx_mesh.cu holds the kernels).  TEST INFRASTRUCTURE: built and loaded by tests/vx_paste_oracle.py with gcc; the
 * product library never links it.  It reads the same slot-indexed world arrays as the region oracle: positions
 * [n_slots][3], voxels [n_slots][32768] (rows of Uniform slots are not read), flags [n_slots] (0 Varied, else 1 + type). */
#include <stdint.h>
#include <string.h>

#define VXO_CHUNK_VOLUME 32768
#define VXO_PASTE_SKIP 0xFF
#define VXO_COORD (1 << 29)
#define VXO_MAX_DIM 1024

typedef struct { /* VxPasteOp */
    int64_t offset;
    int32_t origin[3];
    int32_t dims[3];
    uint8_t replace_mask;
    uint8_t pad[7];
} vxo_paste_op;

/* the box lo .. lo + dims - 1 is valid: every dims[e] in [1, 1024], both corners within [-2^29, 2^29] */
static int box_valid(const int32_t lo[3], const int32_t dims[3]) {
    for (int e = 0; e < 3; ++e) {
        if (dims[e] < 1 || dims[e] > VXO_MAX_DIM) return 0;
        const int64_t hi = (int64_t)lo[e] + dims[e] - 1;
        if (lo[e] < -VXO_COORD || lo[e] > VXO_COORD || hi < -VXO_COORD || hi > VXO_COORD) return 0;
    }
    return 1;
}

/* vx_world_batch_copy_region over the slot-indexed arrays: returns 0, or -1 (VX_ERR_INVALID) before anything is written. */
int vxo_copy_region(const int32_t *positions, const uint8_t *voxels, const uint8_t *flags, int32_t n_slots_total, const int32_t lo[3],
                    const int32_t dims[3], const int32_t *chunk_slots, uint8_t *out) {
    /* invalid arguments */
    if (!box_valid(lo, dims)) return -1;
    int32_t c0[3], n[3];
    for (int e = 0; e < 3; ++e) {
        c0[e] = lo[e] >> 5;
        n[e] = ((lo[e] + dims[e] - 1) >> 5) - c0[e] + 1;
    }
    for (int32_t k = 0; k < n[2]; ++k)
        for (int32_t j = 0; j < n[1]; ++j)
            for (int32_t i = 0; i < n[0]; ++i) {
                const int32_t s = chunk_slots[(k * n[1] + j) * n[0] + i];
                if (s < -1 || s >= n_slots_total) return -1;
                if (s >= 0 && (positions[3 * s] != c0[0] + i || positions[3 * s + 1] != c0[1] + j || positions[3 * s + 2] != c0[2] + k)) return -1;
            }
    /* every voxel of the box, [z][y][x] */
    for (int32_t z = 0; z < dims[2]; ++z)
        for (int32_t y = 0; y < dims[1]; ++y)
            for (int32_t x = 0; x < dims[0]; ++x) {
                const int32_t v[3] = {lo[0] + x, lo[1] + y, lo[2] + z};
                const int32_t s = chunk_slots[(((v[2] >> 5) - c0[2]) * n[1] + ((v[1] >> 5) - c0[1])) * n[0] + ((v[0] >> 5) - c0[0])];
                uint8_t t;
                if (s == -1) t = VXO_PASTE_SKIP;
                else if (flags[s] != 0) t = (uint8_t)(flags[s] - 1);
                else t = voxels[(size_t)s * VXO_CHUNK_VOLUME + (v[2] & 31) * 1024 + (v[1] & 31) * 32 + (v[0] & 31)];
                out[((size_t)z * dims[1] + y) * dims[0] + x] = t;
            }
    return 0;
}

/* vx_world_batch_paste over the slot-indexed arrays: returns 0, or -1 (VX_ERR_INVALID) before anything changes; voxels and
 * flags are updated in place, changed_out (n) receives the change bits of slots[i]. */
int vxo_paste(const int32_t *positions, uint8_t *voxels, uint8_t *flags, int32_t n_slots_total, const vxo_paste_op *ops, int32_t n_ops,
              const uint8_t *templates, int64_t n_template_bytes, const int32_t *slots, int32_t n, uint8_t *changed_out) {
    /* invalid arguments */
    for (int32_t i = 0; i < n; ++i) {
        if (slots[i] < 0 || slots[i] >= n_slots_total) return -1;
        for (int32_t k = 0; k < i; ++k)
            if (slots[k] == slots[i]) return -1;
    }
    for (int32_t i = 0; i < n_ops; ++i) {
        const vxo_paste_op *op = &ops[i];
        if (op->replace_mask > 15) return -1;
        if (!box_valid(op->origin, op->dims)) return -1;
        const int64_t volume = (int64_t)op->dims[0] * op->dims[1] * op->dims[2];
        if (op->offset < 0 || op->offset + volume > n_template_bytes) return -1;
        for (int64_t j = 0; j < volume; ++j) {
            const uint8_t p = templates[op->offset + j];
            if (p > 3 && p != VXO_PASTE_SKIP) return -1;
        }
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
            const vxo_paste_op *op = &ops[k];
            for (int32_t z = 0; z < 32; ++z)
                for (int32_t y = 0; y < 32; ++y)
                    for (int32_t x = 0; x < 32; ++x) {
                        const int64_t v[3] = {(int64_t)positions[3 * s] * 32 + x, (int64_t)positions[3 * s + 1] * 32 + y,
                                              (int64_t)positions[3 * s + 2] * 32 + z};
                        int64_t t[3];
                        int covered = 1;
                        for (int e = 0; e < 3; ++e) {
                            t[e] = v[e] - op->origin[e];
                            if (t[e] < 0 || t[e] >= op->dims[e]) covered = 0;
                        }
                        if (!covered) continue;
                        const uint8_t p = templates[op->offset + (t[2] * op->dims[1] + t[1]) * op->dims[0] + t[0]];
                        uint8_t *c = &cur[z * 1024 + y * 32 + x];
                        if (p == VXO_PASTE_SKIP || !((op->replace_mask >> *c) & 1) || *c == p) continue;
                        *c = p;
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
