// vx_mesh.cu -- binary greedy meshing of 32^3 chunks on sm_100a.
//
// Reference semantics: /root/reference/src/meshing/binary_greedy.rs:83-121 (mesh_chunk_in_world),
// :213-264 (mesh_face), :286-440 (generate_binary_masks), :683-807 (greedy_mesh_slice_into) and
// mesh.rs:283-307 (TinyQuad::new), :369-397 (FaceList::add_quad), :489-523 (ChunkMesh::add_quad).
//
// Design (one CTA per chunk, persistent over the batch):
//   stage 1  every thread streams 32-voxel x-rows with two 128-bit loads and SWAR-packs the two
//            block-type bits of each voxel into two 32-bit words (bits along x) -> 2 x 32 x 32
//            word bit-planes P[y][z] in shared memory (8 KB instead of the 32 KB byte volume).
//            Neighbour chunks contribute six 32x32-bit solid halo planes, transposed on load.
//   stage 2  128 warp-level 32x32 bit transposes (5 shuffle steps) give the two other orientations
//            once per chunk: T[x][y] (bits z) and R[z][x] (bits y), plus slice-occupancy masks.
//   stage 3  a warp owns one (face, slice) unit; its rows in the reference orientation (lane = row,
//            bit = column) are plain loads from T / R, exposure is word logic (A_t & ~S_neighbour).
//            The greedy merge runs with the row words in registers, one iteration per quad: lowest
//            non-empty row by ballot, run mask by carry propagation, row extension with ONE
//            __ballot_sync over all rows below, consumed bits cleared lane-parallel.
//   output   quads are staged per warp and pooled in shared memory; a CTA scan over the 192 unit
//            counts + one atomicAdd on the batch cursor fix the positions and the pool is copied out
//            in exact reference order (face, slice, block type, row, column) as 3-byte TinyQuads.
//            Chunks with more quads than the pool holds re-run the merge and write directly.
#include "vx_common.cuh"

#include <cstddef>
#include <memory>
#include <unordered_set>
#include <vector>

namespace {

#ifndef VX_MESH_MIN_BLOCKS
#define VX_MESH_MIN_BLOCKS 5
#endif
constexpr int MESH_THREADS = 256;
constexpr int MESH_WARPS = MESH_THREADS / 32;
constexpr int PS = 33; // padded row stride of the 32x32 word planes (bank-conflict free both ways)
constexpr int STAGE_CAP = 128;          // quads one (face, slice) unit may stage per warp on the fast path
constexpr int POOL_CAP = 2 * 32 * PS;   // quads of a chunk kept in shared memory on the fast path (aliases P0/P1)
constexpr unsigned FULL = 0xffffffffu;
constexpr int SLICE_ROW = 6 * 33; // slice_offsets per chunk: 32 slice starts + the end, for each face
constexpr int AABB_ROW = 36;      // face_aabb per chunk: min.xyz, max.xyz for each face

// VxMeshBatch::cursor.  The mesh kernel takes quads from `quads`, counts non-empty meshes in `meshes`, sets `overflow` when
// the quad stream is too small and hands out chunks beyond the first wave from `work`.
struct MeshCursor {
    unsigned long long quads, meshes, overflow, work;
};

struct MeshSmem {
    // stage 1: [y*PS + z], bit x = block-type bit 0 / 1.  After stage 2 the space is the chunk's quad pool.
    union {
        struct { uint32_t P0[32 * PS], P1[32 * PS]; } p;
        uint32_t pool[POOL_CAP];
    } u;
    uint32_t T0[32 * PS], T1[32 * PS]; // [x*PS + y], bits z: rows of the +-X units (lane = y) and +-Y units (lane = x)
    uint32_t R0[32 * PS], R1[32 * PS]; // [z*PS + x], bits y: rows of the +-Z units (lane = x)
    uint32_t halo[6][32];              // neighbour solid planes in unit orientation, see load_halos()
    uint32_t stage[MESH_WARPS][STAGE_CAP];
    uint32_t cnt[192];                 // quads per (face, slice)
    uint32_t offs[192];                // exclusive offsets inside the chunk
    uint32_t pstart[192];              // start of the unit's quads in the pool (fast path)
    uint16_t omap[POOL_CAP];           // final position inside the chunk -> pool position (fast path)
    uint32_t faceTot[6], faceBase[6];
    uint32_t faceRows[6], faceCols[6], faceSlices[6];
    uint32_t occ[3]; // bit s: slice s along x / y / z holds a solid voxel
    uint32_t base, total, overflow, pool_used, slow;
    int32_t next_oi; // the chunk this CTA meshes next (fetched from the batch's work counter while the current one is in flight)
};

// 4 voxels (one per byte, values 0..3) -> 4 bits, voxel k -> bit k.  bit = 0 or 1 selects the type bit.
__device__ __forceinline__ uint32_t gather4(uint32_t w, int bit) {
    return (((w >> bit) & 0x01010101u) * 0x01020408u) >> 24;
}

__device__ __forceinline__ void pack_row(const uint4 a, const uint4 b, uint32_t &p0, uint32_t &p1) {
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    p0 = 0;
    p1 = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        p0 |= gather4(w[j], 0) << (4 * j);
        p1 |= gather4(w[j], 1) << (4 * j);
    }
}

__device__ __forceinline__ uint4 ld_stream(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// 32x32 bit-matrix transpose across a warp: in: lane i holds row i (bit j = column j);
// out: lane j holds column j (bit i = row i).
__device__ __forceinline__ uint32_t transpose32(uint32_t x, int lane) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const uint32_t m = s == 16 ? 0x0000ffffu : s == 8 ? 0x00ff00ffu : s == 4 ? 0x0f0f0f0fu : s == 2 ? 0x33333333u : 0x55555555u;
        const uint32_t y = __shfl_xor_sync(FULL, x, s);
        x = (lane & s) ? ((x & ~m) | ((y >> s) & m)) : ((x & m) | ((y << s) & ~m));
    }
    return x;
}

// TinyQuad::new (mesh.rs:283-307) as the three bytes b0 | b1 << 8 | b2 << 16.  b0 = u | (v & 7) << 5,
// b1 = v >> 3 | (w - 1) << 2, b2 = (h - 1) | type << 6: the two pieces of v are adjacent, so the 24-bit value is
// simply u | v << 5 | (w - 1) << 10 | (h - 1) << 16 | type << 22.
__device__ __forceinline__ uint32_t pack_tinyquad(uint32_t u, uint32_t v, uint32_t w, uint32_t h, uint32_t type) {
    return u | (v << 5) | ((w - 1u) << 10) | ((h - 1u) << 16) | (type << 22);
}

// Greedy merge of one 32x32 mask (binary_greedy.rs:683-807).  Lane = row, d = that row's bits.  Returns the quad count.
// One loop iteration per quad: the lowest row that still has bits is the reference's current row (rows are visited in
// ascending order and a row is left only when it is empty), its lowest set bit starts the next run.
//   MODE 0: count only.
//   MODE 1: write TinyQuads (mesh.rs:283-307) of block type `type` to out[3*(pos + k)]; if out4 != nullptr write
//           VxQuad {row, col, width, height} instead.
//   MODE 2: write packed TinyQuads (u32) to stage[pos + k] while pos + k < STAGE_CAP (keeps counting beyond).
template <int MODE>
__device__ __forceinline__ uint32_t greedy_warp(uint32_t d, int lane, uint32_t type, uint8_t *out, uint32_t pos,
                                                VxQuad *out4, uint32_t *stage) {
    uint32_t n = 0;
    for (;;) {
        const uint32_t rows = __ballot_sync(FULL, d != 0);
        if (!rows) break;
        const int r = __clz(__brev(rows)); // lowest row with bits (rows != 0)
        const uint32_t cur = __shfl_sync(FULL, d, r);
        const int col = __clz(__brev(cur));
        // the run of ones that starts at the lowest set bit: adding that bit carries through the run
        const uint32_t m = cur & ~(cur + (cur & (0u - cur)));
        const int h = __popc(m); // trailing_ones of (cur >> col)
        // rows below that still hold the whole run
        const uint32_t ok = __ballot_sync(FULL, lane > r && (d & m) == m);
        const uint32_t below = r == 31 ? 0u : (ok >> (r + 1));
        const int ext = __clz(__brev(~below)); // consecutive rows r+1.. (bits >= 31-r of ~below are 1 -> ext <= 31-r)
        if ((uint32_t)(lane - r) <= (uint32_t)ext) d &= ~m;
        const uint32_t w = 1u + (uint32_t)ext;
        if (MODE == 1) {
            if (out4) {
                if (lane == 0) out4[pos + n] = VxQuad{(uint8_t)r, (uint8_t)col, (uint8_t)w, (uint8_t)h};
            } else {
                const uint32_t packed = pack_tinyquad((uint32_t)r, (uint32_t)col, w, (uint32_t)h, type);
                if (lane < 3) out[3 * (size_t)(pos + n) + lane] = (uint8_t)(packed >> (8 * lane));
            }
        } else if (MODE == 2) {
            if (lane == 0 && pos + n < (uint32_t)STAGE_CAP) stage[pos + n] = pack_tinyquad((uint32_t)r, (uint32_t)col, w, (uint32_t)h, type);
        }
        n++;
    }
    return n;
}

struct ChunkArgs {
    const uint8_t *voxels;
    const int32_t *neighbors;
    const uint8_t *uniform_flags;
    int32_t n_chunks;       // chunks in the voxel / neighbour arrays (what neighbour indices refer to)
    const int32_t *subset;  // chunk ids to mesh (a shard of the world), or null = all n_chunks
    int32_t n_out;          // chunks meshed
    int32_t out_by_chunk;   // 1: per-chunk outputs are written at the chunk's own index (in-place update of a batch)
    uint8_t *quads;
    unsigned long long cap_quads;
    uint32_t *quad_base, *quad_count, *slice_offsets;
    int32_t *face_aabb;
    uint8_t *has_mesh;
    MeshCursor *cursor;
};

// Neighbour solid planes.  First in load order: f=0/1 (+X/-X): i = y, bit z;  f=2/3 (+Y/-Y): i = z, bit x;
// f=4/5 (+Z/-Z): i = y, bit x.  transpose_halos() then brings f = 2..5 into unit orientation:
// f=2/3: i = x, bit z;  f=4/5: i = x, bit y  (f = 0/1 already are: i = y, bit z).
__device__ void load_halos(MeshSmem &sm, const ChunkArgs &a, int chunk, int tid) {
    const int lane = tid & 31, warp = tid >> 5;
    // resolve the six neighbours (warp-uniform values, computed redundantly)
    const uint8_t *nbp[6];
    uint32_t fill[6];
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        const int32_t nb = a.neighbors ? a.neighbors[(size_t)chunk * 6 + f] : VX_NBR_NONE;
        nbp[f] = nullptr;
        fill[f] = 0;
        if (nb >= 0 && nb < a.n_chunks) {
            const uint8_t uf = a.uniform_flags ? a.uniform_flags[nb] : 0;
            if (uf) fill[f] = (uf - 1) != 0 ? FULL : 0u; // Uniform neighbour: is_solid (binary_greedy.rs:305-313)
            else nbp[f] = a.voxels + (size_t)nb * VX_CHUNK_VOLUME;
        } else if (nb == VX_NBR_UNIFORM_SOLID) fill[f] = FULL;
    }
    // +-X: one byte per (y,z): warp task (f, y), lane = z, ballot -> word with bit z
    for (int t = warp; t < 64; t += MESH_WARPS) {
        const int f = t >> 5, y = t & 31;
        uint32_t word = fill[f];
        if (nbp[f]) {
            const uint8_t v = nbp[f][lane * 1024 + y * 32 + (f == 0 ? 0 : 31)];
            word = __ballot_sync(FULL, v != 0);
        }
        if (lane == 0) sm.halo[f][y] = word;
    }
    // +-Y, +-Z: one 32-byte x-row per entry, SWAR packed: thread task (f, i)
    if (tid < 128) {
        const int f = 2 + (tid >> 5), i = tid & 31;
        uint32_t word = fill[f];
        if (nbp[f]) {
            size_t off;
            if (f == 2) off = (size_t)i * 1024;                 // +Y neighbour: row y=0 of plane z=i
            else if (f == 3) off = (size_t)i * 1024 + 31 * 32;  // -Y neighbour: row y=31
            else if (f == 4) off = (size_t)i * 32;              // +Z neighbour: plane z=0, row y=i
            else off = (size_t)31 * 1024 + (size_t)i * 32;      // -Z neighbour: plane z=31
            const uint4 *p = reinterpret_cast<const uint4 *>(nbp[f] + off);
            uint32_t p0, p1;
            pack_row(__ldg(p), __ldg(p + 1), p0, p1);
            word = p0 | p1;
        }
        // (i, bit x) -> (x, bit i): warps 0..3 hold exactly the four planes f = 2..5
        sm.halo[f][lane] = transpose32(word, lane);
    }
}

// exposure words of the three block types of a row against the neighbour row's solid word
__device__ __forceinline__ void exposure(uint32_t a0, uint32_t a1, uint32_t nbS, uint32_t e[3]) {
    const uint32_t open = ~nbS;
    e[0] = a0 & ~a1 & open; // Grass = 1
    e[1] = a1 & ~a0 & open; // Dirt  = 2
    e[2] = a0 & a1 & open;  // Stone = 3
}

// Row words (lane = row, bits = column) of unit (face, slice) for the three block types, straight from the
// pre-transposed planes: axis 0 (X): rows y, cols z;  axis 1 (Y): rows x, cols z;  axis 2 (Z): rows x, cols y
// (binary_greedy.rs:446-458).
__device__ __forceinline__ void unit_rows(const MeshSmem &sm, int face, int slice, int lane, uint32_t d[3]) {
    const int axis = face >> 1;
    const int ns = (face & 1) == 0 ? slice + 1 : slice - 1; // the neighbour slice along the face normal
    const bool inside = ns >= 0 && ns < 32;
    uint32_t a0, a1, nbS;
    if (axis == 0) { // T[x][y], lane = y
        a0 = sm.T0[slice * PS + lane];
        a1 = sm.T1[slice * PS + lane];
        nbS = inside ? (sm.T0[ns * PS + lane] | sm.T1[ns * PS + lane]) : sm.halo[face][lane];
    } else if (axis == 1) { // T[x][y], lane = x
        a0 = sm.T0[lane * PS + slice];
        a1 = sm.T1[lane * PS + slice];
        nbS = inside ? (sm.T0[lane * PS + ns] | sm.T1[lane * PS + ns]) : sm.halo[face][lane];
    } else { // R[z][x], lane = x
        a0 = sm.R0[slice * PS + lane];
        a1 = sm.R1[slice * PS + lane];
        nbS = inside ? (sm.R0[ns * PS + lane] | sm.R1[ns * PS + lane]) : sm.halo[face][lane];
    }
    exposure(a0, a1, nbS, d);
}

// Pass over the 192 (face, slice) units of the chunk, one warp per unit.
//   MODE 2 (fast path): count, and stage / pool the quads in shared memory;  MODE 1 (slow path): re-run the merge and
//   write the quads to their final place (only for chunks whose quads did not fit the pool).
template <int MODE>
__device__ __forceinline__ void process_units(MeshSmem &sm, const ChunkArgs &a, int tid) {
    const int lane = tid & 31, warp = tid >> 5;
    // FaceList AABB inputs, accumulated per warp and flushed when the warp moves on to the next face (its units
    // unit = warp + 8k visit the faces in order, four slices each)
    uint32_t accRows = 0, accCols = 0, accSlices = 0;
    int accFace = 0;
    for (int unit = warp; unit < 192; unit += MESH_WARPS) {
        const int face = unit >> 5, slice = unit & 31;
        if (MODE == 2 && face != accFace) {
            if (lane == 0 && accSlices) {
                atomicOr(&sm.faceRows[accFace], accRows);
                atomicOr(&sm.faceCols[accFace], accCols);
                atomicOr(&sm.faceSlices[accFace], accSlices);
            }
            accRows = accCols = accSlices = 0;
            accFace = face;
        }
        if (MODE == 2) {
            // a slice without a solid voxel has no faces: skip it without touching the planes
            if (!((sm.occ[face >> 1] >> slice) & 1u)) {
                if (lane == 0) sm.cnt[unit] = 0;
                continue;
            }
        }
        uint32_t d[3];
        unit_rows(sm, face, slice, lane, d);
        if (MODE == 2) {
            uint32_t n = 0, colsAny = 0;
            const uint32_t rowsAny = __ballot_sync(FULL, (d[0] | d[1] | d[2]) != 0);
            if (rowsAny) {
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    colsAny |= d[t];
                    n += greedy_warp<2>(d[t], lane, (uint32_t)(t + 1), nullptr, n, nullptr, sm.stage[warp]);
                }
                colsAny = __reduce_or_sync(FULL, colsAny);
            }
            uint32_t start = 0;
            if (lane == 0) {
                sm.cnt[unit] = n;
                if (n) {
                    start = atomicAdd(&sm.pool_used, n);
                    sm.pstart[unit] = start;
                    if (n > (uint32_t)STAGE_CAP || start + n > (uint32_t)POOL_CAP) sm.slow = 1u;
                }
            }
            if (n) {
                accRows |= rowsAny;
                accCols |= colsAny;
                accSlices |= 1u << slice;
                start = __shfl_sync(FULL, start, 0);
                __syncwarp();
                if (n <= (uint32_t)STAGE_CAP && start + n <= (uint32_t)POOL_CAP)
                    for (uint32_t i = lane; i < n; i += 32) sm.u.pool[start + i] = sm.stage[warp][i];
                __syncwarp();
            }
        } else {
            if (sm.cnt[unit] == 0) continue;
            uint32_t pos = sm.base + sm.offs[unit];
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                if (__any_sync(FULL, d[t] != 0)) pos += greedy_warp<1>(d[t], lane, (uint32_t)(t + 1), a.quads, pos, nullptr, nullptr);
            }
        }
    }
    if (MODE == 2 && lane == 0 && accSlices) {
        atomicOr(&sm.faceRows[accFace], accRows);
        atomicOr(&sm.faceCols[accFace], accCols);
        atomicOr(&sm.faceSlices[accFace], accSlices);
    }
}

__global__ void __launch_bounds__(MESH_THREADS, VX_MESH_MIN_BLOCKS) mesh_chunks_kernel(ChunkArgs a) {
    __shared__ MeshSmem sm;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // Chunks are handed out dynamically: every CTA starts with chunk blockIdx.x and draws the following ones from a counter, so
    // a CTA that got a light chunk (a few dozen quads) takes over work a static stride would have left to a CTA still busy
    // with a heavy one (over a thousand).  The world sweep is ~1.1 resident waves of chunks: the second "wave" used to double
    // its duration.  The draw is issued at the start of a chunk and read at its end (latency hidden behind the chunk).
    int oi = blockIdx.x;
    while (oi < a.n_out) {
        __syncthreads(); // everybody is done with the previous chunk and has read next_oi
        if (tid == 0) sm.next_oi = (int32_t)gridDim.x + (int32_t)atomicAdd(&a.cursor->work, 1ull);
        do {
        const int chunk = a.subset ? a.subset[oi] : oi; // input chunk
        const int oo = a.out_by_chunk ? chunk : oi;     // where its outputs go
        uint32_t *so = a.slice_offsets + (size_t)oo * SLICE_ROW;
        int32_t *ab = a.face_aabb + (size_t)oo * AABB_ROW;
        if (a.uniform_flags && a.uniform_flags[chunk]) { // Uniform chunk -> None (binary_greedy.rs:87)
            for (int i = tid; i < SLICE_ROW; i += MESH_THREADS) so[i] = 0;
            if (tid < AABB_ROW) ab[tid] = (tid % 6) < 3 ? 32 : 0;
            if (tid == 0) {
                a.quad_base[oo] = 0;
                a.quad_count[oo] = 0;
                a.has_mesh[oo] = 0;
            }
            break;
        }
        // ---- stage 1: byte volume -> bit planes P[y][z] (bits x)
        const uint4 *src = reinterpret_cast<const uint4 *>(a.voxels + (size_t)chunk * VX_CHUNK_VOLUME);
        uint4 ra[4], rb[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { // issue all loads first (8 x 128-bit in flight per thread)
            const int r = tid + k * MESH_THREADS;
            ra[k] = ld_stream(src + 2 * r);
            rb[k] = ld_stream(src + 2 * r + 1);
        }
        __syncthreads(); // the previous chunk's pool (aliases P0/P1) and counters are no longer read
        if (tid < 18) (&sm.faceRows[0])[tid] = 0; // faceRows, faceCols, faceSlices are contiguous
        if (tid == 0) {
            sm.pool_used = 0;
            sm.slow = 0;
            sm.occ[0] = sm.occ[1] = sm.occ[2] = 0;
        }
        load_halos(sm, a, chunk, tid);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = tid + k * MESH_THREADS; // r = z*32 + y
            uint32_t p0, p1;
            pack_row(ra[k], rb[k], p0, p1);
            const int y = r & 31, z = r >> 5;
            sm.u.p.P0[y * PS + z] = p0;
            sm.u.p.P1[y * PS + z] = p1;
        }
        __syncthreads();

        // ---- stage 2: the two other orientations of the type planes, 128 warp transposes (empty ones skipped)
        //      T[x][y] bits z  <-  for every y: rows z of P (bits x), transposed
        //      R[z][x] bits y  <-  for every z: rows y of P (bits x), transposed
        for (int item = warp; item < 128; item += MESH_WARPS) {
            const int which = item >> 6, plane = (item >> 5) & 1, s = item & 31;
            const uint32_t *P = plane ? sm.u.p.P1 : sm.u.p.P0;
            if (which == 0) { // s = y, lane = z
                uint32_t w = P[s * PS + lane];
                const uint32_t xs = __reduce_or_sync(FULL, w); // x columns present in slice y
                if (xs) {
                    w = transpose32(w, lane);
                    if (lane == 0) {
                        atomicOr(&sm.occ[1], 1u << s);
                        atomicOr(&sm.occ[0], xs);
                    }
                }
                (plane ? sm.T1 : sm.T0)[lane * PS + s] = w; // lane = x
            } else { // s = z, lane = y
                uint32_t w = P[lane * PS + s];
                if (__any_sync(FULL, w != 0)) {
                    w = transpose32(w, lane);
                    if (lane == 0) atomicOr(&sm.occ[2], 1u << s);
                }
                (plane ? sm.R1 : sm.R0)[s * PS + lane] = w; // lane = x
            }
        }
        __syncthreads();

        // ---- stage 3: greedy merge of every (face, slice) unit; quads go to the shared-memory pool
        process_units<2>(sm, a, tid);
        __syncthreads();
        if (tid < 6) {
            uint32_t run = 0;
            for (int s = 0; s < 32; ++s) {
                sm.offs[tid * 32 + s] = run;
                run += sm.cnt[tid * 32 + s];
            }
            sm.faceTot[tid] = run;
        }
        __syncthreads();
        if (tid == 0) {
            uint32_t run = 0;
            for (int f = 0; f < 6; ++f) {
                sm.faceBase[f] = run;
                run += sm.faceTot[f];
            }
            sm.total = run;
            unsigned long long base = 0;
            if (run) {
                base = atomicAdd(&a.cursor->quads, (unsigned long long)run);
                atomicAdd(&a.cursor->meshes, 1ull);
            }
            sm.overflow = (base + run > a.cap_quads) ? 1u : 0u;
            if (sm.overflow) atomicExch(&a.cursor->overflow, 1ull);
            sm.base = (uint32_t)base;
            a.quad_base[oo] = (uint32_t)base;
            a.quad_count[oo] = run;
            a.has_mesh[oo] = run ? 1 : 0; // mesh.is_empty() -> None (binary_greedy.rs:116-120)
        }
        __syncthreads();
        if (tid < 192) {
            const int f = tid >> 5;
            const uint32_t o = sm.offs[tid] + sm.faceBase[f];
            sm.offs[tid] = o;
            so[f * 33 + (tid & 31)] = o;
        }
        if (tid < 6) so[tid * 33 + 32] = sm.faceBase[tid] + sm.faceTot[tid];
        if (tid < 6) { // FaceList::min / max (mesh.rs:369-397) from the occupancy of the exposure masks
            const uint32_t rows = sm.faceRows[tid], cols = sm.faceCols[tid], sl = sm.faceSlices[tid];
            int mn[3] = {32, 32, 32}, mx[3] = {0, 0, 0};
            if (sl) {
                const int axis = tid >> 1, add = (tid & 1) ? 0 : 1; // axis_pos = slice + 1 for positive faces
                const int s0 = __ffs(sl) - 1 + add, s1 = 31 - __clz(sl) + add;
                const int u0 = __ffs(rows) - 1, u1 = 32 - __clz(rows);
                const int v0 = __ffs(cols) - 1, v1 = 32 - __clz(cols);
                if (axis == 0) { mn[0] = s0; mx[0] = s1; mn[1] = u0; mx[1] = u1; mn[2] = v0; mx[2] = v1; }
                else if (axis == 1) { mn[0] = u0; mx[0] = u1; mn[1] = s0; mx[1] = s1; mn[2] = v0; mx[2] = v1; }
                else { mn[0] = u0; mx[0] = u1; mn[1] = v0; mx[1] = v1; mn[2] = s0; mx[2] = s1; }
            }
            for (int k = 0; k < 3; ++k) {
                ab[tid * 6 + k] = mn[k];
                ab[tid * 6 + 3 + k] = mx[k];
            }
        }
        __syncthreads();
        // ---- output in reference order (face, slice, block type, row, column)
        if (sm.total && !sm.overflow) {
            if (!sm.slow) { // pool -> quad stream: one thread per unit lays out the order map, then one thread per quad
                if (tid < 192) {
                    const uint32_t n = sm.cnt[tid], o = sm.offs[tid], ps = sm.pstart[tid];
                    for (uint32_t k = 0; k < n; ++k) sm.omap[o + k] = (uint16_t)(ps + k);
                }
                __syncthreads();
                uint8_t *dst = a.quads + 3 * (size_t)sm.base;
                for (uint32_t t = tid; t < sm.total; t += MESH_THREADS) {
                    const uint32_t q = sm.u.pool[sm.omap[t]];
                    dst[3 * t] = (uint8_t)q;
                    dst[3 * t + 1] = (uint8_t)(q >> 8);
                    dst[3 * t + 2] = (uint8_t)(q >> 16);
                }
            } else {
                process_units<1>(sm, a, tid); // rare: more quads than the pool holds
            }
        }
        } while (0);
        __syncthreads();
        oi = sm.next_oi;
    }
}

// KAT surface: one warp per 32-row mask.
__global__ void greedy_slices_kernel(const uint32_t *masks, int n, VxQuad *out, int32_t *n_out) {
    const int lane = threadIdx.x & 31;
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= n) return;
    const uint32_t d = masks[(size_t)w * 32 + lane];
    const uint32_t c = greedy_warp<1>(d, lane, 0, nullptr, 0, out + (size_t)w * 512, nullptr);
    if (lane == 0) n_out[w] = (int32_t)c;
}

// The per-chunk arrays of a batch: bytes per chunk, and the byte that marks an absent chunk of a world batch.  Every batch
// has the first MESH_ARRAYS; a batch that owns its world copy (vx_mesh_chunks, vx_world_batch_create) has all of them.
struct ChunkArray {
    VxDeviceBuffer VxMeshBatch::*buf;
    size_t row_bytes;
    int absent;
};
constexpr ChunkArray CHUNK_ARRAYS[] = {
    {&VxMeshBatch::quad_base, sizeof(uint32_t), 0},
    {&VxMeshBatch::quad_count, sizeof(uint32_t), 0},
    {&VxMeshBatch::slice_offsets, sizeof(uint32_t) * SLICE_ROW, 0},
    {&VxMeshBatch::face_aabb, sizeof(int32_t) * AABB_ROW, 0},
    {&VxMeshBatch::has_mesh, 1, 0},
    {&VxMeshBatch::positions, sizeof(int32_t) * 3, 0},
    {&VxMeshBatch::world_voxels, VX_CHUNK_VOLUME, 0},
    {&VxMeshBatch::world_neighbors, sizeof(int32_t) * 6, 0xFF}, // VX_NBR_NONE
    {&VxMeshBatch::world_flags, 1, 1},                          // "uniform air"
};
constexpr int MESH_ARRAYS = 6, ALL_ARRAYS = sizeof(CHUNK_ARRAYS) / sizeof(CHUNK_ARRAYS[0]);

struct BatchRelease {
    VxContext *ctx;
    void operator()(VxMeshBatch *b) const { vx_mesh_batch_release(ctx, b); }
};
// a batch under construction: released on every failure exit, handed to the caller with release()
using BatchPtr = std::unique_ptr<VxMeshBatch, BatchRelease>;

// quad stream of a batch that is about to be meshed: a typical terrain chunk has ~200 quads (binary_greedy.rs:91), so start
// with 512 per chunk and regrow on demand
int64_t first_cap_quads(int32_t n) { return (int64_t)(n > 0 ? n : 1) * 512; }

// A new batch of n chunks with the first `arrays` of CHUNK_ARRAYS, the cursor and room for cap_quads quads.
int new_batch(VxContext *ctx, int32_t n, int64_t cap_quads, int arrays, BatchPtr &b) {
    b = BatchPtr(new VxMeshBatch(), BatchRelease{ctx});
    b->n_chunks = n;
    for (int k = 0; k < arrays; ++k) VX_CUDA(ctx, (b.get()->*CHUNK_ARRAYS[k].buf).reserve(CHUNK_ARRAYS[k].row_bytes * (size_t)n));
    VX_CUDA(ctx, b->cursor.reserve(sizeof(MeshCursor)));
    VX_CUDA(ctx, b->quads.reserve(3 * (size_t)cap_quads + 16));
    b->cap_quads = cap_quads;
    return VX_OK;
}

int read_cursor(VxContext *ctx, const VxMeshBatch *b, MeshCursor &h) {
    VX_CUDA(ctx, cudaMemcpyAsync(&h, b->cursor.ptr, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VX_OK;
}

// also waits for everything enqueued before it (h and the caller's host arrays may go out of scope)
int write_cursor(VxContext *ctx, VxMeshBatch *b, const MeshCursor &h) {
    VX_CUDA(ctx, cudaMemcpyAsync(b->cursor.ptr, &h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VX_OK;
}

// What the mesher reads: the voxels of n_chunks chunks, their neighbour rows (null: all VX_NBR_NONE) and Uniform flags
// (null: all Varied).  Neighbour indices refer to these n_chunks.
struct MeshInput {
    const uint8_t *voxels;
    const int32_t *neighbors;
    const uint8_t *uniform_flags;
    int32_t n_chunks;
};

MeshInput world_input(const VxMeshBatch *b) {
    return {b->world_voxels.as<uint8_t>(), b->has_neighbors ? b->world_neighbors.as<int32_t>() : nullptr, b->world_flags.as<uint8_t>(),
            b->n_chunks};
}

enum class MeshMode {
    EveryRowRegrow, // every row; the cursor is read back, and an overflowed quad stream is grown to the exact need and meshed again
    EveryRowSteady, // every row, no read-back: an overflow is reported by the next vx_mesh_batch_info
    AppendListed,   // the listed chunks at their own rows, quads appended behind the stream's end (their old quads become dead space)
};

// Every-row modes: row i of the batch is chunk rows[i] of `in` (chunk i when rows is null), n_rows == b->n_chunks.
// AppendListed: rows lists the n_rows chunks to re-mesh.
int run_mesher(VxContext *ctx, VxMeshBatch *b, const MeshInput &in, MeshMode mode, const int32_t *rows, int32_t n_rows) {
    const bool listed = mode == MeshMode::AppendListed;
    MeshCursor *cursor = b->cursor.as<MeshCursor>();
    for (int attempt = 0; attempt < 2; ++attempt) {
        if (listed) VX_CUDA(ctx, cudaMemsetAsync(&cursor->work, 0, sizeof(cursor->work), ctx->stream));
        else VX_CUDA(ctx, cudaMemsetAsync(cursor, 0, sizeof(MeshCursor), ctx->stream));
        ChunkArgs a;
        a.voxels = in.voxels;
        a.neighbors = in.neighbors;
        a.uniform_flags = in.uniform_flags;
        a.n_chunks = in.n_chunks;
        a.subset = rows;
        a.n_out = n_rows;
        a.out_by_chunk = listed ? 1 : 0;
        a.quads = b->quads.as<uint8_t>();
        a.cap_quads = (unsigned long long)b->cap_quads;
        a.quad_base = b->quad_base.as<uint32_t>();
        a.quad_count = b->quad_count.as<uint32_t>();
        a.slice_offsets = b->slice_offsets.as<uint32_t>();
        a.face_aabb = b->face_aabb.as<int32_t>();
        a.has_mesh = b->has_mesh.as<uint8_t>();
        a.cursor = cursor;
        int per_sm = 0;
        VX_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mesh_chunks_kernel, MESH_THREADS, 0));
        if (per_sm < 1) per_sm = 1;
        int grid = ctx->num_sms * per_sm;
        if (grid > a.n_out) grid = a.n_out;
        if (grid < 1) grid = 1;
        mesh_chunks_kernel<<<grid, MESH_THREADS, 0, ctx->stream>>>(a);
        VX_CHECK_LAUNCH(ctx);
        b->total_quads = -1;
        b->n_meshes = -1;
        if (mode != MeshMode::EveryRowRegrow) return VX_OK;
        MeshCursor h;
        const int rc = read_cursor(ctx, b, h);
        if (rc != VX_OK) return rc;
        if (!h.overflow) {
            b->total_quads = (int64_t)h.quads;
            b->n_meshes = (int32_t)h.meshes;
            return VX_OK;
        }
        if (h.quads >= (1ull << 32)) return vx_fail(ctx, VX_ERR_CAPACITY, "more than 2^32 quads in one batch");
        VX_CUDA(ctx, b->quads.reserve(3 * (size_t)h.quads + 16));
        b->cap_quads = (int64_t)h.quads;
    }
    return vx_fail(ctx, VX_ERR_CAPACITY, "mesher output did not fit after regrow");
}

// Mesh every row of a new batch (EveryRowRegrow; an empty batch has nothing to mesh) and hand it to *out.
int mesh_new_batch(VxContext *ctx, BatchPtr &b, const MeshInput &in, const int32_t *rows, VxMeshBatch **out) {
    if (b->n_chunks > 0) {
        const int rc = run_mesher(ctx, b.get(), in, MeshMode::EveryRowRegrow, rows, b->n_chunks);
        if (rc != VX_OK) return rc;
    } else {
        b->total_quads = 0;
        b->n_meshes = 0;
    }
    *out = b.release();
    return VX_OK;
}

// positions of the batch's chunks from the device array d_positions, or zeros without one
int copy_positions(VxContext *ctx, VxMeshBatch *b, const int32_t *d_positions) {
    const size_t bytes = sizeof(int32_t) * 3 * (size_t)b->n_chunks;
    if (bytes == 0) return VX_OK;
    if (d_positions) VX_CUDA(ctx, cudaMemcpyAsync(b->positions.ptr, d_positions, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    else VX_CUDA(ctx, cudaMemsetAsync(b->positions.ptr, 0, bytes, ctx->stream));
    return VX_OK;
}

struct ShardOffsets {
    uint32_t off[64]; // first quad of rank r's stream in the assembled stream
};

// first quad of every rank's stream in the assembled stream, from the totals the blocks carry (no host round trip): one thread
__global__ void shard_offsets_kernel(int world, const uint8_t *__restrict__ blocks, VxShardLayout L, uint32_t *off /* [64] offsets, [64] totals */,
                                     MeshCursor *cursor, unsigned long long cap_quads) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    unsigned long long run = 0, overflow = 0;
    for (int r = 0; r < world; ++r) {
        unsigned long long t = *reinterpret_cast<const unsigned long long *>(blocks + (size_t)r * (size_t)L.rank_stride + L.off_quads - 16);
        if (t > (unsigned long long)L.quads_capacity) { // the shard outgrew its block: reported by vx_mesh_batch_info
            overflow = 1;
            t = (unsigned long long)L.quads_capacity;
        }
        off[r] = (uint32_t)run;
        off[64 + r] = (uint32_t)t;
        run += t;
    }
    if (run > cap_quads || run >= (1ull << 32)) overflow = 1;
    cursor->quads = run;
    cursor->meshes = 0; // counted by the assemble kernel
    cursor->overflow = overflow;
    cursor->work = 0;
}

// one thread per quad of every rank's stream: move it to its place in the assembled stream
__global__ void __launch_bounds__(256) copy_shard_quads_kernel(const uint8_t *__restrict__ blocks, VxShardLayout L, const uint32_t *__restrict__ off, uint8_t *dst,
                                                               unsigned long long cap_quads) {
    const int r = blockIdx.y;
    const uint32_t n = off[64 + r], base = off[r];
    const uint8_t *src = blocks + (size_t)r * (size_t)L.rank_stride + L.off_quads;
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        if ((unsigned long long)base + q >= cap_quads) return;
        const uint8_t a = src[3 * (size_t)q], b = src[3 * (size_t)q + 1], c = src[3 * (size_t)q + 2];
        uint8_t *d = dst + 3 * ((size_t)base + q);
        d[0] = a; d[1] = b; d[2] = c;
    }
}

// one CTA per chunk of the assembled batch: copy its row from the gathered shard blocks (vx_mesh_batch_assemble_shards)
__global__ void __launch_bounds__(64) assemble_shards_kernel(int n_chunks, int world, ShardOffsets so, const uint8_t *__restrict__ blocks, VxShardLayout L,
                                                             uint32_t *quad_base, uint32_t *quad_count, uint32_t *slice_offsets, int32_t *face_aabb,
                                                             uint8_t *has_mesh, MeshCursor *cursor, unsigned long long total,
                                                             const uint32_t *__restrict__ d_off = nullptr) {
    const int c = blockIdx.x;
    if (c >= n_chunks) return;
    const int r = c % world;
    const size_t j = (size_t)(c / world);
    const uint8_t *blk = blocks + (size_t)r * (size_t)L.rank_stride;
    const uint32_t *g_base = reinterpret_cast<const uint32_t *>(blk + L.off_quad_base), *g_count = reinterpret_cast<const uint32_t *>(blk + L.off_quad_count);
    const uint32_t *g_so = reinterpret_cast<const uint32_t *>(blk + L.off_slice_offsets);
    const int32_t *g_aabb = reinterpret_cast<const int32_t *>(blk + L.off_face_aabb);
    const uint8_t *g_has = blk + L.off_has_mesh;
    for (int i = threadIdx.x; i < SLICE_ROW; i += 64) slice_offsets[(size_t)c * SLICE_ROW + i] = g_so[j * SLICE_ROW + i];
    if (threadIdx.x < AABB_ROW) face_aabb[(size_t)c * AABB_ROW + threadIdx.x] = g_aabb[j * AABB_ROW + threadIdx.x];
    if (threadIdx.x == AABB_ROW) quad_base[c] = g_base[j] + (d_off ? d_off[r] : so.off[r]);
    if (threadIdx.x == AABB_ROW + 1) quad_count[c] = g_count[j];
    if (threadIdx.x == AABB_ROW + 2) {
        has_mesh[c] = g_has[j];
        if (d_off && g_has[j]) atomicAdd(&cursor->meshes, 1ull);
    }
    if (!d_off && c == 0 && threadIdx.x == AABB_ROW + 3) {
        cursor->quads = total;
        cursor->meshes = 0;
        cursor->overflow = 0;
        cursor->work = 0;
    }
}

// The batch an assemble of n_chunks writes: *batch_inout (created for the same n_chunks; its quad stream grown to `want`
// quads after a synchronise when it holds fewer than `need`), or a new one with room for `want`, owned by `fresh`.  The
// positions are copied from d_positions; a new batch without them gets zeros.
int assemble_target(VxContext *ctx, VxMeshBatch *const *batch_inout, int32_t n_chunks, int64_t need, int64_t want,
                    const int32_t *d_positions, BatchPtr &fresh) {
    VxMeshBatch *b = *batch_inout;
    if (!b) {
        const int rc = new_batch(ctx, n_chunks, want > 0 ? want : 1, MESH_ARRAYS, fresh);
        if (rc != VX_OK) return rc;
        b = fresh.get();
    } else if (b->n_chunks != n_chunks) {
        return vx_fail(ctx, VX_ERR_INVALID, "batch was created for another chunk count");
    } else if (need > b->cap_quads) {
        VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        VX_CUDA(ctx, b->quads.reserve(3 * (size_t)want + 16));
        b->cap_quads = want;
    }
    return d_positions || fresh ? copy_positions(ctx, b, d_positions) : VX_OK;
}

// device-to-device copy into a shard block (nothing for an empty section)
cudaError_t to_block(VxContext *ctx, uint8_t *d_block, int64_t off, const void *src, size_t bytes) {
    return bytes ? cudaMemcpyAsync(d_block + off, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream) : cudaSuccess;
}

// the shard's per-chunk arrays into their sections of the block (vx_shard_layout)
int pack_rows(VxContext *ctx, const VxMeshBatch *shard, const VxShardLayout *L, uint8_t *d_block) {
    const size_t n = (size_t)shard->n_chunks;
    VX_CUDA(ctx, to_block(ctx, d_block, L->off_quad_base, shard->quad_base.ptr, 4 * n));
    VX_CUDA(ctx, to_block(ctx, d_block, L->off_quad_count, shard->quad_count.ptr, 4 * n));
    VX_CUDA(ctx, to_block(ctx, d_block, L->off_slice_offsets, shard->slice_offsets.ptr, 4 * SLICE_ROW * n));
    VX_CUDA(ctx, to_block(ctx, d_block, L->off_face_aabb, shard->face_aabb.ptr, 4 * AABB_ROW * n));
    VX_CUDA(ctx, to_block(ctx, d_block, L->off_has_mesh, shard->has_mesh.ptr, n));
    return VX_OK;
}

// one CTA per live chunk: move its quads from the old stream to their place in the compacted one
__global__ void __launch_bounds__(256) compact_quads_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, const uint4 *__restrict__ moves, int n_moves) {
    for (int m = blockIdx.x; m < n_moves; m += gridDim.x) {
        const uint4 mv = moves[m]; // old base, new base, count (quads)
        const uint8_t *s = src + 3 * (size_t)mv.x;
        uint8_t *d = dst + 3 * (size_t)mv.y;
        const uint32_t bytes = 3u * mv.z;
        for (uint32_t i = threadIdx.x; i < bytes; i += blockDim.x) d[i] = s[i];
    }
}

// Drop the dead space of an append-updated quad stream WITHOUT re-meshing (the streaming world keeps meshes that are
// deliberately stale, main.rs:225-280): live quads are copied chunk by chunk into a fresh stream with room for
// `extra_quads` more.
int compact_stream(VxContext *ctx, VxMeshBatch *b, int64_t extra_quads) {
    const size_t n = (size_t)b->n_chunks;
    std::vector<uint32_t> base(n), count(n);
    std::vector<uint8_t> has(n);
    if (n) {
        VX_CUDA(ctx, cudaMemcpyAsync(base.data(), b->quad_base.ptr, 4 * n, cudaMemcpyDeviceToHost, ctx->stream));
        VX_CUDA(ctx, cudaMemcpyAsync(count.data(), b->quad_count.ptr, 4 * n, cudaMemcpyDeviceToHost, ctx->stream));
        VX_CUDA(ctx, cudaMemcpyAsync(has.data(), b->has_mesh.ptr, n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    std::vector<uint4> moves;
    uint64_t live = 0;
    for (size_t i = 0; i < n; ++i) {
        if (has[i] && count[i]) {
            moves.push_back(make_uint4(base[i], (uint32_t)live, count[i], 0u));
            base[i] = (uint32_t)live;
            live += count[i];
        } else {
            base[i] = (uint32_t)live;
        }
    }
    const int64_t want = (int64_t)live * 2 + extra_quads + 4096;
    if (want >= (int64_t)1 << 32) return vx_fail(ctx, VX_ERR_CAPACITY, "more than 2^32 quads in one batch");
    VxDeviceBuffer fresh;
    VX_CUDA(ctx, fresh.reserve(3 * (size_t)want + 16));
    if (!moves.empty()) {
        VX_CUDA(ctx, ctx->tmp_c.reserve(sizeof(uint4) * moves.size()));
        VX_CUDA(ctx, cudaMemcpyAsync(ctx->tmp_c.ptr, moves.data(), sizeof(uint4) * moves.size(), cudaMemcpyHostToDevice, ctx->stream));
        const int grid = (int)(moves.size() < (size_t)ctx->num_sms * 8 ? moves.size() : (size_t)ctx->num_sms * 8);
        compact_quads_kernel<<<grid, 256, 0, ctx->stream>>>(b->quads.as<uint8_t>(), fresh.as<uint8_t>(), ctx->tmp_c.as<uint4>(), (int)moves.size());
        VX_CHECK_LAUNCH(ctx);
    }
    if (n) VX_CUDA(ctx, cudaMemcpyAsync(b->quad_base.ptr, base.data(), 4 * n, cudaMemcpyHostToDevice, ctx->stream));
    MeshCursor h{live, 0ull, 0ull, 0ull};
    for (size_t i = 0; i < n; ++i) h.meshes += has[i] ? 1 : 0;
    const int rc = write_cursor(ctx, b, h); // also waits for the copies from the host vectors above
    if (rc != VX_OK) return rc;
    b->quads.release();
    b->quads = fresh;
    b->cap_quads = want;
    b->total_quads = (int64_t)live;
    b->n_meshes = (int32_t)h.meshes;
    return VX_OK;
}

// ids (in range) without repeats, in first-seen order
std::vector<int32_t> unique_ids(const std::vector<int32_t> &ids, int32_t n_chunks) {
    std::vector<int32_t> list;
    std::vector<uint8_t> seen((size_t)n_chunks, 0);
    for (const int32_t c : ids)
        if (!seen[c]) {
            seen[c] = 1;
            list.push_back(c);
        }
    return list;
}

// Re-mesh exactly the listed chunks of a world-owning batch in place.  Their quads are appended behind the live end of
// the stream; when it has no room for them, the live quads are compacted first (copied, not re-meshed), so every other
// chunk's mesh stays as it is.
int remesh_listed(VxContext *ctx, VxMeshBatch *b, const std::vector<int32_t> &list) {
    if (list.empty()) return VX_OK;
    VxMeshBatchInfo info;
    int rc = vx_mesh_batch_info(ctx, b, &info);
    if (rc != VX_OK) return rc;
    for (int attempt = 0; attempt < 3; ++attempt) {
        // typical chunk: a few hundred quads, so 4096 each is a generous bound that the overflow flag backs up
        const int64_t room = (int64_t)list.size() * (attempt == 0 ? 4096 : 98304); // 98,304 = the most quads a chunk can have
        if (b->total_quads + room > b->cap_quads) {
            rc = compact_stream(ctx, b, room);
            if (rc != VX_OK) return rc;
        }
        const int64_t before = b->total_quads; // live end of the stream (run_mesher invalidates the cached value)
        VX_CUDA(ctx, b->update_ids.reserve(sizeof(int32_t) * list.size()));
        VX_CUDA(ctx, cudaMemcpyAsync(b->update_ids.ptr, list.data(), sizeof(int32_t) * list.size(), cudaMemcpyHostToDevice, ctx->stream));
        rc = run_mesher(ctx, b, world_input(b), MeshMode::AppendListed, b->update_ids.as<int32_t>(), (int32_t)list.size());
        if (rc != VX_OK) return rc;
        MeshCursor h;
        rc = read_cursor(ctx, b, h);
        if (rc != VX_OK) return rc;
        if (!h.overflow) {
            b->total_quads = (int64_t)h.quads; // length of the stream, dead space included
            b->n_meshes = -1;                  // recounted on demand
            return VX_OK;
        }
        // overflow: the chunks of this list that did not fit have no quads; clear the flag, make room, mesh the list again
        h.overflow = 0;
        h.quads = (unsigned long long)before;
        rc = write_cursor(ctx, b, h);
        if (rc != VX_OK) return rc;
        b->total_quads = before;
    }
    return vx_fail(ctx, VX_ERR_CAPACITY, "world batch: quad stream overflow persisted");
}

// vx_world_batch_set_blocks, step 1: one CTA per edited slot.  A Uniform slot gets voxel rows of its block type and becomes
// Varied, so that the edits of step 2 land in a complete chunk.
constexpr int EDIT_THREADS = 256;
__global__ void __launch_bounds__(EDIT_THREADS) materialize_uniform_kernel(uint8_t *voxels, uint8_t *flags, const int32_t *slots) {
    const int32_t s = slots[blockIdx.x];
    const uint8_t flag = flags[s];
    if (flag == 0) return; // uniform across the CTA: no thread reaches the barrier
    const uint32_t t = (uint32_t)(flag - 1) * 0x01010101u;
    uint4 *row = reinterpret_cast<uint4 *>(voxels + (size_t)s * VX_CHUNK_VOLUME);
    for (int k = threadIdx.x; k < VX_CHUNK_VOLUME / 16; k += EDIT_THREADS) row[k] = make_uint4(t, t, t, t);
    __syncthreads(); // every thread has read the flag
    if (threadIdx.x == 0) flags[s] = 0;
}

// step 2: one thread per edit; the host has removed repeated voxels, so no two threads store to the same byte
__global__ void scatter_blocks_kernel(uint8_t *voxels, const int32_t *slot, const int32_t *index, const int32_t *type, int32_t n) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) voxels[(size_t)slot[i] * VX_CHUNK_VOLUME + index[i]] = (uint8_t)type[i];
}

} // namespace

extern "C" {

int vx_mesh_chunks_device(VxContext *ctx, const uint8_t *d_voxels, const int32_t *d_positions,
                          const int32_t *d_neighbors, const uint8_t *d_uniform_flags, int32_t n_chunks,
                          VxMeshBatch **out) {
    if (!ctx || !out || n_chunks < 0 || (n_chunks > 0 && !d_voxels)) return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_chunks_device: bad argument");
    if ((reinterpret_cast<uintptr_t>(d_voxels) & 15) != 0) return vx_fail(ctx, VX_ERR_INVALID, "voxels must be 16-byte aligned");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    BatchPtr b;
    int rc = new_batch(ctx, n_chunks, first_cap_quads(n_chunks), MESH_ARRAYS, b);
    if (rc == VX_OK) rc = copy_positions(ctx, b.get(), d_positions);
    if (rc == VX_OK) rc = mesh_new_batch(ctx, b, {d_voxels, d_neighbors, d_uniform_flags, n_chunks}, nullptr, out);
    return rc;
}

int vx_mesh_chunk_subset_device(VxContext *ctx, const uint8_t *d_voxels, const int32_t *d_positions,
                                const int32_t *d_neighbors, const uint8_t *d_uniform_flags, int32_t n_chunks,
                                const int32_t *d_subset, int32_t n_subset, VxMeshBatch **batch_inout) {
    if (!ctx || !batch_inout || n_chunks < 0 || n_subset < 0 || (n_subset > 0 && (!d_voxels || !d_subset)))
        return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_chunk_subset_device: bad argument");
    if ((reinterpret_cast<uintptr_t>(d_voxels) & 15) != 0) return vx_fail(ctx, VX_ERR_INVALID, "voxels must be 16-byte aligned");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    const MeshInput in{d_voxels, d_neighbors, d_uniform_flags, n_chunks};
    if (*batch_inout) { // steady state: re-mesh the same shard into the existing batch, no allocation
        if ((*batch_inout)->n_chunks != n_subset) return vx_fail(ctx, VX_ERR_INVALID, "batch was created for another subset size");
        if (n_subset == 0) return VX_OK;
        return run_mesher(ctx, *batch_inout, in, MeshMode::EveryRowSteady, d_subset, n_subset);
    }
    BatchPtr b;
    int rc = new_batch(ctx, n_subset, first_cap_quads(n_subset), MESH_ARRAYS, b);
    if (rc != VX_OK) return rc;
    if (d_positions && n_subset > 0) { // positions of the subset, gathered on the host side of the stream (small)
        std::vector<int32_t> ids((size_t)n_subset), pos((size_t)n_chunks * 3), sub((size_t)n_subset * 3);
        VX_CUDA(ctx, cudaMemcpyAsync(ids.data(), d_subset, sizeof(int32_t) * (size_t)n_subset, cudaMemcpyDeviceToHost, ctx->stream));
        VX_CUDA(ctx, cudaMemcpyAsync(pos.data(), d_positions, sizeof(int32_t) * 3 * (size_t)n_chunks, cudaMemcpyDeviceToHost, ctx->stream));
        VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (int32_t i = 0; i < n_subset; ++i) {
            if (ids[i] < 0 || ids[i] >= n_chunks) return vx_fail(ctx, VX_ERR_INVALID, "subset id out of range");
            for (int k = 0; k < 3; ++k) sub[(size_t)i * 3 + k] = pos[(size_t)ids[i] * 3 + k];
        }
        VX_CUDA(ctx, cudaMemcpyAsync(b->positions.ptr, sub.data(), sizeof(int32_t) * 3 * (size_t)n_subset, cudaMemcpyHostToDevice, ctx->stream));
        VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    } else {
        rc = copy_positions(ctx, b.get(), nullptr);
        if (rc != VX_OK) return rc;
    }
    return mesh_new_batch(ctx, b, in, d_subset, batch_inout);
}

int vx_remesh_chunks_device(VxContext *ctx, const uint8_t *d_voxels, const int32_t *d_neighbors,
                            const uint8_t *d_uniform_flags, VxMeshBatch *batch) {
    if (!ctx || !batch || !d_voxels) return vx_fail(ctx, VX_ERR_INVALID, "vx_remesh_chunks_device: bad argument");
    if (batch->n_chunks == 0) return VX_OK;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    return run_mesher(ctx, batch, {d_voxels, d_neighbors, d_uniform_flags, batch->n_chunks}, MeshMode::EveryRowSteady, nullptr, batch->n_chunks);
}

int vx_mesh_chunks(VxContext *ctx, const uint8_t *voxels, const int32_t *positions, const int32_t *neighbors,
                   const uint8_t *uniform_flags, int32_t n_chunks, VxMeshBatch **out) {
    if (!ctx || !out || n_chunks < 0 || (n_chunks > 0 && !voxels)) return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_chunks: bad argument");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)n_chunks;
    // the world copy stays with the batch (vx_mesh_batch_update edits it in place)
    BatchPtr b;
    const int rc = new_batch(ctx, n_chunks, first_cap_quads(n_chunks), ALL_ARRAYS, b);
    if (rc != VX_OK) return rc;
    if (n) {
        VX_CUDA(ctx, cudaMemcpyAsync(b->world_voxels.ptr, voxels, n * VX_CHUNK_VOLUME, cudaMemcpyHostToDevice, ctx->stream));
        if (neighbors) VX_CUDA(ctx, cudaMemcpyAsync(b->world_neighbors.ptr, neighbors, n * 6 * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        if (uniform_flags) VX_CUDA(ctx, cudaMemcpyAsync(b->world_flags.ptr, uniform_flags, n, cudaMemcpyHostToDevice, ctx->stream));
        else VX_CUDA(ctx, cudaMemsetAsync(b->world_flags.ptr, 0, n, ctx->stream));
        if (positions) VX_CUDA(ctx, cudaMemcpyAsync(b->positions.ptr, positions, n * 3 * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        else VX_CUDA(ctx, cudaMemsetAsync(b->positions.ptr, 0, n * 3 * sizeof(int32_t), ctx->stream));
    }
    b->owns_world = true;
    b->has_neighbors = neighbors != nullptr;
    if (neighbors) b->host_neighbors.assign(neighbors, neighbors + n * 6);
    return mesh_new_batch(ctx, b, world_input(b.get()), nullptr, out);
}

int vx_mesh_batch_update(VxContext *ctx, VxMeshBatch *b, const int32_t *chunk_ids, int32_t n_ids, const uint8_t *voxels,
                         const uint8_t *uniform_flags, int32_t *n_remeshed) {
    if (!ctx || !b || n_ids < 0 || (n_ids > 0 && (!chunk_ids || !voxels))) return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_batch_update: bad argument");
    if (!b->owns_world) return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_batch_update: the batch was not created by vx_mesh_chunks (no world copy)");
    if (n_remeshed) *n_remeshed = 0;
    if (n_ids == 0) return VX_OK;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    // edited chunks + the neighbours whose border faces they can change (main.rs:225-280 invalidates the same six)
    std::vector<int32_t> ids(chunk_ids, chunk_ids + n_ids);
    for (const int32_t c : ids)
        if (c < 0 || c >= b->n_chunks) return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_batch_update: chunk id out of range");
    if (b->has_neighbors)
        for (int32_t i = 0; i < n_ids; ++i)
            for (int f = 0; f < 6; ++f) {
                const int32_t nb = b->host_neighbors[(size_t)chunk_ids[i] * 6 + f];
                if (nb >= 0 && nb < b->n_chunks) ids.push_back(nb);
            }
    // new voxel data / uniform flags of the edited chunks into the world copy
    for (int32_t i = 0; i < n_ids; ++i) {
        VX_CUDA(ctx, cudaMemcpyAsync(b->world_voxels.as<uint8_t>() + (size_t)chunk_ids[i] * VX_CHUNK_VOLUME, voxels + (size_t)i * VX_CHUNK_VOLUME,
                                     VX_CHUNK_VOLUME, cudaMemcpyHostToDevice, ctx->stream));
        const uint8_t uf = uniform_flags ? uniform_flags[i] : 0;
        VX_CUDA(ctx, cudaMemsetAsync(b->world_flags.as<uint8_t>() + chunk_ids[i], uf, 1, ctx->stream));
    }
    const std::vector<int32_t> list = unique_ids(ids, b->n_chunks);
    if (n_remeshed) *n_remeshed = (int32_t)list.size();
    return remesh_listed(ctx, b, list);
}

int vx_mesh_batch_info(VxContext *ctx, const VxMeshBatch *b, VxMeshBatchInfo *info) {
    if (!ctx || !b || !info) return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_batch_info: bad argument");
    if (b->total_quads < 0) {
        MeshCursor h;
        const int rc = read_cursor(ctx, b, h);
        if (rc != VX_OK) return rc;
        if (h.overflow) return vx_fail(ctx, VX_ERR_CAPACITY, "remesh overflowed the batch quad stream");
        b->total_quads = (int64_t)h.quads;
        b->n_meshes = (int32_t)h.meshes;
    }
    if (b->n_meshes < 0) { // after an in-place update: count has_mesh
        std::vector<uint8_t> hm((size_t)b->n_chunks);
        if (b->n_chunks) VX_CUDA(ctx, cudaMemcpyAsync(hm.data(), b->has_mesh.ptr, (size_t)b->n_chunks, cudaMemcpyDeviceToHost, ctx->stream));
        VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        int32_t nm = 0;
        for (uint8_t v : hm) nm += v ? 1 : 0;
        b->n_meshes = nm;
    }
    info->n_chunks = b->n_chunks;
    info->n_meshes = b->n_meshes;
    info->total_quads = b->total_quads;
    return VX_OK;
}

int vx_mesh_batch_device(const VxMeshBatch *b, VxMeshBatchDevice *out) {
    if (!b || !out) return VX_ERR_INVALID;
    out->d_quads = b->quads.as<uint8_t>();
    out->d_quad_base = b->quad_base.as<uint32_t>();
    out->d_quad_count = b->quad_count.as<uint32_t>();
    out->d_slice_offsets = b->slice_offsets.as<uint32_t>();
    out->d_face_aabb = b->face_aabb.as<int32_t>();
    out->d_has_mesh = b->has_mesh.as<uint8_t>();
    out->d_positions = b->positions.as<int32_t>();
    return VX_OK;
}

int vx_mesh_batch_download(VxContext *ctx, const VxMeshBatch *b, uint8_t *quads, uint32_t *quad_base,
                           uint32_t *quad_count, uint32_t *slice_offsets, int32_t *face_aabb, uint8_t *has_mesh) {
    if (!ctx || !b) return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_batch_download: bad argument");
    VxMeshBatchInfo info;
    int rc = vx_mesh_batch_info(ctx, b, &info);
    if (rc != VX_OK) return rc;
    const size_t n = (size_t)b->n_chunks;
    if (quads && info.total_quads) VX_CUDA(ctx, cudaMemcpyAsync(quads, b->quads.ptr, 3 * (size_t)info.total_quads, cudaMemcpyDeviceToHost, ctx->stream));
    if (quad_base && n) VX_CUDA(ctx, cudaMemcpyAsync(quad_base, b->quad_base.ptr, 4 * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (quad_count && n) VX_CUDA(ctx, cudaMemcpyAsync(quad_count, b->quad_count.ptr, 4 * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (slice_offsets && n) VX_CUDA(ctx, cudaMemcpyAsync(slice_offsets, b->slice_offsets.ptr, 4 * SLICE_ROW * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (face_aabb && n) VX_CUDA(ctx, cudaMemcpyAsync(face_aabb, b->face_aabb.ptr, 4 * AABB_ROW * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (has_mesh && n) VX_CUDA(ctx, cudaMemcpyAsync(has_mesh, b->has_mesh.ptr, n, cudaMemcpyDeviceToHost, ctx->stream));
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VX_OK;
}

int vx_mesh_batch_upload(VxContext *ctx, const uint8_t *quads, int64_t total_quads, const uint32_t *quad_base,
                         const uint32_t *quad_count, const uint32_t *slice_offsets, const int32_t *face_aabb,
                         const uint8_t *has_mesh, const int32_t *positions, int32_t n_chunks, VxMeshBatch **out) {
    if (!ctx || !out || n_chunks < 0 || total_quads < 0) return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_batch_upload: bad argument");
    if (n_chunks > 0 && (!quad_base || !quad_count || !slice_offsets || !face_aabb || !has_mesh || !positions))
        return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_batch_upload: null array");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    BatchPtr b;
    int rc = new_batch(ctx, n_chunks, total_quads > 0 ? total_quads : 1, MESH_ARRAYS, b);
    if (rc != VX_OK) return rc;
    const size_t n = (size_t)n_chunks;
    auto up = [&](void *dst, const void *src, size_t bytes) -> cudaError_t {
        return bytes ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream) : cudaSuccess;
    };
    VX_CUDA(ctx, up(b->quads.ptr, quads, 3 * (size_t)total_quads));
    VX_CUDA(ctx, up(b->quad_base.ptr, quad_base, 4 * n));
    VX_CUDA(ctx, up(b->quad_count.ptr, quad_count, 4 * n));
    VX_CUDA(ctx, up(b->slice_offsets.ptr, slice_offsets, 4 * SLICE_ROW * n));
    VX_CUDA(ctx, up(b->face_aabb.ptr, face_aabb, 4 * AABB_ROW * n));
    VX_CUDA(ctx, up(b->has_mesh.ptr, has_mesh, n));
    VX_CUDA(ctx, up(b->positions.ptr, positions, 12 * n));
    int32_t nm = 0;
    for (size_t i = 0; i < n; ++i) nm += has_mesh[i] ? 1 : 0;
    rc = write_cursor(ctx, b.get(), MeshCursor{(unsigned long long)total_quads, (unsigned long long)nm, 0ull, 0ull});
    if (rc != VX_OK) return rc;
    b->total_quads = total_quads;
    b->n_meshes = nm;
    *out = b.release();
    return VX_OK;
}

// Chunk-sharded meshing, exchange step (SURVEY 8e; binary_greedy.rs:62-78 returns every mesh to the caller): rank r
// meshed the chunks k with k % world == r into a compact shard batch (row j = chunk r + j * world).  Each rank packs
// its shard into one block (vx_mesh_shard_pack), the blocks are all-gathered (one NCCL collective), and
// vx_mesh_batch_assemble_shards puts them back into one batch in chunk order.  The quad stream is the concatenation
// of the shards' streams (a chunk's quads stay contiguous and in reference order; only quad_base is rebased), so no
// quad is touched more than once.
int vx_shard_layout(int32_t rows_per_rank, int64_t max_shard_quads, VxShardLayout *out) {
    if (!out || rows_per_rank < 0 || max_shard_quads < 0) return VX_ERR_INVALID;
    auto up16 = [](int64_t v) { return (v + 15) & ~(int64_t)15; };
    const int64_t rows = rows_per_rank;
    int64_t o = 0;
    out->rows_per_rank = rows_per_rank;
    out->off_quad_base = o; o = up16(o + 4 * rows);
    out->off_quad_count = o; o = up16(o + 4 * rows);
    out->off_slice_offsets = o; o = up16(o + 4 * SLICE_ROW * rows);
    out->off_face_aabb = o; o = up16(o + 4 * AABB_ROW * rows);
    out->off_has_mesh = o; o = up16(o + rows);
    o += 16; // block[off_quads - 16 .. off_quads - 8): u64 quad total of the shard (vx_mesh_shard_pack_async)
    out->off_quads = o; o = up16(o + 3 * max_shard_quads);
    out->quads_capacity = max_shard_quads;
    out->rank_stride = o;
    return VX_OK;
}

int vx_mesh_shard_pack(VxContext *ctx, const VxMeshBatch *shard, const VxShardLayout *L, uint8_t *d_block) {
    if (!ctx || !shard || !L || !d_block || shard->n_chunks > L->rows_per_rank) return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_shard_pack: bad argument");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    VxMeshBatchInfo info;
    int rc = vx_mesh_batch_info(ctx, shard, &info);
    if (rc != VX_OK) return rc;
    if (info.total_quads > L->quads_capacity) return vx_fail(ctx, VX_ERR_CAPACITY, "shard has more quads than the layout holds");
    rc = pack_rows(ctx, shard, L, d_block);
    if (rc != VX_OK) return rc;
    VX_CUDA(ctx, to_block(ctx, d_block, L->off_quads, shard->quads.ptr, 3 * (size_t)info.total_quads));
    return VX_OK;
}

int vx_mesh_batch_assemble_shards(VxContext *ctx, int32_t n_chunks, int32_t world, const uint8_t *d_blocks, const VxShardLayout *L,
                                  const int64_t *shard_quads, const int32_t *d_positions, VxMeshBatch **batch_inout) {
    if (!ctx || !batch_inout || !L || n_chunks < 0 || world < 1 || world > 64 || !shard_quads || (int64_t)L->rows_per_rank * world < n_chunks ||
        (n_chunks > 0 && !d_blocks))
        return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_batch_assemble_shards: bad argument");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    int64_t total = 0;
    ShardOffsets so;
    memset(&so, 0, sizeof(so));
    for (int r = 0; r < world; ++r) {
        if (shard_quads[r] < 0 || shard_quads[r] > L->quads_capacity) return vx_fail(ctx, VX_ERR_INVALID, "shard quad count exceeds the layout");
        so.off[r] = (uint32_t)total;
        total += shard_quads[r];
    }
    if (total >= (int64_t)1 << 32) return vx_fail(ctx, VX_ERR_CAPACITY, "more than 2^32 quads in one batch");
    BatchPtr fresh;
    const int rc = assemble_target(ctx, batch_inout, n_chunks, total, total + total / 8, d_positions, fresh);
    if (rc != VX_OK) return rc;
    VxMeshBatch *b = fresh ? fresh.get() : *batch_inout;
    if (n_chunks > 0) {
        assemble_shards_kernel<<<n_chunks, 64, 0, ctx->stream>>>(n_chunks, world, so, d_blocks, *L, b->quad_base.as<uint32_t>(), b->quad_count.as<uint32_t>(),
                                                                 b->slice_offsets.as<uint32_t>(), b->face_aabb.as<int32_t>(), b->has_mesh.as<uint8_t>(),
                                                                 b->cursor.as<MeshCursor>(), (unsigned long long)total);
        VX_CHECK_LAUNCH(ctx);
    }
    for (int r = 0; r < world; ++r)
        if (shard_quads[r])
            VX_CUDA(ctx, cudaMemcpyAsync(b->quads.as<uint8_t>() + 3 * (size_t)so.off[r], d_blocks + (size_t)r * (size_t)L->rank_stride + L->off_quads,
                                         3 * (size_t)shard_quads[r], cudaMemcpyDeviceToDevice, ctx->stream));
    b->total_quads = total;
    b->n_meshes = -1; // counted on demand (vx_mesh_batch_info)
    if (fresh) *batch_inout = fresh.release();
    return VX_OK;
}

// The same exchange without a host round trip (steady state of a re-mesh sweep: the block capacity is known from an earlier
// sweep).  pack copies the whole quad section the block has room for and the shard's quad total (its cursor, 8 bytes in front
// of the quad section); assemble reads the totals from the gathered blocks on the device.  A shard that outgrew its block
// sets the batch's overflow flag: the next vx_mesh_batch_info fails with VX_ERR_CAPACITY and the caller sizes the blocks anew.
int vx_mesh_shard_pack_async(VxContext *ctx, const VxMeshBatch *shard, const VxShardLayout *L, uint8_t *d_block) {
    if (!ctx || !shard || !L || !d_block || shard->n_chunks > L->rows_per_rank) return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_shard_pack_async: bad argument");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    const int rc = pack_rows(ctx, shard, L, d_block);
    if (rc != VX_OK) return rc;
    const int64_t q = shard->cap_quads < L->quads_capacity ? shard->cap_quads : L->quads_capacity;
    VX_CUDA(ctx, to_block(ctx, d_block, L->off_quads, shard->quads.ptr, 3 * (size_t)(q > 0 ? q : 0)));
    VX_CUDA(ctx, to_block(ctx, d_block, L->off_quads - 16, shard->cursor.as<uint8_t>() + offsetof(MeshCursor, quads), sizeof(unsigned long long)));
    return VX_OK;
}

int vx_mesh_batch_assemble_shards_async(VxContext *ctx, int32_t n_chunks, int32_t world, const uint8_t *d_blocks, const VxShardLayout *L,
                                        const int32_t *d_positions, VxMeshBatch **batch_inout) {
    if (!ctx || !batch_inout || !L || n_chunks < 0 || world < 1 || world > 64 || (int64_t)L->rows_per_rank * world < n_chunks || (n_chunks > 0 && !d_blocks))
        return vx_fail(ctx, VX_ERR_INVALID, "vx_mesh_batch_assemble_shards_async: bad argument");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t bound = (int64_t)world * L->quads_capacity; // the assembled stream can never need more
    if (bound >= (int64_t)1 << 32) return vx_fail(ctx, VX_ERR_CAPACITY, "more than 2^32 quads in one batch");
    BatchPtr fresh;
    const int rc = assemble_target(ctx, batch_inout, n_chunks, bound, bound, d_positions, fresh);
    if (rc != VX_OK) return rc;
    VxMeshBatch *b = fresh ? fresh.get() : *batch_inout;
    VX_CUDA(ctx, ctx->tmp_d.reserve(sizeof(uint32_t) * 128));
    uint32_t *d_off = ctx->tmp_d.as<uint32_t>();
    shard_offsets_kernel<<<1, 32, 0, ctx->stream>>>(world, d_blocks, *L, d_off, b->cursor.as<MeshCursor>(), (unsigned long long)b->cap_quads);
    VX_CHECK_LAUNCH(ctx);
    if (n_chunks > 0) {
        ShardOffsets none;
        memset(&none, 0, sizeof(none));
        assemble_shards_kernel<<<n_chunks, 64, 0, ctx->stream>>>(n_chunks, world, none, d_blocks, *L, b->quad_base.as<uint32_t>(), b->quad_count.as<uint32_t>(),
                                                                 b->slice_offsets.as<uint32_t>(), b->face_aabb.as<int32_t>(), b->has_mesh.as<uint8_t>(),
                                                                 b->cursor.as<MeshCursor>(), 0ull, d_off);
        VX_CHECK_LAUNCH(ctx);
        const int per_rank = (int)((L->quads_capacity + 255) / 256 < 1 ? 1 : ((L->quads_capacity + 255) / 256 > 1024 ? 1024 : (L->quads_capacity + 255) / 256));
        copy_shard_quads_kernel<<<dim3(per_rank, world), 256, 0, ctx->stream>>>(d_blocks, *L, d_off, b->quads.as<uint8_t>(), (unsigned long long)b->cap_quads);
        VX_CHECK_LAUNCH(ctx);
    }
    b->total_quads = -1; // read from the device on demand (vx_mesh_batch_info), together with the overflow flag
    b->n_meshes = -1;
    if (fresh) *batch_inout = fresh.release();
    return VX_OK;
}

void vx_mesh_batch_release(VxContext *ctx, VxMeshBatch *b) {
    if (!b) return;
    if (ctx) cudaSetDevice(ctx->device);
    for (const ChunkArray &c : CHUNK_ARRAYS) (b->*c.buf).release();
    b->quads.release();
    b->cursor.release();
    b->update_ids.release();
    delete b;
}

int vx_greedy_mesh_slices(VxContext *ctx, const uint32_t *masks, int32_t n_slices, VxQuad *out, int32_t *n_out) {
    if (!ctx || n_slices < 0 || (n_slices > 0 && (!masks || !out || !n_out))) return vx_fail(ctx, VX_ERR_INVALID, "vx_greedy_mesh_slices: bad argument");
    if (n_slices == 0) return VX_OK;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)n_slices;
    VX_CUDA(ctx, ctx->tmp_a.reserve(n * 32 * sizeof(uint32_t)));
    VX_CUDA(ctx, ctx->tmp_b.reserve(n * 512 * sizeof(VxQuad)));
    VX_CUDA(ctx, ctx->tmp_c.reserve(n * sizeof(int32_t)));
    VX_CUDA(ctx, cudaMemcpyAsync(ctx->tmp_a.ptr, masks, n * 32 * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    const int threads = 128;
    const int blocks = (int)((n * 32 + threads - 1) / threads);
    greedy_slices_kernel<<<blocks, threads, 0, ctx->stream>>>(ctx->tmp_a.as<uint32_t>(), n_slices, ctx->tmp_b.as<VxQuad>(), ctx->tmp_c.as<int32_t>());
    VX_CHECK_LAUNCH(ctx);
    VX_CUDA(ctx, cudaMemcpyAsync(n_out, ctx->tmp_c.ptr, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    VX_CUDA(ctx, cudaMemcpyAsync(out, ctx->tmp_b.ptr, n * 512 * sizeof(VxQuad), cudaMemcpyDeviceToHost, ctx->stream));
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VX_OK;
}

// ---- streaming world (SURVEY 8f N2): World::update world.rs:57-100 + the mesh cache of main.rs:225-280 -----------------

int vx_world_batch_create(VxContext *ctx, int32_t capacity, VxMeshBatch **out) {
    if (!ctx || !out || capacity <= 0) return vx_fail(ctx, VX_ERR_INVALID, "vx_world_batch_create: bad argument");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)capacity;
    BatchPtr b;
    int rc = new_batch(ctx, capacity, first_cap_quads(capacity), ALL_ARRAYS, b);
    if (rc != VX_OK) return rc;
    for (const ChunkArray &c : CHUNK_ARRAYS) // every slot starts as an absent chunk: no neighbours, "uniform air", no mesh
        VX_CUDA(ctx, cudaMemsetAsync((b.get()->*c.buf).ptr, c.absent, c.row_bytes * n, ctx->stream));
    rc = write_cursor(ctx, b.get(), MeshCursor{});
    if (rc != VX_OK) return rc;
    b->owns_world = true;
    b->has_neighbors = true;
    b->host_neighbors.assign(n * 6, -1);
    b->total_quads = 0;
    b->n_meshes = 0;
    *out = b.release();
    return VX_OK;
}

// The reference's world is a HashMap that simply grows (world.rs:30-100: a moving camera that keeps hitting
// max_chunks_per_frame never reaches the unload step; World::set_view_distance widens the sphere at run time).  A world
// batch grows the same way: more slots, everything already loaded -- voxels, flags, neighbour rows, meshes, the quad
// stream -- is kept (device-to-device copies), the new slots are absent chunks.
int vx_world_batch_grow(VxContext *ctx, VxMeshBatch *b, int32_t new_capacity) {
    if (!ctx || !b || !b->owns_world || !b->has_neighbors) return vx_fail(ctx, VX_ERR_INVALID, "vx_world_batch_grow: not a world batch");
    if (new_capacity <= b->n_chunks) return VX_OK;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const size_t n0 = (size_t)b->n_chunks, n1 = (size_t)new_capacity;
    auto grow = [&](VxDeviceBuffer &buf, size_t per, int fill) -> cudaError_t {
        VxDeviceBuffer fresh;
        cudaError_t e = fresh.reserve(n1 * per);
        if (e != cudaSuccess) return e;
        e = cudaMemcpyAsync(fresh.ptr, buf.ptr, n0 * per, cudaMemcpyDeviceToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(static_cast<uint8_t *>(fresh.ptr) + n0 * per, fill, (n1 - n0) * per, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) {
            fresh.release();
            return e;
        }
        buf.release();
        buf = fresh;
        return cudaSuccess;
    };
    for (const ChunkArray &c : CHUNK_ARRAYS) VX_CUDA(ctx, grow(b->*c.buf, c.row_bytes, c.absent));
    b->host_neighbors.resize(n1 * 6, -1);
    b->n_chunks = new_capacity;
    return VX_OK;
}

static int world_check_slots(VxContext *ctx, const VxMeshBatch *b, const int32_t *slots, int32_t n, const char *who) {
    if (!ctx || !b || n < 0 || (n > 0 && !slots)) return vx_fail(ctx, VX_ERR_INVALID, who);
    if (!b->owns_world || !b->has_neighbors) return vx_fail(ctx, VX_ERR_INVALID, "not a world batch (vx_world_batch_create)");
    for (int32_t i = 0; i < n; ++i)
        if (slots[i] < 0 || slots[i] >= b->n_chunks) return vx_fail(ctx, VX_ERR_INVALID, "slot out of range");
    return VX_OK;
}

int vx_world_batch_assign(VxContext *ctx, VxMeshBatch *b, const int32_t *slots, int32_t n, const int32_t *positions, const int32_t *neighbors) {
    int rc = world_check_slots(ctx, b, slots, n, "vx_world_batch_assign: bad argument");
    if (rc != VX_OK || n == 0) return rc;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    for (int32_t i = 0; i < n; ++i) {
        const size_t s = (size_t)slots[i];
        if (positions) VX_CUDA(ctx, cudaMemcpyAsync(b->positions.as<int32_t>() + 3 * s, positions + 3 * (size_t)i, 12, cudaMemcpyHostToDevice, ctx->stream));
        if (neighbors) {
            for (int f = 0; f < 6; ++f) {
                const int32_t nb = neighbors[6 * (size_t)i + f];
                if (nb >= b->n_chunks || nb < -3) return vx_fail(ctx, VX_ERR_INVALID, "vx_world_batch_assign: neighbour out of range");
                b->host_neighbors[6 * s + f] = nb;
            }
            VX_CUDA(ctx, cudaMemcpyAsync(b->world_neighbors.as<int32_t>() + 6 * s, neighbors + 6 * (size_t)i, 24, cudaMemcpyHostToDevice, ctx->stream));
        }
    }
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); // the caller's arrays may go away
    return VX_OK;
}

int vx_world_batch_generate(VxContext *ctx, VxMeshBatch *b, const int32_t *slots, int32_t n, const int32_t *positions,
                            const VxTerrainParams *params, uint8_t *uniform_flags_out) {
    int rc = world_check_slots(ctx, b, slots, n, "vx_world_batch_generate: bad argument");
    if (rc != VX_OK || n == 0) return rc;
    if (!positions || !params) return vx_fail(ctx, VX_ERR_INVALID, "vx_world_batch_generate: bad argument");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t nn = (size_t)n;
    VX_CUDA(ctx, ctx->tmp_b.reserve(nn * VX_CHUNK_VOLUME + 16));
    std::vector<uint8_t> flags(nn);
    rc = vx_generate_terrain(ctx, positions, n, params, ctx->tmp_b.as<uint8_t>(), flags.data()); // Chunk::generate_terrain chunk.rs:114-207
    if (rc != VX_OK) return rc;
    for (size_t i = 0; i < nn; ++i) {
        const size_t s = (size_t)slots[i];
        VX_CUDA(ctx, cudaMemcpyAsync(b->world_voxels.as<uint8_t>() + s * VX_CHUNK_VOLUME, ctx->tmp_b.as<uint8_t>() + i * VX_CHUNK_VOLUME, VX_CHUNK_VOLUME,
                                     cudaMemcpyDeviceToDevice, ctx->stream));
        VX_CUDA(ctx, cudaMemsetAsync(b->world_flags.as<uint8_t>() + s, flags[i], 1, ctx->stream));
        VX_CUDA(ctx, cudaMemcpyAsync(b->positions.as<int32_t>() + 3 * s, positions + 3 * i, 12, cudaMemcpyHostToDevice, ctx->stream));
        if (uniform_flags_out) uniform_flags_out[i] = flags[i];
    }
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VX_OK;
}

int vx_world_batch_unload(VxContext *ctx, VxMeshBatch *b, const int32_t *slots, int32_t n) {
    int rc = world_check_slots(ctx, b, slots, n, "vx_world_batch_unload: bad argument");
    if (rc != VX_OK || n == 0) return rc;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    for (int32_t i = 0; i < n; ++i) { // an absent chunk: "uniform air" for any stale neighbour reference, no mesh, no neighbours of its own
        const size_t s = (size_t)slots[i];
        VX_CUDA(ctx, cudaMemsetAsync(b->world_flags.as<uint8_t>() + s, 1, 1, ctx->stream));
        VX_CUDA(ctx, cudaMemsetAsync(b->has_mesh.as<uint8_t>() + s, 0, 1, ctx->stream));
        VX_CUDA(ctx, cudaMemsetAsync(b->quad_count.as<uint32_t>() + s, 0, 4, ctx->stream));
        VX_CUDA(ctx, cudaMemsetAsync(b->world_neighbors.as<int32_t>() + 6 * s, 0xFF, 24, ctx->stream));
        for (int f = 0; f < 6; ++f) b->host_neighbors[6 * s + f] = -1;
    }
    b->n_meshes = -1;
    return VX_OK;
}

int vx_world_batch_remesh(VxContext *ctx, VxMeshBatch *b, const int32_t *slots, int32_t n) {
    int rc = world_check_slots(ctx, b, slots, n, "vx_world_batch_remesh: bad argument");
    if (rc != VX_OK || n == 0) return rc;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    return remesh_listed(ctx, b, unique_ids(std::vector<int32_t>(slots, slots + n), b->n_chunks));
}

int vx_world_batch_set_blocks(VxContext *ctx, VxMeshBatch *b, const int32_t *slots, const int32_t *voxel_index, const uint8_t *block_types,
                              int32_t n) {
    int rc = world_check_slots(ctx, b, slots, n, "vx_world_batch_set_blocks: bad argument");
    if (rc != VX_OK || n == 0) return rc;
    if (!voxel_index || !block_types) return vx_fail(ctx, VX_ERR_INVALID, "vx_world_batch_set_blocks: bad argument");
    for (int32_t i = 0; i < n; ++i) {
        if (voxel_index[i] < 0 || voxel_index[i] >= VX_CHUNK_VOLUME) return vx_fail(ctx, VX_ERR_INVALID, "vx_world_batch_set_blocks: voxel index out of range");
        if (block_types[i] > 3) return vx_fail(ctx, VX_ERR_INVALID, "vx_world_batch_set_blocks: block type out of range");
    }
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    // last edit of a voxel wins: walk the list backwards and keep the first occurrence of each (slot, voxel)
    std::vector<int32_t> es, ei, et;
    std::unordered_set<int64_t> seen;
    for (int32_t i = n - 1; i >= 0; --i)
        if (seen.insert((int64_t)slots[i] * VX_CHUNK_VOLUME + voxel_index[i]).second) {
            es.push_back(slots[i]);
            ei.push_back(voxel_index[i]);
            et.push_back(block_types[i]);
        }
    const std::vector<int32_t> touched = unique_ids(es, b->n_chunks);
    const size_t m = touched.size(), k = es.size();
    std::vector<int32_t> staged; // distinct slots, then slot, voxel index and type of each edit
    staged.reserve(m + 3 * k);
    staged.insert(staged.end(), touched.begin(), touched.end());
    staged.insert(staged.end(), es.begin(), es.end());
    staged.insert(staged.end(), ei.begin(), ei.end());
    staged.insert(staged.end(), et.begin(), et.end());
    VX_CUDA(ctx, ctx->tmp_a.reserve(sizeof(int32_t) * staged.size()));
    int32_t *d = ctx->tmp_a.as<int32_t>();
    VX_CUDA(ctx, cudaMemcpyAsync(d, staged.data(), sizeof(int32_t) * staged.size(), cudaMemcpyHostToDevice, ctx->stream));
    materialize_uniform_kernel<<<(unsigned)m, EDIT_THREADS, 0, ctx->stream>>>(b->world_voxels.as<uint8_t>(), b->world_flags.as<uint8_t>(), d);
    VX_CHECK_LAUNCH(ctx);
    scatter_blocks_kernel<<<(unsigned)((k + 255) / 256), 256, 0, ctx->stream>>>(b->world_voxels.as<uint8_t>(), d + m, d + m + k, d + m + 2 * k,
                                                                                  (int32_t)k);
    VX_CHECK_LAUNCH(ctx);
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); // `staged` goes out of scope
    return VX_OK;
}

} // extern "C"
