// kp_grid.cuh -- device view of the uniform-grid spatial hash (K3) shared by the neighbour
// kernels (kp_grid.cu) and the ICP correspondence kernel (kp_icp.cu).
#pragma once
#include "kp_common.cuh"

struct KpGridDev {
    const float4 *pts;        // sorted by cell key; .w = original index (int bits)
    const uint4 *slots;       // open addressing, 16-byte slots {key lo, key hi, start, end}; key ~0 = empty.
                              // One 128-bit load returns the key AND the cell's [start,end) run in pts.
    uint32_t hmask;
    int sh_x, sh_y;           // key = cx << sh_x | cy << sh_y | cz   (cz is the low field: the cells of a
                              // z-row are adjacent in the sorted array)
    int dim[3];
    int npts;                 // rows of pts (NaN rows, if any, sit at the end)
    const uint2 *cellmap;     // per 32 cells (cell index (cx*dim1 + cy)*dim2 + cz): {~occupancy bits, rank of the
                              // first occupied cell of the word among all occupied cells}; NULL when the grid is
                              // too large (then the hash is used).  rank -> run_start[rank] is the cell's first
                              // point: one 8-byte load + a popcount replaces hashing and probing, and because
                              // ranks follow the sort order a whole z-row resolves to ONE contiguous run.
    const int32_t *run_start; // [occupied cells + 1] first position of each occupied cell's run in pts
    double org[3];
    double cell, inv_cell;
};

#ifdef __CUDACC__
__device__ __forceinline__ int kp_cell_coord(const KpGridDev &g, double v, int c)
{
    return (int)floor(__dmul_rn(__dsub_rn(v, g.org[c]), g.inv_cell));
}
__device__ __forceinline__ uint64_t kp_cell_key(const KpGridDev &g, int cx, int cy, int cz)
{
    return ((uint64_t)(uint32_t)cx << g.sh_x) | ((uint64_t)(uint32_t)cy << g.sh_y) | (uint64_t)(uint32_t)cz;
}
__device__ __forceinline__ uint64_t kp_slot_key(const uint4 &s) { return ((uint64_t)s.y << 32) | s.x; }
// [start,end) of the cells (cx, cy, zlo..zhi), zhi - zlo <= 31, through the cell map.  Branch-free: the two
// map words and the two run boundaries are loaded unconditionally, so lookups of several columns overlap.
__device__ __forceinline__ int2 kp_map_range(const KpGridDev &g, int cx, int cy, int zlo, int zhi)
{
    const long long base = ((long long)cx * g.dim[1] + cy) * g.dim[2];
    const long long lo = base + zlo, hi = base + zhi;
    const long long wa = lo >> 5, wb = hi >> 5;
    const uint2 A = __ldg(g.cellmap + wa);
    const uint2 B = __ldg(g.cellmap + wb);
    const bool same = wa == wb;
    const unsigned below = (1u << (lo & 31)) - 1u, upto = (2u << (hi & 31)) - 1u;
    const unsigned occa = ~A.x, occb = ~B.x;
    const int ca = __popc(occa & ~below & (same ? upto : 0xffffffffu));
    const int cb = same ? 0 : __popc(occb & upto);
    const int cnt = ca + cb;
    int first = ca ? (int)A.y + __popc(occa & below) : (int)B.y;
    first = cnt ? first : 0;
    return make_int2(__ldg(g.run_start + first), __ldg(g.run_start + first + cnt));
}
// fp32 squared distance of the neighbour kernels' candidate passes (relative error < 6e-7, DESIGN §3): it chooses which
// candidates the double expression kp_d2 has to decide, it never decides one itself
__device__ __forceinline__ float hq_d32(float qx, float qy, float qz, const float4 &c)
{
    const float dx = qx - c.x, dy = qy - c.y, dz = qz - c.z;
    return __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, dx * dx));
}
// resolve a probe sequence that starts at slot h with the already loaded slot s
__device__ __forceinline__ int2 kp_slot_resolve(const KpGridDev &g, uint64_t key, uint32_t h, uint4 s)
{
    for (;;) {
        const uint64_t k = kp_slot_key(s);
        if (k == key) return make_int2((int)s.z, (int)s.w);
        if (k == ~0ull) return make_int2(0, 0);
        h = (h + 1) & g.hmask;
        s = __ldg(g.slots + h);
    }
}
// [start,end) of a cell, (0,0) when empty or outside the grid
__device__ __forceinline__ int2 kp_cell_range(const KpGridDev &g, int cx, int cy, int cz)
{
    if ((unsigned)cx >= (unsigned)g.dim[0] || (unsigned)cy >= (unsigned)g.dim[1] || (unsigned)cz >= (unsigned)g.dim[2])
        return make_int2(0, 0);
    if (g.cellmap) return kp_map_range(g, cx, cy, cz, cz);
    const uint64_t key = kp_cell_key(g, cx, cy, cz);
    const uint32_t h = (uint32_t)kp_mix64(key) & g.hmask;
    return kp_slot_resolve(g, key, h, __ldg(g.slots + h));
}
// Merged [start,end) of the z-row (cx, cy, cz-1 .. cz+1): the three cells are adjacent in pts, so the
// union of the non-empty ones is one contiguous run.  Cell-map path: one or two 8-byte loads, then the two
// run boundaries.  Hash path (huge grids): the three first probes are issued together.
__device__ __forceinline__ int2 kp_row_range(const KpGridDev &g, int cx, int cy, int cz)
{
    if ((unsigned)cx >= (unsigned)g.dim[0] || (unsigned)cy >= (unsigned)g.dim[1]) return make_int2(0, 0);
    if (g.cellmap) {
        const int zlo = max(cz - 1, 0), zhi = min(cz + 1, g.dim[2] - 1);
        if (zlo > zhi) return make_int2(0, 0);
        return kp_map_range(g, cx, cy, zlo, zhi);
    }
    bool act[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) act[j] = (unsigned)(cz - 1 + j) < (unsigned)g.dim[2];
    uint64_t key[3];
    uint32_t h[3];
    uint4 s[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        key[j] = kp_cell_key(g, cx, cy, cz - 1 + j);
        h[j] = (uint32_t)kp_mix64(key[j]) & g.hmask;
        s[j] = make_uint4(0xffffffffu, 0xffffffffu, 0u, 0u);
        if (act[j]) s[j] = __ldg(g.slots + h[j]);
    }
    int a = 0x7fffffff, b = 0;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        if (!act[j]) continue;
        const int2 r = kp_slot_resolve(g, key[j], h[j], s[j]);
        if (r.y > r.x) { a = min(a, r.x); b = max(b, r.y); }
    }
    return b > 0 ? make_int2(a, b) : make_int2(0, 0);
}
// [start,end) of the cells (cx, cy, zlo..zhi) (clamped to the grid): one contiguous run of pts
__device__ __forceinline__ int2 kp_span_range(const KpGridDev &g, int cx, int cy, int zlo, int zhi)
{
    if ((unsigned)cx >= (unsigned)g.dim[0] || (unsigned)cy >= (unsigned)g.dim[1]) return make_int2(0, 0);
    zlo = max(zlo, 0); zhi = min(zhi, g.dim[2] - 1);
    if (zlo > zhi) return make_int2(0, 0);
    if (g.cellmap) return kp_map_range(g, cx, cy, zlo, zhi);
    int a = 0x7fffffff, b = 0;
    for (int z = zlo; z <= zhi; ++z) {
        const int2 r = kp_cell_range(g, cx, cy, z);
        if (r.y > r.x) { a = min(a, r.x); b = max(b, r.y); }
    }
    return b > 0 ? make_int2(a, b) : make_int2(0, 0);
}
#endif

KpGridDev kp_grid_dev(const KpGrid &g);
