// kp_engine.cu -- device-driven, batched whole-frame engine behind kp_pipeline_* (BASELINE config C4).
// Per frame: unproject + transform + fuse (preprocessing/data.py:44-58) -> filter_outliers
// (preprocessing/filtering.py:23-24: voxel + SOR) -> floor removal (floor_removal.py:64-73: band,
// segment_plane, invert-select, merge, SOR) -> point-to-plane ICP refinement of every sub extrinsic
// (preprocessing/registration.py:65-86: voxel, normals, registration_icp).
//
// Frames are independent (the reference loop at preprocessing/data.py:35 is a pure map).  The engine processes
// them in BATCHES of B frames: every kernel of a stage is launched once for the whole batch (blockIdx.y = frame
// or cloud), every count a later kernel needs (valid points, voxels, kept points, band sizes, straggler lists,
// RANSAC tallies, ICP convergence) stays in device memory, and grids are persistent over a static capacity.  A
// batch is therefore a fixed launch sequence with NO host round trip: it is captured once as a CUDA graph
// (main branch + a forked ICP branch) and replayed by ONE host thread on a few batch slots, each with its own
// stream pair and buffers, so the GPU always has several batches in flight.
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include "kp_batch.cuh"

int kp_unproject_engine(kp_ctx *ctx, const uint16_t *d_depth, const float *d_xytab, const double *h_T, int B, int S, int64_t P,
                        int flags, double scale, float *d_xyz, float *d_xyz_raw, int32_t *d_slots, int32_t *d_rows,
                        const uint8_t *d_rgb, const double *d_crop_med, double crop_gate);
size_t kp_unproject_engine_slots(int B, int S, int64_t P);
int kp_crop_median_engine(kp_ctx *ctx, const uint16_t *d_depth, const uint32_t *d_vbits, int B, int S, int64_t P, uint32_t *d_hist,
                          double *d_med);
size_t kp_crop_median_hist_elems();
int kp_resample_engine(kp_ctx *ctx, const float *const *d_base, int64_t stride, const int32_t *d_n, int64_t n_step, int B, int64_t N, int mode,
                       uint64_t seed, const int64_t *h_ids, int32_t *d_status, int64_t status_step, uint32_t *keys, uint32_t *hist,
                       void *st, unsigned long long *list, float *d_out);
size_t kp_resample_engine_hist_elems();
size_t kp_resample_engine_state_bytes();
int64_t kp_resample_engine_cap(int64_t N);
bool kp_resample_engine_fits(int64_t N);

namespace {
constexpr int ENG_MAX_S = 6;
constexpr int ENG_MAX_CAND = 16;       // RANSAC hypotheses that may tie on the winning inlier count

// one ICP cloud (frame b, sensor s): [b * S + s], uniform stride so that all of them are segments of one launch
struct EngCloud {
    int32_t nv, n;                      // valid rows of the ICP input, voxel count
    float b6[6];
    KpVoxDev vox;
};
// per-frame state produced and consumed on the device
struct EngDyn {
    int32_t n_fused, n_voxel, n_sor, n_lo, n_rest, n_merged, n_fsor, n_out;
    int32_t status, floor_skip, ymax_enc, n_ror;    // n_ror: survivors of the radius outlier removal (0 when it is off)
    int32_t nocc[4];                    // occupied cells of grid g[0..3]
    int32_t cnt_l0[3], cnt_l1[3];       // level-0 / level-1 leftover lists of the three neighbour searches
    int32_t cnt_lm[3], nocc_m[2], pad3; // leftovers of the mid level; occupied cells of the mid grids
    int32_t n_old[3], pad2;             // points the GRID level 0 has to search: 0 when the voxel-brick index was built
    int32_t ransac_best, ransac_ncand, ransac_cand[ENG_MAX_CAND];
    float b6[6];                        // bounds of the fused cloud
    KpVoxDev vox_fused;
    KpGridDev g[4];                     // [0],[1]: level 0 / 1 of the main branch, [2],[3]: of the ICP target
    KpGridDev gm[2];                    // mid-level grids (main branch, ICP target)
    KpVbiDev vbi[2];                    // voxel-brick index: [0] main branch (SOR clouds), [1] ICP target
    double sor_sum, sor_sq, sor_stats[3];
    double plane[4];
    double cand_sq[ENG_MAX_CAND];
    double icp_T[5][16], icp_fit[5], icp_rmse[5];
    int32_t icp_iters[5], pad1;
    double refit_c[4];                  // floor refit: centroid of the winning hypothesis's inliers, their count
    double floor_plane[4];              // the frame's floor plane (RANSAC mode): kp_frame_result.floor_plane
};

__device__ __forceinline__ int bit_length_dev(long long v)
{
    int b = 0;
    while (v > 0) { ++b; v >>= 1; }
    return b < 1 ? 1 : b;
}

// voxel grid of a cloud from its bounds: the arithmetic of kp_voxel_device (kp_voxel.cu), on the device
__device__ void vox_setup(const float *b6, int nvalid, double voxel, KpVoxDev &vp, int32_t &status)
{
    vp.voxel = voxel; vp.ok = 0; vp.sh_x = vp.sh_y = 0; vp.sentinel = 0xffffffffu;
    for (int c = 0; c < 3; ++c) { vp.minb[c] = 0.0; vp.imax[c] = 0; }
    if (nvalid <= 0) return;
    int bits[3];
    for (int c = 0; c < 3; ++c) {
        vp.minb[c] = __dsub_rn((double)b6[c], __dmul_rn(voxel, 0.5));
        const double maxb = __dadd_rn((double)b6[3 + c], __dmul_rn(voxel, 0.5));
        if (__dmul_rn(voxel, 2147483647.0) < __dsub_rn(maxb, vp.minb[c])) { status = KP_E_RANGE; return; }
        const long long imax = (long long)floor(__ddiv_rn(__dsub_rn((double)b6[3 + c], vp.minb[c]), voxel));
        bits[c] = bit_length_dev(imax);
        vp.imax[c] = (int)(imax < 0x7fffffff ? imax : 0x7fffffff);
    }
    vp.sh_y = bits[2];
    vp.sh_x = bits[2] + bits[1];
    const int total = bits[0] + bits[1] + bits[2];
    if (total + 1 > 32) { status = KP_E_RANGE; return; }     // the engine sorts 32-bit keys (index + one sentinel bit)
    vp.sentinel = 1u << total;
    vp.ok = 1;
}

// ---------------------------------------------------------------- frame setup (one thread per frame)
struct SetupParams {
    EngDyn *dyn; EngCloud *icl; const int32_t *rows;     // K1 bounds rows [B][S][2][8]
    int S; double voxel, icp_voxel; int do_icp;     // do_icp: the rows carry a second set (the ICP inputs)
};
__global__ void k_e_frame_setup(const __grid_constant__ SetupParams p, int B)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= B) return;
    EngDyn &d = p.dyn[f];
    const int sets = p.do_icp ? 2 : 1;
    const int32_t *rows = p.rows + (size_t)f * p.S * sets * 8;
    d.status = KP_OK; d.floor_skip = 0; d.ymax_enc = kp_f2ord(-INFINITY);
    d.n_voxel = d.n_sor = d.n_lo = d.n_rest = d.n_merged = d.n_fsor = d.n_out = 0;
    d.ransac_best = -1; d.ransac_ncand = 0;
    for (int i = 0; i < 3; ++i) { d.cnt_l0[i] = 0; d.cnt_l1[i] = 0; d.cnt_lm[i] = 0; }
    // fused bounds = union over the sensors that saw anything (set 0 rows)
    float b6[6] = {INFINITY, INFINITY, INFINITY, -INFINITY, -INFINITY, -INFINITY};
    int nvalid = 0;
    for (int s = 0; s < p.S; ++s) {
        const int32_t *r = rows + (size_t)(sets * s) * 8;
        if (r[6] <= 0) continue;
        nvalid += r[6];
        for (int c = 0; c < 3; ++c) { b6[c] = fminf(b6[c], kp_ord2f(r[c])); b6[3 + c] = fmaxf(b6[3 + c], kp_ord2f(r[3 + c])); }
    }
    int32_t status = KP_OK;
    for (int c = 0; c < 6; ++c) d.b6[c] = b6[c];
    vox_setup(b6, nvalid, p.voxel, d.vox_fused, status);
    d.n_fused = nvalid;
    for (int s = 0; s < p.S && p.do_icp; ++s) {
        const int32_t *r = rows + (size_t)(2 * s + 1) * 8;
        EngCloud &cl = p.icl[(size_t)f * p.S + s];
        for (int c = 0; c < 6; ++c) cl.b6[c] = kp_ord2f(r[c]);
        cl.nv = r[6];
        cl.n = 0;
        cl.vox.ok = 0;
        if (p.do_icp) vox_setup(cl.b6, r[6], p.icp_voxel, cl.vox, status);
        if (!cl.vox.ok) cl.nv = 0;
    }
    if (!d.vox_fused.ok) d.n_fused = 0;      // empty or out of range: every later stage sees an empty cloud
    d.status = status;
}

// ---------------------------------------------------------------- voxel downsample (keys -> sort -> heads -> mean)
struct VoxArgs {
    const float *xyz; int64_t xyz_stride;      // rows per segment
    int64_t n;                                 // rows per segment (static)
    const KpVoxDev *vp; int64_t vp_stride;     // bytes between the segments' KpVoxDev
    uint32_t *keys; int64_t key_stride;
};
__device__ __forceinline__ const KpVoxDev &vox_of(const KpVoxDev *vp, int64_t stride_bytes, int seg)
{
    return *reinterpret_cast<const KpVoxDev *>(reinterpret_cast<const char *>(vp) + seg * stride_bytes);
}
__device__ __forceinline__ uint32_t vox_key(const KpVoxDev &vp, float x, float y, float z)
{
    if (!vp.ok || isnan(x)) return vp.sentinel;
    const long long ix = (long long)floor(__ddiv_rn(__dsub_rn((double)x, vp.minb[0]), vp.voxel));
    const long long iy = (long long)floor(__ddiv_rn(__dsub_rn((double)y, vp.minb[1]), vp.voxel));
    const long long iz = (long long)floor(__ddiv_rn(__dsub_rn((double)z, vp.minb[2]), vp.voxel));
    return (uint32_t)(((unsigned long long)ix << vp.sh_x) | ((unsigned long long)iy << vp.sh_y) | (unsigned long long)iz);
}
__global__ void __launch_bounds__(256) k_e_voxel_keys(const __grid_constant__ VoxArgs a)
{
    const int seg = blockIdx.y;
    const KpVoxDev vp = vox_of(a.vp, a.vp_stride, seg);
    const float *xyz = a.xyz + 3 * seg * a.xyz_stride;
    uint32_t *keys = a.keys + seg * a.key_stride;
    // A thread owns FOUR CONSECUTIVE rows = 48 bytes = three 16-byte loads, and writes their keys as one 16-byte store; two
    // such groups per trip, all six loads issued before the first division.  (Key strides are multiples of 64 rows and the
    // arenas 256-byte aligned, so every key group is 16-byte aligned.)  The kernel is a stream of 12-byte rows in and
    // 4-byte keys out: the three IEEE double divisions per row are latency, not throughput.
    constexpr int U = 2;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if ((((uintptr_t)xyz) & 15u) != 0u) {
        // The input clouds (fused S * P rows per frame, raw P rows per sensor) are not padded: when P is not a multiple
        // of 4 a segment after the first starts off the 16-byte grid, and its rows are read one by one.
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += stride)
            keys[i] = vox_key(vp, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]);
        return;
    }
    const int64_t groups = a.n / 4;
    const float4 *x4 = reinterpret_cast<const float4 *>(xyz);
    uint4 *k4 = reinterpret_cast<uint4 *>(keys);
    for (int64_t g0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g0 < groups; g0 += U * stride) {
        float4 v[U][3];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t g = g0 + u * stride;
            if (g < groups) { v[u][0] = x4[3 * g]; v[u][1] = x4[3 * g + 1]; v[u][2] = x4[3 * g + 2]; }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t g = g0 + u * stride;
            if (g >= groups) break;
            uint4 k;
            k.x = vox_key(vp, v[u][0].x, v[u][0].y, v[u][0].z);
            k.y = vox_key(vp, v[u][0].w, v[u][1].x, v[u][1].y);
            k.z = vox_key(vp, v[u][1].z, v[u][1].w, v[u][2].x);
            k.w = vox_key(vp, v[u][2].y, v[u][2].z, v[u][2].w);
            k4[g] = k;
        }
    }
    // rows beyond the last full group (n not a multiple of 4)
    if (blockIdx.x == 0)
        for (int64_t i = groups * 4 + threadIdx.x; i < a.n; i += blockDim.x) keys[i] = vox_key(vp, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]);
}
// one thread per voxel run: sums its points in input order (the sort is stable) in double, one division, one rounding
struct VoxMeanArgs {
    const float *xyz; int64_t xyz_stride;
    const int32_t *vals; int64_t val_stride;
    const int32_t *run_start; int64_t rs_stride;
    DCnt R;
    float *out; int64_t out_stride;
    const uint32_t *keys; int64_t key_stride;          // sorted keys (voxel index of a run = key of its first row)
    const KpVoxDev *vp; int64_t vp_stride;
    uint32_t *vijk;                                    // nullable: packed voxel coordinates per output row (stride out_stride)
};
__global__ void __launch_bounds__(128) k_e_voxel_mean(const __grid_constant__ VoxMeanArgs a)
{
    const int seg = blockIdx.y;
    const int R = a.R.at(seg);
    const float *xyz = a.xyz + 3 * seg * a.xyz_stride;
    const int32_t *vals = a.vals + seg * a.val_stride, *rs = a.run_start + seg * a.rs_stride;
    float *out = a.out + 3 * seg * a.out_stride;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < R; r += gridDim.x * blockDim.x) {
        const int lo = rs[r], hi = rs[r + 1];
        double sx = 0, sy = 0, sz = 0;
        for (int t = lo; t < hi; ++t) {
            const int64_t i = vals[t];
            sx = __dadd_rn(sx, (double)xyz[3 * i]);
            sy = __dadd_rn(sy, (double)xyz[3 * i + 1]);
            sz = __dadd_rn(sz, (double)xyz[3 * i + 2]);
        }
        const double cnt = (double)(hi - lo);
        out[3 * (int64_t)r] = (float)__ddiv_rn(sx, cnt);
        out[3 * (int64_t)r + 1] = (float)__ddiv_rn(sy, cnt);
        out[3 * (int64_t)r + 2] = (float)__ddiv_rn(sz, cnt);
        if (a.vijk) {
            const KpVoxDev &vp = vox_of(a.vp, a.vp_stride, seg);
            const uint32_t key = a.keys[seg * a.key_stride + lo];
            const uint32_t ix = key >> vp.sh_x, iy = (key >> vp.sh_y) & ((1u << (vp.sh_x - vp.sh_y)) - 1u), iz = key & ((1u << vp.sh_y) - 1u);
            a.vijk[seg * a.out_stride + r] = (ix << 20) | ((iy & 1023u) << 10) | (iz & 1023u);   // (10 bits each: checked by the index build)
        }
    }
}

// ---------------------------------------------------------------- neighbour grid by counting sort
// Layout on the device (mirror of grid_layout in kp_grid.cu), occupancy bits, ranks by a scan of the word
// popcounts, points per occupied cell by integer atomics, run starts by a scan, scatter.  The order of the points
// INSIDE a cell depends on the atomics' arrival order; every search result is canonical ((d2, index) order,
// certified in double), so the outputs do not.
struct GridArgs {
    KpGridDev *g; int64_t g_stride;            // bytes between the segments' grid structs
    const float *xyz; int64_t xyz_stride;      // rows
    DCnt n;
    const float *b6; int64_t b6_stride;        // floats; NULL -> derive from `parent`
    const KpGridDev *parent; double parent_mult;
    double cell;
    float4 *sorted; int64_t sorted_stride;
    uint2 *cellmap; int64_t map_stride;        // words
    int32_t *cell_cnt; int64_t cnt_stride;     // doubles as run_start after the scan
    int32_t *rank; int32_t *loc; int64_t tmp_stride;
    int64_t cap_cells;
    DOut nocc;
};
__device__ __forceinline__ KpGridDev &grid_of(KpGridDev *g, int64_t stride_bytes, int seg)
{
    return *reinterpret_cast<KpGridDev *>(reinterpret_cast<char *>(g) + seg * stride_bytes);
}
__global__ void k_eg_setup(const __grid_constant__ GridArgs a)
{
    const int seg = blockIdx.x;
    if (threadIdx.x != 0) return;
    KpGridDev &g = grid_of(a.g, a.g_stride, seg);
    const int n = a.n.at(seg);
    double lo[3], hi[3], cell = a.cell;
    if (a.b6) {
        const float *b = a.b6 + seg * a.b6_stride;
        for (int c = 0; c < 3; ++c) { lo[c] = (double)b[c]; hi[c] = (double)b[3 + c]; }
    } else {
        const KpGridDev &pg = grid_of(const_cast<KpGridDev *>(a.parent), a.g_stride, seg);
        for (int c = 0; c < 3; ++c) { lo[c] = (double)(float)pg.org[c]; hi[c] = (double)(float)(pg.org[c] + pg.cell * (double)pg.dim[c]); }
        cell = pg.cell * a.parent_mult;
    }
    g.pts = a.sorted + seg * a.sorted_stride;
    g.slots = nullptr; g.hmask = 0; g.sh_x = 0; g.sh_y = 0;
    g.cellmap = a.cellmap + seg * a.map_stride;
    g.run_start = a.cell_cnt + seg * a.cnt_stride;
    g.npts = n;
    if (n <= 0 || !(cell > 0.0)) {
        for (int c = 0; c < 3; ++c) { g.org[c] = 0.0; g.dim[c] = 0; }
        g.cell = cell > 0.0 ? cell : 1.0; g.inv_cell = 1.0 / g.cell;
        return;
    }
    for (;;) {
        bool ok = true;
        double ncell = 1.0;
        for (int c = 0; c < 3; ++c) {
            double ext = hi[c] - lo[c];
            if (!(ext >= 0)) ext = 0;
            if (ext / cell > 2000000.0) ok = false;
            ncell *= floor(ext / cell) + 2.0;
        }
        if (ok && ncell <= (double)a.cap_cells) break;
        cell *= 2.0;                            // a coarser cell never changes a result, only the cost of a search
    }
    g.cell = cell;
    g.inv_cell = 1.0 / cell;
    for (int c = 0; c < 3; ++c) {
        g.org[c] = lo[c];
        double ext = hi[c] - lo[c];
        if (!(ext >= 0)) ext = 0;
        g.dim[c] = (int)floor(ext * g.inv_cell) + 2;
    }
    // the capacity test above used ext / cell, the dims use ext * (1 / cell): one more doubling if they disagree
    while ((double)g.dim[0] * g.dim[1] * g.dim[2] > (double)a.cap_cells) {
        g.cell *= 2.0; g.inv_cell = 1.0 / g.cell;
        for (int c = 0; c < 3; ++c) { double ext = hi[c] - lo[c]; if (!(ext >= 0)) ext = 0; g.dim[c] = (int)floor(ext * g.inv_cell) + 2; }
    }
}
__device__ __forceinline__ long long grid_words(const KpGridDev &g)
{
    return ((long long)g.dim[0] * g.dim[1] * g.dim[2] + 31) / 32 + 1;
}
__global__ void __launch_bounds__(256) k_eg_clear(const __grid_constant__ GridArgs a)
{
    const int seg = blockIdx.y;
    const KpGridDev &g = grid_of(a.g, a.g_stride, seg);
    const long long words = grid_words(g);
    uint2 *map = a.cellmap + seg * a.map_stride;
    int32_t *cnt = a.cell_cnt + seg * a.cnt_stride;
    const int n = a.n.at(seg);
    const long long stride = (long long)gridDim.x * blockDim.x, t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long w = t0; w < words; w += stride) map[w] = make_uint2(0xffffffffu, 0u);
    for (long long i = t0; i <= n; i += stride) cnt[i] = 0;
}
__device__ __forceinline__ int eg_cell_of(const KpGridDev &g, float x, float y, float z)
{
    const int cx = min(max(kp_cell_coord(g, (double)x, 0), 0), g.dim[0] - 1);
    const int cy = min(max(kp_cell_coord(g, (double)y, 1), 0), g.dim[1] - 1);
    const int cz = min(max(kp_cell_coord(g, (double)z, 2), 0), g.dim[2] - 1);
    return (cx * g.dim[1] + cy) * g.dim[2] + cz;
}
__device__ __forceinline__ void eg_mark_cell(uint2 *map, int cell)
{
    const unsigned bit = 1u << (cell & 31);
    // (neighbouring points share cells: skip the atomic when the bit is already visible as set)
    if (map[cell >> 5].x & bit) atomicAnd(&map[cell >> 5].x, ~bit);
}
__global__ void __launch_bounds__(256) k_eg_mark(const __grid_constant__ GridArgs a)
{
    const int seg = blockIdx.y;
    const KpGridDev g = grid_of(a.g, a.g_stride, seg);
    const int n = a.n.at(seg);
    const float *xyz = a.xyz + 3 * seg * a.xyz_stride;
    uint2 *map = a.cellmap + seg * a.map_stride;
    int32_t *cellidx = a.rank + seg * a.tmp_stride;
    // four consecutive rows per thread: three 16-byte loads in, one 16-byte store of the cell indices out (segment strides
    // are multiples of 64 rows: every group is 16-byte aligned)
    const int groups = n / 4;
    const float4 *x4 = reinterpret_cast<const float4 *>(xyz);
    int4 *c4 = reinterpret_cast<int4 *>(cellidx);
    for (int gidx = blockIdx.x * blockDim.x + threadIdx.x; gidx < groups; gidx += gridDim.x * blockDim.x) {
        const float4 v0 = x4[3 * (int64_t)gidx], v1 = x4[3 * (int64_t)gidx + 1], v2 = x4[3 * (int64_t)gidx + 2];
        int4 c;
        c.x = eg_cell_of(g, v0.x, v0.y, v0.z);
        c.y = eg_cell_of(g, v0.w, v1.x, v1.y);
        c.z = eg_cell_of(g, v1.z, v1.w, v2.x);
        c.w = eg_cell_of(g, v2.y, v2.z, v2.w);
        c4[gidx] = c;
        eg_mark_cell(map, c.x);
        if (c.y != c.x) eg_mark_cell(map, c.y);
        if (c.z != c.y) eg_mark_cell(map, c.z);
        if (c.w != c.z) eg_mark_cell(map, c.w);
    }
    if (blockIdx.x == 0)
        for (int i = groups * 4 + threadIdx.x; i < n; i += blockDim.x) {
            const int cell = eg_cell_of(g, xyz[3 * (int64_t)i], xyz[3 * (int64_t)i + 1], xyz[3 * (int64_t)i + 2]);
            cellidx[i] = cell;
            eg_mark_cell(map, cell);
        }
}
// ranks: exclusive scan of the words' popcounts into .y (tile sums, last CTA scans them, apply)
__device__ __forceinline__ bool eg_last_block(unsigned int *ticket)
{
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1 : 0;
    __syncthreads();
    if (s_last) __threadfence();
    return s_last != 0;
}
__global__ void __launch_bounds__(256) k_eg_rank_reduce(const __grid_constant__ GridArgs a, BScan S)
{
    __shared__ int wc[8];
    __shared__ int carry_s;
    __shared__ int wtot[8];
    const int seg = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const KpGridDev &g = grid_of(a.g, a.g_stride, seg);
    const long long words = grid_words(g);
    const int ntiles = (int)((words + BC_TILE - 1) / BC_TILE);
    const uint2 *map = a.cellmap + seg * a.map_stride;
    int32_t *ts = S.tile_sum + (size_t)seg * S.max_tiles;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        int s = 0;
#pragma unroll
        for (int j = 0; j < BC_ITEMS; ++j) {
            const long long i = (long long)tile * BC_TILE + j * BC_THREADS + threadIdx.x;
            if (i < words) s += __popc(~map[i].x);
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) s += __shfl_xor_sync(KP_FULL, s, d);
        if (lane == 0) wc[w] = s;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int ww = 0; ww < 8; ++ww) t += wc[ww]; ts[tile] = t; }
        __syncthreads();
    }
    if (!eg_last_block(S.ticket + seg)) return;
    // exclusive scan of the tile sums by this CTA
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < ntiles; base += BC_THREADS) {
        const int i = base + threadIdx.x;
        const int x = i < ntiles ? __ldcg(ts + i) : 0;
        int incl = x;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) { const int y = __shfl_up_sync(KP_FULL, incl, s); if (lane >= s) incl += y; }
        if (lane == 31) wtot[w] = incl;
        __syncthreads();
        int woff = 0;
#pragma unroll
        for (int ww = 0; ww < 8; ++ww) woff += ww < w ? wtot[ww] : 0;
        const int excl = carry_s + woff + incl - x;
        if (i < ntiles) ts[i] = excl;
        __syncthreads();
        if (threadIdx.x == BC_THREADS - 1) carry_s = excl + x;
        __syncthreads();
    }
    if (threadIdx.x == 0) { a.nocc.at(seg) = carry_s; S.ticket[seg] = 0; }
}
__global__ void __launch_bounds__(256) k_eg_rank_apply(const __grid_constant__ GridArgs a, BScan S)
{
    __shared__ int wtot[8];
    const int seg = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const KpGridDev &g = grid_of(a.g, a.g_stride, seg);
    const long long words = grid_words(g);
    const int ntiles = (int)((words + BC_TILE - 1) / BC_TILE);
    uint2 *map = a.cellmap + seg * a.map_stride;
    const int32_t *ts = S.tile_sum + (size_t)seg * S.max_tiles;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // thread t owns BC_ITEMS consecutive words
        const long long i0 = (long long)tile * BC_TILE + (long long)threadIdx.x * BC_ITEMS;
        int c[BC_ITEMS];
        int s = 0;
#pragma unroll
        for (int j = 0; j < BC_ITEMS; ++j) { c[j] = i0 + j < words ? __popc(~map[i0 + j].x) : 0; s += c[j]; }
        int incl = s;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(KP_FULL, incl, d); if (lane >= d) incl += y; }
        if (lane == 31) wtot[w] = incl;
        __syncthreads();
        int run = ts[tile] + incl - s;
#pragma unroll
        for (int ww = 0; ww < 8; ++ww) run += ww < w ? wtot[ww] : 0;
#pragma unroll
        for (int j = 0; j < BC_ITEMS; ++j) { if (i0 + j < words) map[i0 + j].y = (unsigned)run; run += c[j]; }
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256) k_eg_count(const __grid_constant__ GridArgs a)
{
    const int seg = blockIdx.y;
    const int n = a.n.at(seg);
    const uint2 *map = a.cellmap + seg * a.map_stride;
    int32_t *rank = a.rank + seg * a.tmp_stride, *loc = a.loc + seg * a.tmp_stride, *cnt = a.cell_cnt + seg * a.cnt_stride;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int cell = rank[i];
        const uint2 wd = map[cell >> 5];
        const int r = (int)wd.y + __popc(~wd.x & ((1u << (cell & 31)) - 1u));
        rank[i] = r;
        loc[i] = atomicAdd(&cnt[r], 1);
    }
}
__global__ void __launch_bounds__(256) k_eg_scatter(const __grid_constant__ GridArgs a)
{
    const int seg = blockIdx.y;
    const int n = a.n.at(seg);
    const float *xyz = a.xyz + 3 * seg * a.xyz_stride;
    const int32_t *rank = a.rank + seg * a.tmp_stride, *loc = a.loc + seg * a.tmp_stride, *rs = a.cell_cnt + seg * a.cnt_stride;
    float4 *sorted = a.sorted + seg * a.sorted_stride;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int pos = rs[rank[i]] + loc[i];
        sorted[pos] = make_float4(xyz[3 * (int64_t)i], xyz[3 * (int64_t)i + 1], xyz[3 * (int64_t)i + 2], __int_as_float(i));
    }
}

// ---------------------------------------------------------------- voxel-brick index (kp_vbi.cuh)
struct VbiArgs {
    KpVbiDev *v; int64_t v_stride;                  // bytes between the segments' index structs
    const float *xyz; int64_t xyz_stride;           // rows
    const uint32_t *vijk; int64_t vijk_stride;
    DCnt n;
    const KpVoxDev *vp; int64_t vp_stride;
    uint2 *bricks; int64_t brick_stride; int64_t cap_bricks;
    float4 *pts; uint32_t *vijk_sorted; int64_t pts_stride;
    int32_t *status; int64_t status_stride;         // int units
};
__device__ __forceinline__ KpVbiDev &vbi_of(KpVbiDev *v, int64_t stride_bytes, int seg)
{
    return *reinterpret_cast<KpVbiDev *>(reinterpret_cast<char *>(v) + seg * stride_bytes);
}
__global__ void k_vbi_setup(const __grid_constant__ VbiArgs a)
{
    const int seg = blockIdx.x;
    if (threadIdx.x != 0) return;
    KpVbiDev &v = vbi_of(a.v, a.v_stride, seg);
    const KpVoxDev &vp = vox_of(a.vp, a.vp_stride, seg);
    const int n = a.n.at(seg);
    v.bricks = a.bricks + seg * a.brick_stride;
    v.pts = a.pts + seg * a.pts_stride;
    v.vijk = a.vijk_sorted + seg * a.pts_stride;
    v.voxel = vp.voxel; v.inv_voxel = 1.0 / vp.voxel;
    v.npts = 0; v.ok = 0; v.eps = 0.0;
    double nbricks = 1.0, M = 0.0;
    bool fits = vp.ok && n > 0;
    for (int c = 0; c < 3; ++c) {
        v.minb[c] = vp.minb[c];
        const int sh = c == 0 ? 1 : 2;                // bricks of 2 x 4 x 4 voxels
        v.nb[c] = (vp.imax[c] >> sh) + 1 + 2 * KP_VBI_PAD;
        v.nvox[c] = ((vp.imax[c] >> sh) + 1) << sh;
        if (vp.imax[c] >= 1024) fits = false;
        nbricks *= (double)v.nb[c];
        M = fmax(M, fmax(fabs(vp.minb[c]), fabs(vp.minb[c] + vp.voxel * (double)v.nvox[c])));
    }
    if (nbricks > (double)a.cap_bricks) fits = false;
    if (!fits) { v.nb[0] = v.nb[1] = v.nb[2] = 0; return; }
    v.eps = M * (1.0 / 4194304.0);                  // 4 ulp of the largest float32 coordinate
    v.npts = n;
    v.ok = 1;
}
__global__ void __launch_bounds__(256) k_vbi_clear(const __grid_constant__ VbiArgs a)
{
    const int seg = blockIdx.y;
    const KpVbiDev &v = vbi_of(a.v, a.v_stride, seg);
    if (!v.ok) return;
    const long long nb = (long long)v.nb[0] * v.nb[1] * v.nb[2];
    uint2 *br = a.bricks + seg * a.brick_stride;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += (long long)gridDim.x * blockDim.x) br[i] = make_uint2(0u, 0u);
}
__device__ __forceinline__ void vbi_locate(const KpVbiDev &v, uint32_t ijk, long long &L, unsigned &bit)
{
    const int ix = (int)(ijk >> 20), iy = (int)((ijk >> 10) & 1023u), iz = (int)(ijk & 1023u);
    L = kp_vbi_brick_index(v, ix >> 1, iy >> 2, iz >> 2);
    bit = (unsigned)((ix & 1) * 16 + (iy & 3) * 4 + (iz & 3));
}
__global__ void __launch_bounds__(256) k_vbi_mark(const __grid_constant__ VbiArgs a)
{
    const int seg = blockIdx.y;
    const KpVbiDev v = vbi_of(a.v, a.v_stride, seg);
    if (!v.ok) return;
    const uint32_t *vijk = a.vijk + seg * a.vijk_stride;
    uint2 *br = a.bricks + seg * a.brick_stride;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < v.npts; i += gridDim.x * blockDim.x) {
        long long L; unsigned bit;
        vbi_locate(v, vijk[i], L, bit);
        const unsigned m = 1u << bit;
        // a second point in the same voxel cannot happen on a voxel-downsampled cloud; if it does, say so
        if (atomicOr(&br[L].x, m) & m) a.status[seg * a.status_stride] = KP_E_RANGE;
    }
}
__global__ void __launch_bounds__(256) k_vbi_rank_reduce(const __grid_constant__ VbiArgs a, BScan S)
{
    __shared__ int wc[8];
    __shared__ int carry_s;
    __shared__ int wtot[8];
    const int seg = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const KpVbiDev &v = vbi_of(a.v, a.v_stride, seg);
    const long long nb = v.ok ? (long long)v.nb[0] * v.nb[1] * v.nb[2] : 0;
    const int ntiles = (int)((nb + BC_TILE - 1) / BC_TILE);
    const uint2 *br = a.bricks + seg * a.brick_stride;
    int32_t *ts = S.tile_sum + (size_t)seg * S.max_tiles;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        int s = 0;
#pragma unroll
        for (int j = 0; j < BC_ITEMS; ++j) {
            const long long i = (long long)tile * BC_TILE + j * BC_THREADS + threadIdx.x;
            if (i < nb) s += __popc(br[i].x);
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) s += __shfl_xor_sync(KP_FULL, s, d);
        if (lane == 0) wc[w] = s;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int ww = 0; ww < 8; ++ww) t += wc[ww]; ts[tile] = t; }
        __syncthreads();
    }
    if (!eg_last_block(S.ticket + seg)) return;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < ntiles; base += BC_THREADS) {
        const int i = base + threadIdx.x;
        const int x = i < ntiles ? __ldcg(ts + i) : 0;
        int incl = x;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) { const int y = __shfl_up_sync(KP_FULL, incl, s); if (lane >= s) incl += y; }
        if (lane == 31) wtot[w] = incl;
        __syncthreads();
        int woff = 0;
#pragma unroll
        for (int ww = 0; ww < 8; ++ww) woff += ww < w ? wtot[ww] : 0;
        const int excl = carry_s + woff + incl - x;
        if (i < ntiles) ts[i] = excl;
        __syncthreads();
        if (threadIdx.x == BC_THREADS - 1) carry_s = excl + x;
        __syncthreads();
    }
    if (threadIdx.x == 0) S.ticket[seg] = 0;
}
__global__ void __launch_bounds__(256) k_vbi_rank_apply(const __grid_constant__ VbiArgs a, BScan S)
{
    __shared__ int wtot[8];
    const int seg = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const KpVbiDev &v = vbi_of(a.v, a.v_stride, seg);
    const long long nb = v.ok ? (long long)v.nb[0] * v.nb[1] * v.nb[2] : 0;
    const int ntiles = (int)((nb + BC_TILE - 1) / BC_TILE);
    uint2 *br = a.bricks + seg * a.brick_stride;
    const int32_t *ts = S.tile_sum + (size_t)seg * S.max_tiles;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long i0 = (long long)tile * BC_TILE + (long long)threadIdx.x * BC_ITEMS;
        int c[BC_ITEMS];
        int s = 0;
#pragma unroll
        for (int j = 0; j < BC_ITEMS; ++j) {
            c[j] = i0 + j < nb ? __popc(br[i0 + j].x) : 0;
            s += c[j];
        }
        int incl = s;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(KP_FULL, incl, d); if (lane >= d) incl += y; }
        if (lane == 31) wtot[w] = incl;
        __syncthreads();
        int run = ts[tile] + incl - s;
#pragma unroll
        for (int ww = 0; ww < 8; ++ww) run += ww < w ? wtot[ww] : 0;
#pragma unroll
        for (int j = 0; j < BC_ITEMS; ++j) { if (c[j]) br[i0 + j].y = (unsigned)run; run += c[j]; }   // only occupied bricks are ever asked
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256) k_vbi_scatter(const __grid_constant__ VbiArgs a)
{
    const int seg = blockIdx.y;
    const KpVbiDev v = vbi_of(a.v, a.v_stride, seg);
    if (!v.ok) return;
    const float *xyz = a.xyz + 3 * seg * a.xyz_stride;
    const uint32_t *vijk = a.vijk + seg * a.vijk_stride;
    const uint2 *br = a.bricks + seg * a.brick_stride;
    float4 *pts = a.pts + seg * a.pts_stride;
    uint32_t *vs = a.vijk_sorted + seg * a.pts_stride;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < v.npts; i += gridDim.x * blockDim.x) {
        long long L; unsigned bit;
        const uint32_t ijk = vijk[i];
        vbi_locate(v, ijk, L, bit);
        const uint2 e = br[L];
        const int pos = (int)e.y + __popc(e.x & ((1u << bit) - 1u));
        pts[pos] = make_float4(xyz[3 * (int64_t)i], xyz[3 * (int64_t)i + 1], xyz[3 * (int64_t)i + 2], __int_as_float(i));
        vs[pos] = ijk;
    }
}

// ---------------------------------------------------------------- SOR mask, floor band, RANSAC
struct SorMaskArgs {
    const double *mean; int64_t mean_stride;
    DCnt n;
    EngDyn *dyn;
    double ratio;
    uint8_t *keep; int64_t keep_stride;
};
__global__ void __launch_bounds__(256) k_e_sor_mask(const __grid_constant__ SorMaskArgs a)
{
    const int seg = blockIdx.y;
    const int n = a.n.at(seg);
    EngDyn &d = a.dyn[seg];
    const double valid = (double)n;
    const double mu = __ddiv_rn(d.sor_sum, valid);
    const double sd = sqrt(__ddiv_rn(d.sor_sq, __dsub_rn(valid, 1.0)));
    const double thr = __dadd_rn(mu, __dmul_rn(a.ratio, sd));
    const double *mean = a.mean + seg * a.mean_stride;
    uint8_t *keep = a.keep + seg * a.keep_stride;
    if (blockIdx.x == 0 && threadIdx.x == 0) { d.sor_stats[0] = mu; d.sor_stats[1] = sd; d.sor_stats[2] = thr; }
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const double m = mean[i];
        keep[i] = (m > 0 && m < thr) ? 1 : 0;
    }
}
// remove_radius_outlier (SURVEY A.4): keep[row] = #{j : d2(i, j) < r2} > nb, the point itself included.  One thread per
// query in the grid's cell-sorted order, so that neighbouring threads read the same candidate cells (L1).  The cell is
// >= the radius: every neighbour lies in the 27-cell block, whose 9 z-columns are one run each.  fp32 chooses and double
// decides: a candidate whose fp32 d2 lies within the 1e-6 margins of r2 is decided by kp_d2 (DESIGN §3).  Counting stops
// at nb + 1, so a dense surface costs a few candidates per query whatever nb is.
struct RorArgs {
    const KpGridDev *g; int64_t g_stride;      // bytes between the segments' grids
    DCnt n;
    int nb; double r2; float r2_lo, r2_hi;     // r2_lo / r2_hi: r2 (1 -+ 1e-6) rounded down / up to fp32
    uint8_t *keep; int64_t keep_stride;
};
__global__ void __launch_bounds__(128, 8) k_e_ror_count(const __grid_constant__ RorArgs a)
{
    const int seg = blockIdx.y;
    const int n = a.n.at(seg);
    const KpGridDev g = *reinterpret_cast<const KpGridDev *>(reinterpret_cast<const char *>(a.g) + seg * a.g_stride);
    uint8_t *keep = a.keep + seg * a.keep_stride;
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < n; w += gridDim.x * blockDim.x) {
        const float4 me = __ldg(g.pts + w);
        int cnt = 0;
        if (!isnan(me.x)) {
            const int cx = min(max(kp_cell_coord(g, (double)me.x, 0), 0), g.dim[0] - 1);
            const int cy = min(max(kp_cell_coord(g, (double)me.y, 1), 0), g.dim[1] - 1);
            const int cz = min(max(kp_cell_coord(g, (double)me.z, 2), 0), g.dim[2] - 1);
            int2 rng[9];
#pragma unroll
            for (int ci = 0; ci < 9; ++ci) {
                constexpr int order[9] = {4, 1, 3, 5, 7, 0, 2, 6, 8};     // own column first: the likeliest to end the count
                rng[ci] = kp_row_range(g, cx + order[ci] / 3 - 1, cy + order[ci] % 3 - 1, cz);
            }
#pragma unroll
            for (int ci = 0; ci < 9; ++ci) {
                // four candidates per trip: their loads are in flight together
                for (int t = rng[ci].x; t < rng[ci].y && cnt <= a.nb; t += 4) {
                    float4 c[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) c[u] = __ldg(g.pts + min(t + u, rng[ci].y - 1));
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (t + u >= rng[ci].y) break;
                        const float d = hq_d32(me.x, me.y, me.z, c[u]);
                        if (d < a.r2_lo) ++cnt;
                        else if (!(d > a.r2_hi) && kp_d2((double)me.x, (double)me.y, (double)me.z, (double)c[u].x, (double)c[u].y, (double)c[u].z) < a.r2)
                            ++cnt;
                    }
                }
            }
        }
        keep[__float_as_int(me.w)] = cnt > a.nb ? 1 : 0;
    }
}

struct BandArgs {
    const float *xyz; int64_t stride; DCnt n; EngDyn *dyn; int axis; double band; int ransac_n;
    uint8_t *lower; int64_t mask_stride;
};
__global__ void __launch_bounds__(256) k_e_axis_max(const __grid_constant__ BandArgs a)
{
    __shared__ float wm[8];
    const int seg = blockIdx.y;
    const int n = a.n.at(seg);
    const float *xyz = a.xyz + 3 * seg * a.stride;
    float m = -INFINITY;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float v = xyz[3 * (int64_t)i + a.axis];
        if (!isnan(xyz[3 * (int64_t)i])) m = fmaxf(m, v);
    }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) m = fmaxf(m, __shfl_xor_sync(KP_FULL, m, s));
    if ((threadIdx.x & 31) == 0) wm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) m = fmaxf(m, wm[w]);
        const int o = kp_f2ord(m);
        int32_t *enc = &a.dyn[seg].ymax_enc;
        if (o > *(volatile int32_t *)enc) atomicMax(enc, o);
    }
}
__global__ void __launch_bounds__(256) k_e_band_mask(const __grid_constant__ BandArgs a)
{
    const int seg = blockIdx.y;
    const int n = a.n.at(seg);
    EngDyn &d = a.dyn[seg];
    const float *xyz = a.xyz + 3 * seg * a.stride;
    uint8_t *lower = a.lower + seg * a.mask_stride;
    const double lim = __dsub_rn((double)kp_ord2f(d.ymax_enc), a.band);
    if (blockIdx.x == 0 && threadIdx.x == 0) d.floor_skip = n < a.ransac_n ? 1 : 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float v = xyz[3 * (int64_t)i + a.axis];
        lower[i] = !isnan(xyz[3 * (int64_t)i]) && (double)v >= lim;
    }
}

#define DM(a, b) __dmul_rn((a), (b))
#define DA(a, b) __dadd_rn((a), (b))
#define DS(a, b) __dsub_rn((a), (b))
#define DD(a, b) __ddiv_rn((a), (b))
constexpr int RS_MAX_N = 64;
struct RansacArgs {
    const float *xyz; int64_t stride; DCnt n; EngDyn *dyn;
    int ransac_n, iters; uint64_t seed; double thr, probability;
    double4 *planes; uint8_t *pvalid; unsigned long long *cnt; int64_t h_stride;   // [seg][iters]
    double *slots; int nblk;                                                       // [seg][ENG_MAX_CAND][nblk]
    uint8_t *mask; int64_t mask_stride;
};
__global__ void __launch_bounds__(128) k_e_ransac_fit(const __grid_constant__ RansacArgs a)
{
    const int seg = blockIdx.y;
    const int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= a.iters) return;
    const int n = a.n.at(seg);
    const float *xyz = a.xyz + 3 * seg * a.stride;
    double4 *planes = a.planes + seg * a.h_stride;
    a.cnt[seg * a.h_stride + h] = 0ull;
    if (n < a.ransac_n) { planes[h] = make_double4(0.0, 0.0, 0.0, NAN); a.pvalid[seg * a.h_stride + h] = 0; return; }
    int ids[RS_MAX_N];
    int got = 0;
    for (uint64_t j = 0; got < a.ransac_n; ++j) {
        const int v = (int)(kp_rng(a.seed, (uint64_t)h, j) % (uint64_t)n);
        bool dup = false;
        for (int t = 0; t < got; ++t) dup |= ids[t] == v;
        if (!dup) ids[got++] = v;
    }
    double pa, pb, pc, pd;
    bool ok = true;
    if (a.ransac_n == 3) {
        const float *p0 = xyz + 3 * (int64_t)ids[0], *p1 = xyz + 3 * (int64_t)ids[1], *p2 = xyz + 3 * (int64_t)ids[2];
        const double e1x = DS((double)p1[0], (double)p0[0]), e1y = DS((double)p1[1], (double)p0[1]), e1z = DS((double)p1[2], (double)p0[2]);
        const double e2x = DS((double)p2[0], (double)p0[0]), e2y = DS((double)p2[1], (double)p0[1]), e2z = DS((double)p2[2], (double)p0[2]);
        pa = DS(DM(e1y, e2z), DM(e1z, e2y));
        pb = DS(DM(e1z, e2x), DM(e1x, e2z));
        pc = DS(DM(e1x, e2y), DM(e1y, e2x));
        const double nn = sqrt(DA(DA(DM(pa, pa), DM(pb, pb)), DM(pc, pc)));
        if (nn == 0.0 || isnan(nn)) ok = false;
        pa = DD(pa, nn); pb = DD(pb, nn); pc = DD(pc, nn);
        pd = -DA(DA(DM(pa, (double)p0[0]), DM(pb, (double)p0[1])), DM(pc, (double)p0[2]));
    } else {
        double cx = 0, cy = 0, cz = 0;
        for (int j = 0; j < a.ransac_n; ++j) {
            const float *p = xyz + 3 * (int64_t)ids[j];
            cx = DA(cx, (double)p[0]); cy = DA(cy, (double)p[1]); cz = DA(cz, (double)p[2]);
        }
        const double m = (double)a.ransac_n;
        cx = DD(cx, m); cy = DD(cy, m); cz = DD(cz, m);
        double xx = 0, xy = 0, xz = 0, yy = 0, yz = 0, zz = 0;
        for (int j = 0; j < a.ransac_n; ++j) {
            const float *p = xyz + 3 * (int64_t)ids[j];
            const double x = DS((double)p[0], cx), y = DS((double)p[1], cy), z = DS((double)p[2], cz);
            xx = DA(xx, DM(x, x)); xy = DA(xy, DM(x, y)); xz = DA(xz, DM(x, z));
            yy = DA(yy, DM(y, y)); yz = DA(yz, DM(y, z)); zz = DA(zz, DM(z, z));
        }
        const double dx = DS(DM(yy, zz), DM(yz, yz)), dy = DS(DM(xx, zz), DM(xz, xz)), dz = DS(DM(xx, yy), DM(xy, xy));
        if (dx >= dy && dx >= dz) { pa = dx; pb = DS(DM(xz, yz), DM(xy, zz)); pc = DS(DM(xy, yz), DM(xz, yy)); }
        else if (dy >= dx && dy >= dz) { pa = DS(DM(xz, yz), DM(xy, zz)); pb = dy; pc = DS(DM(xy, xz), DM(yz, xx)); }
        else { pa = DS(DM(xy, yz), DM(xz, yy)); pb = DS(DM(xy, xz), DM(yz, xx)); pc = dz; }
        const double nn = sqrt(DA(DA(DM(pa, pa), DM(pb, pb)), DM(pc, pc)));
        if (nn == 0.0 || isnan(nn)) ok = false;
        pa = DD(pa, nn); pb = DD(pb, nn); pc = DD(pc, nn);
        pd = -DA(DA(DM(pa, cx), DM(pb, cy)), DM(pc, cz));
    }
    if (!ok) { pa = pb = pc = 0.0; pd = NAN; }
    planes[h] = make_double4(pa, pb, pc, pd);
    a.pvalid[seg * a.h_stride + h] = ok;
}
__device__ __forceinline__ double plane_dist(const double4 &pl, double x, double y, double z)
{
    return fabs(DA(DA(DA(DM(pl.x, x), DM(pl.y, y)), DM(pl.z, z)), pl.w));
}
constexpr int SCORE_THREADS = 256, SCORE_PTS = 4, SCORE_TILE = SCORE_THREADS * SCORE_PTS, SCORE_HC = 512;
__global__ void __launch_bounds__(SCORE_THREADS) k_e_ransac_score(const __grid_constant__ RansacArgs a)
{
    __shared__ double4 pl_s[SCORE_HC];
    __shared__ int cnt_s[SCORE_THREADS / 32][SCORE_HC];
    const int seg = blockIdx.y;
    const int n = a.n.at(seg);
    if (n < a.ransac_n) return;
    const float *xyz = a.xyz + 3 * seg * a.stride;
    const double4 *planes = a.planes + seg * a.h_stride;
    unsigned long long *g_cnt = a.cnt + seg * a.h_stride;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ntiles = (n + SCORE_TILE - 1) / SCORE_TILE;
    if ((int)blockIdx.x >= ntiles) return;
    for (int h0 = 0; h0 < a.iters; h0 += SCORE_HC) {
        const int hc = min(SCORE_HC, a.iters - h0);
        for (int h = tid; h < hc; h += SCORE_THREADS) pl_s[h] = planes[h0 + h];
        for (int h = tid; h < (SCORE_THREADS / 32) * SCORE_HC; h += SCORE_THREADS) (&cnt_s[0][0])[h] = 0;
        __syncthreads();
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            double px[SCORE_PTS], py[SCORE_PTS], pz[SCORE_PTS];
#pragma unroll
            for (int j = 0; j < SCORE_PTS; ++j) {
                const int64_t i = (int64_t)tile * SCORE_TILE + j * SCORE_THREADS + tid;
                if (i < n) { px[j] = (double)xyz[3 * i]; py[j] = (double)xyz[3 * i + 1]; pz[j] = (double)xyz[3 * i + 2]; }
                else { px[j] = py[j] = pz[j] = NAN; }
            }
            for (int h = 0; h < hc; ++h) {
                const double4 pl = pl_s[h];
                int c = 0;
#pragma unroll
                for (int j = 0; j < SCORE_PTS; ++j)
                    c += __popc(__ballot_sync(KP_FULL, plane_dist(pl, px[j], py[j], pz[j]) < a.thr));
                if (lane == 0 && c) cnt_s[warp][h] += c;
            }
        }
        __syncthreads();
        for (int h = tid; h < hc; h += SCORE_THREADS) {
            int s = 0;
#pragma unroll
            for (int w = 0; w < SCORE_THREADS / 32; ++w) s += cnt_s[w][h];
            if (s) atomicAdd(&g_cnt[h0 + h], (unsigned long long)s);
        }
        __syncthreads();
    }
}
// Open3D's sequential best / early-exit rule replayed over the H counts.  The evolution
// of (best fitness, early-exit bound, processed set) does not depend on how ties are broken, only the winner
// among the hypotheses that tie on the final best count does: those are listed for the tie pass.
__global__ void k_e_ransac_select(const __grid_constant__ RansacArgs a)
{
    const int seg = blockIdx.x;
    if (threadIdx.x != 0) return;
    EngDyn &d = a.dyn[seg];
    const int n = a.n.at(seg);
    d.ransac_best = -1; d.ransac_ncand = 0;
    if (n < a.ransac_n) return;
    const unsigned long long *cnt = a.cnt + seg * a.h_stride;
    const uint8_t *pvalid = a.pvalid + seg * a.h_stride;
    double best_fit = 0.0, break_it = (double)a.iters;
    long done = 0;
    int ncand = 0;
    for (int h = 0; h < a.iters; ++h) {
        if ((double)done > break_it) continue;
        if (!pvalid[h]) continue;
        const double fit = (double)cnt[h] / (double)n;
        if (fit > best_fit) {
            best_fit = fit;
            ncand = 0;
            d.ransac_cand[ncand++] = h;
            if (fit < 1.0) {
                const double b = log(1.0 - a.probability) / log(1.0 - pow(fit, (double)a.ransac_n));
                break_it = b < (double)a.iters ? b : (double)a.iters;
            } else break_it = 0;
        } else if (fit == best_fit && ncand > 0) {
            if (ncand < ENG_MAX_CAND) d.ransac_cand[ncand] = h;
            ++ncand;
        }
        ++done;
    }
    if (ncand > ENG_MAX_CAND) { ncand = ENG_MAX_CAND; d.status = KP_E_RANGE; }   // (more exact ties than the tie pass holds)
    d.ransac_ncand = ncand;
    d.ransac_best = ncand > 0 ? d.ransac_cand[0] : -1;
}
// sum of squared inlier distances of the tied hypotheses: per-thread grid-stride sums, warp butterfly, warps in
// order, one slot per CTA; the final kernel adds the slots in CTA order (the shape of kp_ransac.cu's host path)
__global__ void __launch_bounds__(256) k_e_ransac_tie(const __grid_constant__ RansacArgs a)
{
    __shared__ double sh[8];
    const int seg = blockIdx.y;
    const EngDyn &d = a.dyn[seg];
    if (d.ransac_ncand <= 1) return;
    const int n = a.n.at(seg);
    const float *xyz = a.xyz + 3 * seg * a.stride;
    const double4 *planes = a.planes + seg * a.h_stride;
    for (int c = 0; c < d.ransac_ncand; ++c) {
        const double4 pl = planes[d.ransac_cand[c]];
        double v = 0.0;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
            const double dd = plane_dist(pl, (double)xyz[3 * i], (double)xyz[3 * i + 1], (double)xyz[3 * i + 2]);
            if (dd < a.thr) v = DA(v, DM(dd, dd));
        }
        v = kp_butterfly_sum(v);
        if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0;
            for (int w = 0; w < 8; ++w) s = DA(s, sh[w]);
            a.slots[((size_t)seg * ENG_MAX_CAND + c) * a.nblk + blockIdx.x] = s;
        }
        __syncthreads();
    }
}
__global__ void k_e_ransac_final(const __grid_constant__ RansacArgs a)
{
    const int seg = blockIdx.x;
    if (threadIdx.x != 0) return;
    EngDyn &d = a.dyn[seg];
    int best = d.ransac_best;
    if (d.ransac_ncand > 1) {
        // rm = sum d^2 / sqrt(count); the tied hypotheses share the count: a later one wins iff its rm is smaller
        const unsigned long long *cnt = a.cnt + seg * a.h_stride;
        double best_rm = 0.0;
        for (int c = 0; c < d.ransac_ncand; ++c) {
            double s = 0;
            for (int b = 0; b < a.nblk; ++b) s += a.slots[((size_t)seg * ENG_MAX_CAND + c) * a.nblk + b];
            const int h = d.ransac_cand[c];
            const double rm = cnt[h] ? s / sqrt((double)cnt[h]) : 0.0;
            if (c == 0) best_rm = rm;
            else if (rm < best_rm) { best = h; best_rm = rm; }
        }
    }
    d.ransac_best = best;
    if (best >= 0) {
        const double4 pl = a.planes[seg * a.h_stride + best];
        d.plane[0] = pl.x; d.plane[1] = pl.y; d.plane[2] = pl.z; d.plane[3] = pl.w;
    } else {
        d.plane[0] = d.plane[1] = d.plane[2] = 0.0; d.plane[3] = NAN;     // NaN distance: nobody is an inlier
    }
}
__global__ void __launch_bounds__(256) k_e_plane_mask(const __grid_constant__ RansacArgs a)
{
    const int seg = blockIdx.y;
    const int n = a.n.at(seg);
    const EngDyn &d = a.dyn[seg];
    const double4 pl = make_double4(d.plane[0], d.plane[1], d.plane[2], d.plane[3]);
    const float *xyz = a.xyz + 3 * seg * a.stride;
    uint8_t *mask = a.mask + seg * a.mask_stride;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        mask[i] = plane_dist(pl, (double)xyz[3 * i], (double)xyz[3 * i + 1], (double)xyz[3 * i + 2]) < a.thr;
}

// The plane segment_plane returns: the covariance refit on the winning hypothesis's inliers (mask2 over the band), in
// kp_ransac_device's two passes: pass 0 sums the inliers and counts them, pass 1 sums their moments around the
// centroid.  Per-thread grid-stride sums, warp butterfly, warps in order, one slot per CTA; k_e_refit_fold adds the
// slots in CTA order, so the plane is the same run to run and does not depend on the rest of the batch.
constexpr int REFIT_NV = 6;
struct RefitArgs {
    const float *xyz; int64_t stride; DCnt n; EngDyn *dyn; int ransac_n;
    const uint8_t *mask; int64_t mask_stride;
    double *slots; int nblk;                                        // [seg][nblk][REFIT_NV]
};
template <int PASS>
__global__ void __launch_bounds__(256) k_e_refit_sum(const __grid_constant__ RefitArgs a)
{
    constexpr int NV = PASS == 0 ? 4 : 6;                           // x, y, z, count  |  xx, xy, xz, yy, yz, zz
    __shared__ double sh[8][NV];
    const int seg = blockIdx.y;
    const EngDyn &d = a.dyn[seg];
    if (d.ransac_best < 0) return;
    const int n = a.n.at(seg);
    const float *xyz = a.xyz + 3 * seg * a.stride;
    const uint8_t *mask = a.mask + seg * a.mask_stride;
    const double cx = PASS ? d.refit_c[0] : 0.0, cy = PASS ? d.refit_c[1] : 0.0, cz = PASS ? d.refit_c[2] : 0.0;
    double v[NV];
#pragma unroll
    for (int c = 0; c < NV; ++c) v[c] = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (!mask[i]) continue;
        const double x = DS((double)xyz[3 * i], cx), y = DS((double)xyz[3 * i + 1], cy), z = DS((double)xyz[3 * i + 2], cz);
        if constexpr (PASS == 0) {
            v[0] = DA(v[0], x); v[1] = DA(v[1], y); v[2] = DA(v[2], z); v[3] = DA(v[3], 1.0);
        } else {
            v[0] = DA(v[0], DM(x, x)); v[1] = DA(v[1], DM(x, y)); v[2] = DA(v[2], DM(x, z));
            v[3] = DA(v[3], DM(y, y)); v[4] = DA(v[4], DM(y, z)); v[5] = DA(v[5], DM(z, z));
        }
    }
#pragma unroll
    for (int c = 0; c < NV; ++c) v[c] = kp_butterfly_sum(v[c]);
    if ((threadIdx.x & 31) == 0)
        for (int c = 0; c < NV; ++c) sh[threadIdx.x >> 5][c] = v[c];
    __syncthreads();
    if (threadIdx.x < NV) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s = DA(s, sh[w][threadIdx.x]);
        a.slots[((size_t)seg * a.nblk + blockIdx.x) * REFIT_NV + threadIdx.x] = s;
    }
}
// pass 0: the centroid; pass 1: the frame's floor plane (NaN without a band of ransac_n points, 0 without a valid
// hypothesis, the hypothesis when the refit is degenerate)
__global__ void k_e_refit_fold(const __grid_constant__ RefitArgs a, int pass, int B)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= B) return;
    EngDyn &d = a.dyn[f];
    const double *sl = a.slots + (size_t)f * a.nblk * REFIT_NV;
    const int nv = pass == 0 ? 4 : 6;
    double s[REFIT_NV] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    if (d.ransac_best >= 0)
        for (int b = 0; b < a.nblk; ++b)
            for (int c = 0; c < nv; ++c) s[c] = DA(s[c], sl[(size_t)b * REFIT_NV + c]);
    if (pass == 0) {
        if (d.ransac_best >= 0) {
            d.refit_c[0] = DD(s[0], s[3]); d.refit_c[1] = DD(s[1], s[3]); d.refit_c[2] = DD(s[2], s[3]); d.refit_c[3] = s[3];
        }
        return;
    }
    double pl[4] = {0.0, 0.0, 0.0, 0.0};
    if (d.n_lo < a.ransac_n) {
        pl[0] = pl[1] = pl[2] = pl[3] = NAN;
    } else if (d.ransac_best >= 0) {
        for (int c = 0; c < 4; ++c) pl[c] = d.plane[c];
        double rp[4];
        if (d.refit_c[3] >= 1.0 && cov_fit_from_moments(s, d.refit_c[0], d.refit_c[1], d.refit_c[2], rp))
            for (int c = 0; c < 4; ++c) pl[c] = rp[c];
    }
    for (int c = 0; c < 4; ++c) d.floor_plane[c] = pl[c];
}
// pcd_above_plane (floor_removal.py:39-51) on the filter output: keep[i] = ((a*x + b*y) + c*z) + d < 0 in double, no FMA
struct PlaneSideArgs { const float *xyz; int64_t stride; DCnt n; double pl[4]; uint8_t *keep; int64_t mask_stride; };
__global__ void __launch_bounds__(256) k_e_plane_side(const __grid_constant__ PlaneSideArgs a)
{
    const int seg = blockIdx.y;
    const int n = a.n.at(seg);
    const float *xyz = a.xyz + 3 * seg * a.stride;
    uint8_t *keep = a.keep + seg * a.mask_stride;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        keep[i] = kp_affine(a.pl[0], a.pl[1], a.pl[2], a.pl[3], (double)xyz[3 * i], (double)xyz[3 * i + 1], (double)xyz[3 * i + 2]) < 0.0;
}

// rows src[0..n) appended to dst at row offset off[seg]; total[seg] = off + n
struct AppendArgs { const float *src; float *dst; int64_t stride; DCnt n, off; DOut total; const uint32_t *aux_src; uint32_t *aux_dst; };
__global__ void __launch_bounds__(256) k_e_append_rows(const __grid_constant__ AppendArgs a)
{
    const int seg = blockIdx.y;
    const int n = a.n.at(seg), off = a.off.at(seg);
    const float *src = a.src + 3 * seg * a.stride;
    float *dst = a.dst + 3 * (seg * a.stride + off);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < 3LL * n; e += (int64_t)gridDim.x * blockDim.x) dst[e] = src[e];
    if (a.aux_src)
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x)
            a.aux_dst[seg * a.stride + off + e] = a.aux_src[seg * a.stride + e];
    if (blockIdx.x == 0 && threadIdx.x == 0) a.total.at(seg) = off + n;
}
// n_up = n_in - n_lo (n_in: the floor stage's input) is not stored anywhere: a tiny kernel derives the per-frame scalars
// between stages
struct DeriveArgs { EngDyn *dyn; DCnt n_in; int32_t *n_up; int do_floor, do_fsor; };
__global__ void k_e_derive_up(const __grid_constant__ DeriveArgs a, int B)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < B) a.n_up[f] = a.n_in.at(f) - a.dyn[f].n_lo;
}

// points left to the grid level 0: none when the cloud's voxel-brick index was built
struct NoldArgs { const KpVbiDev *vbi; int64_t vbi_stride; DCnt n; DOut n_old; };
__global__ void k_e_nold(const __grid_constant__ NoldArgs a, int nseg)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseg) return;
    const KpVbiDev &v = *reinterpret_cast<const KpVbiDev *>(reinterpret_cast<const char *>(a.vbi) + s * a.vbi_stride);
    a.n_old.at(s) = v.ok ? 0 : a.n.at(s);
}

// final cloud + result record of every frame
struct FinishArgs {
    EngDyn *dyn; kp_frame_result *res; int S;
    const float *filt_out, *merged, *fsor_out; int64_t stride;      // candidates for the final cloud
    DCnt n_filt;                                                    // rows of filt_out (the voxel + SOR [+ ROR] output)
    int do_floor, do_fsor;
    float *out; int64_t out_stride;                                 // rows; NULL -> no copy
    int floor_mode; double floor_plane[4];                          // k_e_finish: the plane mode's plane
};
__device__ __forceinline__ void finish_pick(const FinishArgs &a, int f, const float *&src, int &n)
{
    const EngDyn &d = a.dyn[f];
    if (!a.do_floor || d.floor_skip) { src = a.filt_out + 3 * f * a.stride; n = a.n_filt.at(f); }
    else if (!a.do_fsor) { src = a.merged + 3 * f * a.stride; n = d.n_merged; }
    else { src = a.fsor_out + 3 * f * a.stride; n = d.n_fsor; }
}
__global__ void k_e_finish(const __grid_constant__ FinishArgs a, int B)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= B) return;
    EngDyn &d = a.dyn[f];
    const float *src; int n;
    finish_pick(a, f, src, n);
    d.n_out = n;
    kp_frame_result &r = a.res[f];
    r.n_fused = d.n_fused; r.n_voxel = d.n_voxel; r.n_sor = d.n_sor;
    if (a.floor_mode == KP_FLOOR_PLANE)
        r.n_floor_inliers = a.do_floor ? a.n_filt.at(f) - d.n_merged : 0;
    else
        r.n_floor_inliers = (a.do_floor && !d.floor_skip) ? d.n_lo - d.n_rest : 0;
    r.n_out = n;
    for (int i = 0; i < 5; ++i) {
        for (int e = 0; e < 16; ++e) r.icp_T[i][e] = i < a.S - 1 ? d.icp_T[i][e] : 0.0;
        r.icp_fitness[i] = i < a.S - 1 ? d.icp_fit[i] : 0.0;
        r.icp_rmse[i] = i < a.S - 1 ? d.icp_rmse[i] : 0.0;
        r.icp_iters[i] = i < a.S - 1 ? d.icp_iters[i] : 0;
    }
    r.status = d.status;
    for (int c = 0; c < 4; ++c) r.floor_plane[c] = !a.do_floor ? NAN : (a.floor_mode == KP_FLOOR_PLANE ? a.floor_plane[c] : d.floor_plane[c]);
}
// the final cloud of every frame into the caller's buffer (device memory, or pinned host memory written through
// the unified address space: the row count is only known on the device)
__global__ void __launch_bounds__(256) k_e_copy_out(const __grid_constant__ FinishArgs a)
{
    const int f = blockIdx.y;
    const float *src; int n;
    finish_pick(a, f, src, n);
    if ((int64_t)n > a.out_stride) n = (int)a.out_stride;           // never past the caller's stride (status says so)
    float *dst = a.out + 3 * f * a.out_stride;
    const int64_t e4 = (3LL * n) / 4;
    const bool al = ((((uintptr_t)src) | ((uintptr_t)dst)) & 15u) == 0u;
    if (al) {
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < e4; e += (int64_t)gridDim.x * blockDim.x)
            reinterpret_cast<float4 *>(dst)[e] = reinterpret_cast<const float4 *>(src)[e];
        for (int64_t e = 4 * e4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < 3LL * n; e += (int64_t)gridDim.x * blockDim.x) dst[e] = src[e];
    } else {
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < 3LL * n; e += (int64_t)gridDim.x * blockDim.x) dst[e] = src[e];
    }
}
// where each frame's final cloud starts (the fixed-N resample reads it from there)
__global__ void k_e_final_src(const __grid_constant__ FinishArgs a, int B, const float **src_out)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= B) return;
    int n;
    finish_pick(a, f, src_out[f], n);
}
__global__ void k_e_check_stride(EngDyn *dyn, kp_frame_result *res, int B, int64_t out_stride)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < B && (int64_t)dyn[f].n_out > out_stride) res[f].status = KP_E_RANGE;
}
}  // namespace

// ================================================================= engine
namespace {
template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
};

struct EngSlot {
    kp_ctx *ctx = nullptr, *aux = nullptr;            // main stream, ICP branch stream
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaGraphExec_t graph = nullptr;
    int64_t graph_nodes = 0;
    std::vector<void *> allocs;
    // K1
    uint16_t *d_depth = nullptr;                      // staging for host depth [B][S][P]
    uint8_t *d_rgb = nullptr;                         // crop: staging for host segmentation images [B][S][P][3]
    uint32_t *crop_hist = nullptr;                    // crop: median-pass histograms [B*S][...] (zero between calls)
    double *crop_med = nullptr;                       // crop: median of every (frame, sensor) of the last batch [B][S]
    uint32_t *rs_hist = nullptr;                      // fixed-N output: radix-select histograms [B][...] (zero between calls)
    void *rs_st = nullptr;                            //   per-frame selection state
    unsigned long long *rs_list = nullptr;            //   candidate lists [B][cap]
    const float **fin_src = nullptr;                  //   first row of each frame's final cloud [B]
    int32_t *k1_slots = nullptr, *k1_rows = nullptr;
    float *fused = nullptr, *icp_in = nullptr;        // [B][NP][3]
    EngDyn *dyn = nullptr;
    EngCloud *icl = nullptr;
    kp_frame_result *d_res = nullptr;
    // main branch
    uint32_t *keys = nullptr, *keys_tmp = nullptr;
    int32_t *vals = nullptr, *vals_tmp = nullptr, *run_start = nullptr;
    BSort sortw{nullptr, nullptr};
    BScan scan{nullptr, nullptr, 0};
    float *A = nullptr, *Bb = nullptr, *C = nullptr, *D = nullptr, *E = nullptr, *Fin = nullptr;
    float4 *sorted[2] = {nullptr, nullptr}, *sorted_m = nullptr;
    uint8_t *flags_m = nullptr; int32_t *list_m = nullptr;
    uint2 *cellmap[2] = {nullptr, nullptr};
    int32_t *cell_cnt[2] = {nullptr, nullptr};
    int32_t *g_rank = nullptr, *g_loc = nullptr;
    double *mean = nullptr, *csum_tmp = nullptr;
    uint8_t *flags[2] = {nullptr, nullptr}, *mask = nullptr, *mask2 = nullptr;
    int32_t *list[2] = {nullptr, nullptr};
    int32_t *n_up = nullptr, *sink = nullptr, *isink = nullptr;
    uint32_t *vA = nullptr, *vB = nullptr, *vC = nullptr, *vD = nullptr, *vE = nullptr, *vsorted = nullptr;   // packed voxel coordinates of A, Bb, C, D, E
    uint2 *bricks = nullptr;
    double4 *planes = nullptr; uint8_t *pvalid = nullptr; unsigned long long *hcnt = nullptr; double *tie_slots = nullptr;
    KpKnnBatch knn_sor, knn_fsor, knn_nrm;
    // ICP branch
    uint32_t *ikeys = nullptr, *ikeys_tmp = nullptr;
    int32_t *ivals = nullptr, *ivals_tmp = nullptr, *irun_start = nullptr;
    BSort isortw{nullptr, nullptr};
    BScan iscan{nullptr, nullptr, 0};
    float *ivox = nullptr;                            // [B][S][P][3] voxel-downsampled ICP clouds
    float4 *isorted[2] = {nullptr, nullptr}, *isorted_m = nullptr;
    uint8_t *iflags_m = nullptr; int32_t *ilist_m = nullptr;
    uint2 *icellmap[2] = {nullptr, nullptr};
    int32_t *icell_cnt[2] = {nullptr, nullptr};
    int32_t *ig_rank = nullptr, *ig_loc = nullptr;
    uint8_t *iflags[2] = {nullptr, nullptr};
    int32_t *ilist[2] = {nullptr, nullptr};
    float *nrm = nullptr;                             // [B][P][3]
    uint32_t *ivijk = nullptr, *ivijk_sorted = nullptr;   // packed voxel coordinates of the ICP clouds / of the indexed target
    uint2 *ibricks = nullptr;
    KpIcpBatch icp;
};
}  // namespace

struct kp_pipeline {
    kp_pipeline_cfg cfg;
    int device = 0;
    int B = 1, W = 1;                 // frames per batch, batch slots in flight
    int64_t cap_cells = 1 << 25;
    int64_t cap_bricks = 1 << 23;
    int64_t NPr = 0, Pr = 0;          // row strides of the engine's own arrays: S*P and P rounded up to 64 (aligned vector access)
    bool use_graph = true, profiling = false, use_vbi_icp = false, use_vbi_knn = false;
    double rho_mult_a = 1.15, rho_mult_b = 2.0;
    double knn_mid = 1.5;             // cell of the mid level (x the level-0 cell); 0 = no mid level (KP_KNN_MID)
    int knn_rad = 1;                  // level-0 block radius in cells (KP_KNN_RAD): 1 = 27 cells of the full edge, 2 = 125 cells of half the edge
    std::vector<EngSlot> slots;
    float *d_tab = nullptr;
    uint32_t *d_vbits = nullptr;      // crop: [S][(P + 31) / 32] bit set = finite table entry (z16 = 0 elsewhere)
    std::vector<double> T_fuse, T_icp;
    kp_frame_result *h_res = nullptr;   // pinned staging of the result records
    int64_t h_res_cap = 0;
    int64_t launches = 0;
    std::string err;
    int sm_count = 148;
};

namespace {
#define PL_CUDA(p, call)                                                                         \
    do {                                                                                         \
        cudaError_t e__ = (call);                                                                \
        if (e__ != cudaSuccess) {                                                                \
            (p)->err = std::string(#call) + ": " + cudaGetErrorString(e__);                      \
            return KP_E_CUDA;                                                                    \
        }                                                                                        \
    } while (0)

template <class T>
int slot_alloc(kp_pipeline *pl, EngSlot &s, size_t count, T **out, bool zero = false)
{
    void *p = nullptr;
    const size_t bytes = ((count > 0 ? count : 1) * sizeof(T) + 255) & ~(size_t)255;
    if (cudaMalloc(&p, bytes) != cudaSuccess) {
        pl->err = std::string("frame engine: cudaMalloc failed: ") + cudaGetErrorString(cudaGetLastError());
        return KP_E_NOMEM;
    }
    if (zero && cudaMemset(p, 0, bytes) != cudaSuccess) { pl->err = "frame engine: cudaMemset failed"; return KP_E_CUDA; }
    s.allocs.push_back(p);
    *out = (T *)p;
    return KP_OK;
}

inline int ctas_for(const kp_pipeline *pl, int per_sm) { return pl->sm_count * per_sm; }

// ---- stage: voxel downsample of `nseg` clouds of `n` rows each
int stage_voxel(kp_pipeline *pl, kp_ctx *ctx, int nseg, int64_t n, const float *xyz, int64_t xyz_stride, const KpVoxDev *vp,
                int64_t vp_stride, DCnt nvalid, uint32_t *keys, uint32_t *keys_tmp, int32_t *vals, int32_t *vals_tmp, int64_t kstride,
                const BSort &sw, const BScan &sc, int32_t *run_start, int64_t rs_stride, float *out, int64_t out_stride, DOut m,
                uint32_t *vijk = nullptr)
{
    {
        KP_PROFB(ctx, "voxel_keys", (double)nseg * n * 16.0);
        VoxArgs a{xyz, xyz_stride, n, vp, vp_stride, keys, kstride};
        // ~64 CTAs per SM over ALL segments, every thread with one or two trips (measured: the same 25 M rows as 24 segments x
        // 1184 CTAs, most threads without work, ran at 3.3 TB/s against 4.0 TB/s as 8 x 1184)
        int64_t gx = (n / 4 + 2 * 256 - 1) / (2 * 256);
        const int64_t cap = ctas_for(pl, 64) / (nseg > 0 ? nseg : 1);
        if (gx > cap) gx = cap;
        if (gx < 1) gx = 1;
        k_e_voxel_keys<<<dim3((unsigned)gx, (unsigned)nseg), 256, 0, ctx->stream>>>(a);
        KP_LAUNCH_CHECK(ctx);
    }
    BLaunch L{ctx, nseg, n, ctas_for(pl, 4)};
    KP_TRY(kp_b_sort_pairs_u32(L, sw, n, 4, keys, keys_tmp, vals, vals_tmp, kstride));     // 4 passes: result back in keys / vals
    KP_TRY(kp_b_run_starts_u32(L, sc, nvalid, keys, kstride, run_start, rs_stride, m));
    {
        KP_PROFB(ctx, "voxel_mean", (double)nseg * n * 16.0);
        VoxMeanArgs a{xyz, xyz_stride, vals, kstride, run_start, rs_stride, DCnt{m.p, m.stride}, out, out_stride, keys, kstride, vp, vp_stride, vijk};
        int64_t gx = (n + 127) / 128;
        if (gx > ctas_for(pl, 16)) gx = ctas_for(pl, 16);
        k_e_voxel_mean<<<dim3((unsigned)gx, (unsigned)nseg), 128, 0, ctx->stream>>>(a);
        KP_LAUNCH_CHECK(ctx);
    }
    return KP_OK;
}

// ---- stage: neighbour grid of `nseg` clouds
int stage_grid(kp_pipeline *pl, kp_ctx *ctx, const GridArgs &a, int nseg, int64_t cap_rows, const BScan &sc, DOut sink)
{
    KP_PROFB(ctx, "grid_build", 0.0);
    const int ctas = ctas_for(pl, 4);
    const dim3 grid((unsigned)ctas, (unsigned)nseg);
    k_eg_setup<<<nseg, 32, 0, ctx->stream>>>(a);
    KP_LAUNCH_CHECK(ctx);
    k_eg_clear<<<grid, 256, 0, ctx->stream>>>(a);
    KP_LAUNCH_CHECK(ctx);
    k_eg_mark<<<grid, 256, 0, ctx->stream>>>(a);
    KP_LAUNCH_CHECK(ctx);
    const int64_t word_tiles = (pl->cap_cells / 32 + 1 + BC_TILE - 1) / BC_TILE;
    const dim3 wgrid((unsigned)(word_tiles < ctas ? word_tiles : ctas), (unsigned)nseg);
    k_eg_rank_reduce<<<wgrid, 256, 0, ctx->stream>>>(a, sc);
    KP_LAUNCH_CHECK(ctx);
    k_eg_rank_apply<<<wgrid, 256, 0, ctx->stream>>>(a, sc);
    KP_LAUNCH_CHECK(ctx);
    k_eg_count<<<grid, 256, 0, ctx->stream>>>(a);
    KP_LAUNCH_CHECK(ctx);
    BLaunch L{ctx, nseg, cap_rows + 1, ctas};
    // run starts = exclusive scan of the per-cell counts over the occupied cells; run_start[nocc] = n (the scan's
    // total, also written to `sink`)
    KP_TRY(kp_b_exclusive_scan(L, sc, DCnt{a.nocc.p, a.nocc.stride}, a.cell_cnt, a.cnt_stride, sink));
    k_eg_scatter<<<grid, 256, 0, ctx->stream>>>(a);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}

// ---- stage: voxel-brick index of `nseg` voxel-downsampled clouds
int stage_vbi(kp_pipeline *pl, kp_ctx *ctx, const VbiArgs &a, int nseg, const BScan &sc)
{
    KP_PROFB(ctx, "vbi_build", 0.0);
    const int ctas = ctas_for(pl, 4);
    const dim3 grid((unsigned)ctas, (unsigned)nseg);
    k_vbi_setup<<<nseg, 32, 0, ctx->stream>>>(a);
    KP_LAUNCH_CHECK(ctx);
    k_vbi_clear<<<grid, 256, 0, ctx->stream>>>(a);
    KP_LAUNCH_CHECK(ctx);
    k_vbi_mark<<<grid, 256, 0, ctx->stream>>>(a);
    KP_LAUNCH_CHECK(ctx);
    const int64_t tiles = (a.cap_bricks + BC_TILE - 1) / BC_TILE;
    const dim3 bgrid((unsigned)(tiles < ctas ? tiles : ctas), (unsigned)nseg);
    k_vbi_rank_reduce<<<bgrid, 256, 0, ctx->stream>>>(a, sc);
    KP_LAUNCH_CHECK(ctx);
    k_vbi_rank_apply<<<bgrid, 256, 0, ctx->stream>>>(a, sc);
    KP_LAUNCH_CHECK(ctx);
    k_vbi_scatter<<<grid, 256, 0, ctx->stream>>>(a);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}

// ---- stage: exact k nearest of every point of `nseg` clouds
// level 0 on the voxel-brick index (on the grid for a cloud whose index could not be built) -> level 1 on a coarser
// grid -> ring-expanding stragglers
struct KnnStage {
    const KpKnnBatch *batch;
    bool vbi;                        // the clouds have a voxel-brick index (vbi_args): level 0 runs on it
    VbiArgs vbi_args;
    DOut n_old;                      // points left to the grid level 0 (all of them without an index)
    GridArgs fine, coarse;           // level-0 grid (fallback) and level-1 grid
    bool mid_on;                     // a mid level between them: the level-0 leftovers through the thread-per-query kernel on a
    GridArgs mid;                    // moderately coarser grid, so that only real outliers reach the warp-per-query level 1
    uint8_t *flags0, *flags1, *flags_m; int64_t flag_stride;
    int32_t *list0, *list1, *list_m; int64_t list_stride;
    DOut cnt0, cnt1, cnt_m;
    DCnt n;
};
int stage_knn(kp_pipeline *pl, kp_ctx *ctx, const KnnStage &k, int nseg, int64_t cap_rows, const BScan &sc, DOut sink, bool build_vbi)
{
    BLaunch L{ctx, nseg, cap_rows, ctas_for(pl, 4)};
    if (k.vbi) {
        if (build_vbi) KP_TRY(stage_vbi(pl, ctx, k.vbi_args, nseg, sc));
        NoldArgs na{k.vbi_args.v, k.vbi_args.v_stride, k.n, k.n_old};
        k_e_nold<<<kp_blocks(nseg, 64), 64, 0, ctx->stream>>>(na, nseg);
        KP_LAUNCH_CHECK(ctx);
    }
    KP_TRY(stage_grid(pl, ctx, k.fine, nseg, cap_rows, sc, sink));          // (over n_old points: nothing when the index exists)
    KP_CUDA(ctx, cudaMemsetAsync(k.flags0, 0, (size_t)nseg * k.flag_stride, ctx->stream));
    if (k.vbi) KP_TRY(kp_knn_batch_vbi(ctx, *k.batch, cap_rows));
    KP_TRY(kp_knn_batch_level0(ctx, *k.batch, cap_rows));
    KP_TRY(kp_b_compact_index(L, sc, k.n, k.flags0, k.flag_stride, k.list0, k.list_stride, k.cnt0));
    if (k.mid_on) {
        KP_TRY(stage_grid(pl, ctx, k.mid, nseg, cap_rows, sc, sink));
        KP_CUDA(ctx, cudaMemsetAsync(k.flags_m, 0, (size_t)nseg * k.flag_stride, ctx->stream));
        KP_TRY(kp_knn_batch_mid(ctx, *k.batch, cap_rows));
        KP_TRY(kp_b_compact_index(L, sc, k.n, k.flags_m, k.flag_stride, k.list_m, k.list_stride, k.cnt_m));
    }
    KP_TRY(stage_grid(pl, ctx, k.coarse, nseg, cap_rows, sc, sink));
    KP_CUDA(ctx, cudaMemsetAsync(k.flags1, 0, (size_t)nseg * k.flag_stride, ctx->stream));
    KP_TRY(kp_knn_batch_level1(ctx, *k.batch, cap_rows));
    KP_TRY(kp_b_compact_index(L, sc, k.n, k.flags1, k.flag_stride, k.list1, k.list_stride, k.cnt1));
    KP_TRY(kp_knn_batch_stragglers(ctx, *k.batch));
    return KP_OK;
}

#define DYN_CNT(slot, field) dcnt(&(slot).dyn->field, sizeof(EngDyn))
#define DYN_OUT(slot, field) dout(&(slot).dyn->field, sizeof(EngDyn))

// level 0: cell for the k-neighbour radius, over the points the index did not take; level 1: three times that cell
GridArgs main_grid_args(kp_pipeline *pl, EngSlot &s, int level, const float *xyz, DCnt n, double cell)
{
    const int64_t NPs = pl->NPr;                                 // row stride of every main-branch array
    GridArgs a;
    memset(&a, 0, sizeof a);
    // level 2 = the mid grid: its cell map and run starts reuse the level-0 grid's memory (level 0 is done by then; the
    // level-0 ROWS stay: they are the query points of every later level), its rows have their own array
    a.g = level == 2 ? &s.dyn->gm[0] : &s.dyn->g[level]; a.g_stride = sizeof(EngDyn);
    a.xyz = xyz; a.xyz_stride = NPs; a.n = n;
    a.b6 = s.dyn->b6; a.b6_stride = sizeof(EngDyn) / 4; a.parent = nullptr; a.parent_mult = 1.0;
    a.cell = level == 0 ? cell / (double)pl->knn_rad : (level == 2 ? pl->knn_mid * cell : 3.0 * cell);
    a.sorted = level == 2 ? s.sorted_m : s.sorted[level]; a.sorted_stride = NPs;
    a.cellmap = s.cellmap[level == 2 ? 0 : level]; a.map_stride = pl->cap_cells / 32 + 64;
    a.cell_cnt = s.cell_cnt[level == 2 ? 0 : level]; a.cnt_stride = NPs + 64;
    a.rank = s.g_rank; a.loc = s.g_loc; a.tmp_stride = NPs;
    a.cap_cells = pl->cap_cells;
    a.nocc = level == 2 ? DYN_OUT(s, nocc_m[0]) : DYN_OUT(s, nocc[level]);
    return a;
}

// ---- stage: remove_statistical_outlier of the batch's clouds `in` (n rows each, voxel coordinates vin) -> `out`, n_out
int stage_sor(kp_pipeline *pl, EngSlot &s, int use, const float *in, const uint32_t *vin, DCnt n, int k, double ratio, float *out,
              uint32_t *vout, DOut n_out)
{
    kp_ctx *ctx = s.ctx;
    const int B = pl->B;
    const int64_t NPs = pl->NPr;
    KP_PROF(ctx, use == 0 ? "sor" : "floor_sor");
    // level-0 cell: multiples of the radius that holds k points of a one-point-per-voxel surface (swept per search: KP_KNN_MULT_SOR / _FSOR)
    static const double mult_env[2] = {getenv("KP_KNN_MULT_SOR") ? atof(getenv("KP_KNN_MULT_SOR")) : 0.0, getenv("KP_KNN_MULT_FSOR") ? atof(getenv("KP_KNN_MULT_FSOR")) : 0.0};
    // (swept on the WFOV frame with the mid level in place: 1.3 for k = 20, 1.1 for k = 50; without a mid level 1.5 / 1.3)
    const double mult_def = pl->knn_mid > 0.0 ? (k <= 32 ? 1.3 : 1.1) : (k <= 32 ? 1.5 : 1.3);
    const double cell = pl->cfg.voxel_size * (mult_env[use] > 0.0 ? mult_env[use] : mult_def) * sqrt((double)k / 3.14159265358979);
    KnnStage ks;
    ks.batch = use == 0 ? &s.knn_sor : &s.knn_fsor;
    ks.vbi = pl->use_vbi_knn;
    memset(&ks.vbi_args, 0, sizeof ks.vbi_args);
    if (ks.vbi) {
        VbiArgs &v = ks.vbi_args;
        v.v = &s.dyn->vbi[0]; v.v_stride = sizeof(EngDyn);
        v.xyz = in; v.xyz_stride = NPs; v.vijk = vin; v.vijk_stride = NPs; v.n = n;
        v.vp = &s.dyn->vox_fused; v.vp_stride = sizeof(EngDyn);
        v.bricks = s.bricks; v.brick_stride = pl->cap_bricks; v.cap_bricks = pl->cap_bricks;
        v.pts = s.sorted[0]; v.vijk_sorted = s.vsorted; v.pts_stride = NPs;      // the index's rows ARE the level-0 rows of levels 1 / 2
        v.status = &s.dyn->status; v.status_stride = sizeof(EngDyn) / 4;
    }
    ks.n_old = DYN_OUT(s, n_old[use]);
    ks.fine = main_grid_args(pl, s, 0, in, ks.vbi ? DYN_CNT(s, n_old[use]) : n, cell);
    ks.coarse = main_grid_args(pl, s, 1, in, n, cell);
    ks.mid_on = pl->knn_mid > 0.0;
    ks.mid = main_grid_args(pl, s, 2, in, n, cell);
    ks.flags0 = s.flags[0]; ks.flags1 = s.flags[1]; ks.flags_m = s.flags_m; ks.flag_stride = NPs;
    ks.list0 = s.list[0]; ks.list1 = s.list[1]; ks.list_m = s.list_m; ks.list_stride = NPs;
    ks.cnt0 = DYN_OUT(s, cnt_l0[use]); ks.cnt1 = DYN_OUT(s, cnt_l1[use]); ks.cnt_m = DYN_OUT(s, cnt_lm[use]);
    ks.n = n;
    KP_TRY(stage_knn(pl, ctx, ks, B, NPs, s.scan, dout(s.sink, 4), true));
    {
        KP_PROFB(ctx, "sor_stats", 0.0);
        BLaunch L{ctx, B, NPs, ctas_for(pl, 4)};
        const int64_t tmp_stride = NPs / 1024 + NPs / 1048576 + 16;
        KP_TRY(kp_b_csum(L, n, s.mean, NPs, 1, nullptr, 0, s.csum_tmp, tmp_stride, &s.dyn->sor_sum, sizeof(EngDyn) / 8));
        KP_TRY(kp_b_csum(L, n, s.mean, NPs, 2, &s.dyn->sor_sum, sizeof(EngDyn) / 8, s.csum_tmp, tmp_stride, &s.dyn->sor_sq, sizeof(EngDyn) / 8));
        SorMaskArgs m{s.mean, NPs, n, s.dyn, ratio, s.mask, NPs};
        k_e_sor_mask<<<dim3((unsigned)ctas_for(pl, 4), (unsigned)B), 256, 0, ctx->stream>>>(m);
        KP_LAUNCH_CHECK(ctx);
    }
    BLaunch L{ctx, B, NPs, ctas_for(pl, 4)};
    return kp_b_compact_rows(L, s.scan, n, s.mask, NPs, 0, in, out, NPs, n_out, vout ? vin : nullptr, vout);
}

// the fused branch's filter output, which the floor stage, k_e_finish and the copy-out read: voxel (A) -> SOR (Bb) -> ROR
// (into whichever of A / Bb is not its input)
struct FilterOut { float *xyz; uint32_t *vijk; DCnt n; };
FilterOut filter_output(const kp_pipeline *pl, EngSlot &s)
{
    const kp_pipeline_cfg &c = pl->cfg;
    const bool in_b = (c.sor_k > 0) != (c.ror_nb_points > 0);
    return FilterOut{in_b ? s.Bb : s.A, in_b ? s.vB : s.vA, c.ror_nb_points > 0 ? DYN_CNT(s, n_ror) : DYN_CNT(s, n_sor)};
}

// fp32 bounds of a double: the largest float <= v, the smallest float >= v
inline float f32_down(double v) { const float f = (float)v; return (double)f > v ? nextafterf(f, -INFINITY) : f; }
inline float f32_up(double v) { const float f = (float)v; return (double)f < v ? nextafterf(f, INFINITY) : f; }

// ---- stage: remove_radius_outlier of the batch's clouds `in` (n rows each, voxel coordinates vin) -> `out`, n_ror
int stage_ror(kp_pipeline *pl, EngSlot &s, const float *in, const uint32_t *vin, DCnt n, float *out, uint32_t *vout)
{
    kp_ctx *ctx = s.ctx;
    const kp_pipeline_cfg &c = pl->cfg;
    const int B = pl->B;
    const int64_t NPs = pl->NPr;
    KP_PROF(ctx, "ror");
    // the SOR's level-0 grid arrays (free once it is done); the cell is the radius with kp_radius_mask's margin.  k_eg_setup
    // may double it to fit cap_cells: any cell >= the radius keeps every neighbour inside the 27-cell block.
    GridArgs g = main_grid_args(pl, s, 0, in, n, 0.0);
    g.cell = c.ror_radius * (1.0 + 1e-6);
    KP_TRY(stage_grid(pl, ctx, g, B, NPs, s.scan, dout(s.sink, 4)));
    {
        KP_PROFB(ctx, "ror_count", 0.0);
        const double r2 = c.ror_radius * c.ror_radius;
        RorArgs a{&s.dyn->g[0], sizeof(EngDyn), n, c.ror_nb_points, r2, f32_down(r2 * (1.0 - 1e-6)), f32_up(r2 * (1.0 + 1e-6)), s.mask, NPs};
        int64_t gx = (NPs + 127) / 128;
        if (gx > ctas_for(pl, 8)) gx = ctas_for(pl, 8);
        k_e_ror_count<<<dim3((unsigned)gx, (unsigned)B), 128, 0, ctx->stream>>>(a);
        KP_LAUNCH_CHECK(ctx);
    }
    BLaunch L{ctx, B, NPs, ctas_for(pl, 4)};
    return kp_b_compact_rows(L, s.scan, n, s.mask, NPs, 0, in, out, NPs, DYN_OUT(s, n_ror), vout ? vin : nullptr, vout);
}

// ---- stage: floor removal (band split, RANSAC plane on the band, band outliers + upper part)
int stage_floor(kp_pipeline *pl, EngSlot &s, const float *in, const uint32_t *vin, DCnt n_in)
{
    kp_ctx *ctx = s.ctx;
    const kp_pipeline_cfg &c = pl->cfg;
    const int B = pl->B;
    const int64_t NPs = pl->NPr;
    const dim3 grid((unsigned)ctas_for(pl, 4), (unsigned)B);
    BLaunch L{ctx, B, NPs, ctas_for(pl, 4)};
    {
        KP_PROFB(ctx, "band_mask", 0.0);
        BandArgs a{in, NPs, n_in, s.dyn, 1, c.floor_band, c.ransac_n, s.mask, NPs};
        k_e_axis_max<<<grid, 256, 0, ctx->stream>>>(a);
        KP_LAUNCH_CHECK(ctx);
        k_e_band_mask<<<grid, 256, 0, ctx->stream>>>(a);
        KP_LAUNCH_CHECK(ctx);
    }
    // lower band -> C, upper part -> D
    KP_TRY(kp_b_partition_rows(L, s.scan, n_in, s.mask, NPs, in, s.C, s.D, NPs, DYN_OUT(s, n_lo), vin, s.vC, s.vD));
    {
        DeriveArgs d{s.dyn, n_in, s.n_up, c.do_floor, c.floor_sor_k > 0};
        k_e_derive_up<<<kp_blocks(B, 64), 64, 0, ctx->stream>>>(d, B);
        KP_LAUNCH_CHECK(ctx);
    }
    RansacArgs r;
    memset(&r, 0, sizeof r);
    r.xyz = s.C; r.stride = NPs; r.n = DYN_CNT(s, n_lo); r.dyn = s.dyn;
    r.ransac_n = c.ransac_n; r.iters = c.ransac_iters; r.seed = c.seed; r.thr = c.ransac_thr; r.probability = 0.99999999;
    r.planes = s.planes; r.pvalid = s.pvalid; r.cnt = s.hcnt; r.h_stride = c.ransac_iters;
    r.nblk = pl->sm_count * 2; r.slots = s.tie_slots;
    r.mask = s.mask2; r.mask_stride = NPs;
    {
        KP_PROFB(ctx, "ransac_fit", 0.0);
        k_e_ransac_fit<<<dim3(kp_blocks(c.ransac_iters, 128), (unsigned)B), 128, 0, ctx->stream>>>(r);
        KP_LAUNCH_CHECK(ctx);
    }
    {
        KP_PROFB(ctx, "ransac_score", 0.0);
        k_e_ransac_score<<<dim3((unsigned)r.nblk, (unsigned)B), SCORE_THREADS, 0, ctx->stream>>>(r);
        KP_LAUNCH_CHECK(ctx);
    }
    {
        KP_PROFB(ctx, "ransac_select", 0.0);
        k_e_ransac_select<<<B, 32, 0, ctx->stream>>>(r);
        KP_LAUNCH_CHECK(ctx);
        k_e_ransac_tie<<<dim3((unsigned)r.nblk, (unsigned)B), 256, 0, ctx->stream>>>(r);
        KP_LAUNCH_CHECK(ctx);
        k_e_ransac_final<<<B, 32, 0, ctx->stream>>>(r);
        KP_LAUNCH_CHECK(ctx);
        k_e_plane_mask<<<grid, 256, 0, ctx->stream>>>(r);
        KP_LAUNCH_CHECK(ctx);
    }
    {
        // the reported plane: refit on the inliers (the tie slots are free again: k_e_ransac_final has read them)
        KP_PROFB(ctx, "floor_refit", 0.0);
        RefitArgs f{s.C, NPs, DYN_CNT(s, n_lo), s.dyn, c.ransac_n, s.mask2, NPs, s.tie_slots, r.nblk};
        const dim3 rg((unsigned)r.nblk, (unsigned)B);
        k_e_refit_sum<0><<<rg, 256, 0, ctx->stream>>>(f);
        KP_LAUNCH_CHECK(ctx);
        k_e_refit_fold<<<kp_blocks(B, 32), 32, 0, ctx->stream>>>(f, 0, B);
        KP_LAUNCH_CHECK(ctx);
        k_e_refit_sum<1><<<rg, 256, 0, ctx->stream>>>(f);
        KP_LAUNCH_CHECK(ctx);
        k_e_refit_fold<<<kp_blocks(B, 32), 32, 0, ctx->stream>>>(f, 1, B);
        KP_LAUNCH_CHECK(ctx);
    }
    // outlier_cloud + upper (floor_removal.py:71-72): band outliers first, then the upper part
    KP_TRY(kp_b_compact_rows(L, s.scan, DYN_CNT(s, n_lo), s.mask2, NPs, 1, s.C, s.E, NPs, DYN_OUT(s, n_rest), vin ? s.vC : nullptr, s.vE));
    {
        KP_PROFB(ctx, "merge", 0.0);
        AppendArgs a{s.D, s.E, NPs, DCnt{s.n_up, 1}, DYN_CNT(s, n_rest), DYN_OUT(s, n_merged), vin ? s.vD : nullptr, s.vE};
        k_e_append_rows<<<grid, 256, 0, ctx->stream>>>(a);
        KP_LAUNCH_CHECK(ctx);
    }
    return KP_OK;
}

// ---- stage: floor removal at the caller's plane (pcd_above_plane): the kept rows of the filter output -> E, n_merged
int stage_floor_plane(kp_pipeline *pl, EngSlot &s, const float *in, const uint32_t *vin, DCnt n_in)
{
    kp_ctx *ctx = s.ctx;
    const kp_pipeline_cfg &c = pl->cfg;
    const int B = pl->B;
    const int64_t NPs = pl->NPr;
    {
        KP_PROFB(ctx, "plane_side", 0.0);
        PlaneSideArgs a{in, NPs, n_in, {c.floor_plane[0], c.floor_plane[1], c.floor_plane[2], c.floor_plane[3]}, s.mask, NPs};
        k_e_plane_side<<<dim3((unsigned)ctas_for(pl, 4), (unsigned)B), 256, 0, ctx->stream>>>(a);
        KP_LAUNCH_CHECK(ctx);
    }
    BLaunch L{ctx, B, NPs, ctas_for(pl, 4)};
    return kp_b_compact_rows(L, s.scan, n_in, s.mask, NPs, 0, in, s.E, NPs, DYN_OUT(s, n_merged), vin, vin ? s.vE : nullptr);
}

// ---- stage: ICP branch (voxel of the master and of every raw sub cloud, target grid + normals, all pairs together)
int stage_icp(kp_pipeline *pl, EngSlot &s, kp_ctx *ctx)
{
    const kp_pipeline_cfg &c = pl->cfg;
    const int B = pl->B, S = c.S;
    const int64_t P = c.P, Pr = pl->Pr;                           // rows of one sensor cloud; row stride of the ICP-branch arrays
    KP_PROF(ctx, "icp_branch");
    // the B * S clouds (frame b, sensor s) are the segments of ONE voxel pass
    const DCnt nv = dcnt(&s.icl->nv, sizeof(EngCloud));
    const DOut nvox = dout(&s.icl->n, sizeof(EngCloud));
    KP_TRY(stage_voxel(pl, ctx, B * S, P, s.icp_in, P, &s.icl->vox, sizeof(EngCloud), nv, s.ikeys, s.ikeys_tmp, s.ivals, s.ivals_tmp, Pr,
                       s.isortw, s.iscan, s.irun_start, Pr + 64, s.ivox, Pr, nvox, s.ivijk));
    // voxel-brick index over every frame's target (the master's voxel cloud): normals and ICP correspondences search it;
    // the grid is the fallback for a target whose index could not be built (n_old = its points then, else 0)
    const DCnt ntgt = dcnt(&s.icl->n, sizeof(EngCloud) * S);
    KnnStage ks;
    ks.batch = &s.knn_nrm;
    ks.vbi = pl->use_vbi_icp;
    memset(&ks.vbi_args, 0, sizeof ks.vbi_args);
    if (ks.vbi) {
        VbiArgs &v = ks.vbi_args;
        v.v = &s.dyn->vbi[1]; v.v_stride = sizeof(EngDyn);
        v.xyz = s.ivox; v.xyz_stride = (int64_t)S * Pr; v.vijk = s.ivijk; v.vijk_stride = (int64_t)S * Pr;
        v.n = ntgt;
        v.vp = &s.icl->vox; v.vp_stride = sizeof(EngCloud) * S;
        v.bricks = s.ibricks; v.brick_stride = pl->cap_bricks; v.cap_bricks = pl->cap_bricks;
        v.pts = s.isorted[0]; v.vijk_sorted = s.ivijk_sorted; v.pts_stride = Pr;
        v.status = &s.dyn->status; v.status_stride = sizeof(EngDyn) / 4;
    }
    ks.n_old = DYN_OUT(s, n_old[2]);
    GridArgs g;
    memset(&g, 0, sizeof g);
    g.g = &s.dyn->g[2]; g.g_stride = sizeof(EngDyn);
    g.xyz = s.ivox; g.xyz_stride = (int64_t)S * Pr; g.n = ks.vbi ? DYN_CNT(s, n_old[2]) : ntgt;
    g.b6 = s.icl->b6; g.b6_stride = sizeof(EngCloud) * S / 4; g.parent = nullptr; g.parent_mult = 1.0;
    g.cell = fmax(c.normals_radius * (1.0 + 4e-6), c.icp_max_corr * (1.0 + 1e-6));      // covers the normals radius and the ICP gate
    g.sorted = s.isorted[0]; g.sorted_stride = Pr;
    g.cellmap = s.icellmap[0]; g.map_stride = pl->cap_cells / 32 + 64;
    g.cell_cnt = s.icell_cnt[0]; g.cnt_stride = Pr + 64;
    g.rank = s.ig_rank; g.loc = s.ig_loc; g.tmp_stride = Pr;
    g.cap_cells = pl->cap_cells;
    g.nocc = DYN_OUT(s, nocc[2]);
    ks.fine = g;
    ks.coarse = g;
    ks.coarse.g = &s.dyn->g[3]; ks.coarse.n = ntgt; ks.coarse.cell = 3.0 * g.cell;
    ks.coarse.sorted = s.isorted[1]; ks.coarse.cellmap = s.icellmap[1]; ks.coarse.cell_cnt = s.icell_cnt[1];
    ks.coarse.nocc = DYN_OUT(s, nocc[3]);
    // (normals are a radius-capped search on a grid whose cell covers the radius: level 0 certifies everything but fp32
    // ties, so no mid level here)
    ks.mid_on = false;
    ks.mid = g;
    ks.flags0 = s.iflags[0]; ks.flags1 = s.iflags[1]; ks.flags_m = s.iflags_m; ks.flag_stride = Pr;
    ks.list0 = s.ilist[0]; ks.list1 = s.ilist[1]; ks.list_m = s.ilist_m; ks.list_stride = Pr;
    ks.cnt0 = DYN_OUT(s, cnt_l0[2]); ks.cnt1 = DYN_OUT(s, cnt_l1[2]); ks.cnt_m = DYN_OUT(s, cnt_lm[2]);
    ks.n = ntgt;
    {
        KP_PROF(ctx, "normals");
        KP_TRY(stage_knn(pl, ctx, ks, B, Pr, s.iscan, dout(s.isink, 4), true));
    }
    return kp_icp_batch_run(ctx, s.icp);
}
}  // namespace

// ================================================================= construction, graph, run
namespace {
__global__ void k_e_copy_cnt(DCnt src, DOut dst, int B)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < B) dst.at(f) = src.at(f);
}

int slot_create(kp_pipeline *pl, EngSlot &s)
{
    const kp_pipeline_cfg &c = pl->cfg;
    const int B = pl->B, S = c.S;
    const int64_t P = c.P, NP = (int64_t)S * P, NPr = pl->NPr, Pr = pl->Pr;
    const bool icp = c.do_icp && S > 1;
    int rc = kp_ctx_create(pl->device, &s.ctx);
    if (rc == KP_OK) rc = kp_ctx_create(pl->device, &s.aux);
    if (rc != KP_OK) { pl->err = kp_last_error(nullptr); return rc; }
    PL_CUDA(pl, cudaEventCreateWithFlags(&s.ev_fork, cudaEventDisableTiming));
    PL_CUDA(pl, cudaEventCreateWithFlags(&s.ev_join, cudaEventDisableTiming));
#define SA(ptr, count) KP_TRY(slot_alloc(pl, s, (size_t)(count), &(ptr)))
#define SAZ(ptr, count) KP_TRY(slot_alloc(pl, s, (size_t)(count), &(ptr), true))
    SAZ(s.d_depth, B * NP);
    if (c.do_crop) {
        SAZ(s.d_rgb, B * NP * 3);
        SAZ(s.crop_hist, (size_t)B * S * kp_crop_median_hist_elems());
        SAZ(s.crop_med, (size_t)B * S);
    }
    if (c.resample_n > 0) {
        // (the selection's key array is s.keys: the graph is done with it when the resample runs)
        SAZ(s.rs_hist, (size_t)B * kp_resample_engine_hist_elems());
        uint8_t *st = nullptr;
        SAZ(st, (size_t)B * kp_resample_engine_state_bytes());
        s.rs_st = st;
        SA(s.rs_list, (size_t)B * kp_resample_engine_cap(c.resample_n));
        SA(s.fin_src, B);
    }
    SA(s.k1_slots, kp_unproject_engine_slots(B, S, P));
    SAZ(s.k1_rows, (size_t)B * S * 2 * 8);
    SA(s.fused, B * NP * 3);
    SAZ(s.dyn, B);
    SAZ(s.icl, (size_t)B * S);
    SAZ(s.d_res, B);
    SA(s.keys, B * NPr); SA(s.keys_tmp, B * NPr); SA(s.vals, B * NPr); SA(s.vals_tmp, B * NPr);
    SA(s.run_start, B * (NPr + 64));
    SA(s.sortw.g_hist, (size_t)B * kp_b_sort_hist_elems(NP)); SA(s.sortw.g_tot, B * 256);
    const int64_t word_tiles = (pl->cap_cells / 32 + 1 + BC_TILE - 1) / BC_TILE;
    const int64_t row_tiles = (NPr + 66 + BC_TILE - 1) / BC_TILE;
    const int64_t brick_tiles = (pl->cap_bricks + BC_TILE - 1) / BC_TILE;
    s.scan.max_tiles = (int)((word_tiles > row_tiles ? word_tiles : row_tiles) + 1);
    if (s.scan.max_tiles < brick_tiles + 1) s.scan.max_tiles = (int)brick_tiles + 1;
    SA(s.scan.tile_sum, (size_t)B * s.scan.max_tiles); SAZ(s.scan.ticket, B);
    SA(s.A, B * NPr * 3); SA(s.Bb, B * NPr * 3); SA(s.C, B * NPr * 3); SA(s.D, B * NPr * 3); SA(s.E, B * NPr * 3); SA(s.Fin, B * NPr * 3);
    const int64_t map_stride = pl->cap_cells / 32 + 64;
    for (int l = 0; l < 2; ++l) {
        SA(s.sorted[l], B * NPr); SA(s.cellmap[l], B * map_stride); SA(s.cell_cnt[l], B * (NPr + 64));
        SA(s.flags[l], B * NPr); SA(s.list[l], B * NPr);
    }
    SA(s.g_rank, B * NPr); SA(s.g_loc, B * NPr);
    if (pl->knn_mid > 0.0) { SA(s.sorted_m, B * NPr); SA(s.flags_m, B * NPr); SA(s.list_m, B * NPr); }
    SA(s.mean, B * NPr); SA(s.csum_tmp, B * (NPr / 1024 + NPr / 1048576 + 16));
    SA(s.mask, B * NPr); SA(s.mask2, B * NPr);
    SAZ(s.n_up, B); SAZ(s.sink, B);
    if (pl->use_vbi_knn) {
        SA(s.vA, B * NPr); SA(s.vB, B * NPr); SA(s.vC, B * NPr); SA(s.vD, B * NPr); SA(s.vE, B * NPr); SA(s.vsorted, B * NPr);
        SA(s.bricks, (size_t)B * pl->cap_bricks);
    }
    const int iters = c.ransac_iters > 0 ? c.ransac_iters : 1;
    SA(s.planes, (size_t)B * iters); SA(s.pvalid, (size_t)B * iters); SA(s.hcnt, (size_t)B * iters);
    SA(s.tie_slots, (size_t)B * ENG_MAX_CAND * pl->sm_count * 2);
    std::vector<KpKnnSegDesc> d((size_t)B);
    for (int use = 0; use < 2; ++use) {
        const int k = use == 0 ? c.sor_k : c.floor_sor_k;
        if (k <= 0 || (use == 1 && !c.do_floor)) continue;
        for (int b = 0; b < B; ++b) {
            KpKnnSegDesc &e = d[b];
            memset(&e, 0, sizeof e);
            e.g0 = &s.dyn[b].g[0]; e.g1 = &s.dyn[b].g[1];
            e.vbi = pl->use_vbi_knn ? &s.dyn[b].vbi[0] : nullptr;
            e.pts0 = s.sorted[0] + (size_t)b * NPr;
            e.n = pl->use_vbi_knn ? &s.dyn[b].n_old[use] : (use == 0 ? &s.dyn[b].n_voxel : &s.dyn[b].n_merged);
            e.flags0 = s.flags[0] + (size_t)b * NPr; e.flags1 = s.flags[1] + (size_t)b * NPr;
            e.list0 = s.list[0] + (size_t)b * NPr; e.list1 = s.list[1] + (size_t)b * NPr;
            e.cnt0 = &s.dyn[b].cnt_l0[use]; e.cnt1 = &s.dyn[b].cnt_l1[use];
            if (pl->knn_mid > 0.0) {
                e.gm = &s.dyn[b].gm[0]; e.flags_m = s.flags_m + (size_t)b * NPr; e.list_m = s.list_m + (size_t)b * NPr; e.cnt_m = &s.dyn[b].cnt_lm[use];
            }
            e.mean = s.mean + (size_t)b * NPr;
        }
        // voxel-brick level 0: rho_a certifies the dense parts of the cloud, rho_b the sparse ones (multiples of the radius
        // that holds k points of a one-point-per-voxel surface)
        const double rk = c.voxel_size * sqrt((double)k / 3.14159265358979);
        rc = kp_knn_batch_create(s.ctx, d.data(), B, k, 0, 0.0, pl->rho_mult_a * rk, pl->rho_mult_b * rk, use == 0 ? &s.knn_sor : &s.knn_fsor);
        if (rc != KP_OK) { pl->err = s.ctx->err; return rc; }
    }
    if (icp) {
        SA(s.icp_in, B * NP * 3);
        SA(s.ikeys, (size_t)B * S * Pr); SA(s.ikeys_tmp, (size_t)B * S * Pr); SA(s.ivals, (size_t)B * S * Pr); SA(s.ivals_tmp, (size_t)B * S * Pr);
        SA(s.irun_start, (size_t)B * S * (Pr + 64));
        SA(s.isortw.g_hist, (size_t)B * S * kp_b_sort_hist_elems(P)); SA(s.isortw.g_tot, (size_t)B * S * 256);
        const int64_t irow_tiles = (Pr + 66 + BC_TILE - 1) / BC_TILE;
        s.iscan.max_tiles = (int)((word_tiles > irow_tiles ? word_tiles : irow_tiles) + 1);
        if (s.iscan.max_tiles < brick_tiles + 1) s.iscan.max_tiles = (int)brick_tiles + 1;
        SA(s.iscan.tile_sum, (size_t)B * S * s.iscan.max_tiles); SAZ(s.iscan.ticket, (size_t)B * S);
        SA(s.ivox, (size_t)B * S * Pr * 3);
        for (int l = 0; l < 2; ++l) {
            SA(s.isorted[l], B * Pr); SA(s.icellmap[l], B * map_stride); SA(s.icell_cnt[l], B * (Pr + 64));
            SA(s.iflags[l], B * Pr); SA(s.ilist[l], B * Pr);
        }
        SA(s.ig_rank, B * Pr); SA(s.ig_loc, B * Pr);
        if (pl->knn_mid > 0.0) { SA(s.isorted_m, B * Pr); SA(s.iflags_m, B * Pr); SA(s.ilist_m, B * Pr); }
        SA(s.nrm, B * Pr * 3);
        SA(s.ivijk, (size_t)B * S * Pr); SA(s.ivijk_sorted, B * Pr); SA(s.ibricks, (size_t)B * pl->cap_bricks);
        SAZ(s.isink, (size_t)B * S);
        for (int b = 0; b < B; ++b) {
            KpKnnSegDesc &e = d[b];
            memset(&e, 0, sizeof e);
            e.g0 = &s.dyn[b].g[2]; e.g1 = &s.dyn[b].g[3];
            e.vbi = pl->use_vbi_icp ? &s.dyn[b].vbi[1] : nullptr;
            e.pts0 = s.isorted[0] + (size_t)b * Pr;
            e.n = pl->use_vbi_icp ? &s.dyn[b].n_old[2] : &s.icl[(size_t)b * S].n;
            e.flags0 = s.iflags[0] + (size_t)b * Pr; e.flags1 = s.iflags[1] + (size_t)b * Pr;
            e.list0 = s.ilist[0] + (size_t)b * Pr; e.list1 = s.ilist[1] + (size_t)b * Pr;
            e.cnt0 = &s.dyn[b].cnt_l0[2]; e.cnt1 = &s.dyn[b].cnt_l1[2];
            e.cloud = s.ivox + 3 * (size_t)b * S * Pr;
            e.normals = s.nrm + 3 * (size_t)b * Pr;
        }
        rc = kp_knn_batch_create(s.ctx, d.data(), B, c.normals_max_nn, 1, c.normals_radius, c.normals_radius * 1.001, c.normals_radius * 1.001,
                                 &s.knn_nrm);
        if (rc != KP_OK) { pl->err = s.ctx->err; return rc; }
        std::vector<KpIcpPairDesc> pr;
        for (int b = 0; b < B; ++b)
            for (int sn = 1; sn < S && sn <= 5; ++sn) {
                KpIcpPairDesc e;
                e.tgt_grid = &s.dyn[b].g[2];
                e.tgt_vbi = pl->use_vbi_icp ? &s.dyn[b].vbi[1] : nullptr;
                e.tgt_normals = s.nrm + 3 * (size_t)b * Pr;
                e.src = s.ivox + 3 * ((size_t)b * S + sn) * Pr;
                e.n_src = &s.icl[(size_t)b * S + sn].n;
                for (int i = 0; i < 16; ++i) e.init_T[i] = pl->T_icp[16 * sn + i];
                e.res_T = s.dyn[b].icp_T[sn - 1]; e.res_fit = &s.dyn[b].icp_fit[sn - 1]; e.res_rmse = &s.dyn[b].icp_rmse[sn - 1];
                e.res_iters = &s.dyn[b].icp_iters[sn - 1];
                pr.push_back(e);
            }
        rc = kp_icp_batch_create(s.ctx, pr.data(), (int)pr.size(), P, c.icp_max_corr, c.icp_max_iter, 1e-6, 1e-6, &s.icp);
        if (rc != KP_OK) { pl->err = s.ctx->err; return rc; }
    }
#undef SA
#undef SAZ
    return KP_OK;
}

void slot_destroy(EngSlot &s)
{
    if (s.ctx) cudaStreamSynchronize(s.ctx->stream);
    if (s.aux) cudaStreamSynchronize(s.aux->stream);
    if (s.graph) cudaGraphExecDestroy(s.graph);
    kp_knn_batch_destroy(&s.knn_sor); kp_knn_batch_destroy(&s.knn_fsor); kp_knn_batch_destroy(&s.knn_nrm);
    kp_icp_batch_destroy(&s.icp);
    for (void *p : s.allocs) cudaFree(p);
    s.allocs.clear();
    if (s.ev_fork) cudaEventDestroy(s.ev_fork);
    if (s.ev_join) cudaEventDestroy(s.ev_join);
    if (s.ctx) kp_ctx_destroy(s.ctx);
    if (s.aux) kp_ctx_destroy(s.aux);
    s.ctx = s.aux = nullptr;
}

// the part of a batch that never changes: everything between K1 and the copy-out.  `fork`: run the ICP branch on
// the slot's second stream (joined before the result records are written).
int enqueue_core(kp_pipeline *pl, EngSlot &s, bool fork)
{
    const kp_pipeline_cfg &c = pl->cfg;
    const int B = pl->B, S = c.S;
    const int64_t NP = (int64_t)S * c.P, NPr = pl->NPr;
    const bool icp = c.do_icp && S > 1;
    kp_ctx *ctx = s.ctx;
    {
        SetupParams sp{s.dyn, s.icl, s.k1_rows, S, c.voxel_size, c.icp_voxel, icp ? 1 : 0};
        k_e_frame_setup<<<kp_blocks(B, 32), 32, 0, ctx->stream>>>(sp, B);
        KP_LAUNCH_CHECK(ctx);
    }
    kp_ctx *ictx = ctx;
    if (icp && fork) {
        ictx = s.aux;
        KP_CUDA(ctx, cudaEventRecord(s.ev_fork, ctx->stream));
        KP_CUDA(ctx, cudaStreamWaitEvent(s.aux->stream, s.ev_fork, 0));
    }
    if (icp && fork) KP_TRY(stage_icp(pl, s, ictx));      // enqueued first so that its small kernels interleave with the main branch
    // ---- filter_outliers: voxel + SOR
    KP_TRY(stage_voxel(pl, ctx, B, NP, s.fused, NP, &s.dyn->vox_fused, sizeof(EngDyn), DYN_CNT(s, n_fused), s.keys, s.keys_tmp, s.vals,
                       s.vals_tmp, NPr, s.sortw, s.scan, s.run_start, NPr + 64, s.A, NPr, DYN_OUT(s, n_voxel), s.vA));
    const float *sor_out = s.A;
    const uint32_t *v_sor_out = s.vA;
    if (c.sor_k > 0) {
        KP_TRY(stage_sor(pl, s, 0, s.A, s.vA, DYN_CNT(s, n_voxel), c.sor_k, c.sor_ratio, s.Bb, s.vB, DYN_OUT(s, n_sor)));
        sor_out = s.Bb;
        v_sor_out = s.vB;
    } else {
        k_e_copy_cnt<<<kp_blocks(B, 64), 64, 0, ctx->stream>>>(DYN_CNT(s, n_voxel), DYN_OUT(s, n_sor), B);
        KP_LAUNCH_CHECK(ctx);
    }
    // ---- radius outlier removal (optional): its output replaces the SOR output downstream
    const FilterOut fo = filter_output(pl, s);
    if (c.ror_nb_points > 0) KP_TRY(stage_ror(pl, s, sor_out, v_sor_out, DYN_CNT(s, n_sor), fo.xyz, fo.vijk));
    // ---- floor removal + SOR
    if (c.do_floor) {
        if (c.floor_mode == KP_FLOOR_PLANE) KP_TRY(stage_floor_plane(pl, s, fo.xyz, fo.vijk, fo.n));
        else KP_TRY(stage_floor(pl, s, fo.xyz, fo.vijk, fo.n));
        if (c.floor_sor_k > 0)
            KP_TRY(stage_sor(pl, s, 1, s.E, s.vE, DYN_CNT(s, n_merged), c.floor_sor_k, c.floor_sor_ratio, s.Fin, nullptr, DYN_OUT(s, n_fsor)));
    }
    if (icp && !fork) KP_TRY(stage_icp(pl, s, ctx));
    if (icp && fork) {
        KP_CUDA(ctx, cudaEventRecord(s.ev_join, s.aux->stream));
        KP_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, s.ev_join, 0));
    }
    {
        FinishArgs fa{s.dyn, s.d_res, S, fo.xyz, s.E, s.Fin, NPr, fo.n, c.do_floor, c.floor_sor_k > 0, nullptr, 0, c.floor_mode,
                      {c.floor_plane[0], c.floor_plane[1], c.floor_plane[2], c.floor_plane[3]}};
        k_e_finish<<<kp_blocks(B, 32), 32, 0, ctx->stream>>>(fa, B);
        KP_LAUNCH_CHECK(ctx);
    }
    return KP_OK;
}

int slot_capture(kp_pipeline *pl, EngSlot &s)
{
    const int64_t l0 = s.ctx->launches + s.aux->launches;
    cudaGraph_t g = nullptr;
    PL_CUDA(pl, cudaStreamBeginCapture(s.ctx->stream, cudaStreamCaptureModeThreadLocal));
    int rc = enqueue_core(pl, s, true);
    cudaError_t e = cudaStreamEndCapture(s.ctx->stream, &g);
    if (rc != KP_OK) { pl->err = s.ctx->err.empty() ? s.aux->err : s.ctx->err; if (g) cudaGraphDestroy(g); return rc; }
    if (e != cudaSuccess) { pl->err = std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e); return KP_E_CUDA; }
    e = cudaGraphInstantiate(&s.graph, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) { pl->err = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e); return KP_E_CUDA; }
    s.graph_nodes = s.ctx->launches + s.aux->launches - l0;      // kernel nodes: counted once per replay (run_impl)
    return KP_OK;
}

// K1 of a batch (outside the graph): with the crop, the median pass over the batch's depth first
int enqueue_k1(kp_pipeline *p, EngSlot &s, const uint16_t *d_depth, const uint8_t *d_rgb, int nf)
{
    const kp_pipeline_cfg &c = p->cfg;
    const int S = c.S;
    if (c.do_crop) KP_TRY(kp_crop_median_engine(s.ctx, d_depth, p->d_vbits, nf, S, c.P, s.crop_hist, s.crop_med));
    return kp_unproject_engine(s.ctx, d_depth, p->d_tab, p->T_fuse.data(), nf, S, c.P, c.unproject_flags, c.scale, s.fused,
                               (c.do_icp && S > 1) ? s.icp_in : nullptr, s.k1_slots, s.k1_rows, c.do_crop ? d_rgb : nullptr,
                               s.crop_med, c.crop_gate);
}

int run_impl(kp_pipeline *p, const uint16_t *depth, const uint8_t *rgb, int depth_on_device, int64_t F, const int64_t *h_frame_ids,
             kp_frame_result *h_results, float *out_xyz, int64_t out_stride, float *d_fixed)
{
    if (!p || !h_results || F < 0 || (F > 0 && !depth)) return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_run: bad argument");
    if (out_xyz && out_stride <= 0) { p->err = "kp_pipeline_run: out_stride must be > 0 when an output buffer is given"; return KP_E_ARG; }
    if (F > 0 && !rgb != !p->cfg.do_crop) {
        p->err = p->cfg.do_crop ? "kp_pipeline_run: this pipeline crops: it needs the segmentation images (rgb)"
                                : "kp_pipeline_run: rgb given to a pipeline created without the crop";
        return KP_E_ARG;
    }
    if (d_fixed && p->cfg.resample_n <= 0) { p->err = "kp_pipeline_run: fixed-N output requested from a pipeline with resample_n = 0"; return KP_E_ARG; }
    if (F == 0) return KP_OK;
    const kp_pipeline_cfg &c = p->cfg;
    const int B = p->B, S = c.S;
    const int64_t NP = (int64_t)S * c.P;
    PL_CUDA(p, cudaSetDevice(p->device));
    if (p->h_res_cap < F) {
        if (p->h_res) cudaFreeHost(p->h_res);
        p->h_res = nullptr; p->h_res_cap = 0;
        PL_CUDA(p, cudaMallocHost((void **)&p->h_res, sizeof(kp_frame_result) * (size_t)F));
        p->h_res_cap = F;
    }
    const bool direct = p->profiling || !p->use_graph;
    const int W = p->profiling ? 1 : p->W;
    const int64_t nbatch = (F + B - 1) / B;
    for (int64_t i = 0; i < nbatch; ++i) {
        EngSlot &s = p->slots[(size_t)(i % W)];
        kp_ctx *ctx = s.ctx;
        const int64_t f0 = i * B;
        const int nf = (int)(F - f0 < B ? F - f0 : B);
        const uint16_t *d_depth = depth + f0 * NP;
        const uint8_t *d_rgb = rgb ? rgb + 3 * f0 * NP : nullptr;
        if (!depth_on_device) {
            PL_CUDA(p, cudaMemcpyAsync(s.d_depth, depth + f0 * NP, sizeof(uint16_t) * (size_t)nf * NP, cudaMemcpyHostToDevice, ctx->stream));
            d_depth = s.d_depth;
            if (rgb) {
                PL_CUDA(p, cudaMemcpyAsync(s.d_rgb, d_rgb, 3 * (size_t)nf * NP, cudaMemcpyHostToDevice, ctx->stream));
                d_rgb = s.d_rgb;
            }
        }
        // frames of a short last batch beyond nf: empty bounds rows -> empty clouds, every stage is a no-op for them
        if (nf < B) PL_CUDA(p, cudaMemsetAsync(s.k1_rows, 0, sizeof(int32_t) * (size_t)B * S * 2 * 8, ctx->stream));
        int rc = enqueue_k1(p, s, d_depth, d_rgb, nf);
        if (rc != KP_OK) { p->err = ctx->err; return rc; }
        if (direct) {
            rc = enqueue_core(p, s, !p->profiling);
            if (rc != KP_OK) { p->err = ctx->err.empty() ? s.aux->err : ctx->err; return rc; }
        } else {
            PL_CUDA(p, cudaGraphLaunch(s.graph, ctx->stream));
            p->launches += s.graph_nodes;
        }
        const FilterOut fo = filter_output(p, s);
        if (out_xyz) {
            FinishArgs fa{s.dyn, s.d_res, S, fo.xyz, s.E, s.Fin, p->NPr, fo.n, c.do_floor, c.floor_sor_k > 0, out_xyz + 3 * f0 * out_stride,
                          out_stride};
            k_e_copy_out<<<dim3((unsigned)p->sm_count, (unsigned)nf), 256, 0, ctx->stream>>>(fa);
            ctx->launches++;
            k_e_check_stride<<<kp_blocks(nf, 32), 32, 0, ctx->stream>>>(s.dyn, s.d_res, nf, out_stride);
            ctx->launches++;
        }
        if (d_fixed) {
            // each frame's fixed-N slot from its final cloud, sample stream = its frame id; short / overflowing frames
            // get their status in the result record (written by the graph's k_e_finish just before)
            int64_t ids[16];
            for (int b = 0; b < nf; ++b) ids[b] = h_frame_ids ? h_frame_ids[f0 + b] : f0 + b;
            FinishArgs fa{s.dyn, s.d_res, S, fo.xyz, s.E, s.Fin, p->NPr, fo.n, c.do_floor, c.floor_sor_k > 0, nullptr, 0};
            k_e_final_src<<<kp_blocks(nf, 32), 32, 0, ctx->stream>>>(fa, nf, s.fin_src);
            ctx->launches++;
            rc = kp_resample_engine(ctx, s.fin_src, p->NPr, &s.dyn->n_out, (int64_t)(sizeof(EngDyn) / 4), nf, c.resample_n, c.resample_mode,
                                    c.seed, ids, &s.d_res->status, (int64_t)(sizeof(kp_frame_result) / 4), s.keys, s.rs_hist, s.rs_st,
                                    s.rs_list, d_fixed + 3 * f0 * (int64_t)c.resample_n);
            if (rc != KP_OK) { p->err = ctx->err; return rc; }
        }
        PL_CUDA(p, cudaMemcpyAsync(p->h_res + f0, s.d_res, sizeof(kp_frame_result) * (size_t)nf, cudaMemcpyDeviceToHost, ctx->stream));
    }
    for (int w = 0; w < W && w < (int)p->slots.size(); ++w) {
        PL_CUDA(p, cudaStreamSynchronize(p->slots[w].ctx->stream));
        PL_CUDA(p, cudaStreamSynchronize(p->slots[w].aux->stream));
    }
    memcpy(h_results, p->h_res, sizeof(kp_frame_result) * (size_t)F);
    if (getenv("KP_PIPE_DEBUG")) {
        EngDyn d;
        cudaMemcpy(&d, p->slots[0].dyn, sizeof d, cudaMemcpyDeviceToHost);
        fprintf(stderr, "[kp engine] frame 0 of slot 0: fused %d voxel %d sor %d lo %d rest %d merged %d fsor %d | leftovers L0 %d %d %d  L1 %d %d %d | cells %d %d %d %d | g0 cell %g dims %d %d %d\n",
                d.n_fused, d.n_voxel, d.n_sor, d.n_lo, d.n_rest, d.n_merged, d.n_fsor, d.cnt_l0[0], d.cnt_l0[1], d.cnt_l0[2], d.cnt_l1[0],
                d.cnt_l1[1], d.cnt_l1[2], d.nocc[0], d.nocc[1], d.nocc[2], d.nocc[3], d.g[0].cell, d.g[0].dim[0], d.g[0].dim[1], d.g[0].dim[2]);
    }
    for (int64_t f = 0; f < F; ++f)
        if (h_results[f].status != KP_OK) {
            char buf[160];
            snprintf(buf, sizeof buf, "frame %lld: status %d (%s)", (long long)f, h_results[f].status,
                     h_results[f].status == KP_E_RANGE ? "out_stride smaller than the frame's final cloud, voxel / grid range exceeded, or resample candidate list overflow"
                     : h_results[f].status == KP_E_ARG ? "fewer final points than resample_n (select_points_randomly)" : "error");
            p->err = buf;
            return h_results[f].status;
        }
    return KP_OK;
}
}  // namespace

extern "C" {

int kp_pipeline_create(int device, const kp_pipeline_cfg *cfg, const float *h_xytab, const double *h_T, kp_pipeline **out)
{
    if (!cfg || !h_xytab || !out) return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_create: NULL argument");
    if (cfg->S < 1 || cfg->S > ENG_MAX_S || cfg->P < 1) return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_create: need 1..6 sensors and P >= 1");
    if (!(cfg->voxel_size > 0.0)) return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_create: voxel_size <= 0");
    if (cfg->floor_mode != KP_FLOOR_RANSAC && cfg->floor_mode != KP_FLOOR_PLANE)
        return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_create: floor_mode must be KP_FLOOR_RANSAC or KP_FLOOR_PLANE (got %d)", cfg->floor_mode);
    if (cfg->floor_mode == KP_FLOOR_PLANE && !(isfinite(cfg->floor_plane[0]) && isfinite(cfg->floor_plane[1]) && isfinite(cfg->floor_plane[2]) &&
                                               isfinite(cfg->floor_plane[3])))
        return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_create: the floor plane of KP_FLOOR_PLANE must have finite coefficients");
    if (cfg->do_floor && cfg->floor_mode == KP_FLOOR_RANSAC && (cfg->ransac_n < 3 || cfg->ransac_n > RS_MAX_N || cfg->ransac_iters < 1 || !(cfg->ransac_thr > 0.0)))
        return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_create: segment_plane needs 3 <= ransac_n <= %d, iterations >= 1, threshold > 0", RS_MAX_N);
    if (cfg->do_icp && cfg->S > 1 && (!(cfg->icp_voxel > 0.0) || !(cfg->icp_max_corr > 0.0) || cfg->normals_max_nn < 1 || !(cfg->normals_radius > 0.0)))
        return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_create: ICP needs icp_voxel, icp_max_corr, normals_radius > 0 and normals_max_nn >= 1");
    if (cfg->do_crop && !(cfg->crop_gate >= 0.0))
        return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_create: crop_gate must be >= 0 (millimetres)");
    if (cfg->resample_n != 0 && (cfg->resample_n < 1 || cfg->resample_n > 16384 || !kp_resample_engine_fits(cfg->resample_n)))
        return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_create: resample_n must be 0 (off) or 1..16384 (got %d)", cfg->resample_n);
    if (cfg->resample_n != 0 && cfg->resample_mode != KP_RESAMPLE_RANDOM && cfg->resample_mode != KP_RESAMPLE_PREFIX)
        return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_create: resample_mode must be KP_RESAMPLE_RANDOM or KP_RESAMPLE_PREFIX");
    if (cfg->ror_nb_points < 0 || (cfg->ror_nb_points > 0 && !(cfg->ror_radius > 0.0)))
        return kp_set_err(nullptr, KP_E_ARG, "kp_pipeline_create: ror_nb_points must be >= 0 (0 = off), and ror_radius > 0 when it is on");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        return kp_set_err(nullptr, KP_E_NODEVICE, "no CUDA device visible: kinectpy_b200 has no CPU path");
    }
    if (device < 0 || device >= ndev) return kp_set_err(nullptr, KP_E_ARG, "device %d out of range (have %d)", device, ndev);
    kp_pipeline *p = new kp_pipeline();
    p->cfg = *cfg;
    p->device = device;
    cudaSetDevice(device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) p->sm_count = prop.multiProcessorCount;
    // frames in flight = n_streams: batches of B frames share every launch, W batch slots overlap
    const int fl = cfg->n_streams < 1 ? 1 : (cfg->n_streams > 32 ? 32 : cfg->n_streams);
    int B = fl >= 16 ? 8 : (fl < 4 ? fl : 4);      // (measured: 170-181 frames/s for every B from 1 to 8; larger B = fewer launches per frame)
    if (getenv("KP_PIPE_BATCH")) B = atoi(getenv("KP_PIPE_BATCH"));
    if (B < 1) B = 1;
    if (B > 16) B = 16;
    int W = (fl + B - 1) / B;
    if (getenv("KP_PIPE_SLOTS")) W = atoi(getenv("KP_PIPE_SLOTS"));
    if (W < 1) W = 1;
    if (W > 8) W = 8;
    p->B = B; p->W = W;
    p->use_graph = !(getenv("KP_PIPE_GRAPH") && atoi(getenv("KP_PIPE_GRAPH")) == 0);
    p->use_vbi_icp = getenv("KP_ICP_VBI") && atoi(getenv("KP_ICP_VBI")) != 0;   // 8 % fewer ICP pass time, paid back by the index build: off unless asked for
    p->use_vbi_knn = getenv("KP_KNN_VBI") && atoi(getenv("KP_KNN_VBI")) != 0;   // measured slower than the grid level 0: off unless asked for
    p->knn_rad = (getenv("KP_KNN_RAD") && atoi(getenv("KP_KNN_RAD")) == 2) ? 2 : 1;
    if (getenv("KP_KNN_MID")) p->knn_mid = atof(getenv("KP_KNN_MID"));
    if (getenv("KP_VBI_RHO_A")) p->rho_mult_a = atof(getenv("KP_VBI_RHO_A"));
    if (getenv("KP_VBI_RHO_B")) p->rho_mult_b = atof(getenv("KP_VBI_RHO_B"));
    const int S = cfg->S;
    const size_t NP = (size_t)S * cfg->P;
    int64_t cells = 1 << 20;
    while (cells < (int64_t)NP * 16 && cells < (1 << 25)) cells <<= 1;
    p->cap_cells = cells;
    int64_t bricks = 1 << 16;
    while (bricks < (int64_t)NP * 3 && bricks < (1 << 23)) bricks <<= 1;
    p->cap_bricks = bricks;
    p->NPr = ((int64_t)NP + 63) & ~(int64_t)63;
    p->Pr = (cfg->P + 63) & ~(int64_t)63;
    p->T_fuse.assign(16 * S, 0.0);
    p->T_icp.assign(16 * S, 0.0);
    for (int s = 0; s < S; ++s)
        for (int i = 0; i < 16; ++i) {
            // h_T: [2][S][16] = fusion extrinsics, then ICP initial guesses; NULL -> identity for both
            p->T_fuse[16 * s + i] = h_T ? h_T[16 * s + i] : (i % 5 == 0 ? 1.0 : 0.0);
            p->T_icp[16 * s + i] = h_T ? h_T[16 * (S + s) + i] : (i % 5 == 0 ? 1.0 : 0.0);
        }
    auto fail = [&](int rc) {
        std::string m = p->err;
        kp_pipeline_destroy(p);
        return kp_set_err(nullptr, rc, "kp_pipeline_create: %s", m.c_str());
    };
    if (cudaMalloc((void **)&p->d_tab, sizeof(float) * 2 * NP) != cudaSuccess) { p->err = "table allocation failed"; return fail(KP_E_NOMEM); }
    if (cudaMemcpy(p->d_tab, h_xytab, sizeof(float) * 2 * NP, cudaMemcpyHostToDevice) != cudaSuccess) { p->err = "table copy failed"; return fail(KP_E_CUDA); }
    if (cfg->do_crop) {
        // the crop median counts a pixel outside the table as z = 0: which pixels those are, one bit each
        const int64_t words = (cfg->P + 31) / 32;
        std::vector<uint32_t> bits((size_t)S * words, 0u);
        for (int s = 0; s < S; ++s)
            for (int64_t i = 0; i < cfg->P; ++i) {
                const float *t = h_xytab + 2 * ((size_t)s * cfg->P + i);
                if (!(t[0] != t[0] || t[1] != t[1])) bits[(size_t)s * words + i / 32] |= 1u << (i % 32);
            }
        if (cudaMalloc((void **)&p->d_vbits, sizeof(uint32_t) * bits.size()) != cudaSuccess) { p->err = "table bitmap allocation failed"; return fail(KP_E_NOMEM); }
        if (cudaMemcpy(p->d_vbits, bits.data(), sizeof(uint32_t) * bits.size(), cudaMemcpyHostToDevice) != cudaSuccess) { p->err = "table bitmap copy failed"; return fail(KP_E_CUDA); }
    }
    p->slots.resize((size_t)W);
    for (auto &s : p->slots) {
        int rc = slot_create(p, s);
        if (rc != KP_OK) return fail(rc);
    }
    // One untimed pass over empty frames per slot: loads every kernel outside a capture and proves the launch
    // sequence on the degenerate input; then the sequence is captured as the slot's graph.
    for (auto &s : p->slots) {
        int rc = enqueue_k1(p, s, s.d_depth, s.d_rgb, B);
        if (rc == KP_OK) rc = enqueue_core(p, s, true);
        if (rc != KP_OK) { p->err = s.ctx->err.empty() ? s.aux->err : s.ctx->err; return fail(rc); }
        if (cudaStreamSynchronize(s.ctx->stream) != cudaSuccess || cudaStreamSynchronize(s.aux->stream) != cudaSuccess) {
            p->err = std::string("warm-up pass failed: ") + cudaGetErrorString(cudaGetLastError());
            return fail(KP_E_CUDA);
        }
        s.ctx->launches = 0; s.aux->launches = 0;
        if (p->use_graph) {
            rc = slot_capture(p, s);
            if (rc != KP_OK) return fail(rc);
            s.ctx->launches = 0; s.aux->launches = 0;
        }
    }
    *out = p;
    return KP_OK;
}

int kp_pipeline_destroy(kp_pipeline *p)
{
    if (!p) return KP_OK;
    cudaSetDevice(p->device);
    for (auto &s : p->slots) slot_destroy(s);
    if (p->d_tab) cudaFree(p->d_tab);
    if (p->d_vbits) cudaFree(p->d_vbits);
    if (p->h_res) cudaFreeHost(p->h_res);
    delete p;
    return KP_OK;
}

const char *kp_pipeline_last_error(kp_pipeline *p) { return p ? p->err.c_str() : kp_last_error(nullptr); }

int kp_pipeline_run(kp_pipeline *p, const uint16_t *depth, int depth_on_device, int64_t F, kp_frame_result *h_results,
                    float *d_out_xyz, int64_t out_stride)
{
    return run_impl(p, depth, nullptr, depth_on_device, F, nullptr, h_results, d_out_xyz, out_stride, nullptr);
}

int kp_pipeline_run_ex(kp_pipeline *p, const uint16_t *depth, const uint8_t *rgb, int inputs_on_device, int64_t F,
                       const int64_t *h_frame_ids, kp_frame_result *h_results, float *d_out_xyz, int64_t out_stride, float *d_fixed)
{
    return run_impl(p, depth, rgb, inputs_on_device, F, h_frame_ids, h_results, d_out_xyz, out_stride, d_fixed);
}

int kp_pipeline_run_host(kp_pipeline *p, const uint16_t *h_depth, int64_t F, kp_frame_result *h_results, float *h_out_xyz,
                         int64_t out_stride)
{
    if (p && h_out_xyz) {
        // the final clouds are written by a kernel straight into the caller's buffer (their sizes are only known
        // on the device): it must be pinned host memory (kp_host_alloc), which the device addresses directly
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, h_out_xyz) != cudaSuccess || (at.type != cudaMemoryTypeHost && at.type != cudaMemoryTypeManaged)) {
            cudaGetLastError();
            p->err = "kp_pipeline_run_host: h_out_xyz must be pinned host memory (kp_host_alloc)";
            return KP_E_ARG;
        }
    }
    return run_impl(p, h_depth, nullptr, 0, F, nullptr, h_results, h_out_xyz, out_stride, nullptr);
}

int64_t kp_pipeline_launch_count(kp_pipeline *p)
{
    int64_t n = 0;
    if (p) {
        n = p->launches;
        for (auto &s : p->slots) n += s.ctx->launches + s.aux->launches;
    }
    return n;
}

int kp_pipeline_frames_in_flight(kp_pipeline *p, int *batch, int *slots)
{
    if (!p) return KP_E_ARG;
    if (batch) *batch = p->B;
    if (slots) *slots = p->W;
    return KP_OK;
}

int kp_pipeline_frame_counts(kp_pipeline *p, int64_t *h_counts, int n)
{
    // the device-side counts of the first frame of batch slot 0 after its last batch (diagnostics / byte accounting):
    // n_fused, n_voxel, n_sor, n_lo, n_rest, n_merged, n_fsor, n_out, level-0 leftovers [3], level-1 leftovers [3],
    // valid rows of the S ICP inputs [6], their voxel counts [6]; with n >= 29 also mid-level leftovers [3], with n >= 35
    // twice the crop medians [6], with n >= 36 the radius outlier removal's survivors
    if (!p || !h_counts || n < 26) return KP_E_ARG;
    cudaSetDevice(p->device);
    EngSlot &s = p->slots[0];
    if (cudaStreamSynchronize(s.ctx->stream) != cudaSuccess) return KP_E_CUDA;
    EngDyn d;
    if (cudaMemcpy(&d, s.dyn, sizeof d, cudaMemcpyDeviceToHost) != cudaSuccess) return KP_E_CUDA;
    std::vector<EngCloud> cl((size_t)p->cfg.S);
    if (cudaMemcpy(cl.data(), s.icl, sizeof(EngCloud) * cl.size(), cudaMemcpyDeviceToHost) != cudaSuccess) return KP_E_CUDA;
    const int64_t v[8] = {d.n_fused, d.n_voxel, d.n_sor, d.n_lo, d.n_rest, d.n_merged, d.n_fsor, d.n_out};
    for (int i = 0; i < 8; ++i) h_counts[i] = v[i];
    for (int i = 0; i < 3; ++i) { h_counts[8 + i] = d.cnt_l0[i]; h_counts[11 + i] = d.cnt_l1[i]; }
    for (int i = 0; i < 6; ++i) { h_counts[14 + i] = i < p->cfg.S ? cl[i].nv : 0; h_counts[20 + i] = i < p->cfg.S ? cl[i].n : 0; }
    if (n >= 29)
        for (int i = 0; i < 3; ++i) h_counts[26 + i] = d.cnt_lm[i];
    if (n >= 35) {
        // twice the crop median of each sensor (a multiple of 0.5: exact), 0 without the crop
        double med[ENG_MAX_S] = {0.0};
        if (p->cfg.do_crop && cudaMemcpy(med, s.crop_med, sizeof(double) * p->cfg.S, cudaMemcpyDeviceToHost) != cudaSuccess) return KP_E_CUDA;
        for (int i = 0; i < 6; ++i) h_counts[29 + i] = i < p->cfg.S ? (int64_t)(2.0 * med[i]) : 0;
    }
    if (n >= 36) h_counts[35] = p->cfg.ror_nb_points > 0 ? d.n_ror : 0;
    return KP_OK;
}

int kp_pipeline_profile(kp_pipeline *p, int enable_or_read, int max_entries, const char **h_names, double *h_ms,
                        int64_t *h_calls, double *h_bytes, int *h_n)
{
    // enable_or_read: 1 = enable + reset, 0 = disable, 2 = read.  While enabled, batches run one at a time on slot 0
    // as direct launches (no graph, ICP branch on the main stream) with an event pair around every kernel family.
    if (!p) return KP_E_ARG;
    cudaSetDevice(p->device);
    kp_ctx *ctx = p->slots[0].ctx;
    if (enable_or_read == 1 || enable_or_read == 0) {
        kp_profile_reset(ctx);
        kp_profile_enable(ctx, enable_or_read);
        p->profiling = enable_or_read == 1;
        return KP_OK;
    }
    return kp_profile_read(ctx, max_entries, h_names, h_ms, h_calls, h_bytes, h_n);
}

}  // extern "C"
