// kp_grid.cu -- K3: uniform-grid spatial hash and the exact neighbour kernels built on it
// (kNN / hybrid, statistical outlier removal, radius outlier removal, normal estimation).
// Replaces the nanoflann KD-tree queries Open3D runs under remove_statistical_outlier
// (preprocessing/filtering.py:24, floor_removal.py:73), estimate_normals
// (preprocessing/registration.py:11-13) and remove_radius_outlier.
//
// Search scheme: one warp per query.  The query's 27-cell block is probed by 27 lanes at once
// (one hash probe each), the three cells of a z-row are merged into one contiguous range of the
// cell-sorted point array, and the warp streams those ranges 32 candidates at a time
// (one coalesced 16-byte load per lane).  Candidates that beat the current k-th entry are
// appended to a per-warp shared-memory buffer which is bitonic-sorted and truncated to k when it
// fills and at the end of every ring.  After ring r every point closer than r*cell has been seen,
// so the search stops as soon as the k-th distance is inside that radius; otherwise the next
// shell of cells is probed (isolated outliers -- the points SOR exists to find -- take this path).
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "kp_grid.cuh"
#include "kp_batch.cuh"

KpGridDev kp_grid_dev(const KpGrid &g)
{
    KpGridDev d;
    d.pts = g.d_sorted; d.slots = g.d_slots; d.hmask = g.hmask;
    d.sh_x = g.sh_x; d.sh_y = g.sh_y;
    for (int c = 0; c < 3; ++c) { d.dim[c] = g.dim[c]; d.org[c] = g.org[c]; }
    d.cell = g.cell; d.inv_cell = g.inv_cell;
    d.npts = g.n;
    d.cellmap = g.d_cellmap; d.run_start = g.d_run_start;
    return d;
}

namespace {
// ------------------------------------------------------------- build ------
template <class K>
__global__ void __launch_bounds__(256) k_grid_keys(const float *xyz, int64_t n, const __grid_constant__ KpGridDev g,
                                                   unsigned long long sentinel, K *keys)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
    K key;
    if (isnan(x)) key = (K)sentinel;
    else {
        int cx = min(max(kp_cell_coord(g, (double)x, 0), 0), g.dim[0] - 1);
        int cy = min(max(kp_cell_coord(g, (double)y, 1), 0), g.dim[1] - 1);
        int cz = min(max(kp_cell_coord(g, (double)z, 2), 0), g.dim[2] - 1);
        key = (K)kp_cell_key(g, cx, cy, cz);
    }
    keys[i] = key;
}

template <class K>
__global__ void __launch_bounds__(256) k_grid_insert(const K *keys_sorted, int32_t *run_start, const int32_t *d_R,
                                                     int n, unsigned long long sentinel, int has_sentinel,
                                                     uint4 *slots, uint32_t hmask, uint2 *cellmap, int sh_x, int sh_y,
                                                     int dim1, int dim2)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    int R = *d_R;
    if (r >= R) return;
    if (r == 0) run_start[R] = n;   // closes the last run (read by later kernels only)
    int a = run_start[r], b = (r + 1 < R) ? run_start[r + 1] : n;
    unsigned long long key = (unsigned long long)keys_sorted[a];
    if (has_sentinel && key == sentinel) return;
    if (cellmap) {
        // runs are in key order = cell-index order, so r is the rank of this cell among the occupied ones
        const long long cx = (long long)(key >> sh_x), cy = (long long)((key >> sh_y) & ((1ull << (sh_x - sh_y)) - 1ull)),
                        cz = (long long)(key & ((1ull << sh_y) - 1ull));
        const long long bit = (cx * dim1 + cy) * dim2 + cz;
        atomicAnd(&cellmap[bit >> 5].x, ~(1u << (bit & 31)));
        atomicMin(&cellmap[bit >> 5].y, (unsigned)r);
        return;
    }
    uint32_t h = (uint32_t)kp_mix64(key) & hmask;
    for (;;) {
        // claim the key half of the slot, then fill the value half (readers only run in later kernels)
        unsigned long long prev = atomicCAS((unsigned long long *)(slots + h), ~0ull, key);
        if (prev == ~0ull) { reinterpret_cast<int2 *>(slots + h)[1] = make_int2(a, b); return; }
        h = (h + 1) & hmask;
    }
}

__global__ void __launch_bounds__(256) k_grid_gather(const float *xyz, const int32_t *vals_sorted, int64_t n, float4 *sorted)
{
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    int i = vals_sorted[t];
    sorted[t] = make_float4(xyz[3 * (int64_t)i], xyz[3 * (int64_t)i + 1], xyz[3 * (int64_t)i + 2], __int_as_float(i));
}

int bit_length_u(long long v)
{
    int b = 0;
    while (v > 0) { ++b; v >>= 1; }
    return b < 1 ? 1 : b;
}

template <class K>
int grid_sort_build(kp_ctx *ctx, const float *d_xyz, int64_t n, KpGrid *g, int total_bits, unsigned long long sentinel,
                    int32_t **run_start_out, int32_t **d_R_out, bool build_hash)
{
    K *keys, *keys_tmp, *keys_sorted;
    int32_t *vals, *vals_tmp, *vals_sorted, *run_start, *d_R;
    KP_TRY(kp_ws(ctx, (size_t)n, &keys));
    KP_TRY(kp_ws(ctx, (size_t)n, &keys_tmp));
    KP_TRY(kp_ws(ctx, (size_t)n, &vals));
    KP_TRY(kp_ws(ctx, (size_t)n, &vals_tmp));
    KP_TRY(kp_ws(ctx, (size_t)n + 1, &run_start));
    KP_TRY(kp_ws(ctx, 4, &d_R));
    KpGridDev gd = kp_grid_dev(*g);
    {
        KP_PROFB(ctx, "grid_keys", (double)n * (12.0 + sizeof(K)));
        k_grid_keys<K><<<kp_blocks(n, 256), 256, 0, ctx->stream>>>(d_xyz, n, gd, sentinel, keys);
        KP_LAUNCH_CHECK(ctx);
    }
    if (sizeof(K) == 8) {
        KP_TRY(kp_prim_sort_pairs_u64(ctx, n, total_bits + 1, (uint64_t *)keys, (uint64_t *)keys_tmp, vals, vals_tmp,
                                      (uint64_t **)&keys_sorted, &vals_sorted));
        KP_TRY(kp_prim_run_starts_u64(ctx, n, (const uint64_t *)keys_sorted, run_start, d_R));
    } else {
        KP_TRY(kp_prim_sort_pairs_u32(ctx, n, total_bits + 1, (uint32_t *)keys, (uint32_t *)keys_tmp, vals, vals_tmp,
                                      (uint32_t **)&keys_sorted, &vals_sorted));
        KP_TRY(kp_prim_run_starts_u32(ctx, n, (const uint32_t *)keys_sorted, run_start, d_R));
    }
    if (run_start_out) *run_start_out = run_start;
    if (d_R_out) *d_R_out = d_R;
    if (!build_hash) return KP_OK;
    g->d_run_start = run_start;
    const size_t words = (size_t)(((long long)g->dim[0] * g->dim[1] * g->dim[2] + 31) / 32) + 1;
    const size_t table_bytes = g->d_cellmap ? words * sizeof(uint2) : ((size_t)g->hmask + 1) * sizeof(uint4);
    KP_PROFB(ctx, "grid_hash", (double)table_bytes + (double)n * (4.0 + 12.0 + 16.0));
    KP_CUDA(ctx, cudaMemsetAsync(g->d_cellmap ? (void *)g->d_cellmap : (void *)g->d_slots, 0xff, table_bytes, ctx->stream));
    k_grid_insert<K><<<kp_blocks(n, 256), 256, 0, ctx->stream>>>(keys_sorted, run_start, d_R, (int)n, sentinel, 1, g->d_slots,
                                                                 g->hmask, g->d_cellmap, g->sh_x, g->sh_y, g->dim[1],
                                                                 g->dim[2]);
    KP_LAUNCH_CHECK(ctx);
    k_grid_gather<<<kp_blocks(n, 256), 256, 0, ctx->stream>>>(d_xyz, vals_sorted, n, g->d_sorted);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}

int grid_layout(kp_ctx *ctx, const float *h_bounds6, double cell, KpGrid *g, int *total_bits)
{
    // grow the cell until every axis fits 21 bits
    for (;;) {
        bool ok = true;
        for (int c = 0; c < 3; ++c) {
            double ext = (double)h_bounds6[3 + c] - (double)h_bounds6[c];
            if (!(ext >= 0)) ext = 0;
            if (ext / cell > 2000000.0) ok = false;
        }
        if (ok) break;
        cell *= 2.0;
    }
    g->cell = cell;
    g->inv_cell = 1.0 / cell;
    int bits[3];
    for (int c = 0; c < 3; ++c) {
        g->org[c] = (double)h_bounds6[c];
        double ext = (double)h_bounds6[3 + c] - g->org[c];
        if (!(ext >= 0)) ext = 0;
        g->dim[c] = (int)floor(ext * g->inv_cell) + 2;   // +1 for the top cell, +1 rounding margin
        bits[c] = bit_length_u(g->dim[c] - 1);
    }
    g->sh_y = bits[2];
    g->sh_x = bits[2] + bits[1];
    *total_bits = bits[0] + bits[1] + bits[2];
    (void)ctx;
    return KP_OK;
}
}  // namespace

int kp_grid_build(kp_ctx *ctx, const float *d_xyz, int64_t n, double cell, const float *h_bounds6, KpGrid *g)
{
    *g = KpGrid();
    if (!(cell > 0.0)) return kp_set_err(ctx, KP_E_ARG, "grid cell must be > 0");
    if (n > 2147483000LL) return kp_set_err(ctx, KP_E_ARG, "more than 2^31 points in one call");
    g->n = (int32_t)n;
    if (n <= 0) return KP_OK;
    float b6[6];
    if (!h_bounds6) {
        int64_t nv = 0;
        KP_TRY(kp_prim_bounds_fetch(ctx, d_xyz, n, b6, &nv));
        if (nv == 0) { b6[0] = b6[1] = b6[2] = 0; b6[3] = b6[4] = b6[5] = 0; }
        h_bounds6 = b6;
    }
    int total_bits = 0;
    KP_TRY(grid_layout(ctx, h_bounds6, cell, g, &total_bits));
    unsigned long long sentinel = 1ull << total_bits;   // total_bits <= 63
    // hash capacity: power of two >= 2 * min(n, #cells), in 64 bits (2 * n can exceed 2^32); the probe index is 32-bit
    double ncell = (double)g->dim[0] * g->dim[1] * g->dim[2];
    double want = 2.0 * ((double)n < ncell ? (double)n : ncell);
    uint64_t cap = 1024;
    while ((double)cap < want) cap <<= 1;
    const bool force_hash = getenv("KP_GRID_FORCE_HASH") != nullptr;   // test hook: exercise the huge-grid path
    const bool use_map = ncell <= 134217728.0 && !force_hash;           // <= 32 MiB of cell map
    if (!use_map && cap > (1ull << 31))
        return kp_set_err(ctx, KP_E_RANGE, "grid hash of %llu slots for %lld points over %.3g cells exceeds 2^31 slots",
                          (unsigned long long)cap, (long long)n, ncell);
    KP_TRY(kp_ws(ctx, (size_t)n, &g->d_sorted));
    if (use_map) {
        KP_TRY(kp_ws(ctx, (size_t)(ncell / 32.0) + 2, &g->d_cellmap));
    } else {
        g->hmask = (uint32_t)(cap - 1);
        KP_TRY(kp_ws(ctx, (size_t)cap, &g->d_slots));
    }
    if (total_bits + 1 <= 32) return grid_sort_build<uint32_t>(ctx, d_xyz, n, g, total_bits, sentinel, nullptr, nullptr, true);
    return grid_sort_build<uint64_t>(ctx, d_xyz, n, g, total_bits, sentinel, nullptr, nullptr, true);
}

int kp_grid_build_knn(kp_ctx *ctx, const float *d_xyz, int64_t n, double cell, int k, const float *h_bounds6, KpGrid *g)
{
    static const int want = getenv("KP_KNN_RAD") ? atoi(getenv("KP_KNN_RAD")) : 1;
    const int rad = (k <= 64 && want == 2) ? 2 : 1;
    KP_TRY(kp_grid_build(ctx, d_xyz, n, cell / (double)rad, h_bounds6, g));
    g->rad = rad;
    return KP_OK;
}

int kp_grid_auto_cell(kp_ctx *ctx, const float *d_xyz, int64_t n, const float *h_bounds6, double target_per_cell,
                      double *cell_out)
{
    // Trial grid at extent/256, count occupied cells, rescale assuming the cloud is a 2-D surface
    // (occupancy ~ cell^2).  Only the cost of the search depends on this choice, never its result.
    float b6[6];
    if (!h_bounds6) {
        int64_t nv = 0;
        KP_TRY(kp_prim_bounds_fetch(ctx, d_xyz, n, b6, &nv));
        if (nv == 0) { *cell_out = 1.0; return KP_OK; }
        h_bounds6 = b6;
    }
    double e = 0;
    for (int c = 0; c < 3; ++c) e = fmax(e, (double)h_bounds6[3 + c] - (double)h_bounds6[c]);
    if (!(e > 0)) { *cell_out = 1.0; return KP_OK; }
    KpGrid g;
    g.n = (int32_t)n;
    int total_bits = 0;
    double cell0 = e / 256.0;
    KP_TRY(grid_layout(ctx, h_bounds6, cell0, &g, &total_bits));
    int32_t *d_R = nullptr;
    unsigned long long sentinel = 1ull << total_bits;
    if (total_bits + 1 <= 32) KP_TRY(grid_sort_build<uint32_t>(ctx, d_xyz, n, &g, total_bits, sentinel, nullptr, &d_R, false));
    else KP_TRY(grid_sort_build<uint64_t>(ctx, d_xyz, n, &g, total_bits, sentinel, nullptr, &d_R, false));
    KP_CUDA(ctx, cudaMemcpyAsync(ctx->d_scratch, d_R, sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
    KP_TRY(kp_fetch_scratch(ctx, sizeof(int32_t)));
    int R = *(int32_t *)ctx->h_scratch;
    double occ = R > 0 ? (double)n / (double)R : 1.0;
    double cell = g.cell * sqrt(target_per_cell / occ);
    if (cell < g.cell / 64.0) cell = g.cell / 64.0;
    if (cell > e) cell = e;
    *cell_out = cell;
    return KP_OK;
}

// ============================================================ queries =====
namespace {
constexpr int KQ_WARPS = 4;
enum { KQ_MODE_KNN = 0, KQ_MODE_RADIUS = 1, KQ_MODE_NORMALS = 2 };

struct KnnParams {
    KpGridDev g;
    const float *queries;   // NULL -> the cloud queries itself, in cell-sorted order
    int64_t nq;
    int k, cap, mode;
    int rad;                // level-0 block radius in cells (1: 27 cells, 2: 125 cells) the grid was sized for
    double r2cap;           // > 0: only neighbours with d2 < r2cap
    int32_t *idx; double *d2; int32_t *count; double *mean;
    const float *cloud; float *normals;
    int32_t *rcount;
    const int32_t *qlist; const int32_t *qcount;   // visit only these query positions (rows of qpts)
    uint8_t *strag_flags;                          // thread kernel: flags[q] = 1 for queries it could not certify
    const float4 *qpts;                            // self-query source rows (level-0 cell-sorted array)
    int32_t *dbg;                                  // optional [8] tally of the reasons level 1 hands a query on (KP_DEBUG_KNN)
    // frame engine (batched launches, kp_engine.cu): the grid layout and the query count were produced on the device
    const KpGridDev *gdev;                         // non-NULL: replaces g
    const int32_t *nq_dev;                         // non-NULL: replaces nq
    const KpVbiDev *vbi;                           // voxel-brick index of the cloud (k_knn_vbi_b)
    double rho_a, rho_b;                           // its two search radii
};

// batched launches read their parameter block from device memory (blockIdx.y selects the frame): uniform, cached
// loads of the fields a thread uses, with the device-side grid layout / query count patched in
__device__ __forceinline__ KnnParams knn_params_batched(const KnnParams *__restrict__ pp)
{
    KnnParams p = pp[blockIdx.y];
    if (p.gdev) p.g = *p.gdev;
    if (p.nq_dev) p.nq = *p.nq_dev;
    return p;
}

__device__ __forceinline__ bool kq_less(double d, int i, double td, int ti) { return d < td || (d == td && i < ti); }

// bitonic sort of cap (power of two) entries by (d2, idx), one warp, shared memory
__device__ void kq_sort(double *bd, int *bi, int cap, int lane)
{
    for (int size = 2; size <= cap; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = lane; t < (cap >> 1); t += 32) {
                int i = ((t / stride) * 2 * stride) + (t % stride);
                int j = i + stride;
                bool up = (i & size) == 0;
                double di = bd[i], dj = bd[j];
                int ii = bi[i], ij = bi[j];
                bool sw = kq_less(dj, ij, di, ii) == up;
                if (sw) { bd[i] = dj; bd[j] = di; bi[i] = ij; bi[j] = ii; }
            }
            __syncwarp();
        }
    }
}

struct KqState {
    double *bd; int *bi;
    int n_buf, k, cap;
    double tau_d; int tau_i;
    double qx, qy, qz;
    int lane;
    int rcount;
};

__device__ __forceinline__ void kq_truncate(KqState &s)
{
    for (int t = s.n_buf + s.lane; t < s.cap; t += 32) { s.bd[t] = INFINITY; s.bi[t] = 0x7fffffff; }
    __syncwarp();
    kq_sort(s.bd, s.bi, s.cap, s.lane);
    if (s.n_buf > s.k) s.n_buf = s.k;
    if (s.n_buf == s.k) { s.tau_d = s.bd[s.k - 1]; s.tau_i = s.bi[s.k - 1]; }
    __syncwarp();
}

// ---- buffer maintenance without sorting: the buffer always holds EVERY candidate seen so far that is
// below the bound tau.  When it fills, tau is lowered to a sampled pivot that still has >= k entries at or
// below it (one counting pass + one in-place compaction); the exact order is only established once, by the
// final kq_truncate.  (A bitonic sort per overflow, the first version, cost more than the search itself.)
__device__ __forceinline__ int kq_warp_sum(int c)
{
#pragma unroll
    for (int sft = 16; sft >= 1; sft >>= 1) c += __shfl_xor_sync(KP_FULL, c, sft);
    return c;
}
__device__ __forceinline__ int kq_count_le(const KqState &s, double pd, int pi)
{
    int c = 0;
    for (int t = s.lane; t < s.n_buf; t += 32) c += !kq_less(pd, pi, s.bd[t], s.bi[t]);
    return kq_warp_sum(c);
}
__device__ __forceinline__ int kq_count_d_le(const KqState &s, double lim)
{
    int c = 0;
    for (int t = s.lane; t < s.n_buf; t += 32) c += s.bd[t] <= lim;
    return kq_warp_sum(c);
}
__device__ __forceinline__ void kq_keep_le(KqState &s, double pd, int pi)
{
    int out = 0;
    const unsigned lt = (1u << s.lane) - 1u;
    for (int base = 0; base < s.n_buf; base += 32) {
        const int t = base + s.lane;
        const bool v = t < s.n_buf;
        const double d = v ? s.bd[t] : 0.0;
        const int i = v ? s.bi[t] : 0;
        const bool keep = v && !kq_less(pd, pi, d, i);
        const unsigned m = __ballot_sync(KP_FULL, keep);
        __syncwarp();   // the whole chunk is in registers before anything (at an index <= t) is overwritten
        if (keep) { int pos = out + __popc(m & lt); s.bd[pos] = d; s.bi[pos] = i; }
        out += __popc(m);
        __syncwarp();
    }
    s.n_buf = out;
}
__device__ void kq_tighten(KqState &s)
{
    // 32 evenly spaced samples, sorted across the lanes (bitonic network on shuffles)
    const int si = (int)(((long long)s.lane * s.n_buf) >> 5);
    double sd = s.bd[si];
    int sid = s.bi[si];
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            const double od = __shfl_xor_sync(KP_FULL, sd, stride);
            const int oi = __shfl_xor_sync(KP_FULL, sid, stride);
            const bool keep_min = ((s.lane & stride) == 0) == ((s.lane & size) == 0);
            const bool other_less = kq_less(od, oi, sd, sid);
            if (keep_min ? other_less : kq_less(sd, sid, od, oi)) { sd = od; sid = oi; }
        }
    }
    // lowest sample quantile expected to keep ~1.5 k entries; verify by counting, move up if it keeps too few
    int j = (int)((48LL * s.k) / s.n_buf);
    if (j > 31) j = 31;
    for (int tries = 0; tries < 6; ++tries) {
        const double pd = __shfl_sync(KP_FULL, sd, j);
        const int pi = __shfl_sync(KP_FULL, sid, j);
        const int c = kq_count_le(s, pd, pi);
        if (c >= s.k) {
            if (c < s.n_buf) { kq_keep_le(s, pd, pi); s.tau_d = pd; s.tau_i = pi; }
            break;
        }
        if (j == 31) break;
        j = min(31, 2 * j + 1);
    }
    if (s.n_buf > s.cap - 32) kq_truncate(s);   // unlucky samples: fall back to the exact sort
}

__device__ __forceinline__ void kq_candidate(KqState &s, bool valid, float4 p, int mode)
{
    double d = kp_d2(s.qx, s.qy, s.qz, (double)p.x, (double)p.y, (double)p.z);
    int id = __float_as_int(p.w);
    if (mode == KQ_MODE_RADIUS) {
        s.rcount += __popc(__ballot_sync(KP_FULL, valid && d < s.tau_d));
        return;
    }
    bool pass = valid && kq_less(d, id, s.tau_d, s.tau_i);
    unsigned m = __ballot_sync(KP_FULL, pass);
    if (m == 0) return;
    if (pass) {
        int pos = s.n_buf + __popc(m & ((1u << s.lane) - 1u));
        s.bd[pos] = d; s.bi[pos] = id;
    }
    s.n_buf += __popc(m);
    __syncwarp();
    if (s.n_buf > s.cap - 32) kq_tighten(s);
}

__device__ __forceinline__ void kq_scan_ranges(const KpGridDev &g, int rs, int re, KqState &s, int mode)
{
    unsigned m = __ballot_sync(KP_FULL, re > rs);
    while (m) {
        int j = __ffs(m) - 1;
        m &= m - 1;
        int a = __shfl_sync(KP_FULL, rs, j), b = __shfl_sync(KP_FULL, re, j);
        // four coalesced loads in flight per lane before the (sequential) candidate handling
        for (int t = a; t < b; t += 128) {
            const int i0 = t + s.lane;
            const bool v0 = i0 < b, v1 = i0 + 32 < b, v2 = i0 + 64 < b, v3 = i0 + 96 < b;
            const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 p0 = v0 ? __ldg(g.pts + i0) : z4;
            const float4 p1 = v1 ? __ldg(g.pts + i0 + 32) : z4;
            const float4 p2 = v2 ? __ldg(g.pts + i0 + 64) : z4;
            const float4 p3 = v3 ? __ldg(g.pts + i0 + 96) : z4;
            kq_candidate(s, v0, p0, mode);
            if (t + 32 < b) kq_candidate(s, v1, p1, mode);
            if (t + 64 < b) kq_candidate(s, v2, p2, mode);
            if (t + 96 < b) kq_candidate(s, v3, p3, mode);
        }
    }
}

// analytic smallest-eigenvector of a symmetric 3x3 (SURVEY.md A.6); A = {xx,xy,xz,yy,yz,zz}
__device__ void kq_cross(const double *a, const double *b, double *o)
{
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ void kq_evec0(const double *A, double ev, double *out)
{
    double r0[3] = {A[0] - ev, A[1], A[2]}, r1[3] = {A[1], A[3] - ev, A[4]}, r2[3] = {A[2], A[4], A[5] - ev};
    double c01[3], c02[3], c12[3];
    kq_cross(r0, r1, c01); kq_cross(r0, r2, c02); kq_cross(r1, r2, c12);
    double d0 = c01[0] * c01[0] + c01[1] * c01[1] + c01[2] * c01[2];
    double d1 = c02[0] * c02[0] + c02[1] * c02[1] + c02[2] * c02[2];
    double d2 = c12[0] * c12[0] + c12[1] * c12[1] + c12[2] * c12[2];
    double dm = d0; double b0 = c01[0], b1 = c01[1], b2 = c01[2];
    if (d1 > dm) { dm = d1; b0 = c02[0]; b1 = c02[1]; b2 = c02[2]; }
    if (d2 > dm) { dm = d2; b0 = c12[0]; b1 = c12[1]; b2 = c12[2]; }
    if (dm > 0) { double sq = sqrt(dm); out[0] = b0 / sq; out[1] = b1 / sq; out[2] = b2 / sq; }
    else { out[0] = out[1] = out[2] = 0.0; }
}
__device__ void kq_evec1(const double *A, const double *e0, double ev1, double *out)
{
    double U[3], V[3];
    if (fabs(e0[0]) > fabs(e0[1])) { double il = 1.0 / sqrt(e0[0] * e0[0] + e0[2] * e0[2]); U[0] = -e0[2] * il; U[1] = 0; U[2] = e0[0] * il; }
    else { double il = 1.0 / sqrt(e0[1] * e0[1] + e0[2] * e0[2]); U[0] = 0; U[1] = e0[2] * il; U[2] = -e0[1] * il; }
    kq_cross(e0, U, V);
    double AU[3] = {A[0] * U[0] + A[1] * U[1] + A[2] * U[2], A[1] * U[0] + A[3] * U[1] + A[4] * U[2], A[2] * U[0] + A[4] * U[1] + A[5] * U[2]};
    double AV[3] = {A[0] * V[0] + A[1] * V[1] + A[2] * V[2], A[1] * V[0] + A[3] * V[1] + A[4] * V[2], A[2] * V[0] + A[4] * V[1] + A[5] * V[2]};
    double m00 = U[0] * AU[0] + U[1] * AU[1] + U[2] * AU[2] - ev1;
    double m01 = U[0] * AV[0] + U[1] * AV[1] + U[2] * AV[2];
    double m11 = V[0] * AV[0] + V[1] * AV[1] + V[2] * AV[2] - ev1;
    double a00 = fabs(m00), a01 = fabs(m01), a11 = fabs(m11);
    double cu, cv;
    if (a00 >= a11) {
        if (fmax(a00, a01) > 0) {
            if (a00 >= a01) { m01 /= m00; m00 = 1 / sqrt(1 + m01 * m01); m01 *= m00; }
            else { m00 /= m01; m01 = 1 / sqrt(1 + m00 * m00); m00 *= m01; }
            cu = m01; cv = -m00;
        } else { cu = 1; cv = 0; }
    } else {
        if (fmax(a11, a01) > 0) {
            if (a11 >= a01) { m01 /= m11; m11 = 1 / sqrt(1 + m01 * m01); m01 *= m11; }
            else { m11 /= m01; m01 = 1 / sqrt(1 + m11 * m11); m11 *= m01; }
            cu = m11; cv = -m01;
        } else { cu = 1; cv = 0; }
    }
    for (int c = 0; c < 3; ++c) out[c] = cu * U[c] + cv * V[c];
}
__device__ void kq_smallest_eigvec(const double *cov, double *nrm)
{
    double A[6];
    double mc = cov[0];
    for (int i = 1; i < 6; ++i) if (cov[i] > mc) mc = cov[i];
    if (mc == 0.0) { nrm[0] = nrm[1] = nrm[2] = 0.0; return; }
    for (int i = 0; i < 6; ++i) A[i] = cov[i] / mc;
    double norm = A[1] * A[1] + A[2] * A[2] + A[4] * A[4];
    if (norm > 0) {
        double q = (A[0] + A[3] + A[5]) / 3.0;
        double b00 = A[0] - q, b11 = A[3] - q, b22 = A[5] - q;
        double p = sqrt((b00 * b00 + b11 * b11 + b22 * b22 + norm * 2.0) / 6.0);
        double c00 = b11 * b22 - A[4] * A[4];
        double c01 = A[1] * b22 - A[4] * A[2];
        double c02 = A[1] * A[4] - b11 * A[2];
        double det = (b00 * c00 - A[1] * c01 + A[2] * c02) / (p * p * p);
        double half = det * 0.5;
        half = fmin(fmax(half, -1.0), 1.0);
        double angle = acos(half) / 3.0;
        const double two_thirds_pi = 2.09439510239319549;
        double beta2 = cos(angle) * 2.0;
        double beta0 = cos(angle + two_thirds_pi) * 2.0;
        double beta1 = -(beta0 + beta2);
        double e0 = q + p * beta0, e1 = q + p * beta1, e2 = q + p * beta2;
        double v0[3], v1[3], v2[3];
        if (half >= 0) {
            kq_evec0(A, e2, v2);
            kq_evec1(A, v2, e1, v1);
            kq_cross(v1, v2, v0);
        } else {
            kq_evec0(A, e0, v0);
        }
        nrm[0] = v0[0]; nrm[1] = v0[1]; nrm[2] = v0[2];
    } else {
        if (A[0] < A[3] && A[0] < A[5]) { nrm[0] = 1; nrm[1] = 0; nrm[2] = 0; }
        else if (A[3] < A[0] && A[3] < A[5]) { nrm[0] = 0; nrm[1] = 1; nrm[2] = 0; }
        else { nrm[0] = 0; nrm[1] = 0; nrm[2] = 1; }
    }
}

// Results of one query, written by ONE thread from its list sorted ascending by (d2, index)
// (entry t at bd[t*stride], bi[t*stride]).  Sums run sequentially in that order -- the order Open3D's
// std::accumulate sees (the KD-tree returns neighbours by ascending distance) and the oracle uses.
__device__ void kq_finalize(const KnnParams &p, int64_t row, int cnt, const double *bd, const int *bi, int stride)
{
    if (p.mode == KQ_MODE_KNN) {
        if (p.idx) for (int t = 0; t < p.k; ++t) p.idx[row * p.k + t] = t < cnt ? bi[t * stride] : -1;
        if (p.d2) for (int t = 0; t < p.k; ++t) p.d2[row * p.k + t] = t < cnt ? bd[t * stride] : INFINITY;
        if (p.count) p.count[row] = cnt;
        if (p.mean) {
            double acc = 0.0;
            for (int t = 0; t < cnt; ++t) acc = __dadd_rn(acc, sqrt(bd[t * stride]));
            p.mean[row] = cnt > 0 ? __ddiv_rn(acc, (double)cnt) : -1.0;
        }
        return;
    }
    // normals: covariance from cumulants over the neighbourhood, smallest eigenvector (SURVEY.md A.6)
    double nr[3] = {0.0, 0.0, 1.0};
    if (cnt >= 3) {
        double sm[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (int t = 0; t < cnt; ++t) {
            int64_t j = bi[t * stride];
            double x = (double)p.cloud[3 * j], y = (double)p.cloud[3 * j + 1], z = (double)p.cloud[3 * j + 2];
            sm[0] += x; sm[1] += y; sm[2] += z;
            sm[3] += x * x; sm[4] += x * y; sm[5] += x * z; sm[6] += y * y; sm[7] += y * z; sm[8] += z * z;
        }
        double inv = (double)cnt;
        for (int c = 0; c < 9; ++c) sm[c] /= inv;
        double cov[6] = {sm[3] - sm[0] * sm[0], sm[4] - sm[0] * sm[1], sm[5] - sm[0] * sm[2],
                         sm[6] - sm[1] * sm[1], sm[7] - sm[1] * sm[2], sm[8] - sm[2] * sm[2]};
        kq_smallest_eigvec(cov, nr);
        if (nr[0] == 0.0 && nr[1] == 0.0 && nr[2] == 0.0) nr[2] = 1.0;
    }
    p.normals[3 * row] = (float)nr[0]; p.normals[3 * row + 1] = (float)nr[1]; p.normals[3 * row + 2] = (float)nr[2];
}

// ---- warp-per-query kernel: any k, ring expansion, linear-scan fallback.  Used for large k, for external
// queries and for the stragglers the thread-per-query kernel hands over (qlist / qcount).
__device__ __forceinline__ void knn_warp_body(const KnnParams &p, unsigned char *smem_raw)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const KpGridDev &g = p.g;
    const int64_t nq = p.qcount ? (int64_t)*p.qcount : p.nq;
    for (int64_t w = (int64_t)blockIdx.x * KQ_WARPS + warp; w < nq; w += (int64_t)gridDim.x * KQ_WARPS) {
        const int64_t q = p.qlist ? (int64_t)p.qlist[w] : w;
        KqState s;
        s.bd = reinterpret_cast<double *>(smem_raw) + (size_t)warp * p.cap;
        s.bi = reinterpret_cast<int *>(reinterpret_cast<double *>(smem_raw) + (size_t)KQ_WARPS * p.cap) + (size_t)warp * p.cap;
        s.n_buf = 0; s.k = p.k; s.cap = p.cap; s.lane = lane; s.rcount = 0;
        s.tau_d = p.r2cap > 0 ? p.r2cap : INFINITY;
        s.tau_i = p.r2cap > 0 ? (int)0x80000000 : 0x7fffffff;   // strict d2 < r2cap: equality never passes

        int64_t row;
        if (p.queries) {
            s.qx = (double)p.queries[3 * q]; s.qy = (double)p.queries[3 * q + 1]; s.qz = (double)p.queries[3 * q + 2];
            row = q;
        } else {
            float4 me = __ldg(p.qpts + q);
            s.qx = (double)me.x; s.qy = (double)me.y; s.qz = (double)me.z;
            row = __float_as_int(me.w);
        }
        const bool qnan = isnan(s.qx);
        if (!qnan && g.dim[0] > 0) {
            // Rings are centred on the in-grid cell nearest to the query.  For a query inside the grid that is
            // its own cell; for an outside query, a grid point within distance rho of the query still lies
            // within ceil(rho/cell) cells of the clamped cell on every axis, so the ring-r guarantee
            // ("everything closer than r*cell has been seen") holds unchanged.
            const int cx = min(max(kp_cell_coord(g, s.qx, 0), 0), g.dim[0] - 1);
            const int cy = min(max(kp_cell_coord(g, s.qy, 1), 0), g.dim[1] - 1);
            const int cz = min(max(kp_cell_coord(g, s.qz, 2), 0), g.dim[2] - 1);
            // rings needed to cover the whole grid from this cell
            int maxring = max(max(max(cx, g.dim[0] - 1 - cx), max(cy, g.dim[1] - 1 - cy)), max(cz, g.dim[2] - 1 - cz));
            if (maxring < 1) maxring = 1;
            // ---- ring 0+1: the 27-cell block, z-rows merged
            {
                int2 r = make_int2(0, 0);
                if (lane < 27) r = kp_cell_range(g, cx + lane / 9 - 1, cy + (lane / 3) % 3 - 1, cz + lane % 3 - 1);
                bool ne = r.y > r.x;
                int a = ne ? r.x : 0x7fffffff, b = ne ? r.y : 0;
                int a1 = __shfl_down_sync(KP_FULL, a, 1), b1 = __shfl_down_sync(KP_FULL, b, 1);
                int a2 = __shfl_down_sync(KP_FULL, a, 2), b2 = __shfl_down_sync(KP_FULL, b, 2);
                if (lane < 27 && lane % 3 == 0) { a = min(a, min(a1, a2)); b = max(b, max(b1, b2)); if (b == 0) a = 0; }
                else { a = 0; b = 0; }
                kq_scan_ranges(g, a, b, s, p.mode);
            }
            int ring = 1;
            if (p.mode != KQ_MODE_RADIUS) {
                for (;;) {
                    double safe = (double)ring * g.cell * (1.0 - 1.0 / 1048576.0);
                    double s2 = safe * safe;
                    // certified as soon as k of the candidates seen so far lie inside the scanned radius
                    if (s.n_buf >= s.k && kq_count_d_le(s, s2) >= s.k) break;
                    if (p.r2cap > 0 && p.r2cap <= s2) break;
                    if (ring >= maxring) break;
                    ++ring;
                    {
                        // A shell this large costs more probes than the cloud has points: finish with one exact
                        // linear pass over the sorted array instead (bounds the work of far-away stragglers).
                        const long long w3 = 2LL * ring + 1;
                        if (w3 * w3 * w3 > (long long)g.npts) {
                            s.n_buf = 0;
                            s.tau_d = p.r2cap > 0 ? p.r2cap : INFINITY;
                            s.tau_i = p.r2cap > 0 ? (int)0x80000000 : 0x7fffffff;
                            kq_scan_ranges(g, 0, lane == 0 ? g.npts : 0, s, p.mode);
                            break;
                        }
                    }
                    // ---- shell `ring`: two full slabs dz = +-ring, then the perimeter of every layer in between
                    const long long sw = 2LL * ring + 1;
                    const long long slab = sw * sw, per = 4 * (sw - 1);
                    const long long ncell = 2 * slab + (sw - 2) * per;
                    for (long long e0 = 0; e0 < ncell; e0 += 32) {
                        long long e = e0 + lane;
                        int2 r = make_int2(0, 0);
                        if (e < ncell) {
                            int dx, dy, dz;
                            if (e < 2 * slab) {
                                int sl = (int)(e / slab);
                                long long rem = e % slab;
                                dx = (int)(rem / sw) - ring; dy = (int)(rem % sw) - ring; dz = sl ? ring : -ring;
                            } else {
                                long long e2 = e - 2 * slab;
                                int layer = (int)(e2 / per), pi = (int)(e2 % per);
                                dz = -ring + 1 + layer;
                                int side = pi / (int)(sw - 1), t = pi % (int)(sw - 1);
                                if (side == 0) { dx = -ring + t; dy = -ring; }
                                else if (side == 1) { dx = ring; dy = -ring + t; }
                                else if (side == 2) { dx = ring - t; dy = ring; }
                                else { dx = -ring; dy = ring - t; }
                            }
                            r = kp_cell_range(g, cx + dx, cy + dy, cz + dz);
                        }
                        kq_scan_ranges(g, r.x, r.y, s, p.mode);
                    }
                }
            }
        }
        if (p.mode == KQ_MODE_RADIUS) {
            if (lane == 0) p.rcount[row] = s.rcount;
        } else {
            kq_truncate(s);   // the one exact sort: ascending (d2, index), cut to k
            if (lane == 0) kq_finalize(p, row, qnan ? 0 : s.n_buf, s.bd, s.bi, 1);
        }
        __syncwarp();
    }
}
__global__ void __launch_bounds__(KQ_WARPS * 32) k_knn(const __grid_constant__ KnnParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    knn_warp_body(p, smem_raw);
}
__global__ void __launch_bounds__(KQ_WARPS * 32) k_knn_b(const KnnParams *pp)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const KnnParams p = knn_params_batched(pp);      // thread-local copy: the loops read registers, not shared memory
    knn_warp_body(p, smem_raw);
}

// ---- histogram-select kernels (the fast path: k <= HQ_KMAX, the cloud queries itself).
// Selection never maintains a running top-k.  Pass 1 histograms the fp32 squared distances of the 27-cell
// block over [0, R^2) (R = the radius the block certifies); the first bin b whose cumulative count
// reaches k bounds the k-th distance.  Pass 2 re-walks the block (L1-resident) and collects the
// candidates of bins <= b -- k plus a handful -- counting-sorted by bin through the histogram's prefix
// sums.  Only those are evaluated in double: sorted, checked to be strictly ascending in the canonical
// (d2, index) order, and certified against the lower edge of the uncollected bins.  fp32 is used for
// binning only: a bin index is a monotone function of the fp32 distance, whose relative error (< 6e-7)
// is covered by the 1e-6 margins of the certificate, so the result is the exact double-precision answer
// or the query is handed to the next level (flag), never an approximation.
#ifndef HQ_ROLL
#define HQ_ROLL 1
#endif
constexpr int HQ_THREADS = 128;
constexpr int HQ_KMAX = 64;
constexpr float HQ_MAGIC = 8388608.0f;          // 2^23: adding it leaves round(x) in the low mantissa bits
constexpr int HQ_MAGIC_BITS = 0x4B000000;

__device__ __forceinline__ int hq_bin(float d, float scale)
{
    return __float_as_int(__fmaf_rn(d, scale, HQ_MAGIC)) - HQ_MAGIC_BITS;   // round(d * scale), monotone in d
}
__device__ __forceinline__ bool hq_before(double d, int i, double e, int j) { return d < e || (d == e && i < j); }

// geometry of one query against the grid: own cell, gaps to its faces, certified radius, bin scale
struct HqGeom {
    int cx, cy, cz;
    float flo[3], fhi[3], fcs;   // fp32 lower bounds (shrunk by 1e-6) of the gaps to the own cell's faces and of
                                 // the cell edge: cells are pruned in fp32, always on the safe side
    double R2;          // binning range: min(certified radius^2, cap)
    double Rcert2;      // every point closer than sqrt(Rcert2) lies inside the (2R+1)^3-cell block
    bool cap_binding;   // the radius cap, not the block, ends the range: nothing eligible lies outside it
    float scale;
};
__device__ __forceinline__ void hq_geom(const KpGridDev &g, double qx, double qy, double qz, double r2cap, int nb,
                                        bool clamp, int R, HqGeom &o)
{
    const double shrink = 1.0 - 1.0 / 1048576.0;
    o.cx = kp_cell_coord(g, qx, 0); o.cy = kp_cell_coord(g, qy, 1); o.cz = kp_cell_coord(g, qz, 2);
    if (clamp) {
        o.cx = min(max(o.cx, 0), g.dim[0] - 1); o.cy = min(max(o.cy, 0), g.dim[1] - 1); o.cz = min(max(o.cz, 0), g.dim[2] - 1);
    }
    const double qq[3] = {qx, qy, qz};
    const int cc[3] = {o.cx, o.cy, o.cz};
    double mg = INFINITY;
    const double cs = g.cell * shrink;
    o.fcs = (float)(cs * (1.0 - 1e-6));
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        double f = (qq[c] - g.org[c]) * g.inv_cell - (double)cc[c];
        f = fmin(fmax(f, 0.0), 1.0);
        const double lo = f * cs, hi = (1.0 - f) * cs;
        o.flo[c] = (float)(lo * (1.0 - 1e-6)); o.fhi[c] = (float)(hi * (1.0 - 1e-6));
        mg = fmin(mg, fmin(lo, hi));
    }
    const double safe = (double)R * cs + mg;
    o.Rcert2 = safe * safe;
    o.R2 = o.Rcert2;
    o.cap_binding = false;
    if (r2cap > 0) {
        const double capw = r2cap * (1.0 + 2e-6);      // every candidate with d2 < r2cap has fp32 d2 < capw
        if (capw <= o.Rcert2) { o.R2 = capw; o.cap_binding = true; }
    }
    o.scale = (float)((double)(nb - 1) / o.R2);        // bins 0..nb-1 cover fp32 d2 < R2 * (nb - 0.5) / (nb - 1)
}
// fp32 lower bound of the distance from the query to the cells at offset d (in cells) along axis c
__device__ __forceinline__ float hq_gap(const HqGeom &G, int c, int d)
{
    const float g0 = d < 0 ? G.flo[c] : G.fhi[c];
    return d == 0 ? 0.0f : g0 + (float)(abs(d) - 1) * G.fcs;
}
// fp32 upper bound of a squared-distance budget, with room for the rounding of the fp32 gap arithmetic
__device__ __forceinline__ float hq_budget(double b) { return __double2float_ru(b * (1.0 + 4e-6)); }
// [start,end) of the part of the z-column (cx+dx, cy+dy) that can hold a point with d2 <= budget; (0,0) if none.
// Monotone in budget: a cell visited under a budget is visited under every larger one.
__device__ __forceinline__ int2 hq_column(const KpGridDev &g, const HqGeom &G, int dx, int dy, int R, float budget)
{
    const float gx = hq_gap(G, 0, dx), gy = hq_gap(G, 1, dy);
    const float zb = budget - (gx * gx + gy * gy);
    if (!(zb >= 0.0f)) return make_int2(0, 0);
    int zlo = G.cz, zhi = G.cz;
    for (int j = 1; j <= R; ++j) { const float gz = hq_gap(G, 2, -j); if (gz * gz <= zb) zlo = G.cz - j; else break; }
    for (int j = 1; j <= R; ++j) { const float gz = hq_gap(G, 2, j); if (gz * gz <= zb) zhi = G.cz + j; else break; }
    return kp_span_range(g, G.cx + dx, G.cy + dy, zlo, zhi);
}
// columns of the block: the 9 inner ones first, then the ring at Chebyshev distance 2
__constant__ signed char HQ_COLS[25][2] = {
    {0, 0}, {-1, 0}, {1, 0}, {0, -1}, {0, 1}, {-1, -1}, {1, -1}, {-1, 1}, {1, 1},
    {-2, 0}, {2, 0}, {0, -2}, {0, 2}, {-2, -1}, {-2, 1}, {2, -1}, {2, 1}, {-1, -2}, {1, -2}, {-1, 2}, {1, 2},
    {-2, -2}, {2, -2}, {-2, 2}, {2, 2}};
// smallest double-precision d2 a candidate outside bins 0..b can have
__device__ __forceinline__ double hq_lower_edge(int b, float scale) { return ((double)b + 0.5) / (double)scale * (1.0 - 1e-6); }

// Shared memory of a histogram-kernel CTA of T threads: per thread cap candidate entries (4-byte positions into the point
// array) and then nb 16-bit bins, each strided by T (buf[slot * T], hist[bin * T]: any slot pattern is bank-conflict
// free).  hq_smem(T, cap, 0) is where the bins start.
__host__ __device__ constexpr size_t hq_smem(int T, int cap, int nb) { return (size_t)T * ((size_t)cap * sizeof(unsigned) + (size_t)nb * sizeof(unsigned short)); }

// Orders buf[0..m) -- positions, counting-sorted by bin as collected -- by (fp32 d2, position); entries only move inside
// their bin.  An entry stores no distance: its fp32 d2 is recomputed from the point (an L1 hit, the collection pass just
// read it) exactly as the collection pass computed it.  The key of the last entry of the sorted prefix stays in registers,
// so an entry already in place costs one gather; only a shift reads the entries it passes.
template <int HQT>
__device__ __forceinline__ void hq_sort_buf(unsigned *buf, int m, const float4 *pts, const float4 &me)
{
    unsigned dl = 0u, pl = 0u;   // (d2 bits, position) of buf[i - 1], the largest of the sorted prefix
    for (int i = 0; i < m; ++i) {
        const unsigned pos = buf[i * HQT];
        const unsigned d = __float_as_uint(hq_d32(me.x, me.y, me.z, __ldg(pts + pos)));   // d2 >= 0: bits order as floats
        if (i == 0 || dl < d || (dl == d && pl < pos)) { dl = d; pl = pos; continue; }
        buf[i * HQT] = pl;
        int j = i - 2;
        while (j >= 0) {
            const unsigned o = buf[j * HQT];
            const unsigned od = __float_as_uint(hq_d32(me.x, me.y, me.z, __ldg(pts + o)));
            if (od < d || (od == d && o < pos)) break;
            buf[(j + 1) * HQT] = o;
            --j;
        }
        buf[(j + 1) * HQT] = pos;
    }
}

__device__ void kq_finish_normal(const KnnParams &p, int64_t row, int cnt, double *sm)
{
    double nr[3] = {0.0, 0.0, 1.0};
    if (cnt >= 3) {
        double inv = (double)cnt;
        for (int c = 0; c < 9; ++c) sm[c] /= inv;
        double cov[6] = {sm[3] - sm[0] * sm[0], sm[4] - sm[0] * sm[1], sm[5] - sm[0] * sm[2],
                         sm[6] - sm[1] * sm[1], sm[7] - sm[1] * sm[2], sm[8] - sm[2] * sm[2]};
        kq_smallest_eigvec(cov, nr);
        if (nr[0] == 0.0 && nr[1] == 0.0 && nr[2] == 0.0) nr[2] = 1.0;
    }
    p.normals[3 * row] = (float)nr[0]; p.normals[3 * row + 1] = (float)nr[1]; p.normals[3 * row + 2] = (float)nr[2];
}

template <int NB, int R, int HQT>
__device__ __forceinline__ void hq_query(const KnnParams &p, const KpGridDev &g, const int64_t q, unsigned char *smem_raw)
{
    const int tid = threadIdx.x;
    unsigned *buf = reinterpret_cast<unsigned *>(smem_raw) + tid;
    unsigned short *hist = reinterpret_cast<unsigned short *>(smem_raw + hq_smem(HQT, p.cap, 0)) + tid;
    const int k = p.k;
    const float4 me = __ldg(p.qpts + q);
    const int64_t row = __float_as_int(me.w);
    const double qx = (double)me.x, qy = (double)me.y, qz = (double)me.z;
    if (isnan(me.x)) {
        if (p.mode == KQ_MODE_KNN) kq_finalize(p, row, 0, nullptr, nullptr, 0);
        else { double sm[9]; kq_finish_normal(p, row, 0, sm); }
        return;
    }
    HqGeom G;
    hq_geom(g, qx, qy, qz, p.r2cap, NB, false, R, G);
#pragma unroll
    for (int j = 0; j < NB; ++j) hist[j * HQT] = 0;
    // HQ_U candidates per trip: the loads and the distance chains are independent, so one L1 round trip covers all of them
    constexpr int HQ_U = 4;   // swept: 8 is slower (columns hold 10-40 candidates; longer trips waste on the tail)
    auto count = [&](const int2 rr) {
        if (rr.x >= rr.y) return;
        // the next trip's loads are in flight while this one is binned
        float4 nx[HQ_U];
#pragma unroll
        for (int u = 0; u < HQ_U; ++u) nx[u] = __ldg(g.pts + (rr.y - rr.x > u ? rr.x + u : rr.x));
        for (int t = rr.x; t < rr.y; t += HQ_U) {
            const int m = rr.y - t;
            float4 c[HQ_U];
#pragma unroll
            for (int u = 0; u < HQ_U; ++u) c[u] = nx[u];
            if (m > HQ_U) {
#pragma unroll
                for (int u = 0; u < HQ_U; ++u) nx[u] = __ldg(g.pts + (m - HQ_U > u ? t + HQ_U + u : t + HQ_U));
            }
            int bj[HQ_U];
#pragma unroll
            for (int u = 0; u < HQ_U; ++u) bj[u] = hq_bin(hq_d32(me.x, me.y, me.z, c[u]), G.scale);
            // (shared-memory atomics were measured here: 4x slower than the plain read-modify-write)
#pragma unroll
            for (int u = 0; u < HQ_U; ++u)
                if (m > u && (unsigned)bj[u] < (unsigned)NB) hist[bj[u] * HQT]++;
        }
    };
    int b = -1, m = 0, nput = 0;
    auto collect = [&](const int2 rr) {
        for (int t = rr.x; t < rr.y; t += HQ_U) {
            const int mm = rr.y - t;
            float4 c[HQ_U];
#pragma unroll
            for (int u = 0; u < HQ_U; ++u) c[u] = __ldg(g.pts + (mm > u ? t + u : t));
            float dj[HQ_U];
#pragma unroll
            for (int u = 0; u < HQ_U; ++u) dj[u] = hq_d32(me.x, me.y, me.z, c[u]);
#pragma unroll
            for (int u = 0; u < HQ_U; ++u) {
                const int bu = hq_bin(dj[u], G.scale);
                if (mm > u && (unsigned)bu <= (unsigned)b) {
                    const int slot = hist[bu * HQT];
                    hist[bu * HQT] = (unsigned short)(slot + 1);
                    if (slot < m) buf[slot * HQT] = (unsigned)(t + u);
                    ++nput;
                }
            }
        }
    };
    // the bin that holds the k-th distance; the histogram becomes the scatter offsets of pass 2
    auto select_bin = [&]() {
        int cum = 0;
        for (int j = 0; j < NB; ++j) {
            const int c = (int)hist[j * HQT];
            hist[j * HQT] = (unsigned short)cum;
            cum += c;
            if (cum >= k) { b = j; break; }
        }
        m = cum;
    };
    // Pass 1 histograms the fp32 distances, pass 2 collects bins <= b counting-sorted by bin.  Invariant:
    // every candidate with d2 < budget has been visited by pass 1; pass 2 chooses cells by the same rule with
    // a budget that is never larger, so every collected candidate was counted.
    double budget = G.R2;
    bool bounded = false;                       // pass 1 stopped visiting cells beyond a bound found on the way
    bool all;
    if constexpr (R == 1) {
        // 27 cells = 9 columns.  The nine cell-map lookups are unrolled and requested together, ahead of the first run's
        // candidates; the two candidate loops are NOT unrolled over the columns (HQ_ROLL): nine copies of each made the
        // kernel 107 KB of SASS against a 32 KB L1.5 / 6 KB L0 instruction cache, and with every warp of an SM at a
        // different place in it a quarter of the stall samples were instruction fetches (ncu: stall_no_inst).  The ranges
        // then live in local memory (18 words per thread, L1 hits): one load per column of 10-40 candidates.
        int2 rng[9];
        float gap2[9];
        const float fb = hq_budget(budget);
#pragma unroll
        for (int ci = 0; ci < 9; ++ci) {
            constexpr int order[9] = {4, 1, 3, 5, 7, 0, 2, 6, 8};
            const int dx = order[ci] / 3 - 1, dy = order[ci] % 3 - 1;
            rng[ci] = hq_column(g, G, dx, dy, 1, fb);
            const float gx = hq_gap(G, 0, dx), gy = hq_gap(G, 1, dy);
            gap2[ci] = gx * gx + gy * gy;
        }
#if HQ_ROLL
#pragma unroll 1
#else
#pragma unroll
#endif
        for (int ci = 0; ci < 9; ++ci) count(rng[ci]);
        select_bin();
        all = b < 0;                            // fewer than k in range: the loop ran over every bin, take them all
        if (b < 0) b = NB - 1;
        if (m > p.cap || (m < k && !G.cap_binding)) { p.strag_flags[q] = 1; return; }
        const float fb2 = hq_budget(fmin(budget, ((double)b + 1.0) / (double)G.scale));
#if HQ_ROLL
#pragma unroll 1
#else
#pragma unroll
#endif
        for (int ci = 0; ci < 9; ++ci)
            if (gap2[ci] <= fb2) collect(rng[ci]);
    } else {
        // 125 cells = 25 columns.  Phase A = the 9 inner columns; its histogram bounds the k-th distance, and
        // phase B (the outer ring) only visits the cells that reach inside that bound.
        constexpr int ncols = (2 * R + 1) * (2 * R + 1);
        float fbudget = hq_budget(budget);
        for (int ci = 0; ci < ncols; ++ci) {
            if (ci == 9) {
                int cum = 0;
                for (int j = 0; j < NB; ++j) {
                    cum += hist[j * HQT];
                    if (cum >= k) { budget = fmin(budget, ((double)j + 1.0) / (double)G.scale); bounded = true; break; }
                }
                fbudget = hq_budget(budget);
            }
            count(hq_column(g, G, HQ_COLS[ci][0], HQ_COLS[ci][1], R, fbudget));
        }
        select_bin();
        all = !bounded && b < 0;
        if (b < 0) b = NB - 1;
        if (m > p.cap || (m < k && !G.cap_binding)) { p.strag_flags[q] = 1; return; }
        const float budget2 = hq_budget(fmin(budget, ((double)b + 1.0) / (double)G.scale));
        for (int ci = 0; ci < ncols; ++ci) collect(hq_column(g, G, HQ_COLS[ci][0], HQ_COLS[ci][1], R, budget2));
    }
    // (a bin count that wrapped its 16 bits also ends here: > 65535 puts can never equal m <= cap)
    if (nput != m) { p.strag_flags[q] = 1; return; }
    hq_sort_buf<HQT>(buf, m, g.pts, me);
    // ---- exact evaluation in that order; the canonical (d2, index) order must be strictly ascending
    const bool capped = p.r2cap > 0;
    const bool normals = p.mode == KQ_MODE_NORMALS;
    double pd = -1.0; int pi = -1;
    double acc = 0.0;
    double sm[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    int cnt = 0;
    bool bad = false, closed = false;
    float4 cn = m > 0 ? __ldg(g.pts + buf[0]) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = 0; i < m; ++i) {
        const float4 c = cn;
        if (i + 1 < m) cn = __ldg(g.pts + buf[(i + 1) * HQT]);     // next gather in flight during this evaluation
        const double d = kp_d2(qx, qy, qz, (double)c.x, (double)c.y, (double)c.z);
        const int id = __float_as_int(c.w);
        if (!hq_before(pd, pi, d, id)) bad = true;
        if (capped && !(d < p.r2cap)) closed = true;
        if (cnt < k && !closed) {
            pd = d; pi = id;
            if (normals) {
                const double x = (double)c.x, y = (double)c.y, z = (double)c.z;
                sm[0] += x; sm[1] += y; sm[2] += z;
                sm[3] += x * x; sm[4] += x * y; sm[5] += x * z; sm[6] += y * y; sm[7] += y * z; sm[8] += z * z;
            } else {
                if (p.idx) p.idx[row * k + cnt] = id;
                if (p.d2) p.d2[row * k + cnt] = d;
                acc = __dadd_rn(acc, sqrt(d));
            }
            ++cnt;
        } else if (closed && d < p.r2cap) bad = true;   // an eligible entry behind an ineligible one: order is off
    }
    // exact iff no candidate outside the collected set can precede the k-th entry: the visited-but-uncollected
    // ones lie above the lower edge of bin b+1, the unvisited ones at or above `budget` (>= that edge)
    bool exact;
    if (all && G.cap_binding) exact = true;
    else exact = cnt == k && pd < hq_lower_edge(b, G.scale) && (G.cap_binding || pd < G.Rcert2);
    if (bad || !exact) { p.strag_flags[q] = 1; return; }
    if (normals) { kq_finish_normal(p, row, cnt, sm); return; }
    if (p.idx) for (int t = cnt; t < k; ++t) p.idx[row * k + t] = -1;
    if (p.d2) for (int t = cnt; t < k; ++t) p.d2[row * k + t] = INFINITY;
    if (p.count) p.count[row] = cnt;
    if (p.mean) p.mean[row] = cnt > 0 ? __ddiv_rn(acc, (double)cnt) : -1.0;
}
template <int NB, int R, int HQT>
__global__ void __launch_bounds__(HQT) k_knn_hist(const __grid_constant__ KnnParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int64_t w = (int64_t)blockIdx.x * HQT + threadIdx.x;
    if (w >= p.nq) return;
    hq_query<NB, R, HQT>(p, p.g, w, smem_raw);
}
// batched form: the parameter blocks of up to KNN_ARG_SEGS segments travel BY VALUE (constant bank: the hot loops read
// k, cap, the pointers ... as instruction operands, as in the single-cloud kernel); only the grid layout and the query
// count, which an earlier kernel of the frame produced, are loaded from device memory into registers
constexpr int KNN_ARG_SEGS = 8;
struct KnnBatchArgs { KnnParams p[KNN_ARG_SEGS]; };
#ifndef KNN_MIN_CTAS_T
#define KNN_MIN_CTAS_T 0
#endif
template <int NB, int R, int HQT>
__device__ __forceinline__ void knn_hist_b_body(const KnnBatchArgs &a, unsigned char *smem_raw)
{
    const KnnParams &p = a.p[blockIdx.y];
    const KpGridDev g = *p.gdev;
    // level 0: every point of the cloud; coarser levels: the positions the level before could not certify (qlist)
    const int64_t nq = p.qlist ? (int64_t)*p.qcount : (int64_t)*p.nq_dev;
    for (int64_t w = (int64_t)blockIdx.x * HQT + threadIdx.x; w < nq; w += (int64_t)gridDim.x * HQT)
        hq_query<NB, R, HQT>(p, g, p.qlist ? (int64_t)p.qlist[w] : w, smem_raw);
}
template <int NB, int R, int HQT>
__global__ void __launch_bounds__(HQT, KNN_MIN_CTAS_T > 0 ? KNN_MIN_CTAS_T / HQT : 1) k_knn_hist_b(const __grid_constant__ KnnBatchArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    knn_hist_b_body<NB, R, HQT>(a, smem_raw);
}
// the mid level (leftover list on the 1.5 x grid): the same code under its own name, so that launch lists and profiles
// tell the two levels apart
__global__ void __launch_bounds__(64) k_knn_mid_b(const __grid_constant__ KnnBatchArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    knn_hist_b_body<64, 1, 64>(a, smem_raw);
}

// ---- the same histogram select over the voxel-brick index (kp_vbi.cuh) of a voxel-downsampled cloud.
// The candidates of a query are the occupied voxels inside the voxel box of the ball of radius rho around it:
// per brick one 16-byte load and an AND with the box mask; there are no cell runs to look up and a voxel holds one
// point, so a query reads about a third of the points the 27-cell block of the grid kernel holds.  Two radii: rho_a
// certifies the dense parts of the cloud, rho_b (a wider box, restarted from scratch) the sparse ones; what neither
// certifies goes to level 1 like the grid kernel's leftovers.  Selection, exact evaluation in double and the
// certificate are those of hq_query.
template <int NB, int HQT>
__device__ __forceinline__ void vq_query(const KnnParams &p, const KpVbiDev &v, const int64_t q, unsigned char *smem_raw)
{
    const int tid = threadIdx.x;
    unsigned *buf = reinterpret_cast<unsigned *>(smem_raw) + tid;
    unsigned short *hist = reinterpret_cast<unsigned short *>(smem_raw + hq_smem(HQT, p.cap, 0)) + tid;
    const int k = p.k;
    const float4 me = __ldg(v.pts + q);
    const int64_t row = __float_as_int(me.w);
    const double qx = (double)me.x, qy = (double)me.y, qz = (double)me.z;
    const bool capped = p.r2cap > 0;
    const bool normals = p.mode == KQ_MODE_NORMALS;
    for (int phase = 0; phase < 2; ++phase) {
        const double rho = phase == 0 ? p.rho_a : p.rho_b;
        double R2 = rho * rho;
        bool cap_binding = false;
        if (capped) {
            const double capw = p.r2cap * (1.0 + 2e-6);          // every candidate with d2 < r2cap has fp32 d2 < capw
            if (capw <= R2) { R2 = capw; cap_binding = true; }
        }
        // voxel box of the ball: every point with d2 <= R2 sits in a voxel of it (eps: float32 rounding of the stored means)
        const double rad = sqrt(R2) * (1.0 + 1e-6) + v.eps + v.voxel * 1e-6;
        KpVbiBox box;
        kp_vbi_box(v, qx, qy, qz, rad, box);
        const float scale = (float)((double)(NB - 1) / R2);
#pragma unroll
        for (int j = 0; j < NB; ++j) hist[j * HQT] = 0;
        kp_vbi_visit(v, box, [&](int, const float4 &c) {
            const int bj = hq_bin(hq_d32(me.x, me.y, me.z, c), scale);
            if ((unsigned)bj < (unsigned)NB) hist[bj * HQT]++;
        });
        int b = -1, m = 0;
        {
            int cum = 0;
            for (int j = 0; j < NB; ++j) {
                const int c = (int)hist[j * HQT];
                hist[j * HQT] = (unsigned short)cum;
                cum += c;
                if (cum >= k) { b = j; break; }
            }
            m = cum;
        }
        const bool all = b < 0;                       // fewer than k in range: the loop ran over every bin, take them all
        if (b < 0) b = NB - 1;
        if (m > p.cap) { p.strag_flags[q] = 1; return; }
        if (m < k && !cap_binding) {
            if (phase == 0) continue;
            p.strag_flags[q] = 1;
            return;
        }
        int nput = 0;
        // the collection pass only needs the box of the bins it takes (bins <= b end at fp32 d2 (b + 0.5) / scale)
        kp_vbi_box(v, qx, qy, qz, sqrt(fmin(R2, ((double)b + 1.0) / (double)scale)) * (1.0 + 1e-5) + v.eps + v.voxel * 1e-6, box);
        kp_vbi_visit(v, box, [&](int pos, const float4 &c) {
            const float dj = hq_d32(me.x, me.y, me.z, c);
            const int bu = hq_bin(dj, scale);
            if ((unsigned)bu <= (unsigned)b) {
                const int slot = hist[bu * HQT];
                hist[bu * HQT] = (unsigned short)(slot + 1);
                if (slot < m) buf[slot * HQT] = (unsigned)pos;
                ++nput;
            }
        });
        if (nput != m) { p.strag_flags[q] = 1; return; }
        hq_sort_buf<HQT>(buf, m, v.pts, me);
        // ---- exact evaluation in that order; the canonical (d2, index) order must be strictly ascending
        double pd = -1.0; int pi = -1;
        double acc = 0.0;
        double sm[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        int cnt = 0;
        bool bad = false, closed = false;
        float4 cn = m > 0 ? __ldg(v.pts + buf[0]) : make_float4(0.f, 0.f, 0.f, 0.f);
        for (int i = 0; i < m; ++i) {
            const float4 c = cn;
            if (i + 1 < m) cn = __ldg(v.pts + buf[(i + 1) * HQT]);
            const double d = kp_d2(qx, qy, qz, (double)c.x, (double)c.y, (double)c.z);
            const int id = __float_as_int(c.w);
            if (!hq_before(pd, pi, d, id)) bad = true;
            if (capped && !(d < p.r2cap)) closed = true;
            if (cnt < k && !closed) {
                pd = d; pi = id;
                if (normals) {
                    const double x = (double)c.x, y = (double)c.y, z = (double)c.z;
                    sm[0] += x; sm[1] += y; sm[2] += z;
                    sm[3] += x * x; sm[4] += x * y; sm[5] += x * z; sm[6] += y * y; sm[7] += y * z; sm[8] += z * z;
                } else {
                    acc = __dadd_rn(acc, sqrt(d));
                }
                ++cnt;
            } else if (closed && d < p.r2cap) bad = true;
        }
        // exact iff nothing outside the collected set can precede the k-th entry: the visited-but-uncollected candidates
        // lie above the lower edge of bin b+1, the unvisited ones (and the fp32-out-of-range ones) at or beyond the radius
        bool exact;
        if (all && cap_binding) exact = true;
        else exact = cnt == k && pd < hq_lower_edge(b, scale) && (cap_binding || pd < R2 * (1.0 - 4e-6));
        if (bad) { p.strag_flags[q] = 1; return; }
        if (!exact) {
            if (phase == 0 && !cap_binding) continue;
            p.strag_flags[q] = 1;
            return;
        }
        if (normals) { kq_finish_normal(p, row, cnt, sm); return; }
        if (p.mean) p.mean[row] = cnt > 0 ? __ddiv_rn(acc, (double)cnt) : -1.0;
        return;
    }
}
template <int NB, int HQT>
__global__ void __launch_bounds__(HQT, 512 / HQT) k_knn_vbi_b(const KnnParams *pp)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const KnnParams p = knn_params_batched(pp);
    if (!p.vbi) return;
    const KpVbiDev v = *p.vbi;
    if (!v.ok) return;
    for (int64_t w = (int64_t)blockIdx.x * HQT + threadIdx.x; w < v.npts; w += (int64_t)gridDim.x * HQT) vq_query<NB, HQT>(p, v, w, smem_raw);
}

// ---- warp-per-query best-first histogram select: the level-0 stragglers (isolated points and sparse fringes
// -- what SOR is looking for) against a coarser grid.  Their k-th neighbour can be a metre away, so the block
// to search is found, not assumed:
//   (1) grow a cube of cells around the query, COUNTING points through column lookups only (no point is
//       read), until it holds k of them;
//   (2) histogram the fp32 distances of that cube's points: the bin where the count reaches k is a tight
//       upper bound U on the k-th distance (those are real points);
//   (3) histogram every cell that reaches inside the ball of radius U (columns and z-spans pruned by their
//       distance to the query), find the bin b of the k-th distance, and (4) collect bins <= b.
// The few survivors are sorted once and evaluated exactly in double, as in the thread kernel.  A warp
// streams candidate runs with coalesced 16-byte loads, four in flight per lane; bins are shared-memory
// atomics over 512 bins (few collisions at this fan-out).
constexpr int WH_WARPS = 4;
constexpr int WH_NB = 512;
constexpr int WH_CAP = 128;
constexpr int WH_RMAX = 7;            // cube radius (cells) of step 1; the ball search then needs at most 15

__device__ __forceinline__ void wh_sort(unsigned long long *a, int n2, int lane)
{
    for (int size = 2; size <= n2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = lane; t < (n2 >> 1); t += 32) {
                const int i = ((t / stride) * 2 * stride) + (t % stride), j = i + stride;
                const bool up = (i & size) == 0;
                const unsigned long long x = a[i], y = a[j];
                if ((y < x) == up) { a[i] = y; a[j] = x; }
            }
            __syncwarp();
        }
}

// [start,end) of the part of column (dx, dy) of the cube of radius R that can hold a point with d2 <= budget
// (fp32, conservative, monotone in budget); R <= 15 so that a z-span fits two cell-map words
__device__ __forceinline__ int2 wh_column(const KpGridDev &g, const HqGeom &G, int dx, int dy, int R, float budget)
{
    const float gx = hq_gap(G, 0, dx), gy = hq_gap(G, 1, dy);
    const float zb = budget - (gx * gx + gy * gy);
    if (!(zb >= 0.0f)) return make_int2(0, 0);
    const float reach = sqrtf(zb) * 1.000001f, fR = (float)R;
    const int jlo = reach >= G.flo[2] ? (int)fminf((reach - G.flo[2]) / G.fcs + 1.0f, fR) : 0;
    const int jhi = reach >= G.fhi[2] ? (int)fminf((reach - G.fhi[2]) / G.fcs + 1.0f, fR) : 0;
    return kp_span_range(g, G.cx + dx, G.cy + dy, G.cz - jlo, G.cz + jhi);
}

// visits every candidate of the cube of radius R within `budget` of the query: fn(valid, position, point), warp-uniform
template <class F>
__device__ __forceinline__ void wh_visit(const KpGridDev &g, const HqGeom &G, int R, float budget, int lane, F &&fn)
{
    const int side = 2 * R + 1, ncol = side * side;
    for (int c0 = 0; c0 < ncol; c0 += 32) {
        const int c = c0 + lane;
        int2 rr = make_int2(0, 0);
        if (c < ncol) rr = wh_column(g, G, c / side - R, c % side - R, R, budget);
        for (unsigned mrow = __ballot_sync(KP_FULL, rr.y > rr.x); mrow;) {
            const int j = __ffs(mrow) - 1;
            mrow &= mrow - 1;
            const int ra = __shfl_sync(KP_FULL, rr.x, j), rb = __shfl_sync(KP_FULL, rr.y, j);
            for (int t = ra + lane; t - lane < rb; t += 128) {
                const float4 c0p = __ldg(g.pts + min(t, rb - 1));
                const float4 c1p = __ldg(g.pts + min(t + 32, rb - 1));
                const float4 c2p = __ldg(g.pts + min(t + 64, rb - 1));
                const float4 c3p = __ldg(g.pts + min(t + 96, rb - 1));
                fn(t < rb, t, c0p);
                if (t - lane + 32 < rb) fn(t + 32 < rb, t + 32, c1p);
                if (t - lane + 64 < rb) fn(t + 64 < rb, t + 64, c2p);
                if (t - lane + 96 < rb) fn(t + 96 < rb, t + 96, c3p);
            }
        }
    }
}

// bin in which the running count of hist reaches k (each lane owns WH_NB / 32 consecutive bins); -1 if never.
// cum = count up to and including that bin (or the total)
__device__ __forceinline__ int wh_select(const unsigned int *hist, int k, int lane, int &cum)
{
    constexpr int PER = WH_NB / 32;
    int s = 0;
    for (int j = 0; j < PER; ++j) s += (int)hist[lane * PER + j];
    int inc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(KP_FULL, inc, o); if (lane >= o) inc += v; }
    const int tot = __shfl_sync(KP_FULL, inc, 31);
    const unsigned reach = __ballot_sync(KP_FULL, inc >= k);
    int bb = -1, mm = tot;
    if (reach) {
        const int L = __ffs(reach) - 1;
        if (lane == L) {
            int c = inc - s;
            for (int j = 0; j < PER; ++j) { c += (int)hist[lane * PER + j]; if (c >= k) { bb = lane * PER + j; mm = c; break; } }
        }
        bb = __shfl_sync(KP_FULL, bb, L); mm = __shfl_sync(KP_FULL, mm, L);
    }
    cum = mm;
    return bb;
}

__device__ __forceinline__ void knn_wbf_body(const KnnParams &p)
{
    __shared__ unsigned int s_hist[WH_WARPS][WH_NB];
    __shared__ unsigned long long s_buf[WH_WARPS][WH_CAP];
    __shared__ double s_dd[WH_WARPS][WH_CAP];
    __shared__ int s_ii[WH_WARPS][WH_CAP];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const KpGridDev &g = p.g;
    unsigned int *hist = s_hist[warp];
    unsigned long long *buf = s_buf[warp];
    double *dd = s_dd[warp];
    int *ii = s_ii[warp];
    const int k = p.k;
    const int64_t nq = (int64_t)*p.qcount;
    const unsigned lt = (1u << lane) - 1u;
    for (int64_t w = (int64_t)blockIdx.x * WH_WARPS + warp; w < nq; w += (int64_t)gridDim.x * WH_WARPS) {
        const int64_t q = (int64_t)p.qlist[w];
        const float4 me = __ldg(p.qpts + q);
        const int64_t row = __float_as_int(me.w);
        const double qx = (double)me.x, qy = (double)me.y, qz = (double)me.z;
        HqGeom G;
        hq_geom(g, qx, qy, qz, 0.0, WH_NB, true, 1, G);
        const double cs = g.cell * (1.0 - 1.0 / 1048576.0);
        const double capw = p.r2cap > 0 ? p.r2cap * (1.0 + 2e-6) : INFINITY;   // fp32 d2 of every eligible candidate is below
        bool fail = false;
        // ---- (1) smallest cube with k points (or the cube that covers the whole radius cap)
        int r = 0;
        bool cap_binding = false;        // the cube covers the cap ball: nothing eligible lies outside it
        for (;;) {
            ++r;
            if (r > WH_RMAX) { fail = true; if (p.dbg && lane == 0) atomicAdd(p.dbg + 0, 1); break; }
            const int side = 2 * r + 1, ncol = side * side;
            int cntc = 0;
            for (int c0 = 0; c0 < ncol; c0 += 32) {
                const int c = c0 + lane;
                if (c < ncol) {
                    const int2 rr = kp_span_range(g, G.cx + c / side - r, G.cy + c % side - r, G.cz - r, G.cz + r);
                    cntc += rr.y - rr.x;
                }
            }
            cntc = kq_warp_sum(cntc);
            const double inside = (double)r * cs;            // every point closer than this lies in the cube
            if (p.r2cap > 0 && inside * inside >= capw) { cap_binding = true; break; }
            if (cntc >= k) break;
        }
        int n = 0, bsel = -1, m = 0;
        double U2 = 0.0;
        float scale = 0.0f;
        bool all = false;
        if (!fail) {
            // ---- (2) k-th smallest distance among the cube's points -> upper bound U2 on the k-th distance^2
            const double far = (double)(r + 1) * g.cell;      // no point of the cube is farther than sqrt(3) * far
            double range = fmin(3.0 * far * far, capw);
            scale = (float)((double)(WH_NB - 1) / range);
            for (int j = lane; j < WH_NB; j += 32) hist[j] = 0;
            __syncwarp();
            wh_visit(g, G, r, INFINITY, lane, [&](bool v, int, const float4 &c) {
                const int bj = hq_bin(hq_d32(me.x, me.y, me.z, c), scale);
                if (v && (unsigned)bj < (unsigned)WH_NB) atomicAdd(hist + bj, 1u);
            });
            __syncwarp();
            int cum;
            const int b1 = wh_select(hist, k, lane, cum);
            if (b1 >= 0) U2 = fmin(((double)b1 + 1.0) / (double)scale, capw);
            else if (cap_binding) U2 = capw;                  // fewer than k inside the cap: all of them are wanted
            // no bound: the cube holds k points but, with a radius cap, fewer than k of them lie inside it while the cube does
            // not cover the cap ball (without a cap the cube's k points are all within range, and this cannot happen)
            else { fail = true; if (p.dbg && lane == 0) atomicAdd(p.dbg + 1, 1); }
            cap_binding = p.r2cap > 0 && U2 >= capw;          // step 3 visits the whole cap ball: nothing eligible is missed
        }
        // ---- (3) + (4), retried once with shifted bin edges when the k-th distance sits within rounding of an
        // edge (the certificate then cannot tell collected from uncollected; ~1e-3 of the queries)
        bool done = false;
        for (int attempt = 0; attempt < 2 && !fail && !done; ++attempt) {
            // (3) histogram of everything within U2; the ball needs cells up to R2 away
            int R2 = (int)ceil(sqrt(U2) / cs);
            if (R2 < 1) R2 = 1;
            if (R2 > 15) { fail = true; if (p.dbg && lane == 0) atomicAdd(p.dbg + 2, 1); break; }   // z-span would not fit the two-word cell-map lookup
            const float budget = hq_budget(U2);
            scale = (float)((double)(WH_NB - 1) / U2 * (attempt ? 0.9371 : 1.0));
            n = 0;
            __syncwarp();
            for (int j = lane; j < WH_NB; j += 32) hist[j] = 0;
            __syncwarp();
            wh_visit(g, G, R2, budget, lane, [&](bool v, int, const float4 &c) {
                const int bj = hq_bin(hq_d32(me.x, me.y, me.z, c), scale);
                if (v && (unsigned)bj < (unsigned)WH_NB) atomicAdd(hist + bj, 1u);
            });
            __syncwarp();
            bsel = wh_select(hist, k, lane, m);
            all = bsel < 0;                                // fewer than k in range: take them all
            if (bsel < 0) bsel = WH_NB - 1;
            if (m > WH_CAP || (all && !cap_binding)) {
                fail = true;
                if (p.dbg && lane == 0) atomicAdd(p.dbg + (m > WH_CAP ? 3 : 4), 1);
                break;
            }
            // (4) collect bins <= bsel (cells chosen by the same rule under a budget that is not larger)
            const float budget3 = hq_budget(fmin(U2, ((double)bsel + 1.0) / (double)scale));
            wh_visit(g, G, R2, budget3, lane, [&](bool v, int t, const float4 &c) {
                const float d = hq_d32(me.x, me.y, me.z, c);
                const bool pass = v && (unsigned)hq_bin(d, scale) <= (unsigned)bsel;
                const unsigned pm = __ballot_sync(KP_FULL, pass);
                const int pos = n + __popc(pm & lt);
                if (pass && pos < WH_CAP) buf[pos] = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)t;
                n += __popc(pm);
            });
            if (n != m) { fail = true; if (p.dbg && lane == 0) atomicAdd(p.dbg + 5, 1); break; }   // cannot happen; never trust a scatter blindly
            // ---- exact evaluation of the survivors and ONE exact sort by the canonical (d2, index) order.  (At these
            // distances fp32 squared distances collide -- two of ~100 candidates share a float in a few percent of
            // the queries -- so the fp32 order is only used to choose the set, never to order it.)
            int n2 = 32;
            while (n2 < n) n2 <<= 1;
            __syncwarp();
            for (int t = lane; t < n2; t += 32) {
                if (t < n) {
                    const float4 c = __ldg(g.pts + (unsigned)buf[t]);
                    dd[t] = kp_d2(qx, qy, qz, (double)c.x, (double)c.y, (double)c.z);
                    ii[t] = __float_as_int(c.w);
                } else { dd[t] = INFINITY; ii[t] = 0x7fffffff; }
            }
            __syncwarp();
            kq_sort(dd, ii, n2, lane);
            int within = 0;
            for (int t = lane; t < n; t += 32)
                if (t < k && (p.r2cap <= 0 || dd[t] < p.r2cap)) ++within;
            const int cnt = kq_warp_sum(within);    // sorted ascending: the eligible entries are a prefix
            bool exact;
            if (all && cap_binding) exact = true;
            else exact = cnt == k && dd[k - 1] < hq_lower_edge(bsel, scale) && dd[k - 1] < U2;
            if (exact) {
                done = true;
                if (lane == 0) kq_finalize(p, row, cnt, dd, ii, 1);
            } else if (attempt == 1 || cnt != k) {
                fail = true;
                if (p.dbg && lane == 0) atomicAdd(p.dbg + 7, 1);
            }
            __syncwarp();
        }
        if (fail && lane == 0) p.strag_flags[q] = 1;
        __syncwarp();
    }
}
__global__ void __launch_bounds__(WH_WARPS * 32) k_knn_wbf(const __grid_constant__ KnnParams p) { knn_wbf_body(p); }
__global__ void __launch_bounds__(WH_WARPS * 32) k_knn_wbf_b(const KnnParams *pp)
{
    const KnnParams p = knn_params_batched(pp);
    knn_wbf_body(p);
}

int next_pow2(int v)
{
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

int knn_launch_warp(kp_ctx *ctx, KnnParams &p, int64_t grid_queries)
{
    p.cap = next_pow2(4 * p.k > 128 ? 4 * p.k : 128);
    if ((size_t)KQ_WARPS * p.cap * 12 > 96 * 1024) p.cap = next_pow2(p.k + 64 > 128 ? p.k + 64 : 128);
    size_t smem = (size_t)KQ_WARPS * p.cap * (sizeof(double) + sizeof(int));
    if (smem > 200 * 1024) return kp_set_err(ctx, KP_E_ARG, "k = %d neighbours is too many for the per-warp buffer", p.k);
    if (smem > 48 * 1024) KP_CUDA(ctx, cudaFuncSetAttribute(k_knn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t blocks = (grid_queries + KQ_WARPS - 1) / KQ_WARPS;
    int64_t cap_blocks = (int64_t)ctx->sm_count * 32;
    if (p.qlist && blocks > cap_blocks) blocks = cap_blocks;     // persistent loop over the straggler list
    if (blocks < 1) blocks = 1;
    k_knn<<<(unsigned)blocks, KQ_WARPS * 32, smem, ctx->stream>>>(p);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}

template <int NB, int R>
int knn_launch_hist(kp_ctx *ctx, KnnParams &p)
{
    // the per-thread buffer (k + slack entries) is what limits occupancy for large k: smaller CTAs pack the 227 KB of an
    // SM more tightly
    constexpr int T = NB <= 32 ? 128 : 64;
    static const int slack = getenv("KP_KNN_SLACK") ? atoi(getenv("KP_KNN_SLACK")) : 8;   // swept: 6 / 8 / 12
    p.cap = p.k + slack;
    const size_t smem = hq_smem(T, p.cap, NB);
    if (smem > 48 * 1024) KP_CUDA(ctx, cudaFuncSetAttribute(k_knn_hist<NB, R, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_knn_hist<NB, R, T><<<kp_blocks(p.nq, T), T, smem, ctx->stream>>>(p);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}

// compacts flags[0..n) (in query order) into list, returns the count on the host (one stream sync)
int knn_flag_list(kp_ctx *ctx, int64_t n, const uint8_t *flags, int32_t *list, int32_t *d_count, int32_t *h_count)
{
    KP_TRY(kp_prim_compact_mask(ctx, n, flags, 0, nullptr, nullptr, list, d_count));
    KP_CUDA(ctx, cudaMemcpyAsync(ctx->d_scratch, d_count, sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
    KP_TRY(kp_fetch_scratch(ctx, sizeof(int32_t)));
    *h_count = *(int32_t *)ctx->h_scratch;
    return KP_OK;
}

// d_xyz: the cloud the grid was built from (needed to build the coarser level; may be NULL)
int knn_launch(kp_ctx *ctx, KnnParams &p, const char *name, const float *d_xyz = nullptr)
{
    if (p.nq <= 0) return KP_OK;
    // compulsory HBM traffic: the cell-sorted float4 array once + the per-query outputs
    double out_b = p.mode == KQ_MODE_RADIUS ? 4.0 : p.mode == KQ_MODE_NORMALS ? 12.0 + 12.0
                   : (p.idx ? 4.0 * p.k : 0.0) + (p.d2 ? 8.0 * p.k : 0.0) + (p.count ? 4.0 : 0.0) + (p.mean ? 8.0 : 0.0);
    KP_PROFB(ctx, name, (double)p.g.npts * 16.0 + (double)p.nq * (out_b + (p.queries ? 12.0 : 0.0)));
    p.qlist = nullptr; p.qcount = nullptr; p.strag_flags = nullptr; p.dbg = nullptr;
    p.gdev = nullptr; p.nq_dev = nullptr;
    p.qpts = p.g.pts;
    const bool fast = !p.queries && p.mode != KQ_MODE_RADIUS && p.k <= HQ_KMAX;
    if (!fast) return knn_launch_warp(ctx, p, p.nq);
    const KpGridDev g0 = p.g;
    const int64_t nq0 = p.nq;
    int32_t *listA, *listB, *counts;
    uint8_t *flags;
    KP_TRY(kp_ws(ctx, (size_t)nq0, &listA));
    KP_TRY(kp_ws(ctx, (size_t)nq0, &flags));
    KP_TRY(kp_ws(ctx, 8, &counts));
    KP_CUDA(ctx, cudaMemsetAsync(counts, 0, 8 * sizeof(int32_t), ctx->stream));
    KP_CUDA(ctx, cudaMemsetAsync(flags, 0, (size_t)nq0, ctx->stream));
    // level 0: every query, one thread each, against the caller's grid
    p.strag_flags = flags;
    {
        KP_PROFB(ctx, "knn_level0", (double)p.g.npts * 16.0 + (double)p.nq * out_b);
        if (p.rad == 2) {
            if (p.k <= 32) KP_TRY((knn_launch_hist<32, 2>(ctx, p)));
            else KP_TRY((knn_launch_hist<64, 2>(ctx, p)));
        } else {
            if (p.k <= 32) KP_TRY((knn_launch_hist<32, 1>(ctx, p)));
            else KP_TRY((knn_launch_hist<64, 1>(ctx, p)));
        }
    }
    // A radius-capped search on a grid whose cell covers the radius is always certified unless the exact
    // order is ambiguous in fp32 (ties); the flags still have to be looked at.
    // Queries the 27-cell block could not certify: flying pixels and other isolated points (exactly what SOR is
    // looking for) plus the sparsest fringes of the cloud.  Their k-th neighbour can be many cells away, so
    // level 1 repeats the selection on a COARSER grid with one warp per query; what even that block cannot
    // certify goes to the ring-expanding kernel.  Lists are compacted in query order.
    const double coarse_mult = getenv("KP_KNN_COARSE_MULT") ? atof(getenv("KP_KNN_COARSE_MULT")) : 3.0;
    int32_t n_strag = 0;
    KP_TRY(knn_flag_list(ctx, nq0, flags, listA, counts, &n_strag));
    if (getenv("KP_DEBUG_KNN"))
        fprintf(stderr, "[kp knn] %s k=%d n=%lld cell=%g level-0 uncertified=%d\n", name, p.k, (long long)nq0, g0.cell, n_strag);
    if (n_strag <= 0) return KP_OK;
    p.qpts = g0.pts;
    p.qlist = listA;
    p.qcount = counts;
    p.nq = nq0;
    if (d_xyz && coarse_mult > 1.0) {
        float b6[6];
        for (int c = 0; c < 3; ++c) {
            b6[c] = (float)g0.org[c];
            b6[3 + c] = (float)(g0.org[c] + g0.cell * (double)g0.dim[c]);
        }
        KpGrid gl;
        KP_TRY(kp_grid_build(ctx, d_xyz, g0.npts, g0.cell * (double)p.rad * coarse_mult, b6, &gl));
        p.g = kp_grid_dev(gl);
        KP_TRY(kp_ws(ctx, (size_t)n_strag, &listB));
        KP_CUDA(ctx, cudaMemsetAsync(flags, 0, (size_t)nq0, ctx->stream));
        if (getenv("KP_DEBUG_KNN")) {
            KP_TRY(kp_ws(ctx, 8, &p.dbg));
            KP_CUDA(ctx, cudaMemsetAsync(p.dbg, 0, 8 * sizeof(int32_t), ctx->stream));
        }
        {
            KP_PROF(ctx, "knn_level1");
            int64_t blocks = ((int64_t)n_strag + WH_WARPS - 1) / WH_WARPS;
            const int64_t cap_blocks = (int64_t)ctx->sm_count * 16;
            if (blocks > cap_blocks) blocks = cap_blocks;
            k_knn_wbf<<<(unsigned)blocks, WH_WARPS * 32, 0, ctx->stream>>>(p);
            KP_LAUNCH_CHECK(ctx);
        }
        if (p.dbg) {
            KP_CUDA(ctx, cudaMemcpyAsync(ctx->d_scratch, p.dbg, 8 * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
            KP_TRY(kp_fetch_scratch(ctx, 8 * sizeof(int32_t)));
            const int32_t *d = (const int32_t *)ctx->h_scratch;
            fprintf(stderr, "[kp knn] level-1 hand-overs: cube>%d %d, no-bound %d, ball>15 %d, bin>cap %d, short %d, scatter %d, order %d, uncertified %d\n",
                    WH_RMAX, d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);
            p.dbg = nullptr;
        }
        int32_t n2 = 0;
        KP_TRY(knn_flag_list(ctx, nq0, flags, listB, counts + 1, &n2));
        if (getenv("KP_DEBUG_KNN")) fprintf(stderr, "[kp knn] %s level-1 cell=%g uncertified=%d\n", name, gl.cell, n2);
        if (n2 <= 0) return KP_OK;
        p.qlist = listB;
        p.qcount = counts + 1;
        n_strag = n2;
    }
    {
        KP_PROF(ctx, "knn_stragglers");
        return knn_launch_warp(ctx, p, n_strag);
    }
}

// SOR statistics: the two canonical sums run on transformed views of the mean array (kp_prim_csum_mode)
__global__ void k_sor_mask(const double *mean, int64_t n, const double *sum_p, const double *sq_p, double valid, double ratio,
                           uint8_t *keep, double *stats)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double mu = __ddiv_rn(*sum_p, valid);
    double sd = sqrt(__ddiv_rn(*sq_p, __dsub_rn(valid, 1.0)));
    double thr = __dadd_rn(mu, __dmul_rn(ratio, sd));
    if (i == 0) { stats[0] = mu; stats[1] = sd; stats[2] = thr; }
    if (i < n) { double m = mean[i]; keep[i] = (m > 0 && m < thr) ? 1 : 0; }
}
__global__ void k_radius_mask(const int32_t *cnt, int64_t n, int nb, uint8_t *keep)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keep[i] = cnt[i] > nb;
}
}  // namespace

int kp_knn_device(kp_ctx *ctx, const KpGrid &g, const float *d_queries, int64_t nq, int k, double radius, int32_t *d_idx,
                  double *d_d2, int32_t *d_count, double *d_mean, const float *d_xyz)
{
    KnnParams p;
    p.g = kp_grid_dev(g); p.rad = g.rad;
    p.queries = d_queries; p.nq = d_queries ? nq : g.n; p.k = k; p.mode = KQ_MODE_KNN;
    p.r2cap = radius > 0 ? radius * radius : 0.0;
    p.idx = d_idx; p.d2 = d_d2; p.count = d_count; p.mean = d_mean;
    p.cloud = nullptr; p.normals = nullptr; p.rcount = nullptr;
    return knn_launch(ctx, p, "knn", d_xyz);
}

int kp_sor_device(kp_ctx *ctx, const float *d_xyz, int64_t n, int k, double ratio, double cell_hint,
                  const float *h_bounds6, uint8_t *d_keep, double *d_mean, double *h_stats, int64_t *h_kept)
{
    if (k < 1 || !(ratio > 0.0)) return kp_set_err(ctx, KP_E_ARG, "remove_statistical_outlier: nb_neighbors < 1 or std_ratio <= 0");
    if (h_kept) *h_kept = 0;
    if (n <= 0) return KP_OK;
    // valid = number of points that get a neighbour list (NaN rows do not; compacted clouds have none)
    float b6[6];
    int64_t nvalid = n;
    if (!h_bounds6) {
        KP_TRY(kp_prim_bounds_fetch(ctx, d_xyz, n, b6, &nvalid));
        h_bounds6 = b6;
        if (nvalid == 0) {
            KP_CUDA(ctx, cudaMemsetAsync(d_keep, 0, (size_t)n, ctx->stream));
            return KP_OK;
        }
    }
    double cell = cell_hint;
    if (!(cell > 0.0)) KP_TRY(kp_grid_auto_cell(ctx, d_xyz, n, h_bounds6, 0.5 * k > 4 ? 0.5 * k : 4, &cell));
    KpGrid g;
    KP_TRY(kp_grid_build_knn(ctx, d_xyz, n, cell, k, h_bounds6, &g));
    double *mean = d_mean, *red;
    if (!mean) KP_TRY(kp_ws(ctx, (size_t)n, &mean));
    KP_TRY(kp_ws(ctx, (size_t)n / 1024 + (size_t)n / 1048576 + 16, &red));
    {
        KnnParams p;
        p.g = kp_grid_dev(g); p.rad = g.rad;
        p.queries = nullptr; p.nq = n; p.k = k; p.mode = KQ_MODE_KNN; p.r2cap = 0.0;
        p.idx = nullptr; p.d2 = nullptr; p.count = nullptr; p.mean = mean;
        p.cloud = nullptr; p.normals = nullptr; p.rcount = nullptr;
        KP_TRY(knn_launch(ctx, p, "sor_knn", d_xyz));
    }
    KP_PROFB(ctx, "sor_stats", (double)n * (3.0 * 8.0 + 2.0));   // the mean array read by both sums and the mask pass, keep[] written and counted
    // NaN points never get a neighbour list: they count as "not computed" (mean = -1), like upstream's
    // empty-result branch; valid = number of points with a computed mean
    double *d_sum = (double *)ctx->d_scratch, *d_sq = d_sum + 2, *d_stats = d_sum + 4;
    int32_t *d_cnt = (int32_t *)(d_sum + 8);
    unsigned nb = kp_blocks(n, 256);
    KP_TRY(kp_prim_csum_mode(ctx, mean, n, red, d_sum, 1, nullptr, 1.0));                 // sum of the positive means
    KP_TRY(kp_prim_csum_mode(ctx, mean, n, red, d_sq, 2, d_sum, (double)nvalid));         // sum of (mean - mu)^2 over them
    k_sor_mask<<<nb, 256, 0, ctx->stream>>>(mean, n, d_sum, d_sq, (double)nvalid, ratio, d_keep, d_stats);
    KP_LAUNCH_CHECK(ctx);
    KP_TRY(kp_prim_count_u8(ctx, d_keep, n, d_cnt));
    KP_TRY(kp_fetch_scratch(ctx, 10 * sizeof(double)));
    const double *hs = (const double *)ctx->h_scratch;
    if (h_stats) { h_stats[0] = hs[4]; h_stats[1] = hs[5]; h_stats[2] = hs[6]; }
    if (h_kept) *h_kept = *(const int32_t *)(hs + 8);
    return KP_OK;
}

int kp_normals_device(kp_ctx *ctx, const float *d_xyz, int64_t n, double radius, int max_nn, const float *h_bounds6,
                      float *d_normals)
{
    if (max_nn < 1) return kp_set_err(ctx, KP_E_ARG, "estimate_normals: max_nn < 1");
    if (n <= 0) return KP_OK;
    double cell;
    if (radius > 0) cell = radius * (1.0 + 4e-6);
    else KP_TRY(kp_grid_auto_cell(ctx, d_xyz, n, h_bounds6, 0.5 * max_nn > 4 ? 0.5 * max_nn : 4, &cell));
    KpGrid g;
    KP_TRY(kp_grid_build_knn(ctx, d_xyz, n, cell, max_nn, h_bounds6, &g));
    KnnParams p;
    p.g = kp_grid_dev(g); p.rad = g.rad;
    p.queries = nullptr; p.nq = n; p.k = max_nn; p.mode = KQ_MODE_NORMALS;
    p.r2cap = radius > 0 ? radius * radius : 0.0;
    p.idx = nullptr; p.d2 = nullptr; p.count = nullptr; p.mean = nullptr;
    p.cloud = d_xyz; p.normals = d_normals; p.rcount = nullptr;
    return knn_launch(ctx, p, "normals");
}

// ---------------------------------------------------------------- frame engine: batched neighbour searches
// One parameter block per (level, segment) lives in device memory, written once when the engine is created
// (every pointer in it is static; grid layouts and counts are read through gdev / nq_dev / qcount at run time).
int kp_knn_batch_create(kp_ctx *ctx, const KpKnnSegDesc *segs, int nseg, int k, int mode, double radius, double rho_a, double rho_b,
                        KpKnnBatch *out)
{
    out->nseg = nseg; out->k = k; out->mode = mode;
    out->rad = (getenv("KP_KNN_RAD") && atoi(getenv("KP_KNN_RAD")) == 2) ? 2 : 1;
    static const int slack = getenv("KP_KNN_SLACK") ? atoi(getenv("KP_KNN_SLACK")) : 8;
    out->cap_hist = k + slack;
    int capw = next_pow2(4 * k > 128 ? 4 * k : 128);
    if ((size_t)KQ_WARPS * capw * 12 > 96 * 1024) capw = next_pow2(k + 64 > 128 ? k + 64 : 128);
    out->cap_warp = capw;
    if (k > HQ_KMAX) return kp_set_err(ctx, KP_E_ARG, "frame engine: k = %d neighbours exceeds the histogram kernel's %d", k, HQ_KMAX);
    std::vector<KnnParams> h((size_t)4 * nseg);
    out->has_mid = nseg > 0 && segs[0].gm != nullptr;
    out->cap_mid = k + 24;                       // the mid level's bins are wider: more room behind the k-th entry
    for (int s = 0; s < nseg; ++s) {
        const KpKnnSegDesc &d = segs[s];
        KnnParams p;
        memset(&p, 0, sizeof p);
        p.queries = nullptr; p.nq = 0; p.k = k; p.mode = mode == 1 ? KQ_MODE_NORMALS : KQ_MODE_KNN; p.rad = out->rad;
        p.r2cap = radius > 0 ? radius * radius : 0.0;
        p.mean = d.mean; p.cloud = d.cloud; p.normals = d.normals;
        p.qpts = d.pts0;
        // level 0: every point of the cloud, one thread each, against the level-0 grid
        KnnParams a = p;
        a.cap = out->cap_hist; a.gdev = d.g0; a.nq_dev = d.n; a.strag_flags = d.flags0;
        a.vbi = d.vbi; a.rho_a = rho_a; a.rho_b = rho_b;
        h[s] = a;
        // level 1: the leftovers of the level before (list0, or the mid level's list), one warp each, against the coarse grid
        KnnParams b = p;
        b.cap = out->cap_hist; b.gdev = d.g1; b.qlist = d.gm ? d.list_m : d.list0; b.qcount = d.gm ? d.cnt_m : d.cnt0; b.strag_flags = d.flags1; b.rad = 1;
        h[(size_t)nseg + s] = b;
        // mid level: the level-0 leftovers, one THREAD each, histogram select with 64 bins against a moderately coarser grid
        KnnParams m2 = p;
        m2.cap = out->cap_mid; m2.gdev = d.gm; m2.qlist = d.list0; m2.qcount = d.cnt0; m2.strag_flags = d.flags_m; m2.rad = 1;
        h[(size_t)3 * nseg + s] = m2;
        // stragglers: ring expansion on the coarse grid
        KnnParams c = p;
        c.cap = capw; c.gdev = d.g1; c.qlist = d.list1; c.qcount = d.cnt1;
        h[(size_t)2 * nseg + s] = c;
    }
    KP_CUDA(ctx, cudaMalloc(&out->d_params, sizeof(KnnParams) * h.size()));
    KP_CUDA(ctx, cudaMemcpy(out->d_params, h.data(), sizeof(KnnParams) * h.size(), cudaMemcpyHostToDevice));
    out->h_params = malloc(sizeof(KnnParams) * h.size());
    memcpy(out->h_params, h.data(), sizeof(KnnParams) * h.size());
    // shared-memory opt-ins happen here, not inside a stream capture
    const size_t smem_w = (size_t)KQ_WARPS * capw * (sizeof(double) + sizeof(int));
    if (smem_w > 200 * 1024) return kp_set_err(ctx, KP_E_ARG, "k = %d neighbours is too many for the per-warp buffer", k);
    if (smem_w > 48 * 1024) KP_CUDA(ctx, cudaFuncSetAttribute(k_knn_b, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_w));
    const size_t smem_m = hq_smem(64, out->cap_mid, 64);
    if (smem_m > 48 * 1024) KP_CUDA(ctx, cudaFuncSetAttribute(k_knn_mid_b, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_m));
    const size_t smem_h = k <= 32 ? hq_smem(128, out->cap_hist, 32) : hq_smem(64, out->cap_hist, 64);
    if (smem_h > 48 * 1024) {
        if (k <= 32) {
            KP_CUDA(ctx, cudaFuncSetAttribute(k_knn_hist_b<32, 2, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h));
            KP_CUDA(ctx, cudaFuncSetAttribute(k_knn_hist_b<32, 1, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h));
            KP_CUDA(ctx, cudaFuncSetAttribute(k_knn_vbi_b<32, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h));
        } else {
            KP_CUDA(ctx, cudaFuncSetAttribute(k_knn_hist_b<64, 2, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h));
            KP_CUDA(ctx, cudaFuncSetAttribute(k_knn_hist_b<64, 1, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h));
            KP_CUDA(ctx, cudaFuncSetAttribute(k_knn_vbi_b<64, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h));
        }
    }
    // shared memory / L1 split of the level-0 kernels (percent of the maximum shared memory; unset = the driver's choice)
    if (getenv("KP_KNN_CARVEOUT")) {
        const int pct = atoi(getenv("KP_KNN_CARVEOUT"));
        KP_CUDA(ctx, cudaFuncSetAttribute(k_knn_hist_b<32, 1, 128>, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
        KP_CUDA(ctx, cudaFuncSetAttribute(k_knn_hist_b<64, 1, 64>, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
    }
    return KP_OK;
}
void kp_knn_batch_destroy(KpKnnBatch *b)
{
    if (b && b->d_params) { cudaFree(b->d_params); b->d_params = nullptr; }
    if (b && b->h_params) { free(b->h_params); b->h_params = nullptr; }
}
template <int NB, int R, int T>
static int knn_level0_launch(kp_ctx *ctx, const KpKnnBatch &b, int64_t cap_rows, int per_sm, int level = 0)
{
    const KnnParams *hp = (const KnnParams *)b.h_params + (size_t)level * b.nseg;
    const size_t smem = hq_smem(T, level == 3 ? b.cap_mid : b.cap_hist, NB);
    int64_t gx = (cap_rows + T - 1) / T;
    if (gx > (int64_t)ctx->sm_count * per_sm) gx = (int64_t)ctx->sm_count * per_sm;
    for (int s0 = 0; s0 < b.nseg; s0 += KNN_ARG_SEGS) {
        const int ns = b.nseg - s0 < KNN_ARG_SEGS ? b.nseg - s0 : KNN_ARG_SEGS;
        KnnBatchArgs a;
        memset(&a, 0, sizeof a);
        for (int i = 0; i < ns; ++i) a.p[i] = hp[s0 + i];
        if (level == 3 && NB == 64 && R == 1 && T == 64) k_knn_mid_b<<<dim3((unsigned)(gx > 0 ? gx : 1), (unsigned)ns), T, smem, ctx->stream>>>(a);
        else k_knn_hist_b<NB, R, T><<<dim3((unsigned)(gx > 0 ? gx : 1), (unsigned)ns), T, smem, ctx->stream>>>(a);
        KP_LAUNCH_CHECK(ctx);
    }
    return KP_OK;
}
int kp_knn_batch_level0(kp_ctx *ctx, const KpKnnBatch &b, int64_t cap_rows)
{
    KP_PROFB(ctx, "knn_level0", 0.0);
    // persistent CTAs per SM and segment (KP_KNN_CTAS): fewer leave registers for another batch's kernels on the same SM
    static const int per_sm = getenv("KP_KNN_CTAS") ? atoi(getenv("KP_KNN_CTAS")) : 24;
    if (b.k <= 32) return b.rad == 2 ? knn_level0_launch<32, 2, 128>(ctx, b, cap_rows, per_sm) : knn_level0_launch<32, 1, 128>(ctx, b, cap_rows, per_sm);
    return b.rad == 2 ? knn_level0_launch<64, 2, 64>(ctx, b, cap_rows, per_sm * 4 / 3) : knn_level0_launch<64, 1, 64>(ctx, b, cap_rows, per_sm * 4 / 3);
}
int kp_knn_batch_vbi(kp_ctx *ctx, const KpKnnBatch &b, int64_t cap_rows)
{
    const KnnParams *pp = (const KnnParams *)b.d_params;
    KP_PROFB(ctx, "knn_vbi", 0.0);
    if (b.k <= 32) {
        constexpr int T = 128;
        const size_t smem = hq_smem(T, b.cap_hist, 32);
        int64_t gx = (cap_rows + T - 1) / T;
        if (gx > (int64_t)ctx->sm_count * 24) gx = (int64_t)ctx->sm_count * 24;
        k_knn_vbi_b<32, T><<<dim3((unsigned)(gx > 0 ? gx : 1), (unsigned)b.nseg), T, smem, ctx->stream>>>(pp);
    } else {
        constexpr int T = 64;
        const size_t smem = hq_smem(T, b.cap_hist, 64);
        int64_t gx = (cap_rows + T - 1) / T;
        if (gx > (int64_t)ctx->sm_count * 32) gx = (int64_t)ctx->sm_count * 32;
        k_knn_vbi_b<64, T><<<dim3((unsigned)(gx > 0 ? gx : 1), (unsigned)b.nseg), T, smem, ctx->stream>>>(pp);
    }
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}
// mid level: the level-0 leftovers (compacted list: full warps) through the thread-per-query histogram kernel, 64 bins,
// on a grid whose cell is ~1.7 x the level-0 cell.  A leftover is typically a point of a sparse part of the cloud whose
// k-th neighbour lies just outside the level-0 block; the warp-per-query level 1 costs ~20 x a level-0 query, this ~3 x.
int kp_knn_batch_mid(kp_ctx *ctx, const KpKnnBatch &b, int64_t cap_rows)
{
    KP_PROFB(ctx, "knn_mid", 0.0);
    return knn_level0_launch<64, 1, 64>(ctx, b, cap_rows / 4 + 1, 8, 3);
}
// level 1: the leftovers of the level before (compacted list), one warp each, best-first on the coarse grid
int kp_knn_batch_level1(kp_ctx *ctx, const KpKnnBatch &b, int64_t cap_rows)
{
    KP_PROFB(ctx, "knn_level1", 0.0);
    // measured: the histogram kernel on the coarse grid (KP_KNN_L1=hist) certifies only ~half of the leftovers (one bin of
    // the 9x larger range holds more candidates than the buffer) at 2.8x the time of the best-first kernel: kept as an option
    static const bool wbf = !(getenv("KP_KNN_L1") && !strcmp(getenv("KP_KNN_L1"), "hist"));
    if (wbf) {
        k_knn_wbf_b<<<dim3((unsigned)ctx->sm_count * 8, (unsigned)b.nseg), WH_WARPS * 32, 0, ctx->stream>>>((const KnnParams *)b.d_params + b.nseg);
        KP_LAUNCH_CHECK(ctx);
        return KP_OK;
    }
    // (a fraction of the cloud reaches this level: a quarter of the level-0 grid is plenty)
    if (b.k <= 32) return knn_level0_launch<32, 1, 128>(ctx, b, cap_rows / 4 + 1, 8, 1);
    return knn_level0_launch<64, 1, 64>(ctx, b, cap_rows / 4 + 1, 8, 1);
}
int kp_knn_batch_stragglers(kp_ctx *ctx, const KpKnnBatch &b)
{
    KP_PROFB(ctx, "knn_stragglers", 0.0);
    const size_t smem = (size_t)KQ_WARPS * b.cap_warp * (sizeof(double) + sizeof(int));
    k_knn_b<<<dim3((unsigned)ctx->sm_count * 4, (unsigned)b.nseg), KQ_WARPS * 32, smem, ctx->stream>>>((const KnnParams *)b.d_params + 2 * b.nseg);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}

extern "C" {

int kp_knn(kp_ctx *ctx, const float *d_xyz, int64_t n, const float *d_queries, int64_t nq, int k, double radius,
           double cell_hint, int32_t *d_idx, double *d_d2, int32_t *d_count)
{
    if (!ctx || (n > 0 && !d_xyz)) return kp_set_err(ctx, KP_E_ARG, "kp_knn: NULL argument");
    if (k < 1) return kp_set_err(ctx, KP_E_ARG, "kp_knn: k < 1");
    kp_enter(ctx);
    if (!d_queries) nq = n;
    if (nq <= 0) return KP_OK;
    double cell = cell_hint;
    if (!(cell > 0.0)) {
        if (radius > 0) cell = radius * (1.0 + 4e-6);
        else KP_TRY(kp_grid_auto_cell(ctx, d_xyz, n, nullptr, 0.5 * k > 4 ? 0.5 * k : 4, &cell));
    }
    KpGrid g;
    if (d_queries) KP_TRY(kp_grid_build(ctx, d_xyz, n, cell, nullptr, &g));
    else KP_TRY(kp_grid_build_knn(ctx, d_xyz, n, cell, k, nullptr, &g));
    return kp_knn_device(ctx, g, d_queries, nq, k, radius, d_idx, d_d2, d_count, nullptr, d_xyz);
}

int kp_sor_mask(kp_ctx *ctx, const float *d_xyz, int64_t n, int nb_neighbors, double std_ratio, double cell_hint,
                uint8_t *d_keep, double *d_mean, double *h_stats, int64_t *h_kept)
{
    if (!ctx || (n > 0 && (!d_xyz || !d_keep))) return kp_set_err(ctx, KP_E_ARG, "kp_sor_mask: NULL argument");
    kp_enter(ctx);
    return kp_sor_device(ctx, d_xyz, n, nb_neighbors, std_ratio, cell_hint, nullptr, d_keep, d_mean, h_stats, h_kept);
}

int kp_radius_mask(kp_ctx *ctx, const float *d_xyz, int64_t n, int nb_points, double radius, uint8_t *d_keep,
                   int32_t *d_counts, int64_t *h_kept)
{
    if (!ctx || (n > 0 && (!d_xyz || !d_keep))) return kp_set_err(ctx, KP_E_ARG, "kp_radius_mask: NULL argument");
    if (nb_points < 1 || !(radius > 0.0)) return kp_set_err(ctx, KP_E_ARG, "remove_radius_outlier: nb_points < 1 or radius <= 0");
    kp_enter(ctx);
    if (h_kept) *h_kept = 0;
    if (n <= 0) return KP_OK;
    KpGrid g;
    KP_TRY(kp_grid_build(ctx, d_xyz, n, radius * (1.0 + 1e-6), nullptr, &g));
    int32_t *cnt = d_counts;
    if (!cnt) KP_TRY(kp_ws(ctx, (size_t)n, &cnt));
    KnnParams p;
    p.g = kp_grid_dev(g); p.rad = 1;
    p.queries = nullptr; p.nq = n; p.k = 1; p.mode = KQ_MODE_RADIUS; p.r2cap = radius * radius;
    p.idx = nullptr; p.d2 = nullptr; p.count = nullptr; p.mean = nullptr; p.cloud = nullptr; p.normals = nullptr;
    p.rcount = cnt;
    KP_TRY(knn_launch(ctx, p, "radius_count"));
    k_radius_mask<<<kp_blocks(n, 256), 256, 0, ctx->stream>>>(cnt, n, nb_points, d_keep);
    KP_LAUNCH_CHECK(ctx);
    int32_t *d_tot = (int32_t *)ctx->d_scratch;
    KP_TRY(kp_prim_count_u8(ctx, d_keep, n, d_tot));
    KP_TRY(kp_fetch_scratch(ctx, sizeof(int32_t)));
    if (h_kept) *h_kept = *(int32_t *)ctx->h_scratch;
    return KP_OK;
}

int kp_estimate_normals(kp_ctx *ctx, const float *d_xyz, int64_t n, double radius, int max_nn, float *d_normals)
{
    if (!ctx || (n > 0 && (!d_xyz || !d_normals))) return kp_set_err(ctx, KP_E_ARG, "kp_estimate_normals: NULL argument");
    kp_enter(ctx);
    return kp_normals_device(ctx, d_xyz, n, radius, max_nn, nullptr, d_normals);
}

}  // extern "C"
