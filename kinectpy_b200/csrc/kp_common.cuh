// kp_common.cuh -- internal declarations shared by the kernels of libkinectpy_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include <stdlib.h>
#include <string>
#include <vector>
#include "../../include/kp_api.h"

// ---------------------------------------------------------------- context --
struct KpProfEntry {
    const char *name;
    cudaEvent_t e0, e1;
    double bytes;   // algorithmic bytes moved by the launches inside the scope (DESIGN.md, per-kernel table)
};
struct kp_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    // workspace: bump allocator over one (occasionally more) device blocks, reset per API call
    struct Block { char *ptr; size_t cap; };
    std::vector<Block> blocks;
    size_t ws_off = 0;
    // small pinned host mirror + device scratch for scalars that must come back to the host
    char *h_scratch = nullptr;
    char *d_scratch = nullptr;
    size_t scratch_bytes = 1 << 16;
    std::string err;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    cudaEvent_t ev_block = nullptr;   // blocking-sync event of kp_stream_wait
    int64_t launches = 0;
    void *l2_flush = nullptr;
    // profiling
    bool prof_on = false;
    std::vector<KpProfEntry> prof;
    std::vector<cudaEvent_t> ev_pool;
    int sm_count = 148;
    // decoupled look-back state of the single-pass scans (kp_primitives.cu): one 64-bit word per tile
    // {epoch:30, flag:2, value:32}; never cleared between calls, the epoch invalidates old words
    unsigned long long *d_lb_state = nullptr;
    unsigned int lb_epoch = 0;
    static constexpr int LB_TILES = 1 << 16;
    int icp_passes_hint = 0;          // passes the last ICP on this context executed (sizes the next call's first batch)
};

int kp_set_err(kp_ctx *ctx, int code, const char *fmt, ...);
#define KP_CUDA(ctx, call)                                                                    \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess)                                                               \
            return kp_set_err(ctx, KP_E_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call,      \
                              cudaGetErrorString(e__));                                       \
    } while (0)
#define KP_TRY(expr)                 \
    do {                             \
        int rc__ = (expr);           \
        if (rc__ != KP_OK) return rc__; \
    } while (0)
#define KP_LAUNCH_CHECK(ctx)                      \
    do {                                          \
        (ctx)->launches++;                        \
        KP_CUDA(ctx, cudaGetLastError());         \
    } while (0)

void kp_ws_reset(kp_ctx *ctx);
int kp_ws_alloc(kp_ctx *ctx, size_t bytes, void **out);  // 256-byte aligned, valid until next kp_ws_reset
template <class T>
static inline int kp_ws(kp_ctx *ctx, size_t count, T **out)
{
    void *p = nullptr;
    int rc = kp_ws_alloc(ctx, count * sizeof(T) + 16, &p);
    *out = (T *)p;
    return rc;
}
// copies `bytes` from device scratch (offset 0) to pinned host scratch and waits
int kp_fetch_scratch(kp_ctx *ctx, size_t bytes);
// waits for everything enqueued on the context's stream (spinning or sleeping, see kp_ctx.cu)
int kp_stream_wait(kp_ctx *ctx);
// every public entry point starts here: bind the device, recycle the workspace
static inline void kp_enter(kp_ctx *ctx)
{
    cudaSetDevice(ctx->device);
    kp_ws_reset(ctx);
}

struct KpProfScope {
    kp_ctx *ctx;
    size_t idx;
    bool on;
    KpProfScope(kp_ctx *c, const char *name, double bytes = 0.0);
    ~KpProfScope();
    void add_bytes(double b) { if (on) ctx->prof[idx].bytes += b; }
};
#define KP_PROF(ctx, name) KpProfScope prof_scope__(ctx, name)
#define KP_PROFB(ctx, name, bytes) KpProfScope prof_scope__(ctx, name, (double)(bytes))

static inline unsigned kp_blocks(int64_t n, int per_block) { return (unsigned)((n + per_block - 1) / per_block); }

// ----------------------------------------------------- device primitives --
// (kp_primitives.cu)  All asynchronous on ctx->stream unless stated.
// exclusive positions of set flags; d_total[0] receives the number kept
int kp_prim_compact_mask(kp_ctx *ctx, int64_t n, const uint8_t *d_mask, int invert, const float *d_nan_src,
                         int32_t *d_pos_out /*[n] position or -1*/, int32_t *d_index_out /*[kept] nullable*/,
                         int32_t *d_total);
int kp_prim_gather3(kp_ctx *ctx, int64_t n, const int32_t *d_pos, const float *d_in, float *d_out);
// LSD radix sort of (key,value) pairs on bits [0,bits); result always lands in (*keys,*vals) buffers
// passed as `out`; `tmp` buffers are scratch of the same size.
int kp_prim_sort_pairs_u64(kp_ctx *ctx, int64_t n, int bits, uint64_t *d_keys, uint64_t *d_keys_tmp,
                           int32_t *d_vals, int32_t *d_vals_tmp, uint64_t **d_keys_sorted, int32_t **d_vals_sorted);
int kp_prim_sort_pairs_u32(kp_ctx *ctx, int64_t n, int bits, uint32_t *d_keys, uint32_t *d_keys_tmp,
                           int32_t *d_vals, int32_t *d_vals_tmp, uint32_t **d_keys_sorted, int32_t **d_vals_sorted);
// run heads over sorted keys[0..n): d_run_start[r] = first position of run r, d_run_start[R] = n; d_total[0] = R
int kp_prim_run_starts_u64(kp_ctx *ctx, int64_t n, const uint64_t *d_keys, int32_t *d_run_start, int32_t *d_total);
int kp_prim_run_starts_u32(kp_ctx *ctx, int64_t n, const uint32_t *d_keys, int32_t *d_run_start, int32_t *d_total);
// bounds: d_bounds_enc int32[8] = ordered-encoded min xyz, max xyz, count (slot 6); must be initialised by kp_prim_bounds_init
int kp_prim_bounds(kp_ctx *ctx, const float *d_xyz, int64_t n, int32_t *d_bounds_enc);
int kp_prim_bounds_fetch(kp_ctx *ctx, const float *d_xyz, int64_t n, float *h_bounds6, int64_t *h_nvalid);
// canonical double sum (see DESIGN.md "canonical reductions"); result in d_out[0]; d_tmp >= ceil(n/1024)+ceil(n/1M)+2 doubles
int kp_prim_csum(kp_ctx *ctx, const double *d_x, int64_t n, double *d_tmp, double *d_out);
// the same tree over a transformed view: mode 1: max(x, 0); mode 2: x > 0 ? (x - *d_aux / aux_div)^2 : 0
int kp_prim_csum_mode(kp_ctx *ctx, const double *d_x, int64_t n, double *d_tmp, double *d_out, int mode, const double *d_aux,
                      double aux_div);
int kp_prim_count_u8(kp_ctx *ctx, const uint8_t *d_mask, int64_t n, int32_t *d_total);

// ------------------------------------------------------- K1 / K2 device --
// internal flag of kp_unproject_device: d_bounds_enc is [B][S][8], one row per sensor (the frame pipeline needs the
// bounds of the master cloud and of every raw sub cloud as well as the fused ones: all come out of K1)
constexpr int KP_UP_BOUNDS_PER_SENSOR = 1 << 16;
int kp_unproject_device(kp_ctx *ctx, const uint16_t *d_depth, const float *d_xytab, const double *h_T, int B, int S,
                        int64_t P, int flags, double scale, float *d_xyz, uint8_t *d_valid, int16_t *d_xyz16,
                        int32_t *d_bounds_enc);
// h_bounds6 / nvalid: min xyz, max xyz and count of the non-NaN points (from kp_prim_bounds_fetch or K1)
int kp_voxel_device(kp_ctx *ctx, const float *d_xyz, const float *d_colors, const float *d_normals, int64_t n,
                    double voxel, const float *h_bounds6, int64_t nvalid, float *d_xyz_out, float *d_colors_out,
                    float *d_normals_out, int32_t *d_ijk, int32_t *d_point_voxel, double *h_min_bound, int64_t *h_m);

// ------------------------------------------------------------ grid (K3) --
struct KpGrid {
    int32_t n = 0;            // points in the sorted arrays (NaN points excluded)
    double org[3] = {0, 0, 0};
    double cell = 0, inv_cell = 0;
    int32_t dim[3] = {0, 0, 0};
    int sh_x = 0, sh_y = 0;      // packed cell key layout (cz low)
    float4 *d_sorted = nullptr;      // xyz + original index (int bits in .w), sorted by cell key
    uint4 *d_slots = nullptr;        // open addressing table of 16-byte slots {key lo, key hi, start, end}
    uint32_t hmask = 0;
    int32_t n_cells = 0;
    uint2 *d_cellmap = nullptr;      // {~occupancy bits, first rank} per 32 cells (NULL when dim0*dim1*dim2 is too large)
    int32_t *d_run_start = nullptr;  // [occupied cells + 1]
    int rad = 1;                     // block radius (in cells) the cell edge was chosen for: a search covers (2 rad + 1)^3 cells
};
// builds a grid over d_xyz in workspace memory (valid until kp_ws_reset). cell > 0 required.
// h_bounds6: min/max xyz enclosing every non-NaN point (may be conservative); NULL -> computed here (one sync).
int kp_grid_build(kp_ctx *ctx, const float *d_xyz, int64_t n, double cell, const float *h_bounds6, KpGrid *g);
// grid for a neighbour search whose 27-cell block would have edge `cell`: builds it with rad = 2 and half
// the edge when the histogram kernels will run the search (k <= 64), so that the block can be pruned column by column
int kp_grid_build_knn(kp_ctx *ctx, const float *d_xyz, int64_t n, double cell, int k, const float *h_bounds6, KpGrid *g);
// picks a cell edge so that an occupied cell holds ~target points (one trial sort)
int kp_grid_auto_cell(kp_ctx *ctx, const float *d_xyz, int64_t n, const float *h_bounds6, double target_per_cell,
                      double *cell_out);
// cell edge for a k-nearest search on a cloud that was voxel-downsampled at `voxel`
// (1.5 x the k-neighbour radius of an ideal 1-point-per-voxel surface: sensor clouds are sparser than the
// voxel grid far from the camera; sweep in profiles/r01_c_knn_base_coarse_sweep.log)
static inline double kp_knn_cell_from_voxel(double voxel, int k)
{
    static const double mult = getenv("KP_KNN_CELL_MULT") ? atof(getenv("KP_KNN_CELL_MULT")) : 1.5;
    return voxel * mult * sqrt((double)k / 3.14159265358979);
}

// internal forms used by the public API and by the frame pipeline (device pointers, async)
int kp_knn_device(kp_ctx *ctx, const KpGrid &g, const float *d_queries, int64_t nq, int k, double radius,
                  int32_t *d_idx, double *d_d2, int32_t *d_count, double *d_mean /*nullable: mean sqrt dist*/,
                  const float *d_xyz = nullptr /*cloud behind the grid: enables the coarse-level cascade*/);
int kp_sor_device(kp_ctx *ctx, const float *d_xyz, int64_t n, int k, double ratio, double cell_hint,
                  const float *h_bounds6, uint8_t *d_keep, double *d_mean, double *h_stats, int64_t *h_kept);
int kp_normals_device(kp_ctx *ctx, const float *d_xyz, int64_t n, double radius, int max_nn, const float *h_bounds6,
                      float *d_normals);

// ---------------------------------------------------- K4 / K5 device ----
int kp_ransac_device(kp_ctx *ctx, const float *d_xyz, int64_t n, double thr, int ransac_n, int iters, double probability,
                     uint64_t seed, double *h_plane, uint8_t *d_inlier_mask, int64_t *h_ninliers, int32_t *h_best_iter,
                     int64_t *d_counts);
int kp_band_mask_device(kp_ctx *ctx, const float *d_xyz, int64_t n, int axis, double band, uint8_t *d_lower,
                        double *h_axis_max, int64_t *h_nlower);
// point-to-point / coloured variants of the ICP pass (NULL -> point-to-plane)
struct KpIcpExtra {
    int mode = 0;                         // 0 plane, 1 point-to-point, 2 coloured
    const float *src_colors = nullptr;    // [n_src][3]
    const float *tgt_intensity = nullptr; // [n_tgt]
    const float *tgt_grad = nullptr;      // [n_tgt][3]
    double lambda_geometric = 0.968;
};
int kp_icp_device(kp_ctx *ctx, const float *d_src, int64_t n_src, const KpGrid &tgt_grid, const float *d_tgt_normals,
                  double max_corr, const double *h_init16, int max_iter, double rel_fitness, double rel_rmse,
                  double *h_T_out, double *h_fitness, double *h_rmse, int *h_iters, int64_t *h_ncorr,
                  const KpIcpExtra *extra = nullptr);
// intensity = (r+g+b)/3 and the tangent-plane colour gradient of every point (coloured ICP target preparation)
int kp_color_gradient_device(kp_ctx *ctx, const float *d_xyz, const float *d_colors, const float *d_normals, int64_t n,
                             double radius, int max_nn, float *d_intensity, float *d_grad);

// ------------------------------------------------------- device helpers --
#ifdef __CUDACC__
#define KP_FULL 0xffffffffu
__device__ __forceinline__ int kp_f2ord(float f)
{
    int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float kp_ord2f(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }
__host__ __device__ __forceinline__ uint64_t kp_mix64(uint64_t z)
{
    z += 0x9E3779B97F4A7C15ULL;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ uint64_t kp_rng(uint64_t seed, uint64_t a, uint64_t b)
{
    return kp_mix64(kp_mix64(kp_mix64(seed) + a) + b);
}
// canonical butterfly: every lane ends with the same value (IEEE add is commutative)
__device__ __forceinline__ double kp_butterfly_sum(double v)
{
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) v = __dadd_rn(v, __shfl_xor_sync(KP_FULL, v, s));
    return v;
}
// squared distance in double, fixed order, no FMA
__device__ __forceinline__ double kp_d2(double ax, double ay, double az, double bx, double by, double bz)
{
    double dx = __dsub_rn(ax, bx), dy = __dsub_rn(ay, by), dz = __dsub_rn(az, bz);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}
// ((a*x + b*y) + c*z) + d without contraction
__device__ __forceinline__ double kp_affine(double a, double b, double c, double d, double x, double y, double z)
{
    return __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(a, x), __dmul_rn(b, y)), __dmul_rn(c, z)), d);
}
// covariance-determinant plane fit on pre-reduced centred moments m = (xx, xy, xz, yy, yz, zz) around (cx, cy, cz):
// Open3D's segment_plane refit.  false: degenerate (zero or NaN normal).  Shared by kp_ransac_device (host) and the
// frame engine's batched refit (device); the build has no FMA contraction on either side.
__host__ __device__ __forceinline__ bool cov_fit_from_moments(const double *m, double cx, double cy, double cz, double *pl)
{
    const double xx = m[0], xy = m[1], xz = m[2], yy = m[3], yz = m[4], zz = m[5];
    const double dx = yy * zz - yz * yz, dy = xx * zz - xz * xz, dz = xx * yy - xy * xy;
    double a, b, c;
    if (dx >= dy && dx >= dz) { a = dx; b = xz * yz - xy * zz; c = xy * yz - xz * yy; }
    else if (dy >= dx && dy >= dz) { a = xz * yz - xy * zz; b = dy; c = xy * xz - yz * xx; }
    else { a = xy * yz - xz * yy; b = xy * xz - yz * xx; c = dz; }
    const double nn = sqrt((a * a + b * b) + c * c);
    if (nn == 0.0 || nn != nn) return false;
    a /= nn; b /= nn; c /= nn;
    pl[0] = a; pl[1] = b; pl[2] = c;
    pl[3] = -((a * cx + b * cy) + c * cz);
    return true;
}
__device__ __forceinline__ double kp_dot3(double a, double b, double c, double x, double y, double z)
{
    return __dadd_rn(__dadd_rn(__dmul_rn(a, x), __dmul_rn(b, y)), __dmul_rn(c, z));
}
#endif
