// kp_batch.cuh -- device-driven, batched building blocks of the frame engine (kp_engine.cu).
//
// Everything here obeys one launch convention: blockIdx.y = segment (one cloud of one frame of the batch),
// every array of a stage is laid out [segment][capacity] at a fixed stride, and every element COUNT lives in
// device memory (DCnt) because it was produced by an earlier kernel of the same frame.  No kernel argument
// depends on data, so a whole frame batch is a static launch sequence: it is enqueued without a single host
// round trip and captured once as a CUDA graph.  Grids are persistent (a CTA loops over the tiles its segment
// really has), so a loose capacity costs nothing.
#pragma once
#include "kp_common.cuh"
#include "kp_grid.cuh"
#include "kp_vbi.cuh"

// count of segment s = p[s * stride]  (stride in int32 units: counts usually sit in a per-frame state struct)
struct DCnt {
    const int32_t *p;
    int stride;
#ifdef __CUDACC__
    __device__ __forceinline__ int at(int s) const { return p[(size_t)s * stride]; }
#endif
};
struct DOut {
    int32_t *p;
    int stride;
#ifdef __CUDACC__
    __device__ __forceinline__ int32_t &at(int s) const { return p[(size_t)s * stride]; }
#endif
};
static inline DCnt dcnt(const int32_t *p, size_t stride_bytes) { return DCnt{p, (int)(stride_bytes / 4)}; }
static inline DOut dout(int32_t *p, size_t stride_bytes) { return DOut{p, (int)(stride_bytes / 4)}; }

// voxel grid of one cloud, computed on the device from the cloud's bounds (mirror of kp_voxel.cu's host code)
struct KpVoxDev {
    double minb[3];
    double voxel;
    int sh_x, sh_y;
    unsigned int sentinel;     // key of absent (NaN) rows: one bit above the packed index
    int imax[3];               // largest voxel index per axis
    int ok;                    // 0: the cloud is empty or its extent does not fit 31 key bits
};

// launch bookkeeping shared by every batched primitive
struct BLaunch {
    kp_ctx *ctx;               // stream, launch counter, profiling scopes
    int nseg;                  // segments in this launch (grid.y)
    int64_t cap;               // capacity (rows) of one segment
    int ctas;                  // persistent CTAs per segment (grid.x upper bound)
};

constexpr int BC_THREADS = 256;
constexpr int BC_ITEMS = 8;
constexpr int BC_TILE = BC_THREADS * BC_ITEMS;

// scratch of the two-kernel compaction / scans: per segment [max_tiles] tile sums + one ticket word
struct BScan {
    int32_t *tile_sum;         // [nseg][max_tiles]
    unsigned int *ticket;      // [nseg], zero between launches
    int max_tiles;
};

// ---- compaction family (count + last-CTA scan, then scatter): no CTA ever waits for another one
// rows of `in` whose mask byte (xor invert) is set -> packed into `out`; total[seg] = rows kept.  mask NULL: the rows whose
// x is not NaN
// aux_in / aux_out (nullable): a 4-byte payload per row (its packed voxel coordinates) that travels with the row
int kp_b_compact_rows(const BLaunch &L, const BScan &S, DCnt n, const uint8_t *mask, int64_t mask_stride, int invert,
                      const float *in, float *out, int64_t row_stride, DOut total, const uint32_t *aux_in = nullptr,
                      uint32_t *aux_out = nullptr);
// rows with mask set -> out_true (packed), the others -> out_false (packed, order kept); total[seg] = rows in out_true
int kp_b_partition_rows(const BLaunch &L, const BScan &S, DCnt n, const uint8_t *mask, int64_t mask_stride, const float *in,
                        float *out_true, float *out_false, int64_t row_stride, DOut total, const uint32_t *aux_in = nullptr,
                        uint32_t *aux_true = nullptr, uint32_t *aux_false = nullptr);
// positions of set mask bytes -> list[seg][..] (ascending); total[seg] = list length
int kp_b_compact_index(const BLaunch &L, const BScan &S, DCnt n, const uint8_t *mask, int64_t mask_stride, int32_t *list,
                       int64_t list_stride, DOut total);
// run heads of sorted u32 keys[0..n): run_start[r] = first position of run r, run_start[R] = n; total[seg] = R
int kp_b_run_starts_u32(const BLaunch &L, const BScan &S, DCnt n, const uint32_t *keys, int64_t key_stride, int32_t *run_start,
                        int64_t rs_stride, DOut total);
// exclusive scan of v[0..n) in place, v[n] = total, total[seg] = total (n <= cap - 1)
int kp_b_exclusive_scan(const BLaunch &L, const BScan &S, DCnt n, int32_t *v, int64_t v_stride, DOut total);

// ---- stable LSD radix sort of (u32 key, iota) pairs, `n` rows per segment (static), 8 bits per pass, `passes`
// passes; result in (keys, vals) when passes is even, else in (keys_tmp, vals_tmp)
struct BSort {
    int32_t *g_hist;           // [nseg][256][nb]
    int32_t *g_tot;            // [nseg][256]
};
int kp_b_sort_pairs_u32(const BLaunch &L, const BSort &W, int64_t n, int passes, uint32_t *keys, uint32_t *keys_tmp,
                        int32_t *vals, int32_t *vals_tmp, int64_t stride);
size_t kp_b_sort_hist_elems(int64_t n);   // int32 elements of g_hist for one segment

// ---- canonical double sum (kp_primitives.cu's tree, bit for bit) of x[0..n) with n on the device
// mode 0: x   1: max(x, 0)   2: x > 0 ? (x - aux / n)^2 : 0      tmp: [nseg][tmp_stride] doubles
int kp_b_csum(const BLaunch &L, DCnt n, const double *x, int64_t x_stride, int mode, const double *aux, int64_t aux_stride,
              double *tmp, int64_t tmp_stride, double *out, int64_t out_stride);

// Neighbour lists the normals search hands to the ICP (both run on the same grid over the target): for every target
// position p whose search level 0 certified, up to KP_NLIST entries {position, d2 rounded down to float} of its certified
// neighbours in canonical (d2, index) order, p itself left out, closed by a {-1, +inf} entry when shorter; and rho2[p], a
// float lower bound of a squared radius inside which every other target point is in the list (0: no list).
constexpr int KP_NLIST = 12;

// ---- batched neighbour searches (kp_grid.cu): level 0 (thread per query, histogram select) -> level 1 (warp per
// leftover query on a coarser grid) -> ring-expanding stragglers; the engine runs the list compactions and the
// coarse grid build in between
struct KpKnnSegDesc {
    const KpGridDev *g0, *g1;     // device: level-0 / level-1 grid of this cloud
    const KpVbiDev *vbi;          // device, nullable: voxel-brick index of this cloud (level 0 runs on it when it was built)
    const float4 *pts0;           // the level-0 grid's cell-sorted rows (static pointer)
    const int32_t *n;             // device: points in the cloud (every point is a query)
    uint8_t *flags0, *flags1;     // [cap] "not certified at level 0 / 1", indexed by level-0 position
    int32_t *list0, *list1;       // [cap] compacted positions
    const int32_t *cnt0, *cnt1;   // device: lengths of the lists
    const KpGridDev *gm;          // optional mid level (NULL = none): grid, flags, list and count of what it leaves
    uint8_t *flags_m; int32_t *list_m; const int32_t *cnt_m;
    double *mean;                 // SOR: mean distance to the k nearest (by original index)
    const float *cloud;           // normals mode: the cloud, by original index
    float *normals;               // normals mode: output
    int2 *nlist; float *nrho;     // normals mode, nullable: [cap][KP_NLIST] neighbour lists and [cap] rho2, by level-0 position
};
struct KpKnnBatch {
    void *d_params = nullptr, *h_params = nullptr;     // [3 levels][nseg] parameter blocks on the device and their host copy
    int nseg = 0, k = 0, mode = 0, cap_hist = 0, cap_warp = 0, rad = 1, cap_mid = 0, has_mid = 0;
    int lists = 0;                // level 0 writes the neighbour lists (nlist / nrho of the segments)
};
// mode 0: mean distance of the k nearest (SOR); mode 1: normals from the <= k nearest inside `radius`
// rho_a / rho_b: the two search radii of the voxel-brick level 0 (ignored without an index)
int kp_knn_batch_create(kp_ctx *ctx, const KpKnnSegDesc *segs, int nseg, int k, int mode, double radius, double rho_a, double rho_b,
                        KpKnnBatch *out);
int kp_knn_batch_vbi(kp_ctx *ctx, const KpKnnBatch &b, int64_t cap_rows);
void kp_knn_batch_destroy(KpKnnBatch *b);
int kp_knn_batch_level0(kp_ctx *ctx, const KpKnnBatch &b, int64_t cap_rows);
int kp_knn_batch_mid(kp_ctx *ctx, const KpKnnBatch &b, int64_t cap_rows);
int kp_knn_batch_level1(kp_ctx *ctx, const KpKnnBatch &b, int64_t cap_rows);
int kp_knn_batch_stragglers(kp_ctx *ctx, const KpKnnBatch &b);

// ---- batched point-to-plane ICP (kp_icp.cu): every pair of the batch advances in the same launches
// (blockIdx.y = pair); max_iter + 1 identical pass launches, a converged pair's CTAs return at once
struct KpIcpPairDesc {
    const KpGridDev *tgt_grid;    // device: grid over the target (cell >= max_corr)
    const KpVbiDev *tgt_vbi;      // device, nullable: voxel-brick index over the target (preferred when it was built)
    const float *tgt_normals;     // by original target index
    const int2 *tgt_list;         // nullable: neighbour lists of the target's grid positions (KP_NLIST per position)
    const float *tgt_rho;         // with tgt_list: their rho2
    const float *src;             // source cloud (device), n_src rows
    const int32_t *n_src;         // device
    double init_T[16];
    double *res_T, *res_fit, *res_rmse; int32_t *res_iters;   // device: where the pair's converged state goes
};
struct KpIcpBatch {
    void *d_params = nullptr, *d_work = nullptr;
    int npairs = 0, max_iter = 0, grid = 0;
    int64_t cap_src = 0;
    int32_t *d_tally = nullptr;   // KP_DEBUG_ICP: [npairs][max_iter + 1][2] points decided by the list / searched in the grid
};
int kp_icp_batch_create(kp_ctx *ctx, const KpIcpPairDesc *pairs, int npairs, int64_t cap_src, double max_corr, int max_iter,
                        double rel_fitness, double rel_rmse, KpIcpBatch *out);
void kp_icp_batch_destroy(KpIcpBatch *b);
int kp_icp_batch_run(kp_ctx *ctx, const KpIcpBatch &b);
