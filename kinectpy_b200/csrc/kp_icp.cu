// kp_icp.cu -- K5: point-to-plane ICP, every iteration on the device.
// Replaces o3d.pipelines.registration.registration_icp(source, target, max_corr, init,
// TransformationEstimationPointToPlane()) at preprocessing/registration.py:78-84 (SURVEY.md A.7).
//
// One kernel launch per pass (k_icp_iter, one thread per source point).  A pass (i) applies the update found by the previous pass to the
// moving copy of the source (double, in place, like upstream's pcd.Transform(update)),
// (ii) finds each source point's nearest target point inside max_corr through the target's grid
// hash (27 cells, z-rows merged, one thread per source point), (iii) accumulates the 21+6+2
// normal-equation scalars in double, reduced with warp shuffles (xor butterfly), then a fixed-order
// sum over the warps of the CTA, then per-CTA slots; (iv) the last CTA to finish (integer ticket)
// adds the slots in a fixed order, evaluates fitness / rmse / the convergence test, solves the 6x6
// system cooperatively (one thread per matrix element, the operations of the scalar elimination in the
// same order), composes T and publishes the next update, the pass counter and a `done` flag.  The host enqueues
// max_iter+1 passes without reading anything back; passes after `done` return immediately.
#include <math.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <vector>
#include "kp_grid.cuh"
#include "kp_batch.cuh"
#include "kp_umeyama.cuh"

namespace {
#ifndef ICP_THREADS_N
#define ICP_THREADS_N 256
#endif
constexpr int ICP_THREADS = ICP_THREADS_N;
#ifndef ICP_MIN_CTAS
#define ICP_MIN_CTAS 4
#endif
constexpr int ICP_GROUP = 32;  // CTAs per group of the two-level hand-over at the end of a pass
constexpr int ICP_NV = 29;   // 21 upper-triangular JtJ + 6 Jtr + sum d^2 + count
                             // (point-to-point: 3 sum s + 3 sum t + 9 sum t s^T in slots 0..14, same two tail slots)
enum { ICP_PLANE = 0, ICP_POINT = 1, ICP_COLORED = 2 };

struct IcpState {
    double T[16];
    double U[16];
    double fitness, rmse;
    long long ncorr;
    int done, iters;
    unsigned int ticket;
    int pass;                   // number of the pass the next launch executes (advanced by the last CTA)
    double slack;               // frame engine: the fp32 pre-test slack, computed on the device from the grid extent
};

struct IcpParams {
    KpGridDev g;
    const float *tgt_normals;   // indexed by original target index
    int mode;                   // ICP_PLANE / ICP_POINT / ICP_COLORED
    const float *src_int;       // colored: source intensity (r+g+b)/3, in the (re-ordered) order of cur
    const float *tgt_int;       // colored: target intensity, by original target index
    const float *tgt_grad;      // colored: target colour gradient [nt][3], by original target index
    double sqrt_lg, sqrt_lp;    // colored: sqrt(lambda_geometric), sqrt(1 - lambda_geometric)
    double *cur;                // [ns][3] moving source
    int32_t *corr;              // [ns] position of the matched target point in g.pts, -1 = none
    int ns;
    double r2;
    double slack;               // bound on (fp32 d2) - d2 for d2 <= max_corr^2, points near the grid
    int max_iter;
    double rel_fit, rel_rmse;
    IcpState *st;
    double *slots;              // [gridDim.x][ICP_NV]
    double *gslots;             // [groups][ICP_NV] group rows
    unsigned int *gticket;      // [groups] zero between passes
    // frame engine (batched launches, blockIdx.y = pair): values produced on the device
    const KpGridDev *gdev;      // non-NULL: replaces g
    const int32_t *ns_dev;      // non-NULL: replaces ns
    const float *src;           // source cloud of the pair
    double max_corr;
    double init_T[16];
    double *res_T, *res_fit, *res_rmse; int32_t *res_iters;   // where the converged state of the pair goes
    const KpVbiDev *vbi;        // voxel-brick index over the target (device); used instead of the grid when it was built
    const int2 *tlist;          // nullable: the target's neighbour lists by grid position (kp_batch.cuh, KP_NLIST)
    const float *trho;          // with tlist: their rho2
    int32_t *tally;             // nullable (KP_DEBUG_ICP): [max_iter + 1][2] points decided by the list / searched in the grid
};

__device__ __forceinline__ double icp_slack(const KpGridDev &g, double max_corr)
{
    // fp32 rounding of a coordinate of magnitude <= M costs <= M * 2^-24 per operand; 8 x that covers the
    // three axes, both operands and the fp32 arithmetic with room to spare
    double M = 0.0;
    for (int c = 0; c < 3; ++c)
        M = fmax(M, fmax(fabs(g.org[c]), fabs(g.org[c] + g.cell * (double)g.dim[c])) + 2.0 * max_corr);
    const double eps = 8.0 * M / 16777216.0;          // bound on |sqrt(fp32 d2) - sqrt(d2)|
    return eps * (2.0 * max_corr + eps) * 1.000001 + 4e-6 * (max_corr * max_corr);
}

// batched launches: the parameter block of pair blockIdx.y straight from device memory (uniform, cached loads of the
// fields a thread uses: no shared-memory copy, no barrier), with the device-side grid layout, source count and slack
__device__ __forceinline__ IcpParams icp_params_batched(const IcpParams *__restrict__ pp)
{
    IcpParams p = pp[blockIdx.y];
    p.g = *p.gdev;
    p.ns = *p.ns_dev;
    p.slack = p.st->slack;
    return p;
}

__global__ void __launch_bounds__(256) k_icp_init(const float *src, int ns, const __grid_constant__ IcpParams p, IcpState init,
                                                  double *out)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *p.st = init;
    if (i >= ns) return;
    const double *T = init.T;
    double X = src[3 * (int64_t)i], Y = src[3 * (int64_t)i + 1], Z = src[3 * (int64_t)i + 2];
    out[3 * (int64_t)i] = kp_affine(T[0], T[1], T[2], T[3], X, Y, Z);
    out[3 * (int64_t)i + 1] = kp_affine(T[4], T[5], T[6], T[7], X, Y, Z);
    out[3 * (int64_t)i + 2] = kp_affine(T[8], T[9], T[10], T[11], X, Y, Z);
}

// nearest target point inside max_corr (position in g.pts, -1 = none); `prev` = last pass's partner or -1.
// Exhaustive and exact in double: a column (or a cell of it) is skipped only when its nearest face is farther
// than the best match known when the lookups are issued, and the fp32 pre-test only rejects candidates that
// cannot win (slack bounds the error of the fp32 squared distance: the moving source is double, the test runs
// on its float rounding).  The cell-map lookups of all needed columns are issued together (branch-free), so
// their memory round trips overlap instead of queueing behind one another.
__device__ __forceinline__ int icp_nearest(const KpGridDev &g, double sx, double sy, double sz, double r2, double slack, int prev)
{
    int bpos = -1;
    const int cx = kp_cell_coord(g, sx, 0), cy = kp_cell_coord(g, sy, 1), cz = kp_cell_coord(g, sz, 2);
    double bd = INFINITY;
    int bi = -1;
    const float fx32 = (float)sx, fy32 = (float)sy, fz32 = (float)sz;
    // Warm start: after the first passes the update is tiny and most points keep their partner.  The previous
    // partner is a valid candidate, so its distance is an upper bound that prunes almost every other cell.
    if (prev >= 0) {
        const float4 q = __ldg(g.pts + prev);
        const double d2 = kp_d2(sx, sy, sz, (double)q.x, (double)q.y, (double)q.z);
        if (d2 < r2) { bd = d2; bi = __float_as_int(q.w); bpos = prev; }
    }
    // fp32 lower bounds of the distances to the faces of the own cell (shrunk, so rounding in the cell
    // assignment or in the fp32 arithmetic can never hide a closer point)
    float flo[3], fhi[3];
    {
        const double cs = g.cell * (1.0 - 3.0 / 1048576.0);
        const double ss[3] = {sx, sy, sz};
        const int cc[3] = {cx, cy, cz};
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double f = fmin(fmax((ss[c] - g.org[c]) * g.inv_cell - (double)cc[c], 0.0), 1.0);
            flo[c] = (float)(f * cs); fhi[c] = (float)((1.0 - f) * cs);
        }
    }
    const double lim0 = fmin(bd, r2);
    const float budget = __double2float_ru(lim0 * (1.0 + 4e-6));
    int2 rng[9];
#pragma unroll
    for (int oi = 0; oi < 9; ++oi) {
        const int dx = oi / 3 - 1, dy = oi % 3 - 1;
        const float gx = dx < 0 ? flo[0] : (dx > 0 ? fhi[0] : 0.0f), gy = dy < 0 ? flo[1] : (dy > 0 ? fhi[1] : 0.0f);
        const float zb = budget - (gx * gx + gy * gy);
        const int zlo = flo[2] * flo[2] <= zb ? cz - 1 : cz, zhi = fhi[2] * fhi[2] <= zb ? cz + 1 : cz;
        rng[oi] = zb >= 0.0f ? kp_span_range(g, cx + dx, cy + dy, zlo, zhi) : make_int2(0, 0);
    }
    float lim32 = __double2float_ru(lim0 + slack), cur = budget;
    const int order[9] = {4, 1, 3, 5, 7, 0, 2, 6, 8};   // own column first: it tightens the bound for the others
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const int oi = order[k], dx = oi / 3 - 1, dy = oi % 3 - 1;
        const float gx = dx < 0 ? flo[0] : (dx > 0 ? fhi[0] : 0.0f), gy = dy < 0 ? flo[1] : (dy > 0 ? fhi[1] : 0.0f);
        if (gx * gx + gy * gy > cur) continue;
        // four candidates per trip: the loads are issued together, so a column costs one memory round trip per four
        // candidates instead of one each (the warp stalls at the first use of a loaded value)
        for (int t = rng[oi].x; t < rng[oi].y; t += 4) {
            const int m = rng[oi].y - t;
            float4 q[4];
            q[0] = __ldg(g.pts + t);
            q[1] = __ldg(g.pts + (m > 1 ? t + 1 : t));
            q[2] = __ldg(g.pts + (m > 2 ? t + 2 : t));
            q[3] = __ldg(g.pts + (m > 3 ? t + 3 : t));
            float d32[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float ex = fx32 - q[u].x, ey = fy32 - q[u].y, ez = fz32 - q[u].z;
                d32[u] = __fmaf_rn(ez, ez, __fmaf_rn(ey, ey, ex * ex));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (u >= m || d32[u] > lim32) continue;
                const double d2 = kp_d2(sx, sy, sz, (double)q[u].x, (double)q[u].y, (double)q[u].z);
                const int id = __float_as_int(q[u].w);
                if (d2 < r2 && (d2 < bd || (d2 == bd && id < bi))) {
                    bd = d2; bi = id; bpos = t + u;
                    lim32 = __double2float_ru(bd + slack); cur = __double2float_ru(bd * (1.0 + 4e-6));
                }
            }
        }
    }
    return bpos;
}

// The same answer from the neighbour list of the previous partner t (position prev, squared distance d2t < r2 from the
// point), for a point with 4 * d2t * (1 + 1e-6) < rho2(t): every target point at least as close as t lies within 2
// sqrt(d2t) of t (triangle inequality), so inside rho(t), so in t's list, which is in canonical order; the scan stops at
// the first entry beyond that bound.  Candidates are tested exactly as in icp_nearest, so the result is the same.
__device__ __forceinline__ int icp_nearest_list(const KpGridDev &g, const int4 *__restrict__ list, double sx, double sy, double sz,
                                                double r2, double slack, int prev, double d2t, int idt, float stop)
{
    double bd = d2t;
    int bi = idt, bpos = prev;
    const float fx32 = (float)sx, fy32 = (float)sy, fz32 = (float)sz;
    float lim32 = __double2float_ru(bd + slack);
    // four entries (one 32-byte sector) per trip, their points requested together
    for (int j = 0; j < KP_NLIST; j += 4) {
        const int4 e01 = __ldg(list + (size_t)prev * (KP_NLIST / 2) + j / 2), e23 = __ldg(list + (size_t)prev * (KP_NLIST / 2) + j / 2 + 1);
        const int pos[4] = {e01.x, e01.z, e23.x, e23.z};
        const float ed[4] = {__int_as_float(e01.y), __int_as_float(e01.w), __int_as_float(e23.y), __int_as_float(e23.w)};
        // an entry counts only while every entry before it did: the closing {-1, +inf} entry ends the list, and the
        // words behind it were never written
        bool in[4];
        in[0] = ed[0] <= stop;
#pragma unroll
        for (int u = 1; u < 4; ++u) in[u] = in[u - 1] && ed[u] <= stop;
        float4 q[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) q[u] = __ldg(g.pts + (in[u] ? pos[u] : prev));
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (!in[u]) break;                           // the first entry beyond the bound, or the end of the list
            const float ex = fx32 - q[u].x, ey = fy32 - q[u].y, ez = fz32 - q[u].z;
            if (__fmaf_rn(ez, ez, __fmaf_rn(ey, ey, ex * ex)) > lim32) continue;
            const double d2 = kp_d2(sx, sy, sz, (double)q[u].x, (double)q[u].y, (double)q[u].z);
            const int id = __float_as_int(q[u].w);
            if (d2 < r2 && (d2 < bd || (d2 == bd && id < bi))) {
                bd = d2; bi = id; bpos = pos[u];
                lim32 = __double2float_ru(bd + slack);
            }
        }
        if (!in[3]) break;
    }
    return bpos;
}

// The same search through the voxel-brick index of the (voxel-downsampled) target: the ball of radius
// min(best so far, max_corr) around the source point is boxed in voxel coordinates, each brick the box touches
// costs one 16-byte load and an AND of its occupancy word with the box mask, and only the voxels that survive are
// looked at.  With the warm start the ball is a few millimetres wide: one or two bricks, one or two candidates.
__device__ __forceinline__ int icp_nearest_vbi(const KpVbiDev &v, double sx, double sy, double sz, double r2, double slack, int prev)
{
    int bpos = -1, bi = -1;
    double bd = INFINITY;
    if (prev >= 0) {
        const float4 q = __ldg(v.pts + prev);
        const double d2 = kp_d2(sx, sy, sz, (double)q.x, (double)q.y, (double)q.z);
        if (d2 < r2) { bd = d2; bi = __float_as_int(q.w); bpos = prev; }
    }
    const double lim0 = fmin(bd, r2);
    // every point with d2 <= lim0 lies in a voxel whose box (widened by eps) meets the ball of this radius
    const double rad = sqrt(lim0) * (1.0 + 1e-6) + v.eps + v.voxel * 1e-6;
    KpVbiBox box;
    if (!kp_vbi_box(v, sx, sy, sz, rad, box)) return bpos;
    const float fx32 = (float)sx, fy32 = (float)sy, fz32 = (float)sz;
    float lim32 = __double2float_ru(lim0 + slack);
    kp_vbi_visit(v, box, [&](int pos, const float4 &q) {
        const float ex = fx32 - q.x, ey = fy32 - q.y, ez = fz32 - q.z;
        const float d32 = __fmaf_rn(ez, ez, __fmaf_rn(ey, ey, ex * ex));
        if (d32 > lim32) return;
        const double d2 = kp_d2(sx, sy, sz, (double)q.x, (double)q.y, (double)q.z);
        const int id = __float_as_int(q.w);
        if (d2 < r2 && (d2 < bd || (d2 == bd && id < bi))) {
            bd = d2; bi = id; bpos = pos;
            lim32 = __double2float_ru(bd + slack);
        }
    });
    return bpos;
}

// last CTA, all threads: fitness / rmse / convergence test, 6x6 solve, next update
// 6x6 solve by Gaussian elimination with partial pivoting on the augmented matrix M[6][7] in shared memory,
// executed by the whole (last) CTA: thread (r, j) = tid / 7, tid % 7 owns one element.  Every step performs
// exactly the operations of the scalar loop nest (f = M[r][c] / M[c][c]; M[r][j] -= f * M[c][j] for j >= c),
// element-parallel, so the result is the one a single thread would get, without its serial latency chain.
// Returns (to every thread) whether the system was solvable; x[] is valid then.
__device__ bool icp_solve6_cta(double (*M)[7], double *x, int tid)
{
    const int r = tid / 7, j = tid % 7;
    const bool own = tid < 42;
    bool ok = true;
    for (int c = 0; c < 6; ++c) {
        int pv = c;
        double best = fabs(M[c][c]);
        for (int rr = c + 1; rr < 6; ++rr) {
            const double v = fabs(M[rr][c]);
            if (v > best) { best = v; pv = rr; }
        }
        if (!(best > 1e-300)) { ok = false; break; }          // uniform: every thread read the same column
        __syncthreads();
        if (own && r == c && pv != c) { const double t = M[c][j]; M[c][j] = M[pv][j]; M[pv][j] = t; }
        __syncthreads();
        double nv = 0.0;
        const bool upd = own && r > c && j >= c;
        if (upd) { const double f = M[r][c] / M[c][c]; nv = M[r][j] - f * M[c][j]; }
        __syncthreads();
        if (upd) M[r][j] = nv;
        __syncthreads();
    }
    if (ok && tid == 0) {
        for (int rr = 5; rr >= 0; --rr) {
            double sacc = M[rr][6];
            for (int jj = rr + 1; jj < 6; ++jj) sacc -= M[rr][jj] * x[jj];
            x[rr] = sacc / M[rr][rr];
        }
    }
    __syncthreads();
    if (ok)
        for (int rr = 0; rr < 6; ++rr) if (!isfinite(x[rr])) ok = false;
    return ok;
}

// last CTA, all threads: fitness / rmse / convergence test, 6x6 solve, next update
__device__ void icp_finish(const IcpParams &p, IcpState *st, const double *tot, int pass, int tid)
{
    __shared__ double M[6][7];
    __shared__ double x[6];
    __shared__ double Un[16];
    __shared__ int s_done;
    const double nc = tot[28];
    if (tid == 0) {
        const double fit = p.ns > 0 ? nc / (double)p.ns : 0.0;
        const double rmse = nc > 0 ? sqrt(tot[27] / nc) : 0.0;
        const double pfit = st->fitness, prmse = st->rmse;
        st->fitness = fit; st->rmse = rmse; st->ncorr = (long long)nc;
        st->ticket = 0;
        st->pass = pass + 1;
        bool done = false;
        if (pass > 0) {
            st->iters = pass;
            if (fabs(pfit - fit) < p.rel_fit && fabs(prmse - rmse) < p.rel_rmse) done = true;
        }
        if (pass >= p.max_iter) done = true;
        if (done) st->done = 1;
        s_done = done ? 1 : 0;
    }
    if (tid < 16) Un[tid] = (tid % 5 == 0) ? 1.0 : 0.0;
    if (tid < 6) x[tid] = 0.0;
    __syncthreads();
    if (s_done) return;
    if (p.mode == ICP_POINT) {
        if (tid == 0 && nc > 0) kp_umeyama(tot, nc, Un);
    } else {
        if (tid < 42) {
            const int r = tid / 7, j = tid % 7;
            if (j == 6) M[r][6] = -tot[21 + r];
            else {
                const int a = r < j ? r : j, b = r < j ? j : r;
                M[r][j] = tot[a * 6 - (a * (a - 1)) / 2 + (b - a)];   // packed upper triangle, row-major
            }
        }
        __syncthreads();
        const bool ok = icp_solve6_cta(M, x, tid);
        if (ok && nc > 0 && tid == 0) {
            double ca = cos(x[0]), sa = sin(x[0]), cb = cos(x[1]), sb = sin(x[1]), cg = cos(x[2]), sg = sin(x[2]);
            Un[0] = cg * cb; Un[1] = cg * sb * sa - sg * ca; Un[2] = cg * sb * ca + sg * sa; Un[3] = x[3];
            Un[4] = sg * cb; Un[5] = sg * sb * sa + cg * ca; Un[6] = sg * sb * ca - cg * sa; Un[7] = x[4];
            Un[8] = -sb;     Un[9] = cb * sa;                Un[10] = cb * ca;               Un[11] = x[5];
        }
    }
    __syncthreads();
    double tn = 0.0;
    if (tid < 16) {
        const int i2 = tid >> 2, j = tid & 3;
        for (int k = 0; k < 4; ++k) tn = tn + Un[4 * i2 + k] * st->T[4 * k + j];
    }
    __syncthreads();                    // every T element has been read
    if (tid < 16) { st->T[tid] = tn; st->U[tid] = Un[tid]; }
    __threadfence();
}

// The per-point terms of one tile of ICP_THREADS source points (point i of this thread at (sx, sy, sz), partner bpos),
// reduced over each warp into sh[warp][*].  Warp reduction of the 29 scalars by halving exchange: at step s a lane keeps
// one half of its values and trades the other half with lane^s, so 32 values are fully reduced in 31 exchanges (lane L
// ends up with the warp total of value L) instead of 32 butterflies of 5.  Fixed tree -> deterministic.
template <int MODE>
__device__ __forceinline__ void icp_tile_terms(const IcpParams &p, const float4 *tpts, int i, double sx, double sy, double sz, int bpos,
                                               double (*sh)[ICP_NV], int lane, int warp)
{
    bool has = false;
    // plane / colored: J (6) and r of the geometric term; colored adds the photometric row J2, r2;
    // point-to-point: J[0..2] = s, J[3..5] = t
    double J[6] = {0, 0, 0, 0, 0, 0}, r = 0.0, bd = 0.0;
    double J2[6] = {0, 0, 0, 0, 0, 0}, r2v = 0.0;
    if (i < p.ns) {
        p.corr[i] = bpos;
        if (bpos >= 0) {
            has = true;
            const float4 q = __ldg(tpts + bpos);
            const int bi = __float_as_int(q.w);
            const double ex = sx - (double)q.x, ey = sy - (double)q.y, ez = sz - (double)q.z;
            bd = (ex * ex + ey * ey) + ez * ez;
            if (MODE == ICP_POINT) {
                J[0] = sx; J[1] = sy; J[2] = sz; J[3] = (double)q.x; J[4] = (double)q.y; J[5] = (double)q.z;
            } else {
                const double nx = (double)__ldg(p.tgt_normals + 3 * (int64_t)bi), ny = (double)__ldg(p.tgt_normals + 3 * (int64_t)bi + 1),
                             nz = (double)__ldg(p.tgt_normals + 3 * (int64_t)bi + 2);
                r = (ex * nx + ey * ny) + ez * nz;
                J[0] = sy * nz - sz * ny; J[1] = sz * nx - sx * nz; J[2] = sx * ny - sy * nx; J[3] = nx; J[4] = ny; J[5] = nz;
                if (MODE == ICP_COLORED) {
                    // TransformationEstimationForColoredICP (registration.py:108-113): the geometric row weighted
                    // by sqrt(lambda), plus the photometric row of the colour projected onto the target's tangent plane
                    const double is = (double)__ldg(p.src_int + i), it = (double)__ldg(p.tgt_int + bi);
                    const double gx = (double)__ldg(p.tgt_grad + 3 * (int64_t)bi), gy = (double)__ldg(p.tgt_grad + 3 * (int64_t)bi + 1),
                                 gz = (double)__ldg(p.tgt_grad + 3 * (int64_t)bi + 2);
                    // vs_proj - vt = e - (e.n) n ;  is_proj = grad.(vs_proj - vt) + it
                    const double px = ex - r * nx, py = ey - r * ny, pz = ez - r * nz;
                    const double is_proj = ((gx * px + gy * py) + gz * pz) + it;
                    // ditM = -(I - n n^T) grad
                    const double gn = (gx * nx + gy * ny) + gz * nz;
                    const double mx = -(gx - gn * nx), my = -(gy - gn * ny), mz = -(gz - gn * nz);
                    J2[0] = p.sqrt_lp * (sy * mz - sz * my); J2[1] = p.sqrt_lp * (sz * mx - sx * mz); J2[2] = p.sqrt_lp * (sx * my - sy * mx);
                    J2[3] = p.sqrt_lp * mx; J2[4] = p.sqrt_lp * my; J2[5] = p.sqrt_lp * mz;
                    r2v = p.sqrt_lp * (is - is_proj);
#pragma unroll
                    for (int a = 0; a < 6; ++a) J[a] *= p.sqrt_lg;
                    r *= p.sqrt_lg;
                }
            }
        }
    }
    if (__any_sync(KP_FULL, has)) {
        double v[32];
        if (MODE == ICP_POINT) {
#pragma unroll
            for (int a = 0; a < 6; ++a) v[a] = J[a];
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int b = 0; b < 3; ++b) v[6 + 3 * a + b] = J[3 + a] * J[b];
#pragma unroll
            for (int a = 15; a < 27; ++a) v[a] = 0.0;
        } else {
            int k = 0;
#pragma unroll
            for (int a = 0; a < 6; ++a)
#pragma unroll
                for (int b = a; b < 6; ++b) { v[k] = J[a] * J[b]; if (MODE == ICP_COLORED) v[k] += J2[a] * J2[b]; ++k; }
#pragma unroll
            for (int a = 0; a < 6; ++a) { v[21 + a] = J[a] * r; if (MODE == ICP_COLORED) v[21 + a] += J2[a] * r2v; }
        }
        v[27] = bd; v[28] = has ? 1.0 : 0.0; v[29] = 0.0; v[30] = 0.0; v[31] = 0.0;
#pragma unroll
        for (int s = 16; s >= 1; s >>= 1) {
            const bool upper = (lane & s) != 0;
#pragma unroll
            for (int j = 0; j < s; ++j) {
                const double send = upper ? v[j] : v[j + s];
                const double keep = upper ? v[j + s] : v[j];
                v[j] = keep + __shfl_xor_sync(KP_FULL, send, s);
            }
        }
        if (lane < ICP_NV) sh[warp][lane] = v[0];
    } else if (lane < ICP_NV) {
        sh[warp][lane] = 0.0;
    }
}

// One pass: update + correspondence + accumulation, one thread per source point of a tile of ICP_THREADS; every tile
// leaves one slot row; the last CTA solves and publishes the next update.
// QUEUE (batched kernel): a CTA owns ICP_B_TILES tiles.  A point whose partner the target's neighbour list decides skips
// the grid search (icp_nearest_list); the others are packed into a CTA-wide queue and searched by consecutive threads,
// so the searches run in dense warps and a CTA's threads each search about once per pass however many points the lists
// decide.  Each result goes back to the point's slot, and its own thread then goes on as without the queue: the same
// per-point terms and the same per-tile reduction tree, so the sums are bit-identical.
constexpr int ICP_B_TILES = 4;
constexpr int ICP_PENDING = -2;    // queue path: a point waiting for its grid search
template <int MODE, bool QUEUE = false>
__device__ __forceinline__ void icp_iter_body(const IcpParams &p)
{
    constexpr int TPC = QUEUE ? ICP_B_TILES : 1;       // tiles per CTA
    constexpr int W = ICP_THREADS / 32;
    __shared__ double sh[ICP_THREADS / 32][ICP_NV];
    __shared__ double part[ICP_THREADS / 32][32];
    __shared__ double tot[ICP_NV];
    __shared__ unsigned int s_ticket;
    IcpState *st = p.st;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned ntiles = max(1u, ((unsigned)p.ns + ICP_THREADS - 1) / ICP_THREADS);
    const KpGridDev &g = p.g;
    const bool use_vbi = p.vbi != nullptr && p.vbi->ok;
    const float4 *tpts = use_vbi ? p.vbi->pts : g.pts;
    int pass;
    if constexpr (!QUEUE) {
        const int i = blockIdx.x * ICP_THREADS + tid;
        // the point, its last partner and the state words are requested together: one memory round trip before the
        // first arithmetic instead of two (a pass launched after `done` only wastes these few loads)
        double sx = 0.0, sy = 0.0, sz = 0.0;
        int prev0 = -1;
        if (i < p.ns) {
            sx = p.cur[3 * (int64_t)i]; sy = p.cur[3 * (int64_t)i + 1]; sz = p.cur[3 * (int64_t)i + 2];
            prev0 = p.corr[i];              // (not yet written in pass 0: ignored there)
        }
        if (st->done) return;
        pass = st->pass;                    // advanced only after every CTA has taken its ticket
        int bpos = -1;
        if (i < p.ns) {
            const int prev = pass > 0 ? prev0 : -1;
            if (pass > 0) {
                const double *U = st->U;
                const double x2 = kp_affine(U[0], U[1], U[2], U[3], sx, sy, sz);
                const double y2 = kp_affine(U[4], U[5], U[6], U[7], sx, sy, sz);
                const double z2 = kp_affine(U[8], U[9], U[10], U[11], sx, sy, sz);
                sx = x2; sy = y2; sz = z2;
                p.cur[3 * (int64_t)i] = sx; p.cur[3 * (int64_t)i + 1] = sy; p.cur[3 * (int64_t)i + 2] = sz;
            }
            if (use_vbi) {
                if (!isnan(sx)) { const KpVbiDev v = *p.vbi; bpos = icp_nearest_vbi(v, sx, sy, sz, p.r2, p.slack, prev); }
            } else if (!isnan(sx) && g.dim[0] > 0) bpos = icp_nearest(g, sx, sy, sz, p.r2, p.slack, prev);
        }
        icp_tile_terms<MODE>(p, tpts, i, sx, sy, sz, bpos, sh, lane, warp);
        __syncthreads();
        if (tid < ICP_NV) {
            double s = 0;
            for (int w = 0; w < W; ++w) s += sh[w][tid];
            p.slots[(size_t)blockIdx.x * ICP_NV + tid] = s;
        }
    } else {
        constexpr int NPC = TPC * ICP_THREADS;
        __shared__ double s_x[NPC], s_y[NPC], s_z[NPC];
        __shared__ int s_prev[NPC], s_bpos[NPC], s_queue[NPC], s_wn[TPC * W];
        if (st->done) return;
        pass = st->pass;
        const double *U = st->U;
        // 1. update every point; the list decides what it can, the rest is marked pending
#pragma unroll 1
        for (int h = 0; h < TPC; ++h) {
            const int i = (blockIdx.x * TPC + h) * ICP_THREADS + tid, slot = h * ICP_THREADS + tid;
            double sx = 0.0, sy = 0.0, sz = 0.0;
            int prev = -1, bpos = -1;
            bool listed = false;
            if (i < p.ns) {
                sx = p.cur[3 * (int64_t)i]; sy = p.cur[3 * (int64_t)i + 1]; sz = p.cur[3 * (int64_t)i + 2];
                if (pass > 0) {
                    prev = p.corr[i];
                    const double x2 = kp_affine(U[0], U[1], U[2], U[3], sx, sy, sz);
                    const double y2 = kp_affine(U[4], U[5], U[6], U[7], sx, sy, sz);
                    const double z2 = kp_affine(U[8], U[9], U[10], U[11], sx, sy, sz);
                    sx = x2; sy = y2; sz = z2;
                    p.cur[3 * (int64_t)i] = sx; p.cur[3 * (int64_t)i + 1] = sy; p.cur[3 * (int64_t)i + 2] = sz;
                }
                if (!isnan(sx) && (use_vbi || g.dim[0] > 0)) {
                    bpos = ICP_PENDING;
                    if (p.tlist && prev >= 0) {
                        const float4 t = __ldg(g.pts + prev);
                        const float rho2 = __ldg(p.trho + prev);
                        const double d2t = kp_d2(sx, sy, sz, (double)t.x, (double)t.y, (double)t.z);
                        // 4 d2t (1 + 1e-6), rounded up: the 1e-6 covers the rounding of the distances and of rho2 (DESIGN §3)
                        const float stop = __double2float_ru(4.0 * d2t * (1.0 + 1e-6));
                        if (d2t < p.r2 && stop < rho2) {
                            bpos = icp_nearest_list(g, reinterpret_cast<const int4 *>(p.tlist), sx, sy, sz, p.r2, p.slack, prev, d2t, __float_as_int(t.w), stop);
                            listed = true;
                        }
                    }
                }
            }
            s_x[slot] = sx; s_y[slot] = sy; s_z[slot] = sz; s_prev[slot] = prev; s_bpos[slot] = bpos;
            const unsigned need = __ballot_sync(KP_FULL, bpos == ICP_PENDING);
            if (lane == 0) s_wn[h * W + warp] = __popc(need);
            if (p.tally) {
                const unsigned nl = __ballot_sync(KP_FULL, listed);
                if (lane == 0) { atomicAdd(p.tally + 2 * pass, __popc(nl)); atomicAdd(p.tally + 2 * pass + 1, __popc(need)); }
            }
        }
        __syncthreads();
        // 2. the pending points into the queue, in slot order
        int nq = 0;
#pragma unroll
        for (int w = 0; w < TPC * W; ++w) nq += s_wn[w];
#pragma unroll 1
        for (int h = 0; h < TPC; ++h) {
            const int slot = h * ICP_THREADS + tid;
            const bool pend = s_bpos[slot] == ICP_PENDING;
            const unsigned need = __ballot_sync(KP_FULL, pend);
            int base = 0;
            for (int w = 0; w < h * W + warp; ++w) base += s_wn[w];
            if (pend) s_queue[base + __popc(need & ((1u << lane) - 1u))] = slot;
        }
        __syncthreads();
        // 3. the grid searches, one per thread in turn
        for (int j = tid; j < nq; j += ICP_THREADS) {
            const int o = s_queue[j];
            if (use_vbi) { const KpVbiDev v = *p.vbi; s_bpos[o] = icp_nearest_vbi(v, s_x[o], s_y[o], s_z[o], p.r2, p.slack, s_prev[o]); }
            else s_bpos[o] = icp_nearest(g, s_x[o], s_y[o], s_z[o], p.r2, p.slack, s_prev[o]);
        }
        __syncthreads();
        // 4. per tile: the terms of the thread's own point, the tile's slot row
#pragma unroll 1
        for (int h = 0; h < TPC; ++h) {
            const int tile = blockIdx.x * TPC + h, slot = h * ICP_THREADS + tid;
            icp_tile_terms<MODE>(p, tpts, tile * ICP_THREADS + tid, s_x[slot], s_y[slot], s_z[slot], s_bpos[slot], sh, lane, warp);
            __syncthreads();
            if (tid < ICP_NV && (unsigned)tile < ntiles) {
                double s = 0;
                for (int w = 0; w < W; ++w) s += sh[w][tid];
                p.slots[(size_t)tile * ICP_NV + tid] = s;
            }
            if (h + 1 < TPC) __syncthreads();          // sh is written again by the next tile
        }
    }
    // ---- two-level hand-over.  Tiles form groups of ICP_GROUP consecutive slot rows; the last CTA of a group to
    // finish (group ticket) folds the group's slot rows into one group row, then takes the global ticket; the last
    // group folds the group rows.  Each fold is one round of loads (a row per warp-slot, fixed order), instead of
    // one CTA walking ~2000 rows; the tickets see ICP_GROUP / TPC and gridDim/ICP_GROUP atomics per address instead of
    // gridDim.  Fixed tree -> the sums do not depend on which CTA does the folding.
    // (the CTAs that own source points: a batched launch is sized for the capacity and the rest left at once)
    constexpr unsigned CG = ICP_GROUP / TPC;           // CTAs per group
    const unsigned nact = (ntiles + TPC - 1) / TPC;
    const unsigned group = blockIdx.x / CG, ngroups = (nact + CG - 1) / CG;
    const unsigned gsize = min(CG, nact - group * CG);
    const unsigned t0 = group * ICP_GROUP, grows = min((unsigned)ICP_GROUP, ntiles - t0);
    auto fold = [&](const double *rows, unsigned nrows, double *dst_sh) {
        // warp w adds rows w, w + W, ... (all its loads in flight together), then the W partial sums in order
        double sacc = 0;
        if (lane < ICP_NV) {
            unsigned r = warp;
            for (; r + 3 * W < nrows; r += 4 * W) {
                double t[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) t[u] = __ldcg(rows + (size_t)(r + u * W) * ICP_NV + lane);
#pragma unroll
                for (int u = 0; u < 4; ++u) sacc += t[u];
            }
            for (; r < nrows; r += W) sacc += __ldcg(rows + (size_t)r * ICP_NV + lane);
        }
        part[warp][lane] = sacc;
        __syncthreads();
        if (tid < ICP_NV) {
            double t = 0;
            for (int w = 0; w < W; ++w) t += part[w][tid];
            dst_sh[tid] = t;
        }
        __syncthreads();
    };
    __threadfence();
    __syncthreads();
    if (tid == 0) s_ticket = atomicAdd(&p.gticket[group], 1u);
    __syncthreads();
    if (s_ticket != gsize - 1) return;
    __threadfence();
    fold(p.slots + (size_t)t0 * ICP_NV, grows, tot);
    if (tid < ICP_NV) p.gslots[(size_t)group * ICP_NV + tid] = tot[tid];
    if (tid == 0) p.gticket[group] = 0;             // re-armed for the next pass
    __threadfence();
    __syncthreads();
    if (tid == 0) s_ticket = atomicAdd(&st->ticket, 1u);
    __syncthreads();
    if (s_ticket != ngroups - 1) return;
    __threadfence();
    fold(p.gslots, ngroups, tot);
    __syncthreads();
    icp_finish(p, st, tot, pass, tid);
}
template <int MODE>
__global__ void __launch_bounds__(ICP_THREADS, ICP_MIN_CTAS) k_icp_iter(const __grid_constant__ IcpParams p)
{
    icp_iter_body<MODE>(p);
}
#ifndef ICP_B_CTAS
#define ICP_B_CTAS 3   // resident CTAs per SM the batched pass is compiled for (measured: 2 -> 2.71, 3 -> 2.15, 4 -> 2.02 ms alone but no gain for the frame)
#endif
template <int MODE>
__global__ void __launch_bounds__(ICP_THREADS, ICP_B_CTAS) k_icp_iter_b(const IcpParams *pp)
{
    // CTAs beyond the pair's source count, and every CTA of a converged pair, leave before touching anything else
    const IcpParams *me = pp + blockIdx.y;
    const int ns = *me->ns_dev;
    if (blockIdx.x * (ICP_B_TILES * ICP_THREADS) >= (unsigned)max(ns, 1) || me->st->done) return;
    const IcpParams p = icp_params_batched(pp);      // thread-local copy: the loops read registers, not shared memory
    icp_iter_body<MODE, true>(p);
}
// batched init: moving source = init * src, state reset, slack from the device-side grid
__global__ void __launch_bounds__(256) k_icp_init_b(const IcpParams *pp)
{
    const IcpParams *p = pp + blockIdx.y;
    const int ns = *p->ns_dev;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        IcpState init;
        memset(&init, 0, sizeof init);
        for (int i = 0; i < 16; ++i) { init.T[i] = p->init_T[i]; init.U[i] = (i % 5 == 0) ? 1.0 : 0.0; }
        if (p->vbi && p->vbi->ok) {
            // the same bound from the index's extent (the grid is empty when the index took the cloud)
            const KpVbiDev &v = *p->vbi;
            double M = 0.0;
            for (int c = 0; c < 3; ++c)
                M = fmax(M, fmax(fabs(v.minb[c]), fabs(v.minb[c] + v.voxel * (double)v.nvox[c])) + 2.0 * p->max_corr);
            const double eps = 8.0 * M / 16777216.0;
            init.slack = eps * (2.0 * p->max_corr + eps) * 1.000001 + 4e-6 * (p->max_corr * p->max_corr);
        } else init.slack = icp_slack(*p->gdev, p->max_corr);
        *p->st = init;
    }
    const double *T = p->init_T;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += gridDim.x * blockDim.x) {
        const double X = p->src[3 * (int64_t)i], Y = p->src[3 * (int64_t)i + 1], Z = p->src[3 * (int64_t)i + 2];
        p->cur[3 * (int64_t)i] = kp_affine(T[0], T[1], T[2], T[3], X, Y, Z);
        p->cur[3 * (int64_t)i + 1] = kp_affine(T[4], T[5], T[6], T[7], X, Y, Z);
        p->cur[3 * (int64_t)i + 2] = kp_affine(T[8], T[9], T[10], T[11], X, Y, Z);
    }
}
__global__ void k_icp_results_b(const IcpParams *pp, int npairs)
{
    // one thread per pair: the converged state into the frame's result rows
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npairs) return;
    const IcpParams &p = pp[i];
    const IcpState *st = p.st;
    for (int e = 0; e < 16; ++e) p.res_T[e] = st->T[e];
    *p.res_fit = st->fitness; *p.res_rmse = st->rmse; *p.res_iters = st->iters;
}
}  // namespace

// ---------------------------------------------------------------- frame engine: batched point-to-plane ICP
int kp_icp_batch_create(kp_ctx *ctx, const KpIcpPairDesc *pairs, int npairs, int64_t cap_src, double max_corr, int max_iter,
                        double rel_fitness, double rel_rmse, KpIcpBatch *out)
{
    out->npairs = npairs; out->max_iter = max_iter < 0 ? 0 : max_iter; out->cap_src = cap_src;
    const int grid = (int)kp_blocks(cap_src > 0 ? cap_src : 1, ICP_THREADS);
    const int ngroups = (grid + ICP_GROUP - 1) / ICP_GROUP;
    out->grid = grid;
    const size_t per_pair = (size_t)cap_src * 3 * sizeof(double) + (size_t)cap_src * sizeof(int32_t) + (size_t)grid * ICP_NV * sizeof(double) +
                            (size_t)ngroups * ICP_NV * sizeof(double) + (size_t)ngroups * sizeof(unsigned int) + sizeof(IcpState) + 1024;
    KP_CUDA(ctx, cudaMalloc(&out->d_work, per_pair * (size_t)npairs));
    KP_CUDA(ctx, cudaMemset(out->d_work, 0, per_pair * (size_t)npairs));
    if (getenv("KP_DEBUG_ICP")) {
        // tally of the list-decided and the grid-searched points per pass, summed over every run; printed at destroy
        const size_t bytes = sizeof(int32_t) * 2 * (size_t)(out->max_iter + 1) * (size_t)npairs;
        KP_CUDA(ctx, cudaMalloc(&out->d_tally, bytes));
        KP_CUDA(ctx, cudaMemset(out->d_tally, 0, bytes));
    }
    std::vector<IcpParams> h((size_t)npairs);
    char *w = (char *)out->d_work;
    auto take = [&](size_t bytes) { char *r = w; w += (bytes + 255) & ~(size_t)255; return r; };
    for (int i = 0; i < npairs; ++i) {
        IcpParams p;
        memset(&p, 0, sizeof p);
        p.tgt_normals = pairs[i].tgt_normals; p.mode = ICP_PLANE;
        p.sqrt_lg = 1.0; p.sqrt_lp = 0.0;
        p.cur = (double *)take((size_t)cap_src * 3 * sizeof(double));
        p.corr = (int32_t *)take((size_t)cap_src * sizeof(int32_t));
        p.slots = (double *)take((size_t)grid * ICP_NV * sizeof(double));
        p.gslots = (double *)take((size_t)ngroups * ICP_NV * sizeof(double));
        p.gticket = (unsigned int *)take((size_t)ngroups * sizeof(unsigned int));
        p.st = (IcpState *)take(sizeof(IcpState));
        p.r2 = max_corr * max_corr; p.max_corr = max_corr;
        p.max_iter = out->max_iter; p.rel_fit = rel_fitness; p.rel_rmse = rel_rmse;
        p.gdev = pairs[i].tgt_grid; p.ns_dev = pairs[i].n_src; p.src = pairs[i].src; p.vbi = pairs[i].tgt_vbi;
        p.tlist = pairs[i].tgt_list; p.trho = pairs[i].tgt_rho;
        p.tally = out->d_tally ? out->d_tally + (size_t)i * 2 * (out->max_iter + 1) : nullptr;
        for (int e = 0; e < 16; ++e) p.init_T[e] = pairs[i].init_T[e];
        p.res_T = pairs[i].res_T; p.res_fit = pairs[i].res_fit; p.res_rmse = pairs[i].res_rmse; p.res_iters = pairs[i].res_iters;
        h[i] = p;
    }
    KP_CUDA(ctx, cudaMalloc(&out->d_params, sizeof(IcpParams) * h.size()));
    KP_CUDA(ctx, cudaMemcpy(out->d_params, h.data(), sizeof(IcpParams) * h.size(), cudaMemcpyHostToDevice));
    return KP_OK;
}
void kp_icp_batch_destroy(KpIcpBatch *b)
{
    if (!b) return;
    if (b->d_tally) {
        const int np = b->max_iter + 1;
        std::vector<int32_t> t((size_t)2 * np * b->npairs);
        if (cudaMemcpy(t.data(), b->d_tally, sizeof(int32_t) * t.size(), cudaMemcpyDeviceToHost) == cudaSuccess)
            for (int i = 0; i < b->npairs; ++i)
                for (int k = 0; k < np; ++k) {
                    const int32_t *r = t.data() + ((size_t)i * np + k) * 2;
                    if (r[0] || r[1]) fprintf(stderr, "[kp icp] pair %d pass %d list %d grid %d\n", i, k, r[0], r[1]);
                }
        cudaFree(b->d_tally);
        b->d_tally = nullptr;
    }
    if (b->d_params) cudaFree(b->d_params);
    if (b->d_work) cudaFree(b->d_work);
    b->d_params = b->d_work = nullptr;
}
int kp_icp_batch_run(kp_ctx *ctx, const KpIcpBatch &b)
{
    KpProfScope prof_scope__(ctx, "icp");
    const IcpParams *pp = (const IcpParams *)b.d_params;
    int64_t gi = (b.cap_src + 255) / 256;
    if (gi > (int64_t)ctx->sm_count * 8) gi = (int64_t)ctx->sm_count * 8;
    k_icp_init_b<<<dim3((unsigned)(gi > 0 ? gi : 1), (unsigned)b.npairs), 256, 0, ctx->stream>>>(pp);
    KP_LAUNCH_CHECK(ctx);
    for (int i = 0; i <= b.max_iter; ++i) {
        k_icp_iter_b<ICP_PLANE><<<dim3((unsigned)((b.grid + ICP_B_TILES - 1) / ICP_B_TILES), (unsigned)b.npairs), ICP_THREADS, 0, ctx->stream>>>(pp);
        KP_LAUNCH_CHECK(ctx);
    }
    k_icp_results_b<<<kp_blocks(b.npairs, 64), 64, 0, ctx->stream>>>(pp, b.npairs);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}


// internal form: the target grid is built by the caller (pipeline reuses it for both subs)
namespace {
__global__ void __launch_bounds__(256) k_intensity(const float *colors, int64_t n, const int32_t *order, float *out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t j = order ? order[i] : i;
    // (r + g + b) / 3 in double on the float32-stored colours, rounded once
    out[i] = (float)((((double)colors[3 * j] + (double)colors[3 * j + 1]) + (double)colors[3 * j + 2]) / 3.0);
}

// InitializePointCloudForColoredICP: per target point, least-squares colour gradient in the tangent plane over
// its hybrid neighbourhood (rows: projected neighbour offsets -> intensity differences, plus the
// orthogonality row (nn - 1) n -> 0); fewer than 4 neighbours -> zero gradient.
__global__ void __launch_bounds__(128) k_color_gradient(const float *xyz, const float *inten, const float *nrm, int64_t n,
                                                        const int32_t *idx, const int32_t *cnt, int k, float *grad)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int nn = cnt[i];
    double x[3] = {0, 0, 0};
    if (nn >= 4 && !isnan(xyz[3 * i])) {
        const double vx = xyz[3 * i], vy = xyz[3 * i + 1], vz = xyz[3 * i + 2];
        const double nx = nrm[3 * i], ny = nrm[3 * i + 1], nz = nrm[3 * i + 2];
        const double it = inten[i];
        double A[6] = {0, 0, 0, 0, 0, 0}, b[3] = {0, 0, 0};   // AtA (xx xy xz yy yz zz), Atb
        for (int t = 1; t < nn; ++t) {
            const int64_t j = idx[i * k + t];
            const double ax = (double)xyz[3 * j] - vx, ay = (double)xyz[3 * j + 1] - vy, az = (double)xyz[3 * j + 2] - vz;
            const double dn = (ax * nx + ay * ny) + az * nz;
            const double px = ax - dn * nx, py = ay - dn * ny, pz = az - dn * nz;
            const double di = (double)inten[j] - it;
            A[0] += px * px; A[1] += px * py; A[2] += px * pz; A[3] += py * py; A[4] += py * pz; A[5] += pz * pz;
            b[0] += px * di; b[1] += py * di; b[2] += pz * di;
        }
        const double w = (double)(nn - 1);
        A[0] += w * nx * w * nx; A[1] += w * nx * w * ny; A[2] += w * nx * w * nz;
        A[3] += w * ny * w * ny; A[4] += w * ny * w * nz; A[5] += w * nz * w * nz;
        // 3x3 symmetric solve (Gaussian elimination with partial pivoting)
        double M[3][4] = {{A[0], A[1], A[2], b[0]}, {A[1], A[3], A[4], b[1]}, {A[2], A[4], A[5], b[2]}};
        bool ok = true;
        for (int c = 0; c < 3 && ok; ++c) {
            int pv = c;
            for (int r2 = c + 1; r2 < 3; ++r2) if (fabs(M[r2][c]) > fabs(M[pv][c])) pv = r2;
            if (!(fabs(M[pv][c]) > 1e-300)) { ok = false; break; }
            if (pv != c) for (int j = 0; j < 4; ++j) { const double tv = M[c][j]; M[c][j] = M[pv][j]; M[pv][j] = tv; }
            for (int r2 = c + 1; r2 < 3; ++r2) { const double f = M[r2][c] / M[c][c]; for (int j = c; j < 4; ++j) M[r2][j] -= f * M[c][j]; }
        }
        if (ok) {
            x[2] = M[2][3] / M[2][2];
            x[1] = (M[1][3] - M[1][2] * x[2]) / M[1][1];
            x[0] = (M[0][3] - M[0][1] * x[1] - M[0][2] * x[2]) / M[0][0];
            if (!(isfinite(x[0]) && isfinite(x[1]) && isfinite(x[2]))) x[0] = x[1] = x[2] = 0.0;
        }
    }
    grad[3 * i] = (float)x[0]; grad[3 * i + 1] = (float)x[1]; grad[3 * i + 2] = (float)x[2];
}
}  // namespace

int kp_color_gradient_device(kp_ctx *ctx, const float *d_xyz, const float *d_colors, const float *d_normals, int64_t n,
                             double radius, int max_nn, float *d_intensity, float *d_grad)
{
    if (n <= 0) return KP_OK;
    if (max_nn < 1 || !(radius > 0.0)) return kp_set_err(ctx, KP_E_ARG, "colour gradient: radius <= 0 or max_nn < 1");
    k_intensity<<<kp_blocks(n, 256), 256, 0, ctx->stream>>>(d_colors, n, nullptr, d_intensity);
    KP_LAUNCH_CHECK(ctx);
    KpGrid g;
    KP_TRY(kp_grid_build_knn(ctx, d_xyz, n, radius * (1.0 + 4e-6), max_nn, nullptr, &g));
    int32_t *idx, *cnt;
    KP_TRY(kp_ws(ctx, (size_t)n * (size_t)max_nn, &idx));
    KP_TRY(kp_ws(ctx, (size_t)n, &cnt));
    KP_TRY(kp_knn_device(ctx, g, nullptr, n, max_nn, radius, idx, nullptr, cnt, nullptr, d_xyz));
    KP_PROFB(ctx, "color_gradient", (double)n * (4.0 * max_nn + 12.0 + 12.0 + 4.0 + 12.0));
    k_color_gradient<<<kp_blocks(n, 128), 128, 0, ctx->stream>>>(d_xyz, d_intensity, d_normals, n, idx, cnt, max_nn, d_grad);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}

int kp_icp_device(kp_ctx *ctx, const float *d_src, int64_t n_src, const KpGrid &tgt_grid, const float *d_tgt_normals,
                  double max_corr, const double *h_init16, int max_iter, double rel_fitness, double rel_rmse,
                  double *h_T_out, double *h_fitness, double *h_rmse, int *h_iters, int64_t *h_ncorr, const KpIcpExtra *extra)
{
    if (n_src > 2147483000LL) return kp_set_err(ctx, KP_E_ARG, "more than 2^31 points in one call");
    if (max_iter < 0) max_iter = 0;
    KpProfScope prof_scope__(ctx, "icp");
    IcpParams p;
    memset(&p, 0, sizeof p);
    p.g = kp_grid_dev(tgt_grid);
    if (tgt_grid.n <= 0) p.g.dim[0] = p.g.dim[1] = p.g.dim[2] = 0;
    p.tgt_normals = d_tgt_normals;
    p.mode = extra ? extra->mode : ICP_PLANE;
    p.src_int = nullptr; p.tgt_int = extra ? extra->tgt_intensity : nullptr; p.tgt_grad = extra ? extra->tgt_grad : nullptr;
    const double lg = extra ? extra->lambda_geometric : 1.0;
    p.sqrt_lg = sqrt(lg); p.sqrt_lp = sqrt(1.0 - lg);
    p.ns = (int)n_src;
    p.r2 = max_corr * max_corr;
    {
        // fp32 rounding of a coordinate of magnitude <= M costs <= M * 2^-24 per operand; 8 x that covers the
        // three axes, both operands and the fp32 arithmetic with room to spare
        double M = 0.0;
        for (int c = 0; c < 3; ++c)
            M = fmax(M, fmax(fabs(p.g.org[c]), fabs(p.g.org[c] + p.g.cell * (double)p.g.dim[c])) + 2.0 * max_corr);
        const double eps = 8.0 * M / 16777216.0;          // bound on |sqrt(fp32 d2) - sqrt(d2)|
        p.slack = eps * (2.0 * max_corr + eps) * 1.000001 + 4e-6 * p.r2;
    }
    p.max_iter = max_iter;
    p.rel_fit = rel_fitness; p.rel_rmse = rel_rmse;
    const int grid = (int)kp_blocks(n_src > 0 ? n_src : 1, ICP_THREADS);
    KP_TRY(kp_ws(ctx, (size_t)(n_src > 0 ? n_src : 1) * 3, &p.cur));
    KP_TRY(kp_ws(ctx, (size_t)(n_src > 0 ? n_src : 1), &p.corr));
    KP_TRY(kp_ws(ctx, (size_t)grid * ICP_NV, &p.slots));
    const int ngroups = (grid + ICP_GROUP - 1) / ICP_GROUP;
    KP_TRY(kp_ws(ctx, (size_t)ngroups * ICP_NV, &p.gslots));
    KP_TRY(kp_ws(ctx, (size_t)ngroups, &p.gticket));
    KP_CUDA(ctx, cudaMemsetAsync(p.gticket, 0, sizeof(unsigned int) * (size_t)ngroups, ctx->stream));
    KP_TRY(kp_ws(ctx, 1, &p.st));
    IcpState init;
    memset(&init, 0, sizeof init);
    for (int i = 0; i < 16; ++i) { init.T[i] = h_init16[i]; init.U[i] = (i % 5 == 0) ? 1.0 : 0.0; }
    {
        // moving source = init * src.  (Re-ordering the source by target-grid cell was measured: the voxel order the
        // source arrives in is already coherent, and the extra sort cost more than the lookups it saved.)
        const size_t nn = (size_t)(n_src > 0 ? n_src : 1);
        k_icp_init<<<kp_blocks(nn, 256), 256, 0, ctx->stream>>>(d_src, (int)n_src, p, init, p.cur);
        KP_LAUNCH_CHECK(ctx);
        if (p.mode == ICP_COLORED && n_src > 0) {
            float *si;
            KP_TRY(kp_ws(ctx, nn, &si));
            k_intensity<<<kp_blocks(nn, 256), 256, 0, ctx->stream>>>(extra->src_colors, n_src, nullptr, si);
            KP_LAUNCH_CHECK(ctx);
            p.src_int = si;
        }
    }
    // Passes are identical launches (the pass number lives in the device state), enqueued without reading anything
    // back; a pass launched after `done` returns at once but still costs a launch slot (~3.5 us).  So the first
    // batch is sized from the previous call on this context (consecutive frames converge alike) and the state is
    // fetched once after it; only a call that needs more passes than expected pays a second round trip.
    const IcpState *hs = (const IcpState *)ctx->h_scratch;
    int launched = 0;
    int batch = ctx->icp_passes_hint > 0 ? ctx->icp_passes_hint + 2 : 16;
    for (;;) {
        if (batch > max_iter + 1 - launched) batch = max_iter + 1 - launched;
        for (int i = 0; i < batch; ++i) {
            if (p.mode == ICP_POINT) k_icp_iter<ICP_POINT><<<grid, ICP_THREADS, 0, ctx->stream>>>(p);
            else if (p.mode == ICP_COLORED) k_icp_iter<ICP_COLORED><<<grid, ICP_THREADS, 0, ctx->stream>>>(p);
            else k_icp_iter<ICP_PLANE><<<grid, ICP_THREADS, 0, ctx->stream>>>(p);
            KP_LAUNCH_CHECK(ctx);
        }
        launched += batch;
        KP_CUDA(ctx, cudaMemcpyAsync(ctx->d_scratch, p.st, sizeof(IcpState), cudaMemcpyDeviceToDevice, ctx->stream));
        KP_TRY(kp_fetch_scratch(ctx, sizeof(IcpState)));
        if (hs->done || launched > max_iter) break;
        batch = 6;
    }
    ctx->icp_passes_hint = hs->pass;        // passes executed
    // per executed pass: moving source read + write-back (48 B) and, per match, target point + normal (28 B)
    prof_scope__.add_bytes((double)(hs->iters + 1) * 76.0 * (double)n_src);
    if (h_T_out) memcpy(h_T_out, hs->T, sizeof(double) * 16);
    if (h_fitness) *h_fitness = hs->fitness;
    if (h_rmse) *h_rmse = hs->rmse;
    if (h_iters) *h_iters = hs->iters;
    if (h_ncorr) *h_ncorr = hs->ncorr;
    return KP_OK;
}

extern "C" {

int kp_icp_point_to_plane(kp_ctx *ctx, const float *d_src, int64_t n_src, const float *d_tgt,
                          const float *d_tgt_normals, int64_t n_tgt, double max_corr, const double *h_init16,
                          int max_iter, double rel_fitness, double rel_rmse, double *h_T_out,
                          double *h_fitness, double *h_rmse, int *h_iters, int64_t *h_ncorr)
{
    if (!ctx || !h_init16) return kp_set_err(ctx, KP_E_ARG, "kp_icp_point_to_plane: NULL argument");
    if (!(max_corr > 0.0)) return kp_set_err(ctx, KP_E_ARG, "registration_icp: max_correspondence_distance <= 0");
    if (!d_tgt_normals) return kp_set_err(ctx, KP_E_ARG, "TransformationEstimationPointToPlane requires target normals");
    kp_enter(ctx);
    KpGrid g;
    KP_TRY(kp_grid_build(ctx, d_tgt, n_tgt, max_corr * (1.0 + 1e-6), nullptr, &g));
    return kp_icp_device(ctx, d_src, n_src, g, d_tgt_normals, max_corr, h_init16, max_iter, rel_fitness, rel_rmse, h_T_out,
                         h_fitness, h_rmse, h_iters, h_ncorr, nullptr);
}

int kp_icp_point_to_point(kp_ctx *ctx, const float *d_src, int64_t n_src, const float *d_tgt, int64_t n_tgt,
                          double max_corr, const double *h_init16, int max_iter, double rel_fitness, double rel_rmse,
                          double *h_T_out, double *h_fitness, double *h_rmse, int *h_iters, int64_t *h_ncorr)
{
    if (!ctx || !h_init16) return kp_set_err(ctx, KP_E_ARG, "kp_icp_point_to_point: NULL argument");
    if (!(max_corr > 0.0)) return kp_set_err(ctx, KP_E_ARG, "registration_icp: max_correspondence_distance <= 0");
    kp_enter(ctx);
    KpGrid g;
    KP_TRY(kp_grid_build(ctx, d_tgt, n_tgt, max_corr * (1.0 + 1e-6), nullptr, &g));
    KpIcpExtra ex;
    ex.mode = ICP_POINT;
    return kp_icp_device(ctx, d_src, n_src, g, nullptr, max_corr, h_init16, max_iter, rel_fitness, rel_rmse, h_T_out,
                         h_fitness, h_rmse, h_iters, h_ncorr, &ex);
}

int kp_color_gradient(kp_ctx *ctx, const float *d_xyz, const float *d_colors, const float *d_normals, int64_t n,
                      double radius, int max_nn, float *d_grad)
{
    if (!ctx || (n > 0 && (!d_xyz || !d_colors || !d_normals || !d_grad))) return kp_set_err(ctx, KP_E_ARG, "kp_color_gradient: NULL argument");
    kp_enter(ctx);
    float *inten;
    KP_TRY(kp_ws(ctx, (size_t)(n > 0 ? n : 1), &inten));
    return kp_color_gradient_device(ctx, d_xyz, d_colors, d_normals, n, radius, max_nn, inten, d_grad);
}

int kp_icp_colored(kp_ctx *ctx, const float *d_src, const float *d_src_colors, int64_t n_src, const float *d_tgt,
                   const float *d_tgt_colors, const float *d_tgt_normals, int64_t n_tgt, double max_corr,
                   double lambda_geometric, const double *h_init16, int max_iter, double rel_fitness, double rel_rmse,
                   double *h_T_out, double *h_fitness, double *h_rmse, int *h_iters, int64_t *h_ncorr)
{
    if (!ctx || !h_init16) return kp_set_err(ctx, KP_E_ARG, "kp_icp_colored: NULL argument");
    if (!(max_corr > 0.0)) return kp_set_err(ctx, KP_E_ARG, "registration_colored_icp: max_correspondence_distance <= 0");
    if (!d_tgt_normals || !d_tgt_colors || !d_src_colors)
        return kp_set_err(ctx, KP_E_ARG, "registration_colored_icp requires source colours and target colours + normals");
    if (!(lambda_geometric >= 0.0 && lambda_geometric <= 1.0)) return kp_set_err(ctx, KP_E_ARG, "lambda_geometric outside [0, 1]");
    kp_enter(ctx);
    float *inten, *grad;
    KP_TRY(kp_ws(ctx, (size_t)(n_tgt > 0 ? n_tgt : 1), &inten));
    KP_TRY(kp_ws(ctx, (size_t)(n_tgt > 0 ? n_tgt : 1) * 3, &grad));
    // InitializePointCloudForColoredICP(target, KDTreeSearchParamHybrid(2 * max_distance, 30))
    KP_TRY(kp_color_gradient_device(ctx, d_tgt, d_tgt_colors, d_tgt_normals, n_tgt, 2.0 * max_corr, 30, inten, grad));
    KpGrid g;
    KP_TRY(kp_grid_build(ctx, d_tgt, n_tgt, max_corr * (1.0 + 1e-6), nullptr, &g));
    KpIcpExtra ex;
    ex.mode = ICP_COLORED; ex.src_colors = d_src_colors; ex.tgt_intensity = inten; ex.tgt_grad = grad;
    ex.lambda_geometric = lambda_geometric;
    return kp_icp_device(ctx, d_src, n_src, g, d_tgt_normals, max_corr, h_init16, max_iter, rel_fitness, rel_rmse, h_T_out,
                         h_fitness, h_rmse, h_iters, h_ncorr, &ex);
}

}  // extern "C"
