// kp_ransac.cu -- K4: RANSAC plane segmentation with batched hypotheses, plus the floor-band and
// plane-side masks.  Replaces PointCloud.segment_plane at floor_removal.py:70, the band split at
// floor_removal.py:64-66 and pcd_above_plane at floor_removal.py:39-51  (SURVEY.md A.5).
//
// All H hypotheses are sampled (counter-based RNG), fitted and scored in one batch: the scoring
// kernel keeps a chunk of planes in shared memory, every thread holds four points in registers
// and walks the planes; inlier counts are warp ballots + popc accumulated per warp in shared
// memory (single writer, no atomics) and flushed once per CTA.  The sequential best / early-exit
// rule of Open3D is then replayed on the host over the H counts, which gives exactly the result of
// evaluating hypotheses one after the other.
#include <math.h>
#include <vector>
#include "kp_common.cuh"

namespace {
constexpr int RS_MAX_N = 64;     // ransac_n upper bound (reference uses 30, BASELINE 3)
constexpr int SCORE_THREADS = 256;
constexpr int SCORE_PTS = 4;
constexpr int SCORE_TILE = SCORE_THREADS * SCORE_PTS;
constexpr int SCORE_HC = 512;    // hypotheses per shared-memory chunk (16 KB planes + 16 KB counters)

#define DM(a, b) __dmul_rn((a), (b))
#define DA(a, b) __dadd_rn((a), (b))
#define DS(a, b) __dsub_rn((a), (b))
#define DD(a, b) __ddiv_rn((a), (b))

__global__ void __launch_bounds__(128) k_ransac_fit(const float *xyz, int n, int ransac_n, int iters, uint64_t seed,
                                                    double4 *planes, uint8_t *pvalid)
{
    int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= iters) return;
    int ids[RS_MAX_N];
    int got = 0;
    for (uint64_t j = 0; got < ransac_n; ++j) {
        int v = (int)(kp_rng(seed, (uint64_t)h, j) % (uint64_t)n);
        bool dup = false;
        for (int t = 0; t < got; ++t) dup |= ids[t] == v;
        if (!dup) ids[got++] = v;
    }
    double a, b, c, d;
    bool ok = true;
    if (ransac_n == 3) {
        const float *p0 = xyz + 3 * (int64_t)ids[0], *p1 = xyz + 3 * (int64_t)ids[1], *p2 = xyz + 3 * (int64_t)ids[2];
        double e1x = DS((double)p1[0], (double)p0[0]), e1y = DS((double)p1[1], (double)p0[1]), e1z = DS((double)p1[2], (double)p0[2]);
        double e2x = DS((double)p2[0], (double)p0[0]), e2y = DS((double)p2[1], (double)p0[1]), e2z = DS((double)p2[2], (double)p0[2]);
        a = DS(DM(e1y, e2z), DM(e1z, e2y));
        b = DS(DM(e1z, e2x), DM(e1x, e2z));
        c = DS(DM(e1x, e2y), DM(e1y, e2x));
        double nn = sqrt(DA(DA(DM(a, a), DM(b, b)), DM(c, c)));
        if (nn == 0.0 || isnan(nn)) ok = false;
        a = DD(a, nn); b = DD(b, nn); c = DD(c, nn);
        d = -DA(DA(DM(a, (double)p0[0]), DM(b, (double)p0[1])), DM(c, (double)p0[2]));
    } else {
        double cx = 0, cy = 0, cz = 0;
        for (int j = 0; j < ransac_n; ++j) {
            const float *p = xyz + 3 * (int64_t)ids[j];
            cx = DA(cx, (double)p[0]); cy = DA(cy, (double)p[1]); cz = DA(cz, (double)p[2]);
        }
        double m = (double)ransac_n;
        cx = DD(cx, m); cy = DD(cy, m); cz = DD(cz, m);
        double xx = 0, xy = 0, xz = 0, yy = 0, yz = 0, zz = 0;
        for (int j = 0; j < ransac_n; ++j) {
            const float *p = xyz + 3 * (int64_t)ids[j];
            double x = DS((double)p[0], cx), y = DS((double)p[1], cy), z = DS((double)p[2], cz);
            xx = DA(xx, DM(x, x)); xy = DA(xy, DM(x, y)); xz = DA(xz, DM(x, z));
            yy = DA(yy, DM(y, y)); yz = DA(yz, DM(y, z)); zz = DA(zz, DM(z, z));
        }
        double dx = DS(DM(yy, zz), DM(yz, yz)), dy = DS(DM(xx, zz), DM(xz, xz)), dz = DS(DM(xx, yy), DM(xy, xy));
        if (dx >= dy && dx >= dz) { a = dx; b = DS(DM(xz, yz), DM(xy, zz)); c = DS(DM(xy, yz), DM(xz, yy)); }
        else if (dy >= dx && dy >= dz) { a = DS(DM(xz, yz), DM(xy, zz)); b = dy; c = DS(DM(xy, xz), DM(yz, xx)); }
        else { a = DS(DM(xy, yz), DM(xz, yy)); b = DS(DM(xy, xz), DM(yz, xx)); c = dz; }
        double nn = sqrt(DA(DA(DM(a, a), DM(b, b)), DM(c, c)));
        if (nn == 0.0 || isnan(nn)) ok = false;
        a = DD(a, nn); b = DD(b, nn); c = DD(c, nn);
        d = -DA(DA(DM(a, cx), DM(b, cy)), DM(c, cz));
    }
    if (!ok) { a = b = c = 0.0; d = NAN; }   // NaN distance: nobody is an inlier
    planes[h] = make_double4(a, b, c, d);
    pvalid[h] = ok;
}

__device__ __forceinline__ double plane_dist(const double4 &pl, double x, double y, double z)
{
    return fabs(DA(DA(DA(DM(pl.x, x), DM(pl.y, y)), DM(pl.z, z)), pl.w));
}

__global__ void __launch_bounds__(SCORE_THREADS) k_ransac_score(const float *xyz, int n, const double4 *planes, int iters,
                                                                double thr, unsigned long long *g_cnt)
{
    __shared__ double4 pl_s[SCORE_HC];
    __shared__ int cnt_s[SCORE_THREADS / 32][SCORE_HC];   // one counter row per warp: single writer
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ntiles = (n + SCORE_TILE - 1) / SCORE_TILE;
    for (int h0 = 0; h0 < iters; h0 += SCORE_HC) {
        const int hc = min(SCORE_HC, iters - h0);
        for (int h = tid; h < hc; h += SCORE_THREADS) pl_s[h] = planes[h0 + h];
        for (int h = tid; h < (SCORE_THREADS / 32) * SCORE_HC; h += SCORE_THREADS) (&cnt_s[0][0])[h] = 0;
        __syncthreads();
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            double px[SCORE_PTS], py[SCORE_PTS], pz[SCORE_PTS];
#pragma unroll
            for (int j = 0; j < SCORE_PTS; ++j) {
                int64_t i = (int64_t)tile * SCORE_TILE + j * SCORE_THREADS + tid;
                if (i < n) { px[j] = (double)xyz[3 * i]; py[j] = (double)xyz[3 * i + 1]; pz[j] = (double)xyz[3 * i + 2]; }
                else { px[j] = py[j] = pz[j] = NAN; }
            }
            for (int h = 0; h < hc; ++h) {
                const double4 pl = pl_s[h];
                int c = 0;
#pragma unroll
                for (int j = 0; j < SCORE_PTS; ++j)
                    c += __popc(__ballot_sync(KP_FULL, plane_dist(pl, px[j], py[j], pz[j]) < thr));
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

// fixed-shape partial sums: per-thread sequential (grid-stride), warp butterfly, warps added in
// order by thread 0; one slot per block, summed in block order on the host -> run-to-run stable.
template <int NV>
__device__ __forceinline__ void block_slots(double (&v)[NV], double *slots)
{
    __shared__ double sh[32][NV];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int c = 0; c < NV; ++c) v[c] = kp_butterfly_sum(v[c]);
    if (lane == 0)
        for (int c = 0; c < NV; ++c) sh[warp][c] = v[c];
    __syncthreads();
    if (threadIdx.x < NV) {
        double s = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s = DA(s, sh[w][threadIdx.x]);
        slots[(size_t)blockIdx.x * NV + threadIdx.x] = s;
    }
}

__global__ void __launch_bounds__(256) k_plane_mask(const float *xyz, int n, double4 pl, double thr, uint8_t *mask, double *slots)
{
    // slots: [block][2] = {count, sum d^2}
    double v[2] = {0, 0};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double d = plane_dist(pl, (double)xyz[3 * i], (double)xyz[3 * i + 1], (double)xyz[3 * i + 2]);
        bool in = d < thr;
        if (mask) mask[i] = in;
        if (in) { v[0] += 1.0; v[1] = DA(v[1], DM(d, d)); }
    }
    block_slots<2>(v, slots);
}

__global__ void __launch_bounds__(256) k_masked_moments(const float *xyz, const uint8_t *mask, int n, double cx, double cy,
                                                        double cz, double *slots)
{
    // slots: [block][10] = {sum dx, dy, dz, xx, xy, xz, yy, yz, zz, count} with d = p - c
    double v[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (!mask[i]) continue;
        double x = DS((double)xyz[3 * i], cx), y = DS((double)xyz[3 * i + 1], cy), z = DS((double)xyz[3 * i + 2], cz);
        v[0] = DA(v[0], x); v[1] = DA(v[1], y); v[2] = DA(v[2], z);
        v[3] = DA(v[3], DM(x, x)); v[4] = DA(v[4], DM(x, y)); v[5] = DA(v[5], DM(x, z));
        v[6] = DA(v[6], DM(y, y)); v[7] = DA(v[7], DM(y, z)); v[8] = DA(v[8], DM(z, z));
        v[9] += 1.0;
    }
    block_slots<10>(v, slots);
}

__global__ void k_axis_max(const float *xyz, int64_t n, int axis, int32_t *enc)
{
    float m = -INFINITY;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float v = xyz[3 * i + axis];
        if (!isnan(xyz[3 * i])) m = fmaxf(m, v);
    }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) m = fmaxf(m, __shfl_xor_sync(KP_FULL, m, s));
    // one atomic per CTA, and only if it would raise the word (same-address atomics serialise at ~5 ns each)
    __shared__ float wm[32];
    if ((threadIdx.x & 31) == 0) wm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmaxf(m, wm[w]);
        const int o = kp_f2ord(m);
        if (o > *(volatile int32_t *)enc) atomicMax(enc, o);
    }
}
__global__ void k_axis_max_init(int32_t *enc) { *enc = kp_f2ord(-INFINITY); }
__global__ void k_band_mask(const float *xyz, int64_t n, int axis, double band, const int32_t *enc, uint8_t *lower)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double mx = (double)kp_ord2f(*enc);
    double lim = DS(mx, band);
    float v = xyz[3 * i + axis];
    lower[i] = !isnan(xyz[3 * i]) && (double)v >= lim;
}
__global__ void k_plane_side(const float *xyz, int64_t n, double a, double b, double c, double d, uint8_t *mask)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double v = DA(DA(DA(DM(a, (double)xyz[3 * i]), DM(b, (double)xyz[3 * i + 1])), DM(c, (double)xyz[3 * i + 2])), d);
    mask[i] = v < 0.0;
}

}  // namespace

// internal form (no workspace reset): used by the public entry and the frame pipeline
int kp_ransac_device(kp_ctx *ctx, const float *d_xyz, int64_t n, double thr, int ransac_n, int iters, double probability,
                     uint64_t seed, double *h_plane, uint8_t *d_inlier_mask, int64_t *h_ninliers, int32_t *h_best_iter,
                     int64_t *d_counts)
{
    if (ransac_n < 3 || n < ransac_n) return kp_set_err(ctx, KP_E_ARG, "segment_plane: ransac_n < 3 or fewer points than ransac_n");
    if (ransac_n > RS_MAX_N) return kp_set_err(ctx, KP_E_ARG, "segment_plane: ransac_n > %d not supported", RS_MAX_N);
    if (!(thr > 0.0) || iters < 1) return kp_set_err(ctx, KP_E_ARG, "segment_plane: bad threshold or iteration count");
    if (n > 2147483000LL) return kp_set_err(ctx, KP_E_ARG, "more than 2^31 points in one call");
    double4 *planes;
    uint8_t *pvalid;
    unsigned long long *cnt;
    double *slots;
    const int nblk = ctx->sm_count * 2;
    KP_TRY(kp_ws(ctx, (size_t)iters, &planes));
    KP_TRY(kp_ws(ctx, (size_t)iters, &pvalid));
    KP_TRY(kp_ws(ctx, (size_t)iters, &cnt));
    KP_TRY(kp_ws(ctx, (size_t)nblk * 10, &slots));
    {
        KP_PROFB(ctx, "ransac_fit", (double)iters * (ransac_n * 12.0 + 33.0));
        KP_CUDA(ctx, cudaMemsetAsync(cnt, 0, sizeof(unsigned long long) * (size_t)iters, ctx->stream));
        k_ransac_fit<<<kp_blocks(iters, 128), 128, 0, ctx->stream>>>(d_xyz, (int)n, ransac_n, iters, seed, planes, pvalid);
        KP_LAUNCH_CHECK(ctx);
    }
    {
        KP_PROFB(ctx, "ransac_score", (double)n * 12.0 + (double)iters * 40.0);
        int ntiles = (int)((n + SCORE_TILE - 1) / SCORE_TILE);
        int grid = ntiles < nblk ? ntiles : nblk;
        k_ransac_score<<<grid, SCORE_THREADS, 0, ctx->stream>>>(d_xyz, (int)n, planes, iters, thr, cnt);
        KP_LAUNCH_CHECK(ctx);
    }
    std::vector<unsigned long long> h_cnt(iters);
    std::vector<double4> h_planes(iters);
    std::vector<uint8_t> h_valid(iters);
    KP_CUDA(ctx, cudaMemcpyAsync(h_cnt.data(), cnt, sizeof(unsigned long long) * iters, cudaMemcpyDeviceToHost, ctx->stream));
    KP_CUDA(ctx, cudaMemcpyAsync(h_planes.data(), planes, sizeof(double4) * iters, cudaMemcpyDeviceToHost, ctx->stream));
    KP_CUDA(ctx, cudaMemcpyAsync(h_valid.data(), pvalid, (size_t)iters, cudaMemcpyDeviceToHost, ctx->stream));
    if (d_counts) KP_CUDA(ctx, cudaMemcpyAsync(d_counts, cnt, sizeof(int64_t) * iters, cudaMemcpyDeviceToDevice, ctx->stream));
    KP_TRY(kp_stream_wait(ctx));

    // sum of squared inlier distances, needed only when two hypotheses tie on the inlier count
    std::vector<double> sq(iters, -1.0);
    auto sumsq = [&](int h) -> int {
        if (sq[h] >= 0) return KP_OK;
        k_plane_mask<<<nblk, 256, 0, ctx->stream>>>(d_xyz, (int)n, h_planes[h], thr, nullptr, slots);
        KP_LAUNCH_CHECK(ctx);
        std::vector<double> hs((size_t)nblk * 2);
        KP_CUDA(ctx, cudaMemcpyAsync(hs.data(), slots, sizeof(double) * hs.size(), cudaMemcpyDeviceToHost, ctx->stream));
        KP_TRY(kp_stream_wait(ctx));
        double s = 0;
        for (int b = 0; b < nblk; ++b) s += hs[2 * b + 1];
        sq[h] = s;
        return KP_OK;
    };
    // sequential replay of Open3D's best / early-exit rule (oracle: kpo_ransac_plane)
    int best = -1;
    double best_fit = 0, best_rmse = 0;
    double break_it = (double)iters;
    long done = 0;
    for (int h = 0; h < iters; ++h) {
        if ((double)done > break_it) continue;
        if (!h_valid[h]) continue;                // degenerate sample: skipped, not counted
        {
            double fit = (double)h_cnt[h] / (double)n;
            bool better = fit > best_fit;
            if (!better && fit == best_fit && best >= 0) {
                KP_TRY(sumsq(h));
                KP_TRY(sumsq(best));
                double rm = h_cnt[h] ? sq[h] / sqrt((double)h_cnt[h]) : 0.0;
                best_rmse = h_cnt[best] ? sq[best] / sqrt((double)h_cnt[best]) : 0.0;
                better = rm < best_rmse;
            }
            if (better) {
                best = h; best_fit = fit;
                if (fit < 1.0) {
                    double b = log(1.0 - probability) / log(1.0 - pow(fit, (double)ransac_n));
                    break_it = b < (double)iters ? b : (double)iters;
                } else break_it = 0;
            }
        }
        ++done;
    }
    if (h_best_iter) *h_best_iter = best;
    if (best < 0) {
        if (d_inlier_mask) KP_CUDA(ctx, cudaMemsetAsync(d_inlier_mask, 0, (size_t)n, ctx->stream));
        if (h_plane) h_plane[0] = h_plane[1] = h_plane[2] = h_plane[3] = 0.0;
        if (h_ninliers) *h_ninliers = 0;
        return KP_OK;
    }
    KP_PROFB(ctx, "ransac_refit", (double)n * (13.0 + 2.0 * 13.0));
    uint8_t *mask = d_inlier_mask;
    if (!mask) KP_TRY(kp_ws(ctx, (size_t)n, &mask));
    k_plane_mask<<<nblk, 256, 0, ctx->stream>>>(d_xyz, (int)n, h_planes[best], thr, mask, slots);
    KP_LAUNCH_CHECK(ctx);
    std::vector<double> hs((size_t)nblk * 10);
    KP_CUDA(ctx, cudaMemcpyAsync(hs.data(), slots, sizeof(double) * nblk * 2, cudaMemcpyDeviceToHost, ctx->stream));
    KP_TRY(kp_stream_wait(ctx));
    double ninl = 0;
    for (int b = 0; b < nblk; ++b) ninl += hs[2 * b];
    if (h_ninliers) *h_ninliers = (int64_t)ninl;
    double pl[4] = {h_planes[best].x, h_planes[best].y, h_planes[best].z, h_planes[best].w};
    if (ninl >= 1) {
        // refit on the final inliers (covariance fit, two passes: centroid, centred moments)
        k_masked_moments<<<nblk, 256, 0, ctx->stream>>>(d_xyz, mask, (int)n, 0.0, 0.0, 0.0, slots);
        KP_LAUNCH_CHECK(ctx);
        KP_CUDA(ctx, cudaMemcpyAsync(hs.data(), slots, sizeof(double) * nblk * 10, cudaMemcpyDeviceToHost, ctx->stream));
        KP_TRY(kp_stream_wait(ctx));
        double c3[3] = {0, 0, 0};
        for (int b = 0; b < nblk; ++b) for (int c = 0; c < 3; ++c) c3[c] += hs[10 * b + c];
        for (int c = 0; c < 3; ++c) c3[c] /= ninl;
        k_masked_moments<<<nblk, 256, 0, ctx->stream>>>(d_xyz, mask, (int)n, c3[0], c3[1], c3[2], slots);
        KP_LAUNCH_CHECK(ctx);
        KP_CUDA(ctx, cudaMemcpyAsync(hs.data(), slots, sizeof(double) * nblk * 10, cudaMemcpyDeviceToHost, ctx->stream));
        KP_TRY(kp_stream_wait(ctx));
        double m6[6] = {0, 0, 0, 0, 0, 0};
        for (int b = 0; b < nblk; ++b) for (int c = 0; c < 6; ++c) m6[c] += hs[10 * b + 3 + c];
        double rp[4];
        if (cov_fit_from_moments(m6, c3[0], c3[1], c3[2], rp)) { pl[0] = rp[0]; pl[1] = rp[1]; pl[2] = rp[2]; pl[3] = rp[3]; }
    }
    if (h_plane) { h_plane[0] = pl[0]; h_plane[1] = pl[1]; h_plane[2] = pl[2]; h_plane[3] = pl[3]; }
    return KP_OK;
}

int kp_band_mask_device(kp_ctx *ctx, const float *d_xyz, int64_t n, int axis, double band, uint8_t *d_lower,
                        double *h_axis_max, int64_t *h_nlower)
{
    if (axis < 0 || axis > 2) return kp_set_err(ctx, KP_E_ARG, "kp_band_mask: axis must be 0, 1 or 2");
    if (h_nlower) *h_nlower = 0;
    if (n <= 0) return KP_OK;
    KP_PROFB(ctx, "band_mask", (double)n * (12.0 + 12.0 + 2.0));
    int32_t *enc = (int32_t *)ctx->d_scratch;
    int32_t *d_tot = enc + 1;
    k_axis_max_init<<<1, 1, 0, ctx->stream>>>(enc);
    KP_LAUNCH_CHECK(ctx);
    unsigned nb = kp_blocks(n, 256 * 8);
    if (nb > (unsigned)ctx->sm_count * 8) nb = ctx->sm_count * 8;
    k_axis_max<<<nb, 256, 0, ctx->stream>>>(d_xyz, n, axis, enc);
    KP_LAUNCH_CHECK(ctx);
    k_band_mask<<<kp_blocks(n, 256), 256, 0, ctx->stream>>>(d_xyz, n, axis, band, enc, d_lower);
    KP_LAUNCH_CHECK(ctx);
    KP_TRY(kp_prim_count_u8(ctx, d_lower, n, d_tot));
    KP_TRY(kp_fetch_scratch(ctx, 2 * sizeof(int32_t)));
    const int32_t *h = (const int32_t *)ctx->h_scratch;
    if (h_axis_max) {
        int32_t b = h[0] >= 0 ? h[0] : h[0] ^ 0x7fffffff;
        float f;
        memcpy(&f, &b, 4);
        *h_axis_max = (double)f;
    }
    if (h_nlower) *h_nlower = h[1];
    return KP_OK;
}

extern "C" {

int kp_ransac_plane(kp_ctx *ctx, const float *d_xyz, int64_t n, double distance_threshold, int ransac_n,
                    int num_iterations, double probability, uint64_t seed, double *h_plane, uint8_t *d_inlier_mask,
                    int64_t *h_ninliers, int32_t *h_best_iter, int64_t *d_counts)
{
    if (!ctx || !d_xyz) return kp_set_err(ctx, KP_E_ARG, "kp_ransac_plane: NULL argument");
    kp_enter(ctx);
    return kp_ransac_device(ctx, d_xyz, n, distance_threshold, ransac_n, num_iterations, probability, seed, h_plane,
                            d_inlier_mask, h_ninliers, h_best_iter, d_counts);
}

int kp_plane_side_mask(kp_ctx *ctx, const float *d_xyz, int64_t n, double a, double b, double c, double d,
                       uint8_t *d_mask, int64_t *h_kept)
{
    if (!ctx || (n > 0 && (!d_xyz || !d_mask))) return kp_set_err(ctx, KP_E_ARG, "kp_plane_side_mask: NULL argument");
    kp_enter(ctx);
    if (h_kept) *h_kept = 0;
    if (n <= 0) return KP_OK;
    KP_PROFB(ctx, "plane_side", (double)n * 14.0);
    k_plane_side<<<kp_blocks(n, 256), 256, 0, ctx->stream>>>(d_xyz, n, a, b, c, d, d_mask);
    KP_LAUNCH_CHECK(ctx);
    int32_t *d_tot = (int32_t *)ctx->d_scratch;
    KP_TRY(kp_prim_count_u8(ctx, d_mask, n, d_tot));
    KP_TRY(kp_fetch_scratch(ctx, sizeof(int32_t)));
    if (h_kept) *h_kept = *(int32_t *)ctx->h_scratch;
    return KP_OK;
}

int kp_band_mask(kp_ctx *ctx, const float *d_xyz, int64_t n, int axis, double band, uint8_t *d_lower,
                 double *h_axis_max, int64_t *h_nlower)
{
    if (!ctx || (n > 0 && (!d_xyz || !d_lower))) return kp_set_err(ctx, KP_E_ARG, "kp_band_mask: NULL argument");
    kp_enter(ctx);
    return kp_band_mask_device(ctx, d_xyz, n, axis, band, d_lower, h_axis_max, h_nlower);
}

}  // extern "C"
