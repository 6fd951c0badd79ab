// kp_unproject.cu -- K1: depth -> XYZ through the xy-table + extrinsic + fusion order, the int16
// `_depth.dat` entry, the human-crop mask, PointCloud.transform, bounds and ordered compaction.
#include <math.h>
#include "kp_common.cuh"

namespace {
constexpr int UP_THREADS = 256;
constexpr int UP_PPT = 8;                      // pixels per thread: one 128-bit depth load
constexpr int UP_TILE = UP_THREADS * UP_PPT;   // 2048 pixels -> 16 KB of table per CTA
constexpr int UP_MAX_S = 8;

struct UnprojParams {
    const uint16_t *depth;
    const float2 *tab;
    int B, S;
    int64_t P;
    int flags;
    int has_T;
    double scale;
    float *xyz;
    uint8_t *valid;
    int16_t *xyz16;
    int32_t *bounds_enc;   // BOUNDS variants: [B][S][sets][tiles][warps][8] slots of ordered-int min xyz, max xyz, count, pad
    float *xyz_raw;        // RAW variant (frame engine): second output [B][S][P][3] = the same points BEFORE the extrinsic for
                           // s >= 1 (the ICP sources, in their own sensor frame) and the transformed master for s = 0;
                           // its bounds go to slot set 1
    double T[UP_MAX_S][12];
    // CROP variant (frame engine, human crop of preprocessing/data.py:165-178): uint8 [B][S][P][3] segmentation image
    // and the (frame, sensor) median of the int16 z column [B][S]; kept after the fields above so that the other
    // variants address their parameters exactly as before
    const uint8_t *rgb;
    const double *crop_med;
    double crop_gate;
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// The CTA's slice of the calibration table is fetched once with a TMA bulk copy
// (cp.async.bulk -> SASS UBLKCP) that completes on an mbarrier, kept stationary (registers) and
// reused for every frame of the batch; depth streams through with one 128-bit load per thread.
// Compile-time variants (k4a int16 rounding, drop-any-zero rule, extrinsic, bounds) so a launch carries only its
// own arithmetic: the flag tests and the dead branches they guard were a fifth of the instructions.
// rows of a warp's 256 pixels through a warp-private shared-memory stage: every lane parks its 24 floats (row stride
// 25: conflict-free), then the warp writes them back out as six fully coalesced 512-byte float4 rows.  (The direct
// form -- every lane storing its own 96 contiguous bytes -- half-fills 32 sectors per store instruction.)  Only a
// __syncwarp on either side: no CTA barrier in the frame loop.
__device__ __forceinline__ void up_store_rows(float *stage, const float *vals, float *dst_warp, int lane)
{
#pragma unroll
    for (int j = 0; j < UP_PPT * 3; ++j) stage[lane * 25 + j] = vals[j];
    __syncwarp();
    float4 *d4 = reinterpret_cast<float4 *>(dst_warp);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const int e0 = 4 * (32 * k + lane);
        const float *sp = stage + (e0 / 24) * 25 + (e0 % 24);
        d4[32 * k + lane] = make_float4(sp[0], sp[1], sp[2], sp[3]);
    }
    __syncwarp();
}

// CROP: a pixel reaches the fused cloud only if its segmentation colour is non-black in all three channels and its
// int16 z (0 outside the table) is <= median + gate; the ICP inputs (xyz_raw) and their bounds set ignore the crop.
template <bool INT16, bool DROP, bool HAS_T, bool BOUNDS, bool RAW = false, bool CROP = false>
__global__ void __launch_bounds__(UP_THREADS, RAW ? 2 : 3) k_unproject(const __grid_constant__ UnprojParams p)
{
    __shared__ __align__(128) float2 tab_s[UP_TILE];
    __shared__ __align__(8) uint64_t mbar;
    __shared__ float stage_s[UP_THREADS / 32][32 * 25];
    const int tid = threadIdx.x, lane = tid & 31;
    const int s = blockIdx.y;
    const int64_t p0 = (int64_t)blockIdx.x * UP_TILE;
    const int npx = (int)min((int64_t)UP_TILE, p.P - p0);
    const float2 *gtab = p.tab + (int64_t)s * p.P + p0;
    const uint32_t bytes = (uint32_t)npx * 8u;
    const bool bulk = (bytes % 16u == 0u) && ((((uintptr_t)gtab) & 15u) == 0u);

    if (bulk) {
        if (tid == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbar)));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (tid == 0) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&mbar)), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(smem_u32(tab_s)), "l"(gtab), "r"(bytes), "r"(smem_u32(&mbar)) : "memory");
        }
    } else {
        for (int i = tid; i < npx; i += UP_THREADS) tab_s[i] = gtab[i];
    }

    double T[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) T[i] = p.T[s][i];

    const int px0 = tid * UP_PPT;
    const bool full = px0 + UP_PPT <= npx;
    const bool vec_ok = (p.P % 8 == 0) && ((((uintptr_t)p.depth) & 15u) == 0u);
    const bool vst_ok = (p.P % 4 == 0) && ((((uintptr_t)p.xyz) & 15u) == 0u);
    // the first frame's depth word is requested before waiting for the table tile (two independent DRAM round
    // trips overlap); after that the next frame's word is in flight while the current frame is computed and stored
    const bool fast_ld = full && vec_ok;
    uint4 vnext = make_uint4(0u, 0u, 0u, 0u);
    if (fast_ld && p.B > 0) vnext = __ldg(reinterpret_cast<const uint4 *>(p.depth + ((int64_t)s * p.P + p0 + px0)));

    if (bulk) {
        uint32_t done = 0;
        while (!done) {
            asm volatile("{ .reg .pred q; mbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2; selp.u32 %0, 1, 0, q; }"
                         : "=r"(done) : "r"(smem_u32(&mbar)), "r"(0u) : "memory");
        }
    } else {
        __syncthreads();
    }

    float2 tb[UP_PPT];
#pragma unroll
    for (int j = 0; j < UP_PPT; ++j) tb[j] = (px0 + j < npx) ? tab_s[px0 + j] : make_float2(NAN, NAN);

    for (int b = 0; b < p.B; ++b) {
        const int64_t row = ((int64_t)b * p.S + s) * p.P + p0 + px0;   // first pixel of this thread
        uint16_t dz[UP_PPT];
        if (fast_ld) {
            const uint4 v = vnext;
            if (b + 1 < p.B) vnext = __ldg(reinterpret_cast<const uint4 *>(p.depth + row + (int64_t)p.S * p.P));
            dz[0] = v.x & 0xffff; dz[1] = v.x >> 16; dz[2] = v.y & 0xffff; dz[3] = v.y >> 16;
            dz[4] = v.z & 0xffff; dz[5] = v.z >> 16; dz[6] = v.w & 0xffff; dz[7] = v.w >> 16;
        } else {
#pragma unroll
            for (int j = 0; j < UP_PPT; ++j) dz[j] = (px0 + j < npx) ? p.depth[row + j] : (uint16_t)0;
        }
        float out[UP_PPT * 3];
        float raw[RAW ? UP_PPT * 3 : 1];
        float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
        float rmn[3] = {INFINITY, INFINITY, INFINITY}, rmx[3] = {-INFINITY, -INFINITY, -INFINITY};
        int cnt = 0;
        unsigned okmask = 0;
        // CROP: the master's ICP-input bounds (without the crop), the ICP-input count, the crop's pixel mask
        float cmn[3] = {INFINITY, INFINITY, INFINITY}, cmx[3] = {-INFINITY, -INFINITY, -INFINITY};
        int rcnt = 0;
        unsigned cropmask = 0;
        if (CROP) {
            uint8_t c[UP_PPT * 3];
            const uint8_t *src = p.rgb + 3 * row;
            if (full && (row % 8 == 0) && ((((uintptr_t)p.rgb) & 7u) == 0u)) {
                const uint2 *s8 = reinterpret_cast<const uint2 *>(src);
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    const uint2 w = __ldg(s8 + q);
#pragma unroll
                    for (int k = 0; k < 4; ++k) { c[8 * q + k] = (w.x >> (8 * k)) & 0xffu; c[8 * q + 4 + k] = (w.y >> (8 * k)) & 0xffu; }
                }
            } else {
#pragma unroll
                for (int j = 0; j < UP_PPT * 3; ++j) c[j] = (px0 + j / 3 < npx) ? src[j] : (uint8_t)0;
            }
            const double lim = __dadd_rn(p.crop_med[(int64_t)b * p.S + s], p.crop_gate);
#pragma unroll
            for (int j = 0; j < UP_PPT; ++j) {
                const int16_t z16 = (isnan(tb[j].x) || isnan(tb[j].y)) ? (int16_t)0 : (int16_t)dz[j];
                if (c[3 * j] != 0 && c[3 * j + 1] != 0 && c[3 * j + 2] != 0 && (double)z16 <= lim) cropmask |= 1u << j;
            }
        }
#pragma unroll
        for (int j = 0; j < UP_PPT; ++j) {
            const float xt = tb[j].x, yt = tb[j].y;
            const uint16_t z = dz[j];
            bool ok = !(isnan(xt) || isnan(yt)) && z != 0;
            double X, Y, Z;
            int16_t xi = 0, yi = 0, zi = 0;
            if (INT16) {
                const float zf = (float)z;
                const float fx = __fmul_rn(xt, zf), fy = __fmul_rn(yt, zf);   // no FMA: k4a rounds the product first
                if (ok) {
                    xi = (int16_t)(int32_t)floorf(__fadd_rn(fx, 0.5f));
                    yi = (int16_t)(int32_t)floorf(__fadd_rn(fy, 0.5f));
                    zi = (int16_t)z;
                }
                X = __dmul_rn((double)xi, p.scale);
                Y = __dmul_rn((double)yi, p.scale);
                Z = __dmul_rn((double)zi, p.scale);
            } else {
                X = __dmul_rn(__dmul_rn((double)xt, (double)z), p.scale);
                Y = __dmul_rn(__dmul_rn((double)yt, (double)z), p.scale);
                Z = __dmul_rn((double)z, p.scale);
            }
            if (INT16 && p.xyz16 && px0 + j < npx) {
                int16_t *o = p.xyz16 + 3 * (row + j);
                o[0] = xi; o[1] = yi; o[2] = zi;
            }
            if (DROP && (X == 0.0 || Y == 0.0 || Z == 0.0)) ok = false;
            if (RAW && s > 0) {
                const float rx = ok ? (float)X : NAN, ry = ok ? (float)Y : NAN, rz = ok ? (float)Z : NAN;
                raw[3 * j] = rx; raw[3 * j + 1] = ry; raw[3 * j + 2] = rz;
                if (ok) {
                    rmn[0] = fminf(rmn[0], rx); rmn[1] = fminf(rmn[1], ry); rmn[2] = fminf(rmn[2], rz);
                    rmx[0] = fmaxf(rmx[0], rx); rmx[1] = fmaxf(rmx[1], ry); rmx[2] = fmaxf(rmx[2], rz);
                    if (CROP) ++rcnt;
                }
            }
            if (HAS_T && ok) {
                const double x2 = kp_affine(T[0], T[1], T[2], T[3], X, Y, Z);
                const double y2 = kp_affine(T[4], T[5], T[6], T[7], X, Y, Z);
                const double z2 = kp_affine(T[8], T[9], T[10], T[11], X, Y, Z);
                X = x2; Y = y2; Z = z2;
            }
            if (CROP && RAW && s == 0) {
                // the master's ICP input is the transformed master without the crop
                const float rx = ok ? (float)X : NAN, ry = ok ? (float)Y : NAN, rz = ok ? (float)Z : NAN;
                raw[3 * j] = rx; raw[3 * j + 1] = ry; raw[3 * j + 2] = rz;
                if (ok) {
                    cmn[0] = fminf(cmn[0], rx); cmn[1] = fminf(cmn[1], ry); cmn[2] = fminf(cmn[2], rz);
                    cmx[0] = fmaxf(cmx[0], rx); cmx[1] = fmaxf(cmx[1], ry); cmx[2] = fmaxf(cmx[2], rz);
                    ++rcnt;
                }
            }
            if (CROP) ok = ok && ((cropmask >> j) & 1u);      // the crop is for the fused cloud only
            float fx3 = ok ? (float)X : NAN, fy3 = ok ? (float)Y : NAN, fz3 = ok ? (float)Z : NAN;
            out[3 * j] = fx3; out[3 * j + 1] = fy3; out[3 * j + 2] = fz3;
            if (RAW && !CROP && s == 0) { raw[3 * j] = fx3; raw[3 * j + 1] = fy3; raw[3 * j + 2] = fz3; }
            if (ok) okmask |= 1u << j;
            if (BOUNDS && ok) {
                ++cnt;
                mn[0] = fminf(mn[0], fx3); mn[1] = fminf(mn[1], fy3); mn[2] = fminf(mn[2], fz3);
                mx[0] = fmaxf(mx[0], fx3); mx[1] = fmaxf(mx[1], fy3); mx[2] = fmaxf(mx[2], fz3);
            }
        }
        float *o = p.xyz + 3 * row;
        const bool tile_full = npx == UP_TILE;          // CTA-uniform: every lane of every warp owns 8 pixels
        if (tile_full && vst_ok) {
            up_store_rows(stage_s[tid >> 5], out, o - 3 * (lane * UP_PPT), lane);
        } else if (full && vst_ok) {
            float4 *o4 = reinterpret_cast<float4 *>(o);
#pragma unroll
            for (int q = 0; q < 6; ++q) o4[q] = make_float4(out[4 * q], out[4 * q + 1], out[4 * q + 2], out[4 * q + 3]);
        } else {
#pragma unroll
            for (int j = 0; j < UP_PPT; ++j)
                if (px0 + j < npx) { o[3 * j] = out[3 * j]; o[3 * j + 1] = out[3 * j + 1]; o[3 * j + 2] = out[3 * j + 2]; }
        }
        if (RAW) {
            float *r = p.xyz_raw + 3 * row;
            if (tile_full && vst_ok && ((((uintptr_t)p.xyz_raw) & 15u) == 0u)) {
                up_store_rows(stage_s[tid >> 5], raw, r - 3 * (lane * UP_PPT), lane);
            } else if (full && vst_ok && ((((uintptr_t)p.xyz_raw) & 15u) == 0u)) {
                float4 *r4 = reinterpret_cast<float4 *>(r);
#pragma unroll
                for (int q = 0; q < 6; ++q) r4[q] = make_float4(raw[4 * q], raw[4 * q + 1], raw[4 * q + 2], raw[4 * q + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < UP_PPT; ++j)
                    if (px0 + j < npx) { r[3 * j] = raw[3 * j]; r[3 * j + 1] = raw[3 * j + 1]; r[3 * j + 2] = raw[3 * j + 2]; }
            }
        }
        if (p.valid) {
            if (full && (row % 8 == 0) && ((((uintptr_t)p.valid) & 7u) == 0u)) {
                uint2 v;
                v.x = ((okmask >> 0) & 1u) | (((okmask >> 1) & 1u) << 8) | (((okmask >> 2) & 1u) << 16) | (((okmask >> 3) & 1u) << 24);
                v.y = ((okmask >> 4) & 1u) | (((okmask >> 5) & 1u) << 8) | (((okmask >> 6) & 1u) << 16) | (((okmask >> 7) & 1u) << 24);
                *reinterpret_cast<uint2 *>(p.valid + row) = v;
            } else {
#pragma unroll
                for (int j = 0; j < UP_PPT; ++j)
                    if (px0 + j < npx) p.valid[row + j] = (okmask >> j) & 1u;
            }
        }
        if (BOUNDS) {
            // warp shuffles, then lane 0 parks the warp's 7 numbers in its own 32-byte slot; a small kernel folds
            // the slots of a frame afterwards.  No CTA barrier and no atomics inside the frame loop (thousands of
            // warps hitting the frame's 7 words with atomics cost more than the whole unprojection).
            int enc[7] = {kp_f2ord(mn[0]), kp_f2ord(mn[1]), kp_f2ord(mn[2]), kp_f2ord(mx[0]), kp_f2ord(mx[1]), kp_f2ord(mx[2]), cnt};
            // (order-preserving integer images of the floats: one warp-reduce instruction per number instead of five
            // shuffle + min steps)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                enc[c] = __reduce_min_sync(KP_FULL, enc[c]);
                enc[3 + c] = __reduce_max_sync(KP_FULL, enc[3 + c]);
            }
            enc[6] = __reduce_add_sync(KP_FULL, enc[6]);
            constexpr int NSETS = RAW ? 2 : 1;
            if (lane == 0) {
                int4 *slot = reinterpret_cast<int4 *>(p.bounds_enc) +
                             2 * (((((int64_t)b * p.S + s) * NSETS) * gridDim.x + blockIdx.x) * (UP_THREADS / 32) + (tid >> 5));
                slot[0] = make_int4(enc[0], enc[1], enc[2], enc[3]);
                slot[1] = make_int4(enc[4], enc[5], enc[6], 0);
            }
            if (RAW) {
                // set 1: bounds of what went to xyz_raw (without the crop the master's are those of set 0)
                int renc[6] = {kp_f2ord(s ? rmn[0] : (CROP ? cmn[0] : mn[0])), kp_f2ord(s ? rmn[1] : (CROP ? cmn[1] : mn[1])),
                               kp_f2ord(s ? rmn[2] : (CROP ? cmn[2] : mn[2])), kp_f2ord(s ? rmx[0] : (CROP ? cmx[0] : mx[0])),
                               kp_f2ord(s ? rmx[1] : (CROP ? cmx[1] : mx[1])), kp_f2ord(s ? rmx[2] : (CROP ? cmx[2] : mx[2]))};
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    renc[c] = __reduce_min_sync(KP_FULL, renc[c]);
                    renc[3 + c] = __reduce_max_sync(KP_FULL, renc[3 + c]);
                }
                if (CROP) rcnt = __reduce_add_sync(KP_FULL, rcnt);
                if (lane == 0) {
                    int4 *slot = reinterpret_cast<int4 *>(p.bounds_enc) +
                                 2 * (((((int64_t)b * p.S + s) * NSETS + 1) * gridDim.x + blockIdx.x) * (UP_THREADS / 32) + (tid >> 5));
                    slot[0] = make_int4(renc[0], renc[1], renc[2], renc[3]);
                    slot[1] = make_int4(renc[4], renc[5], CROP ? rcnt : enc[6], 0);
                }
            }
        }
    }
}

// folds `per_row` consecutive slots {min xyz, max xyz, count, -} into one row of the same layout
__global__ void __launch_bounds__(256) k_bounds_fold(const int32_t *slots, int64_t per_row, int32_t *rows)
{
    __shared__ int red[7][8];
    const int32_t *src = slots + (int64_t)blockIdx.x * per_row * 8;
    int v[7] = {kp_f2ord(INFINITY), kp_f2ord(INFINITY), kp_f2ord(INFINITY), kp_f2ord(-INFINITY), kp_f2ord(-INFINITY),
                kp_f2ord(-INFINITY), 0};
    for (int64_t e = threadIdx.x; e < per_row; e += blockDim.x) {
        const int4 a = reinterpret_cast<const int4 *>(src)[2 * e], c = reinterpret_cast<const int4 *>(src)[2 * e + 1];
        v[0] = min(v[0], a.x); v[1] = min(v[1], a.y); v[2] = min(v[2], a.z);
        v[3] = max(v[3], a.w); v[4] = max(v[4], c.x); v[5] = max(v[5], c.y);
        v[6] += c.z;
    }
#pragma unroll
    for (int sft = 16; sft >= 1; sft >>= 1) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            v[c] = min(v[c], __shfl_xor_sync(KP_FULL, v[c], sft));
            v[3 + c] = max(v[3 + c], __shfl_xor_sync(KP_FULL, v[3 + c], sft));
        }
        v[6] += __shfl_xor_sync(KP_FULL, v[6], sft);
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int c = 0; c < 7; ++c) red[c][threadIdx.x >> 5] = v[c];
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        const int c = threadIdx.x;
        int r = 0;
        if (c < 7) {
            r = red[c][0];
            for (int w = 1; w < 8; ++w) r = c < 3 ? min(r, red[c][w]) : (c < 6 ? max(r, red[c][w]) : r + red[c][w]);
        }
        rows[8 * (int64_t)blockIdx.x + c] = r;
    }
}

// ---- cloud input of the frame engine: the load stage in place of K1
// Frame f of the batch is rows off[f] .. off[f + 1] of `xyz` (a CSR batch of float32 [n][3] clouds).  CTA (tile, f) owns
// rows [2048 tile, 2048 tile + 2048) of the frame, a warp 256 consecutive rows, a lane 8.  A warp's rows are 768
// consecutive floats that start at any 4-byte offset (a CSR start is a multiple of 12 bytes, and the caller's pointer
// need not be 16-byte aligned): the warp reads the 16-byte-aligned float4s that cover them, coalesced, through the
// warp-private stage of up_store_rows (a float4 that is not wholly inside the warp's rows is read float by float, so
// nothing outside the cloud is touched), then every lane takes its 8 rows from the stage.  Bounds and count of the
// valid rows (x not NaN) go to the warp's slot in K1's format, which k_bounds_fold folds per frame; no atomics.
constexpr int CL_MAX_B = 16;
struct CloudLoadParams {
    const float *xyz;
    int64_t off[CL_MAX_B + 1];     // rows relative to xyz; a frame beyond the batch's clouds has an empty range
    int64_t P;                     // capacity (rows) of one cloud
    int64_t stride;                // rows between the frames' output segments (a multiple of 64)
    int nan_fill;                  // 1: rows [n_f, P) of the segment are set to NaN (the voxel keys read all P rows)
    float *out;                    // [B][stride][3]
    int32_t *slots;                // [B][tiles][8 warps][8]
    int32_t *n_rows;               // [B]: rows of each cloud, valid or not
};
__global__ void __launch_bounds__(UP_THREADS) k_e_load_clouds(const __grid_constant__ CloudLoadParams p)
{
    __shared__ float stage_s[UP_THREADS / 32][32 * 25];
    const int f = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t lo = p.off[f], n = p.off[f + 1] - lo;
    const int64_t w0 = (int64_t)blockIdx.x * UP_TILE + (int64_t)warp * (32 * UP_PPT);       // the warp's first row
    const int nrw = (int)max((int64_t)0, min((int64_t)(32 * UP_PPT), n - w0));              // its rows of the cloud
    float *stage = stage_s[warp];
    if (blockIdx.x == 0 && tid == 0) p.n_rows[f] = (int32_t)n;
    float v[UP_PPT * 3];
    if (nrw > 0) {
        const float *src = p.xyz + 3 * (lo + w0);
        const int mis = (int)((((uintptr_t)src) >> 2) & 3u);          // floats between the aligned float4 and src
        const float4 *a4 = reinterpret_cast<const float4 *>(src - mis);
        const int nf = 3 * nrw;
#pragma unroll
        for (int k = 0; k < 7; ++k) {                                   // 7 x 32 float4 cover 768 + 3 floats
            const int q = 32 * k + lane, e0 = 4 * q - mis;              // first float of this float4, relative to src
            if (e0 >= nf || e0 + 4 <= 0) continue;
            float t[4];
            if (e0 >= 0 && e0 + 4 <= nf) {
                const float4 x = __ldg(a4 + q);
                t[0] = x.x; t[1] = x.y; t[2] = x.z; t[3] = x.w;
            } else {
#pragma unroll
                for (int c = 0; c < 4; ++c) t[c] = (e0 + c >= 0 && e0 + c < nf) ? __ldg(src + e0 + c) : 0.0f;
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int e = e0 + c;
                if (e >= 0 && e < nf) stage[(e / 24) * 25 + e % 24] = t[c];
            }
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < UP_PPT * 3; ++j) v[j] = stage[lane * 25 + j];
        __syncwarp();
    }
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < UP_PPT; ++j) {
        if (lane * UP_PPT + j < nrw) {
            if (!isnan(v[3 * j])) {
                ++cnt;
#pragma unroll
                for (int c = 0; c < 3; ++c) { mn[c] = fminf(mn[c], v[3 * j + c]); mx[c] = fmaxf(mx[c], v[3 * j + c]); }
            }
        } else {
            v[3 * j] = v[3 * j + 1] = v[3 * j + 2] = NAN;
        }
    }
    // rows out: the cloud's rows, and with nan_fill NaN up to P
    const int nout = p.nan_fill ? (int)max((int64_t)0, min((int64_t)(32 * UP_PPT), p.P - w0)) : nrw;
    float *dst = p.out + 3 * ((int64_t)f * p.stride + w0);
    if (nout == 32 * UP_PPT) {
        up_store_rows(stage, v, dst, lane);
    } else {
#pragma unroll
        for (int j = 0; j < UP_PPT; ++j)
            if (lane * UP_PPT + j < nout) {
                float *o = dst + 3 * (lane * UP_PPT + j);
                o[0] = v[3 * j]; o[1] = v[3 * j + 1]; o[2] = v[3 * j + 2];
            }
    }
    int enc[7] = {kp_f2ord(mn[0]), kp_f2ord(mn[1]), kp_f2ord(mn[2]), kp_f2ord(mx[0]), kp_f2ord(mx[1]), kp_f2ord(mx[2]), cnt};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        enc[c] = __reduce_min_sync(KP_FULL, enc[c]);
        enc[3 + c] = __reduce_max_sync(KP_FULL, enc[3 + c]);
    }
    enc[6] = __reduce_add_sync(KP_FULL, enc[6]);
    if (lane == 0) {
        int4 *slot = reinterpret_cast<int4 *>(p.slots) + 2 * (((int64_t)f * gridDim.x + blockIdx.x) * (UP_THREADS / 32) + warp);
        slot[0] = make_int4(enc[0], enc[1], enc[2], enc[3]);
        slot[1] = make_int4(enc[4], enc[5], enc[6], 0);
    }
}

__global__ void k_bounds_decode_batch(const int32_t *enc, int B, float *bounds, int32_t *nvalid)
{
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    if (bounds) for (int c = 0; c < 6; ++c) bounds[6 * b + c] = kp_ord2f(enc[8 * b + c]);
    if (nvalid) nvalid[b] = enc[8 * b + 6];
}

struct Xyz16Params {
    const int16_t *xyz16; int64_t n; int flags; int has_T; double scale; const uint8_t *keep;
    float *xyz; uint8_t *valid; double T[12];
};
__global__ void __launch_bounds__(256) k_points_from_xyz16(const __grid_constant__ Xyz16Params p)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    int16_t xi = p.xyz16[3 * i], yi = p.xyz16[3 * i + 1], zi = p.xyz16[3 * i + 2];
    double X = __dmul_rn((double)xi, p.scale), Y = __dmul_rn((double)yi, p.scale), Z = __dmul_rn((double)zi, p.scale);
    bool ok = true;
    if ((p.flags & KP_UNPROJECT_DROP_ANY_ZERO) && (X == 0.0 || Y == 0.0 || Z == 0.0)) ok = false;
    if (p.keep && !p.keep[i]) ok = false;
    if (ok && p.has_T) {
        const double x2 = kp_affine(p.T[0], p.T[1], p.T[2], p.T[3], X, Y, Z);
        const double y2 = kp_affine(p.T[4], p.T[5], p.T[6], p.T[7], X, Y, Z);
        const double z2 = kp_affine(p.T[8], p.T[9], p.T[10], p.T[11], X, Y, Z);
        X = x2; Y = y2; Z = z2;
    }
    p.xyz[3 * i] = ok ? (float)X : NAN;
    p.xyz[3 * i + 1] = ok ? (float)Y : NAN;
    p.xyz[3 * i + 2] = ok ? (float)Z : NAN;
    if (p.valid) p.valid[i] = ok;
}

struct XformParams { float *xyz; int64_t n; int rotate_only; double T[12]; };
__global__ void __launch_bounds__(256) k_transform(const __grid_constant__ XformParams p)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    double X = p.xyz[3 * i], Y = p.xyz[3 * i + 1], Z = p.xyz[3 * i + 2];
    double x2 = kp_dot3(p.T[0], p.T[1], p.T[2], X, Y, Z);
    double y2 = kp_dot3(p.T[4], p.T[5], p.T[6], X, Y, Z);
    double z2 = kp_dot3(p.T[8], p.T[9], p.T[10], X, Y, Z);
    if (!p.rotate_only) { x2 = __dadd_rn(x2, p.T[3]); y2 = __dadd_rn(y2, p.T[7]); z2 = __dadd_rn(z2, p.T[11]); }
    p.xyz[3 * i] = (float)x2; p.xyz[3 * i + 1] = (float)y2; p.xyz[3 * i + 2] = (float)z2;
}

// ---- human crop (preprocessing/data.py:165-178): histogram of int16 z, median, mask
__global__ void k_hist_i16z(const int16_t *xyz16, int64_t n, uint32_t *hist)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        atomicAdd(&hist[(int)xyz16[3 * i + 2] + 32768], 1u);
}
__global__ void __launch_bounds__(1024) k_median_from_hist(const uint32_t *hist, int64_t n, double *median)
{
    __shared__ unsigned long long part[1024];
    unsigned long long s = 0;
    for (int j = 0; j < 64; ++j) s += hist[threadIdx.x * 64 + j];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        // numpy.median: odd n -> element n//2; even n -> mean of elements n/2-1 and n/2 (0-based, sorted)
        int64_t r_hi = n / 2, r_lo = (n % 2) ? n / 2 : n / 2 - 1;
        double vals[2];
        int64_t ranks[2] = {r_lo, r_hi};
        for (int q = 0; q < 2; ++q) {
            unsigned long long acc = 0;
            int c = 0;
            while (c < 1023 && acc + part[c] <= (unsigned long long)ranks[q]) { acc += part[c]; ++c; }
            int bin = c * 64;
            while (bin < 65535 && acc + hist[bin] <= (unsigned long long)ranks[q]) { acc += hist[bin]; ++bin; }
            vals[q] = (double)(bin - 32768);
        }
        *median = n > 0 ? (vals[0] + vals[1]) * 0.5 : 0.0;
    }
}
__global__ void k_crop_mask(const uint8_t *rgb, const int16_t *xyz16, int64_t n, const double *median, double gate, uint8_t *keep)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool nonblack = rgb[3 * i] != 0 && rgb[3 * i + 1] != 0 && rgb[3 * i + 2] != 0;
    // data.py:170-171: (z <= med + gate) | (z <= med - gate)  ==  z <= med + gate for gate >= 0; keep both terms
    double z = (double)xyz16[3 * i + 2], m = *median;
    bool depth_ok = (z <= m + gate) || (z <= m - gate);
    keep[i] = nonblack && depth_ok;
}

// ---- frame engine: the crop median of every (frame, sensor) of a batch, numpy.median over all P int16 z values
// (zeros included; 0 outside the table).  Two-level radix select on key = (uint16)z16 ^ 0x8000 (signed order):
// a histogram of the high byte over all pixels, then one of the low byte over the pixels whose high byte is that
// of one of the two middle ranks.  Histograms: [B*S][CM_BINS] uint32, zero on entry, cleared again by the pick.
constexpr int CM_THREADS = 256;
constexpr int CM_BINS = 256 + 2 * 256;          // level 1 | level 2 of rank lo | level 2 of rank hi

struct CropMedParams {
    const uint16_t *depth;      // [B][S][P]
    const uint32_t *vbits;      // [S][words]: bit i of sensor s = table entry i is finite
    int S; int64_t P, words;
    uint32_t *hist;             // [B*S][CM_BINS]
    double *med;                // [B*S]
};

__device__ __forceinline__ void cm_ranks(int64_t P, uint32_t r[2])
{
    r[1] = (uint32_t)(P / 2);
    r[0] = (P % 2) ? r[1] : r[1] - 1;
}

// the bin of `h` (256 counts, one per thread) that holds rank r[q], and the count before it; every thread gets both
__device__ void cm_find(const uint32_t *h, const uint32_t r[2], uint32_t *sh_scan /*[CM_THREADS / 32]*/, int bin[2], uint32_t before[2])
{
    __shared__ int s_bin[2];
    __shared__ uint32_t s_before[2];
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const uint32_t c = h[t];
    uint32_t inc = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(KP_FULL, inc, d);
        if (lane >= d) inc += v;
    }
    if (lane == 31) sh_scan[w] = inc;
    __syncthreads();
    uint32_t base = 0;
    for (int i = 0; i < w; ++i) base += sh_scan[i];
    const uint32_t lo = base + inc - c;           // exclusive prefix of bin t
#pragma unroll
    for (int q = 0; q < 2; ++q)
        if (lo <= r[q] && r[q] < lo + c) { s_bin[q] = t; s_before[q] = lo; }
    __syncthreads();
    for (int q = 0; q < 2; ++q) { bin[q] = s_bin[q]; before[q] = s_before[q]; }
    __syncthreads();
}

template <int LEVEL>
__global__ void __launch_bounds__(CM_THREADS) k_crop_hist(const __grid_constant__ CropMedParams p)
{
    constexpr int NB = LEVEL == 0 ? 256 : 512;
    constexpr int NW = CM_THREADS / 32;
    __shared__ uint32_t h[NW][NB];                 // one histogram per warp: the depths of a frame cluster in a few bins
    __shared__ uint32_t scan[NW];
    const int bs = blockIdx.y, s = bs % p.S;
    const int w = threadIdx.x >> 5;
    for (int e = threadIdx.x; e < NW * NB; e += CM_THREADS) (&h[0][0])[e] = 0;
    int pre[2] = {-1, -1};
    if (LEVEL == 1) {
        uint32_t r[2], before[2];
        cm_ranks(p.P, r);
        cm_find(p.hist + (size_t)bs * CM_BINS, r, scan, pre, before);
        if (pre[1] == pre[0]) pre[1] = -1;        // both ranks in one bin: the rank-lo histogram serves both
    }
    __syncthreads();
    const uint16_t *d = p.depth + (size_t)bs * p.P;
    const uint32_t *vb = p.vbits + (size_t)s * p.words;
    const int64_t ngroups = (p.P + 7) / 8;
    const bool vec = (p.P % 8 == 0) && ((((uintptr_t)p.depth) & 15u) == 0u);
    for (int64_t g = (int64_t)blockIdx.x * CM_THREADS + threadIdx.x; g < ngroups; g += (int64_t)gridDim.x * CM_THREADS) {
        const int64_t i0 = 8 * g;
        uint16_t z[8];
        if (vec) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(d + i0));
            z[0] = v.x & 0xffff; z[1] = v.x >> 16; z[2] = v.y & 0xffff; z[3] = v.y >> 16;
            z[4] = v.z & 0xffff; z[5] = v.z >> 16; z[6] = v.w & 0xffff; z[7] = v.w >> 16;
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) z[j] = i0 + j < p.P ? d[i0 + j] : (uint16_t)0;
        }
        const uint32_t bits = (uint32_t)(vb[i0 >> 5] >> (i0 & 31)) & 0xffu;    // i0 % 8 == 0: 8 bits of one word
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (i0 + j >= p.P) break;
            const uint32_t key = (((bits >> j) & 1u) ? (uint32_t)z[j] : 0u) ^ 0x8000u;
            if (LEVEL == 0) {
                atomicAdd(&h[w][key >> 8], 1u);
            } else {
                const int hi = (int)(key >> 8);
                if (hi == pre[0]) atomicAdd(&h[w][key & 0xffu], 1u);
                else if (hi == pre[1]) atomicAdd(&h[w][256 + (key & 0xffu)], 1u);
            }
        }
    }
    __syncthreads();
    uint32_t *gh = p.hist + (size_t)bs * CM_BINS + (LEVEL == 0 ? 0 : 256);
    for (int e = threadIdx.x; e < NB; e += CM_THREADS) {
        uint32_t v = 0;
#pragma unroll
        for (int k = 0; k < NW; ++k) v += h[k][e];
        if (v) atomicAdd(gh + e, v);
    }
}

// one CTA per (frame, sensor): the two middle values from the histograms -> median; clears the histograms
__global__ void __launch_bounds__(CM_THREADS) k_crop_median(const __grid_constant__ CropMedParams p)
{
    __shared__ uint32_t scan[CM_THREADS / 32];
    __shared__ uint32_t h2[2][256];
    const int bs = blockIdx.x, t = threadIdx.x;
    uint32_t *gh = p.hist + (size_t)bs * CM_BINS;
    uint32_t r[2], before[2];
    int pre[2], lo[2];
    cm_ranks(p.P, r);
    cm_find(gh, r, scan, pre, before);
    h2[0][t] = gh[256 + t];
    h2[1][t] = gh[512 + t];
    __syncthreads();
    for (int e = t; e < CM_BINS; e += CM_THREADS) gh[e] = 0;
    // rank q inside its high-byte bin; rank hi has its own low-byte histogram only when its bin differs from rank lo's
    const uint32_t rr[2] = {r[0] - before[0], r[1] - before[1]};
    uint32_t unused[2];
    cm_find(h2[0], rr, scan, lo, unused);
    if (pre[1] != pre[0]) {
        const uint32_t r1[2] = {rr[1], rr[1]};
        int l1[2];
        cm_find(h2[1], r1, scan, l1, unused);
        lo[1] = l1[1];
    }
    if (t == 0) {
        const double v0 = (double)(int16_t)(uint16_t)((((uint32_t)pre[0] << 8) | (uint32_t)lo[0]) ^ 0x8000u);
        const double v1 = (double)(int16_t)(uint16_t)((((uint32_t)pre[1] << 8) | (uint32_t)lo[1]) ^ 0x8000u);
        p.med[bs] = (v0 + v1) * 0.5;
    }
}

static void fill_T12(const double *h_T16, double *T12)
{
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 4; ++c) T12[4 * r + c] = h_T16 ? h_T16[4 * r + c] : (r == c ? 1.0 : 0.0);
}
}  // namespace

// internal (no ws reset): used by the frame pipeline as well
int kp_unproject_device(kp_ctx *ctx, const uint16_t *d_depth, const float *d_xytab, const double *h_T, int B, int S,
                        int64_t P, int flags, double scale, float *d_xyz, uint8_t *d_valid, int16_t *d_xyz16,
                        int32_t *d_bounds_enc /*[B][8] nullable, initialised here*/)
{
    if (B <= 0 || S <= 0 || P <= 0) return KP_OK;
    if (S > UP_MAX_S) return kp_set_err(ctx, KP_E_ARG, "kp_unproject_transform: at most %d sensors per call (got %d)", UP_MAX_S, S);
    if (d_xyz16 && !(flags & KP_UNPROJECT_INT16)) return kp_set_err(ctx, KP_E_ARG, "d_xyz16 output needs KP_UNPROJECT_INT16");
    KP_PROFB(ctx, "unproject_transform", (double)B * S * P * (2.0 + 12.0 + (d_valid ? 1.0 : 0.0) + (d_xyz16 ? 6.0 : 0.0)) +
                                             (double)S * P * 8.0);
    UnprojParams p;
    p.depth = d_depth; p.tab = (const float2 *)d_xytab; p.B = B; p.S = S; p.P = P; p.flags = flags;
    p.has_T = h_T != nullptr; p.scale = scale; p.xyz = d_xyz; p.valid = d_valid; p.xyz16 = d_xyz16; p.xyz_raw = nullptr;
    // bounds: the kernel leaves one slot per warp and frame, folded into d_bounds_enc's rows afterwards
    const int64_t ntiles = kp_blocks(P, UP_TILE);
    const int64_t nslots = (int64_t)B * S * ntiles * (UP_THREADS / 32);
    int32_t *slots = nullptr;
    if (d_bounds_enc) KP_TRY(kp_ws(ctx, (size_t)nslots * 8, &slots));
    p.bounds_enc = slots;
    for (int s = 0; s < UP_MAX_S; ++s) fill_T12(h_T && s < S ? h_T + 16 * s : nullptr, p.T[s]);
    dim3 grid(kp_blocks(P, UP_TILE), (unsigned)S);
    const int variant = ((flags & KP_UNPROJECT_INT16) ? 1 : 0) | ((flags & KP_UNPROJECT_DROP_ANY_ZERO) ? 2 : 0) |
                        (h_T ? 4 : 0) | (d_bounds_enc ? 8 : 0);
#define KP_UP_CASE(v)                                                                                                 \
    case v: k_unproject<((v) & 1) != 0, ((v) & 2) != 0, ((v) & 4) != 0, ((v) & 8) != 0><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    switch (variant) {
        KP_UP_CASE(0) KP_UP_CASE(1) KP_UP_CASE(2) KP_UP_CASE(3) KP_UP_CASE(4) KP_UP_CASE(5) KP_UP_CASE(6) KP_UP_CASE(7)
        KP_UP_CASE(8) KP_UP_CASE(9) KP_UP_CASE(10) KP_UP_CASE(11) KP_UP_CASE(12) KP_UP_CASE(13) KP_UP_CASE(14) KP_UP_CASE(15)
    }
#undef KP_UP_CASE
    KP_LAUNCH_CHECK(ctx);
    if (d_bounds_enc) {
        const int rows = (flags & KP_UP_BOUNDS_PER_SENSOR) ? B * S : B;
        k_bounds_fold<<<rows, 256, 0, ctx->stream>>>(slots, nslots / rows, d_bounds_enc);
        KP_LAUNCH_CHECK(ctx);
    }
    return KP_OK;
}

// frame engine: B frames in one launch; fused cloud [B][S*P][3] in the master frame + ICP inputs [B][S][P][3]
// (s = 0: the transformed master, s >= 1: the sub cloud in its own frame) + bounds rows [B][S][2][8] (set 0: fused
// coordinates of sensor s, set 1: what went to the ICP input).  d_slots: [B*S*2*tiles*8 warps][8] int32 scratch.
int kp_unproject_engine(kp_ctx *ctx, const uint16_t *d_depth, const float *d_xytab, const double *h_T, int B, int S, int64_t P,
                        int flags, double scale, float *d_xyz, float *d_xyz_raw, int32_t *d_slots, int32_t *d_rows,
                        const uint8_t *d_rgb, const double *d_crop_med, double crop_gate)
{
    if (B <= 0 || S <= 0 || P <= 0) return KP_OK;
    if (S > UP_MAX_S) return kp_set_err(ctx, KP_E_ARG, "frame engine: at most %d sensors (got %d)", UP_MAX_S, S);
    KP_PROFB(ctx, "unproject_transform", (double)B * S * P * (2.0 + 12.0 + 12.0 + (d_rgb ? 3.0 : 0.0)) + (double)S * P * 8.0);
    UnprojParams p;
    p.depth = d_depth; p.tab = (const float2 *)d_xytab; p.B = B; p.S = S; p.P = P; p.flags = flags;
    p.has_T = 1; p.scale = scale; p.xyz = d_xyz; p.valid = nullptr; p.xyz16 = nullptr; p.xyz_raw = d_xyz_raw;
    p.bounds_enc = d_slots;
    p.rgb = d_rgb; p.crop_med = d_crop_med; p.crop_gate = crop_gate;
    for (int s = 0; s < UP_MAX_S; ++s) fill_T12(h_T && s < S ? h_T + 16 * s : nullptr, p.T[s]);
    const int64_t ntiles = kp_blocks(P, UP_TILE);
    dim3 grid((unsigned)ntiles, (unsigned)S);
    const int variant = ((flags & KP_UNPROJECT_INT16) ? 1 : 0) | ((flags & KP_UNPROJECT_DROP_ANY_ZERO) ? 2 : 0) | (d_xyz_raw ? 4 : 0) |
                        (d_rgb ? 8 : 0);
    switch (variant) {
    case 0: k_unproject<false, false, true, true, false><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 1: k_unproject<true, false, true, true, false><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 2: k_unproject<false, true, true, true, false><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 3: k_unproject<true, true, true, true, false><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 4: k_unproject<false, false, true, true, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 5: k_unproject<true, false, true, true, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 6: k_unproject<false, true, true, true, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 7: k_unproject<true, true, true, true, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 8: k_unproject<false, false, true, true, false, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 9: k_unproject<true, false, true, true, false, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 10: k_unproject<false, true, true, true, false, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 11: k_unproject<true, true, true, true, false, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 12: k_unproject<false, false, true, true, true, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 13: k_unproject<true, false, true, true, true, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    case 14: k_unproject<false, true, true, true, true, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    default: k_unproject<true, true, true, true, true, true><<<grid, UP_THREADS, 0, ctx->stream>>>(p); break;
    }
    KP_LAUNCH_CHECK(ctx);
    // rows [B][S][sets][8]: one set without the ICP inputs, two with
    k_bounds_fold<<<B * S * (d_xyz_raw ? 2 : 1), 256, 0, ctx->stream>>>(d_slots, ntiles * (UP_THREADS / 32), d_rows);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}
size_t kp_unproject_engine_slots(int B, int S, int64_t P)
{
    return (size_t)B * S * 2 * kp_blocks(P, UP_TILE) * (UP_THREADS / 32) * 8;
}

// frame engine, cloud input: frame f of the batch = rows h_off[f] .. h_off[f + 1] of d_xyz (h_off [B + 1] on the host,
// relative to d_xyz) -> segment f of d_out (row stride `stride`, NaN over rows [n_f, P) with nan_fill), bounds rows
// [B][8] in K1's layout, d_nrows [B].  d_slots: kp_unproject_engine_slots(B, 1, P) int32 scratch.
int kp_load_clouds_engine(kp_ctx *ctx, const float *d_xyz, const int64_t *h_off, int B, int64_t P, int64_t stride, int nan_fill,
                          float *d_out, int32_t *d_slots, int32_t *d_rows, int32_t *d_nrows)
{
    if (B <= 0 || P <= 0) return KP_OK;
    if (B > CL_MAX_B) return kp_set_err(ctx, KP_E_ARG, "frame engine: at most %d clouds per batch (got %d)", CL_MAX_B, B);
    const int64_t rows = h_off[B] - h_off[0];
    const int64_t ntiles = kp_blocks(P, UP_TILE);
    // algorithmic bytes: the rows in, the rows (and the NaN fill) out, one 32-byte slot per warp, the row counts
    KP_PROFB(ctx, "cloud_load", (double)rows * 12.0 + (nan_fill ? (double)B * P : (double)rows) * 12.0 +
                                    (double)B * ntiles * (UP_THREADS / 32) * 32.0 + (double)B * 4.0);
    CloudLoadParams p;
    p.xyz = d_xyz;
    for (int f = 0; f <= CL_MAX_B; ++f) p.off[f] = h_off[f < B ? f : B];
    p.P = P; p.stride = stride; p.nan_fill = nan_fill; p.out = d_out; p.slots = d_slots; p.n_rows = d_nrows;
    k_e_load_clouds<<<dim3((unsigned)ntiles, (unsigned)B), UP_THREADS, 0, ctx->stream>>>(p);
    KP_LAUNCH_CHECK(ctx);
    k_bounds_fold<<<B, 256, 0, ctx->stream>>>(d_slots, ntiles * (UP_THREADS / 32), d_rows);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}

// frame engine: crop medians d_med [B][S] of the batch's depth (d_vbits [S][(P + 31) / 32]: finite table entries;
// d_hist [B*S][kp_crop_median_hist_elems()] zero on entry and on return)
int kp_crop_median_engine(kp_ctx *ctx, const uint16_t *d_depth, const uint32_t *d_vbits, int B, int S, int64_t P, uint32_t *d_hist,
                          double *d_med)
{
    if (B <= 0 || S <= 0 || P <= 0) return KP_OK;
    KP_PROFB(ctx, "crop_median", (double)B * S * P * (2.0 + 2.0) + 2.0 * (double)S * P / 8.0);
    CropMedParams p{d_depth, d_vbits, S, P, (P + 31) / 32, d_hist, d_med};
    // about four CTAs per SM over the batch, each streaming whole 16-byte groups of 8 pixels
    int64_t gx = ((int64_t)ctx->sm_count * 4 + (int64_t)B * S - 1) / ((int64_t)B * S);
    const int64_t gmax = kp_blocks((P + 7) / 8, CM_THREADS);
    if (gx > gmax) gx = gmax;
    if (gx < 1) gx = 1;
    const dim3 grid((unsigned)gx, (unsigned)(B * S));
    k_crop_hist<0><<<grid, CM_THREADS, 0, ctx->stream>>>(p);
    KP_LAUNCH_CHECK(ctx);
    k_crop_hist<1><<<grid, CM_THREADS, 0, ctx->stream>>>(p);
    KP_LAUNCH_CHECK(ctx);
    k_crop_median<<<B * S, CM_THREADS, 0, ctx->stream>>>(p);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}
size_t kp_crop_median_hist_elems() { return CM_BINS; }

extern "C" {

int kp_unproject_transform(kp_ctx *ctx, const uint16_t *d_depth, const float *d_xytab, const double *h_T, int B,
                           int S, int64_t P, int flags, double scale, float *d_xyz, uint8_t *d_valid,
                           int16_t *d_xyz16, float *d_bounds, int32_t *d_nvalid)
{
    if (!ctx || !d_depth || !d_xytab || !d_xyz) return kp_set_err(ctx, KP_E_ARG, "kp_unproject_transform: NULL argument");
    if (B < 0 || S < 0 || P < 0) return kp_set_err(ctx, KP_E_ARG, "kp_unproject_transform: negative size");
    kp_enter(ctx);
    int32_t *enc = nullptr;
    if (d_bounds || d_nvalid) KP_TRY(kp_ws(ctx, (size_t)B * 8, &enc));
    KP_TRY(kp_unproject_device(ctx, d_depth, d_xytab, h_T, B, S, P, flags, scale, d_xyz, d_valid, d_xyz16, enc));
    if (enc && B > 0) {
        k_bounds_decode_batch<<<kp_blocks(B, 128), 128, 0, ctx->stream>>>(enc, B, d_bounds, d_nvalid);
        KP_LAUNCH_CHECK(ctx);
    }
    return KP_OK;
}

int kp_points_from_xyz16(kp_ctx *ctx, const int16_t *d_xyz16, int64_t n, const double *h_T, int flags, double scale,
                         const uint8_t *d_keep, float *d_xyz, uint8_t *d_valid)
{
    if (!ctx || (n > 0 && (!d_xyz16 || !d_xyz))) return kp_set_err(ctx, KP_E_ARG, "kp_points_from_xyz16: NULL argument");
    kp_enter(ctx);
    if (n <= 0) return KP_OK;
    KP_PROFB(ctx, "points_from_xyz16", (double)n * (6.0 + 12.0 + (d_valid ? 1.0 : 0.0) + (d_keep ? 1.0 : 0.0)));
    Xyz16Params p;
    p.xyz16 = d_xyz16; p.n = n; p.flags = flags; p.has_T = h_T != nullptr; p.scale = scale; p.keep = d_keep;
    p.xyz = d_xyz; p.valid = d_valid;
    fill_T12(h_T, p.T);
    k_points_from_xyz16<<<kp_blocks(n, 256), 256, 0, ctx->stream>>>(p);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}

int kp_crop_mask(kp_ctx *ctx, const uint8_t *d_rgb, const int16_t *d_xyz16, int64_t n, double gate, uint8_t *d_keep,
                 double *h_median)
{
    if (!ctx || (n > 0 && (!d_rgb || !d_xyz16 || !d_keep))) return kp_set_err(ctx, KP_E_ARG, "kp_crop_mask: NULL argument");
    kp_enter(ctx);
    if (n <= 0) { if (h_median) *h_median = NAN; return KP_OK; }
    KP_PROFB(ctx, "crop_mask", (double)n * (2.0 + 3.0 + 2.0 + 1.0));
    uint32_t *hist;
    KP_TRY(kp_ws(ctx, 65536, &hist));
    double *d_med = (double *)ctx->d_scratch;
    KP_CUDA(ctx, cudaMemsetAsync(hist, 0, 65536 * sizeof(uint32_t), ctx->stream));
    unsigned nb = kp_blocks(n, 256 * 8);
    if (nb > (unsigned)ctx->sm_count * 8) nb = ctx->sm_count * 8;
    k_hist_i16z<<<nb, 256, 0, ctx->stream>>>(d_xyz16, n, hist);
    KP_LAUNCH_CHECK(ctx);
    k_median_from_hist<<<1, 1024, 0, ctx->stream>>>(hist, n, d_med);
    KP_LAUNCH_CHECK(ctx);
    k_crop_mask<<<kp_blocks(n, 256), 256, 0, ctx->stream>>>(d_rgb, d_xyz16, n, d_med, gate, d_keep);
    KP_LAUNCH_CHECK(ctx);
    if (h_median) {
        KP_TRY(kp_fetch_scratch(ctx, sizeof(double)));
        *h_median = *(double *)ctx->h_scratch;
    }
    return KP_OK;
}

int kp_transform_points(kp_ctx *ctx, float *d_xyz, int64_t n, const double *h_T16, int rotate_only)
{
    if (!ctx || !h_T16 || (n > 0 && !d_xyz)) return kp_set_err(ctx, KP_E_ARG, "kp_transform_points: NULL argument");
    kp_enter(ctx);
    if (n <= 0) return KP_OK;
    KP_PROFB(ctx, "transform", (double)n * 24.0);
    XformParams p;
    p.xyz = d_xyz; p.n = n; p.rotate_only = rotate_only;
    fill_T12(h_T16, p.T);
    k_transform<<<kp_blocks(n, 256), 256, 0, ctx->stream>>>(p);
    KP_LAUNCH_CHECK(ctx);
    return KP_OK;
}

int kp_bounds(kp_ctx *ctx, const float *d_xyz, int64_t n, float *h_bounds, int64_t *h_nvalid)
{
    if (!ctx || !h_bounds) return kp_set_err(ctx, KP_E_ARG, "kp_bounds: NULL argument");
    kp_enter(ctx);
    return kp_prim_bounds_fetch(ctx, d_xyz, n, h_bounds, h_nvalid);
}

int kp_compact(kp_ctx *ctx, int64_t n, const uint8_t *d_mask, int invert, const float *d_a0, float *d_a0_out,
               const float *d_a1, float *d_a1_out, const float *d_a2, float *d_a2_out, int32_t *d_index_out,
               int64_t *h_count)
{
    if (!ctx) return kp_set_err(ctx, KP_E_ARG, "kp_compact: NULL ctx");
    if (!d_mask && !d_a0) return kp_set_err(ctx, KP_E_ARG, "kp_compact: need a mask or points (NaN test)");
    kp_enter(ctx);
    int32_t *d_pos = nullptr;
    int32_t *d_total = (int32_t *)ctx->d_scratch;
    if (n > 0) KP_TRY(kp_ws(ctx, (size_t)n, &d_pos));
    KP_TRY(kp_prim_compact_mask(ctx, n, d_mask, invert, d_a0, d_pos, d_index_out, d_total));
    if (n > 0) {
        if (d_a0 && d_a0_out) KP_TRY(kp_prim_gather3(ctx, n, d_pos, d_a0, d_a0_out));
        if (d_a1 && d_a1_out) KP_TRY(kp_prim_gather3(ctx, n, d_pos, d_a1, d_a1_out));
        if (d_a2 && d_a2_out) KP_TRY(kp_prim_gather3(ctx, n, d_pos, d_a2, d_a2_out));
    }
    if (h_count) {
        KP_TRY(kp_fetch_scratch(ctx, sizeof(int32_t)));
        *h_count = *(int32_t *)ctx->h_scratch;
    }
    return KP_OK;
}

}  // extern "C"
