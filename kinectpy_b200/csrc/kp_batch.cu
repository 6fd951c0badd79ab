// kp_batch.cu -- batched, device-count primitives of the frame engine (see kp_batch.cuh).
// Ordered compaction / partition / run heads / exclusive scan in TWO kernels each (tile counts with the scan of
// the tile totals done by whichever CTA finishes last, then the scatter): no CTA ever waits for another one, so
// the result does not depend on the order in which the hardware dispatches CTAs.  Canonical double sums with the
// element count read on the device.
#include "kp_batch.cuh"

namespace {
// ------------------------------------------------------------------ helpers
// true in the last CTA of the segment (grid.x CTAs per segment) to arrive; every thread of the CTA calls it
__device__ __forceinline__ bool bc_last_block(unsigned int *ticket)
{
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1 : 0;
    __syncthreads();
    const bool last = s_last != 0;
    if (last) __threadfence();
    return last;
}
// in-place exclusive scan of v[0..m) (written by other CTAs of this launch) by one CTA; total to every thread
__device__ int bc_cta_excl_scan(int32_t *v, int m)
{
    __shared__ int wtot[BC_THREADS / 32];
    __shared__ int carry_s;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < m; base += BC_THREADS) {
        const int i = base + threadIdx.x;
        const int x = i < m ? __ldcg(v + i) : 0;
        int incl = x;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const int y = __shfl_up_sync(KP_FULL, incl, s);
            if (lane >= s) incl += y;
        }
        if (lane == 31) wtot[w] = incl;
        __syncthreads();
        int woff = 0;
#pragma unroll
        for (int ww = 0; ww < BC_THREADS / 32; ++ww) woff += ww < w ? wtot[ww] : 0;
        const int excl = carry_s + woff + incl - x;
        if (i < m) v[i] = excl;
        __syncthreads();
        if (threadIdx.x == BC_THREADS - 1) carry_s = excl + x;
        __syncthreads();
    }
    return carry_s;
}

// ------------------------------------------------------------------ flags and emitters
struct FMask {
    const uint8_t *mask; int64_t stride; int invert;
    __device__ bool operator()(int seg, int64_t i) const { return (mask[seg * stride + i] != 0) != (invert != 0); }
};
struct FValid {                 // rows whose x is not NaN (kp_b_compact_rows without a mask)
    const float *in; int64_t stride;
    __device__ bool operator()(int seg, int64_t i) const { return !isnan(in[3 * (seg * stride + i)]); }
};
struct FRunHead {
    const uint32_t *keys; int64_t stride;
    __device__ bool operator()(int seg, int64_t i) const
    {
        const uint32_t *k = keys + seg * stride;
        return i == 0 || k[i] != k[i - 1];
    }
};
struct ERows {
    const float *in; float *out; int64_t stride;     // stride in rows
    const uint32_t *aux_in; uint32_t *aux_out;
    __device__ void operator()(int seg, int64_t i, bool f, int pos) const
    {
        if (!f) return;
        const float *a = in + 3 * (seg * stride + i);
        float *o = out + 3 * (seg * stride + pos);
        const float x = a[0], y = a[1], z = a[2];
        o[0] = x; o[1] = y; o[2] = z;
        if (aux_in) aux_out[seg * stride + pos] = aux_in[seg * stride + i];
    }
};
struct EPart {
    const float *in; float *out_t; float *out_f; int64_t stride;
    const uint32_t *aux_in; uint32_t *aux_t; uint32_t *aux_f;
    __device__ void operator()(int seg, int64_t i, bool f, int pos) const
    {
        // pos = number of set flags before i: a cleared row lands at i - pos among the cleared ones
        const float *a = in + 3 * (seg * stride + i);
        const int64_t dst = seg * stride + (f ? (int64_t)pos : i - pos);
        float *o = (f ? out_t : out_f) + 3 * dst;
        const float x = a[0], y = a[1], z = a[2];
        o[0] = x; o[1] = y; o[2] = z;
        if (aux_in) (f ? aux_t : aux_f)[dst] = aux_in[seg * stride + i];
    }
};
struct EIndex {
    int32_t *list; int64_t stride;
    __device__ void operator()(int seg, int64_t i, bool f, int pos) const
    {
        if (f) list[seg * stride + pos] = (int32_t)i;
    }
};

// ------------------------------------------------------------------ count (+ scan of the tile totals) / scatter
template <class Flag>
__global__ void __launch_bounds__(BC_THREADS) k_bc_count(Flag flag, DCnt n, BScan S, DOut total, int32_t *closing,
                                                         int64_t closing_stride)
{
    __shared__ int wc[BC_THREADS / 32];
    const int seg = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t nn = n.at(seg);
    const int ntiles = (int)((nn + BC_TILE - 1) / BC_TILE);
    int32_t *ts = S.tile_sum + (size_t)seg * S.max_tiles;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t base = (int64_t)tile * BC_TILE;
        int cnt = 0;
#pragma unroll
        for (int j = 0; j < BC_ITEMS; ++j) {
            const int64_t i = base + j * BC_THREADS + threadIdx.x;
            const bool f = i < nn && flag(seg, i);
            cnt += __popc(__ballot_sync(KP_FULL, f));
        }
        if (lane == 0) wc[w] = cnt;
        __syncthreads();
        if (threadIdx.x == 0) {
            int s = 0;
#pragma unroll
            for (int ww = 0; ww < BC_THREADS / 32; ++ww) s += wc[ww];
            ts[tile] = s;
        }
        __syncthreads();
    }
    if (bc_last_block(S.ticket + seg)) {
        const int tot = bc_cta_excl_scan(ts, ntiles);
        if (threadIdx.x == 0) {
            total.at(seg) = tot;
            if (closing) closing[seg * closing_stride + tot] = (int32_t)nn;
            S.ticket[seg] = 0;
        }
    }
}

template <class Flag, class Emit>
__global__ void __launch_bounds__(BC_THREADS) k_bc_scatter(Flag flag, Emit emit, DCnt n, BScan S)
{
    __shared__ int cnt[BC_ITEMS * (BC_THREADS / 32)];
    const int seg = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t nn = n.at(seg);
    const int ntiles = (int)((nn + BC_TILE - 1) / BC_TILE);
    const int32_t *ts = S.tile_sum + (size_t)seg * S.max_tiles;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t base = (int64_t)tile * BC_TILE;
        const int tile_off = ts[tile];
        bool f[BC_ITEMS];
        int rank[BC_ITEMS];
#pragma unroll
        for (int j = 0; j < BC_ITEMS; ++j) {
            const int64_t i = base + j * BC_THREADS + threadIdx.x;
            f[j] = i < nn && flag(seg, i);
            const unsigned b = __ballot_sync(KP_FULL, f[j]);
            rank[j] = __popc(b & ((1u << lane) - 1u));
            if (lane == 0) cnt[j * (BC_THREADS / 32) + w] = __popc(b);
        }
        __syncthreads();
        if (w == 0) {
            // element order inside the tile is (j, warp, lane) = entry order of cnt[]; a lane owns two entries
            const int c0 = cnt[2 * lane], c1 = cnt[2 * lane + 1];
            const int s = c0 + c1;
            int incl = s;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = __shfl_up_sync(KP_FULL, incl, d);
                if (lane >= d) incl += y;
            }
            cnt[2 * lane] = tile_off + incl - s;
            cnt[2 * lane + 1] = tile_off + incl - s + c0;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < BC_ITEMS; ++j) {
            const int64_t i = base + j * BC_THREADS + threadIdx.x;
            if (i < nn) emit(seg, i, f[j], cnt[j * (BC_THREADS / 32) + w] + rank[j]);
        }
        __syncthreads();
    }
}

template <class Flag, class Emit>
int bc_run(const BLaunch &L, const BScan &S, DCnt n, Flag flag, Emit emit, DOut total, int32_t *closing = nullptr,
           int64_t closing_stride = 0)
{
    if (L.nseg <= 0) return KP_OK;
    const int64_t tiles = (L.cap + BC_TILE - 1) / BC_TILE;
    if (tiles > S.max_tiles) return kp_set_err(L.ctx, KP_E_ARG, "batched compaction: %lld tiles exceed the scratch (%d)", (long long)tiles, S.max_tiles);
    const dim3 grid((unsigned)(tiles < L.ctas ? (tiles > 0 ? tiles : 1) : L.ctas), (unsigned)L.nseg);
    k_bc_count<<<grid, BC_THREADS, 0, L.ctx->stream>>>(flag, n, S, total, closing, closing_stride);
    KP_LAUNCH_CHECK(L.ctx);
    k_bc_scatter<<<grid, BC_THREADS, 0, L.ctx->stream>>>(flag, emit, n, S);
    KP_LAUNCH_CHECK(L.ctx);
    return KP_OK;
}

// ------------------------------------------------------------------ exclusive scan of an int32 array
// thread t of a tile owns BC_ITEMS consecutive values (two 16-byte loads)
__global__ void __launch_bounds__(BC_THREADS) k_bs_reduce(const int32_t *v, int64_t v_stride, DCnt n, BScan S, DOut total,
                                                          int32_t *closing_v)
{
    __shared__ int wc[BC_THREADS / 32];
    const int seg = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t nn = n.at(seg);
    const int ntiles = (int)((nn + BC_TILE - 1) / BC_TILE);
    int32_t *ts = S.tile_sum + (size_t)seg * S.max_tiles;
    const int32_t *vs = v + seg * v_stride;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t i0 = (int64_t)tile * BC_TILE + (int64_t)threadIdx.x * BC_ITEMS;
        int s = 0;
        if (i0 + BC_ITEMS <= nn) {
            const int4 a = *reinterpret_cast<const int4 *>(vs + i0), b = *reinterpret_cast<const int4 *>(vs + i0 + 4);
            s = a.x + a.y + a.z + a.w + b.x + b.y + b.z + b.w;
        } else {
            for (int j = 0; j < BC_ITEMS; ++j) if (i0 + j < nn) s += vs[i0 + j];
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) s += __shfl_xor_sync(KP_FULL, s, d);
        if (lane == 0) wc[w] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
#pragma unroll
            for (int ww = 0; ww < BC_THREADS / 32; ++ww) t += wc[ww];
            ts[tile] = t;
        }
        __syncthreads();
    }
    if (bc_last_block(S.ticket + seg)) {
        const int tot = bc_cta_excl_scan(ts, ntiles);
        if (threadIdx.x == 0) {
            total.at(seg) = tot;
            if (closing_v) closing_v[seg * v_stride + nn] = tot;     // v[n] = total (written after every read of v)
            S.ticket[seg] = 0;
        }
    }
}
__global__ void __launch_bounds__(BC_THREADS) k_bs_apply(int32_t *v, int64_t v_stride, DCnt n, BScan S)
{
    __shared__ int wtot[BC_THREADS / 32];
    const int seg = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t nn = n.at(seg);
    const int ntiles = (int)((nn + BC_TILE - 1) / BC_TILE);
    const int32_t *ts = S.tile_sum + (size_t)seg * S.max_tiles;
    int32_t *vs = v + seg * v_stride;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t i0 = (int64_t)tile * BC_TILE + (int64_t)threadIdx.x * BC_ITEMS;
        int x[BC_ITEMS];
        const bool full = i0 + BC_ITEMS <= nn;
        if (full) {
            const int4 a = *reinterpret_cast<const int4 *>(vs + i0), b = *reinterpret_cast<const int4 *>(vs + i0 + 4);
            x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
        } else {
#pragma unroll
            for (int j = 0; j < BC_ITEMS; ++j) x[j] = i0 + j < nn ? vs[i0 + j] : 0;
        }
        int s = 0;
#pragma unroll
        for (int j = 0; j < BC_ITEMS; ++j) s += x[j];
        int incl = s;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(KP_FULL, incl, d);
            if (lane >= d) incl += y;
        }
        if (lane == 31) wtot[w] = incl;
        __syncthreads();
        int run = ts[tile] + incl - s;
#pragma unroll
        for (int ww = 0; ww < BC_THREADS / 32; ++ww) run += ww < w ? wtot[ww] : 0;
        int o[BC_ITEMS];
#pragma unroll
        for (int j = 0; j < BC_ITEMS; ++j) { o[j] = run; run += x[j]; }
        if (full) {
            *reinterpret_cast<int4 *>(vs + i0) = make_int4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<int4 *>(vs + i0 + 4) = make_int4(o[4], o[5], o[6], o[7]);
        } else {
#pragma unroll
            for (int j = 0; j < BC_ITEMS; ++j) if (i0 + j < nn) vs[i0 + j] = o[j];
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ canonical sums (tree of kp_primitives.cu)
__global__ void __launch_bounds__(256) k_bcsum_level(const double *x, int64_t x_stride, DCnt n, double *tmp, int64_t tmp_stride,
                                                     double *out, int64_t out_stride, int mode, const double *aux, int64_t aux_stride)
{
    const int seg = blockIdx.y, lane = threadIdx.x & 31;
    const int64_t nn = n.at(seg);
    const int64_t groups = (nn + 1023) / 1024;
    const double *xs = x + seg * x_stride;
    const double mu = mode == 2 ? __ddiv_rn(aux[seg * aux_stride], (double)nn) : 0.0;
    if (nn <= 0) {
        if (blockIdx.x == 0 && threadIdx.x == 0) out[seg * out_stride] = 0.0;
        return;
    }
    double *dst = groups == 1 ? out + seg * out_stride : tmp + seg * tmp_stride;
    for (int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); g < groups; g += (int64_t)gridDim.x * (blockDim.x >> 5)) {
        const int64_t lo = g * 1024;
        double acc = 0.0;
#pragma unroll 4
        for (int r = 0; r < 32; ++r) {
            const int64_t i = lo + r * 32 + lane;
            if (i < nn) {
                double v = xs[i];
                if (mode == 1) v = v > 0 ? v : 0.0;
                else if (mode == 2) { const double d = __dsub_rn(v, mu); v = v > 0 ? __dmul_rn(d, d) : 0.0; }
                acc = __dadd_rn(acc, v);
            }
        }
        acc = kp_butterfly_sum(acc);
        if (lane == 0) dst[g] = acc;
    }
}
__global__ void __launch_bounds__(1024) k_bcsum_rest(DCnt n, double *tmp, int64_t tmp_stride, double *out, int64_t out_stride)
{
    const int seg = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t nn = n.at(seg);
    int64_t cn = (nn + 1023) / 1024;
    if (cn <= 1) return;                      // the first level already wrote the result
    double *cur = tmp + seg * tmp_stride, *nxt = cur + cn;
    for (;;) {
        const int64_t groups = (cn + 1023) / 1024;
        double *dst = groups == 1 ? out + seg * out_stride : nxt;
        for (int64_t g = warp; g < groups; g += 32) {
            const int64_t lo = g * 1024;
            double acc = 0.0;
            for (int r = 0; r < 32; ++r) {
                const int64_t i = lo + r * 32 + lane;
                if (i < cn) acc = __dadd_rn(acc, cur[i]);
            }
            acc = kp_butterfly_sum(acc);
            if (lane == 0) dst[g] = acc;
        }
        if (groups == 1) break;
        __syncthreads();
        cur = nxt; nxt = nxt + groups; cn = groups;
    }
}
}  // namespace

int kp_b_compact_rows(const BLaunch &L, const BScan &S, DCnt n, const uint8_t *mask, int64_t mask_stride, int invert,
                      const float *in, float *out, int64_t row_stride, DOut total, const uint32_t *aux_in, uint32_t *aux_out)
{
    KP_PROFB(L.ctx, "compact_rows", 0.0);
    if (!mask) return bc_run(L, S, n, FValid{in, row_stride}, ERows{in, out, row_stride, aux_in, aux_out}, total);
    return bc_run(L, S, n, FMask{mask, mask_stride, invert}, ERows{in, out, row_stride, aux_in, aux_out}, total);
}
int kp_b_partition_rows(const BLaunch &L, const BScan &S, DCnt n, const uint8_t *mask, int64_t mask_stride, const float *in,
                        float *out_true, float *out_false, int64_t row_stride, DOut total, const uint32_t *aux_in,
                        uint32_t *aux_true, uint32_t *aux_false)
{
    KP_PROFB(L.ctx, "compact_rows", 0.0);
    return bc_run(L, S, n, FMask{mask, mask_stride, 0}, EPart{in, out_true, out_false, row_stride, aux_in, aux_true, aux_false}, total);
}
int kp_b_compact_index(const BLaunch &L, const BScan &S, DCnt n, const uint8_t *mask, int64_t mask_stride, int32_t *list,
                       int64_t list_stride, DOut total)
{
    KP_PROFB(L.ctx, "compact_index", 0.0);
    return bc_run(L, S, n, FMask{mask, mask_stride, 0}, EIndex{list, list_stride}, total);
}
int kp_b_run_starts_u32(const BLaunch &L, const BScan &S, DCnt n, const uint32_t *keys, int64_t key_stride, int32_t *run_start,
                        int64_t rs_stride, DOut total)
{
    KP_PROFB(L.ctx, "run_heads", 0.0);
    return bc_run(L, S, n, FRunHead{keys, key_stride}, EIndex{run_start, rs_stride}, total, run_start, rs_stride);
}
int kp_b_exclusive_scan(const BLaunch &L, const BScan &S, DCnt n, int32_t *v, int64_t v_stride, DOut total)
{
    if (L.nseg <= 0) return KP_OK;
    const int64_t tiles = (L.cap + BC_TILE - 1) / BC_TILE;
    if (tiles > S.max_tiles) return kp_set_err(L.ctx, KP_E_ARG, "batched scan: %lld tiles exceed the scratch (%d)", (long long)tiles, S.max_tiles);
    const dim3 grid((unsigned)(tiles < L.ctas ? (tiles > 0 ? tiles : 1) : L.ctas), (unsigned)L.nseg);
    k_bs_reduce<<<grid, BC_THREADS, 0, L.ctx->stream>>>(v, v_stride, n, S, total, v);
    KP_LAUNCH_CHECK(L.ctx);
    k_bs_apply<<<grid, BC_THREADS, 0, L.ctx->stream>>>(v, v_stride, n, S);
    KP_LAUNCH_CHECK(L.ctx);
    return KP_OK;
}

int kp_b_csum(const BLaunch &L, DCnt n, const double *x, int64_t x_stride, int mode, const double *aux, int64_t aux_stride,
              double *tmp, int64_t tmp_stride, double *out, int64_t out_stride)
{
    if (L.nseg <= 0) return KP_OK;
    const int64_t groups = (L.cap + 1023) / 1024;
    int64_t gx = (groups + 7) / 8;
    if (gx > L.ctas) gx = L.ctas;
    if (gx < 1) gx = 1;
    k_bcsum_level<<<dim3((unsigned)gx, (unsigned)L.nseg), 256, 0, L.ctx->stream>>>(x, x_stride, n, tmp, tmp_stride, out, out_stride, mode,
                                                                                 aux, aux_stride);
    KP_LAUNCH_CHECK(L.ctx);
    k_bcsum_rest<<<(unsigned)L.nseg, 1024, 0, L.ctx->stream>>>(n, tmp, tmp_stride, out, out_stride);
    KP_LAUNCH_CHECK(L.ctx);
    return KP_OK;
}
