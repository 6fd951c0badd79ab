// kp_resample.cu -- K6: fixed-N point resampling feeding PointNet (BASELINE config C5).
// Replaces select_points_randomly (utils/processing.py:259-275: np.random.choice(n, N, replace=False),
// called at datasets/kinect_dataset.py:103-104) and the prefix variant `points[:N]` of
// datasets/kinect_dataset_npz.py:96-97.
//
// np.random.choice draws from numpy's global Mersenne state, which no parallel machine reproduces;
// the subset here is defined by a counter-based key instead: point i of sample stream s gets
// key = min(kp_rng(seed, s, i) >> 32, 2^32 - 2), NaN rows get 2^32 - 1, and the sample is the N
// points with the smallest (key, index), in that order -- a uniformly random N-subset in uniformly
// random order, like the reference's, and one a CPU restatement can replay bit for bit.
//
// Selection (all clouds of a batch in the same launches, blockIdx.y = cloud; HBM-bound streaming):
//   keys     one pass over the points -> 32-bit key per point (+ count of valid points)
//   3 x (histogram + pick): radix-select of the N-th smallest key, 11 + 11 + 10 bits, the histogram of a
//            pass restricted to the keys that match the prefix found so far; no data moves
//   collect  keys <= threshold appended (warp-aggregated atomics) as 64-bit (key << 32 | index)
//   sort     one CTA per cloud: bitonic sort of those ~N entries in shared memory, gather of the first N
// The clouds of a batch are either CSR rows of one array (kp_resample_batch) or the fixed-stride final clouds of the
// frame engine with their row counts in device memory (RselClouds).  For CSR input, a cloud whose candidate list
// overflows (more than 2048 keys tie with the threshold: never for hashed keys) or whose N exceeds the
// shared-memory sort falls back to a full stable radix sort of (key, index); the engine has no host round trip, so
// there a short cloud or an overflow is the frame's status and its slot is zero-filled.
#include <string.h>
#include <vector>
#include "kp_common.cuh"

namespace {
constexpr int RSEL_BINS = 2048;

struct RselState {
    uint32_t prefix;      // key bits fixed so far (left-aligned value, see shift)
    uint32_t need;        // how many keys are still to be taken inside the current prefix
    uint32_t nvalid;      // non-NaN points
    uint32_t count;       // entries appended by collect
};

constexpr int RSEL_MAX_IDS = 16;       // frame ids carried in the launch parameters (the engine's frames per launch)

// where cloud b lives: CSR rows off[b] .. off[b+1] of the points, or n_dev[b * n_step] rows (a count the device
// wrote) from base[b] (a pointer the device wrote) with keys at b * stride; sample stream first_stream + b, or ids[b];
// status (nullable): int32 per cloud at b * status_step
struct RselClouds {
    const int64_t *off;
    const float *const *base;
    int64_t stride;
    const int32_t *n_dev; int64_t n_step;
    uint64_t first_stream;
    int use_ids;
    uint64_t ids[RSEL_MAX_IDS];
    int32_t *status; int64_t status_step;
};
// o: first key of the cloud; pts: its first point
__device__ __forceinline__ void rsel_cloud(const RselClouds &c, const float *xyz, int b, int64_t &o, int64_t &n, const float *&pts)
{
    if (c.off) { o = c.off[b]; n = c.off[b + 1] - o; pts = xyz + 3 * o; }
    else { o = (int64_t)b * c.stride; n = c.n_dev[(int64_t)b * c.n_step]; pts = c.base[b]; }
}
__device__ __forceinline__ uint64_t rsel_stream(const RselClouds &c, int b) { return c.use_ids ? c.ids[b] : c.first_stream + (uint64_t)b; }

__device__ __forceinline__ uint32_t resample_key(const float *xyz, int64_t i, uint64_t seed, uint64_t stream)
{
    uint32_t key = 0xffffffffu;
    if (!isnan(xyz[3 * i])) {
        key = (uint32_t)(kp_rng(seed, stream, (uint64_t)i) >> 32);
        if (key == 0xffffffffu) key = 0xfffffffeu;
    }
    return key;
}

__global__ void __launch_bounds__(256) k_resample_keys(const float *xyz, int64_t n, uint64_t seed, uint64_t stream,
                                                       uint32_t *keys, int32_t *vals)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = resample_key(xyz, i, seed, stream);
    if (vals) vals[i] = (int32_t)i;
}

// batched: keys of every cloud + per-cloud valid count + first-pass histogram (top 11 bits)
__global__ void __launch_bounds__(256) k_rsel_keys(const float *xyz, const __grid_constant__ RselClouds c, uint64_t seed,
                                                   uint32_t *keys, uint32_t *hist, RselState *st)
{
    __shared__ uint32_t sh[RSEL_BINS];
    const int b = blockIdx.y;
    int64_t o, n;
    const float *pts;
    rsel_cloud(c, xyz, b, o, n, pts);
    for (int e = threadIdx.x; e < RSEL_BINS; e += 256) sh[e] = 0;
    __syncthreads();
    int valid = 0;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        const uint32_t key = resample_key(pts, i, seed, rsel_stream(c, b));
        keys[o + i] = key;
        valid += key != 0xffffffffu;
        atomicAdd(&sh[key >> 21], 1u);
    }
    __syncthreads();
    for (int e = threadIdx.x; e < RSEL_BINS; e += 256) if (sh[e]) atomicAdd(&hist[(size_t)b * RSEL_BINS + e], sh[e]);
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) valid += __shfl_xor_sync(KP_FULL, valid, s);
    if ((threadIdx.x & 31) == 0 && valid) atomicAdd(&st[b].nvalid, (uint32_t)valid);
}

// histogram of the next digit over the keys that match the prefix (pass 1: bits 20..10, pass 2: bits 9..0)
__global__ void __launch_bounds__(256) k_rsel_hist(const uint32_t *keys, const __grid_constant__ RselClouds c, int pass, uint32_t *hist,
                                                   const RselState *st)
{
    __shared__ uint32_t sh[RSEL_BINS];
    const int b = blockIdx.y;
    int64_t o, n;
    const float *pts;
    rsel_cloud(c, nullptr, b, o, n, pts);
    for (int e = threadIdx.x; e < RSEL_BINS; e += 256) sh[e] = 0;
    __syncthreads();
    const uint32_t prefix = st[b].prefix;
    const int pshift = pass == 1 ? 21 : 10;             // bits above this position are fixed
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        const uint32_t key = keys[o + i];
        if ((key >> pshift) == prefix) atomicAdd(&sh[pass == 1 ? (key >> 10) & 0x7ffu : key & 0x3ffu], 1u);
    }
    __syncthreads();
    for (int e = threadIdx.x; e < RSEL_BINS; e += 256) if (sh[e]) atomicAdd(&hist[(size_t)b * RSEL_BINS + e], sh[e]);
}

// one CTA per cloud: the bin where the running count reaches `need`; extends the prefix, clears the histogram
__global__ void __launch_bounds__(256) k_rsel_pick(uint32_t *hist, int pass, uint32_t N, RselState *st)
{
    __shared__ uint32_t part[256];
    const int b = blockIdx.x, tid = threadIdx.x;
    uint32_t *h = hist + (size_t)b * RSEL_BINS;
    const uint32_t need = pass == 0 ? N : st[b].need;
    constexpr int PER = RSEL_BINS / 256;
    uint32_t loc[PER], s = 0;
#pragma unroll
    for (int j = 0; j < PER; ++j) { loc[j] = h[tid * PER + j]; s += loc[j]; h[tid * PER + j] = 0; }
    part[tid] = s;
    __syncthreads();
    if (tid == 0) {
        uint32_t run = 0;
        for (int t = 0; t < 256; ++t) { const uint32_t c = part[t]; part[t] = run; run += c; }
    }
    __syncthreads();
    uint32_t run = part[tid];
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        if (run < need && need <= run + loc[j]) {       // exactly one (tid, j) satisfies this when need <= total
            const uint32_t digit = (uint32_t)(tid * PER + j);
            st[b].prefix = pass == 0 ? digit : (pass == 1 ? (st[b].prefix << 11) | digit : (st[b].prefix << 10) | digit);
            st[b].need = need - run;
        }
        run += loc[j];
    }
}

// keys <= threshold -> list[b][cap] as (key << 32 | index), any order
__global__ void __launch_bounds__(256) k_rsel_collect(const uint32_t *keys, const __grid_constant__ RselClouds c, RselState *st,
                                                      unsigned long long *list, int cap)
{
    const int b = blockIdx.y;
    int64_t o, n;
    const float *pts;
    rsel_cloud(c, nullptr, b, o, n, pts);
    const uint32_t T = st[b].prefix;                    // after three picks: the full 32-bit threshold key
    const int lane = threadIdx.x & 31;
    for (int64_t i0 = (int64_t)blockIdx.x * 256 + (threadIdx.x & ~31); i0 < n; i0 += (int64_t)gridDim.x * 256) {
        const int64_t i = i0 + lane;
        const uint32_t key = i < n ? keys[o + i] : 0xffffffffu;
        const bool take = i < n && key <= T && key != 0xffffffffu;
        const unsigned m = __ballot_sync(KP_FULL, take);
        if (m == 0) continue;
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&st[b].count, (uint32_t)__popc(m));
        base = __shfl_sync(KP_FULL, base, 0);
        const uint32_t pos = base + (uint32_t)__popc(m & ((1u << lane) - 1u));
        if (take && pos < (uint32_t)cap) list[(size_t)b * cap + pos] = ((unsigned long long)key << 32) | (uint32_t)i;
    }
}

// one CTA per cloud: sort of the candidate list in shared memory, then the first N rows are gathered.  The sorting
// network is the bitonic one whose merges all run ascending (each merge starts by comparing i with its mirror in the
// block), so the entries past the list -- +inf in a power-of-two array -- never move and are never stored: the buffer
// holds `cap` entries, not the next power of two.  A cloud with fewer than N valid points or an overflowing list
// returns untouched (the host checks the state), or, with a status array, gets that status and a zero slot.
__global__ void __launch_bounds__(1024) k_rsel_sort_gather(const float *xyz, const __grid_constant__ RselClouds c, const RselState *st,
                                                           const unsigned long long *list, int cap, int cap2, int64_t N,
                                                           float *out, int32_t *index_out)
{
    extern __shared__ unsigned long long sm[];
    const int b = blockIdx.x;
    const uint32_t cnt = st[b].count;
    if (st[b].nvalid < (uint32_t)N || cnt > (uint32_t)cap) {
        if (c.status) {
            if (threadIdx.x == 0) {
                int32_t *sp = c.status + (int64_t)b * c.status_step;
                if (*sp == KP_OK) *sp = st[b].nvalid < (uint32_t)N ? KP_E_ARG : KP_E_RANGE;
            }
            for (int64_t e = threadIdx.x; e < 3 * N; e += 1024) out[3 * (size_t)b * (size_t)N + (size_t)e] = 0.0f;
        }
        return;
    }
    for (int e = threadIdx.x; e < cap; e += 1024) sm[e] = (uint32_t)e < cnt ? list[(size_t)b * cap + e] : ~0ull;
    __syncthreads();
    for (int size = 2; size <= cap2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < (cap2 >> 1); t += 1024) {
                int i, j;
                if (stride == (size >> 1)) {            // first step of a merge: i against its mirror in the block
                    i = (t / stride) * size + (t % stride);
                    j = (t / stride) * size + size - 1 - (t % stride);
                } else {
                    i = ((t / stride) * 2 * stride) + (t % stride);
                    j = i + stride;
                }
                if (j < cap) {
                    const unsigned long long x = sm[i], y = sm[j];
                    if (y < x) { sm[i] = y; sm[j] = x; }
                }
            }
            __syncthreads();
        }
    int64_t o, n;
    const float *src;
    rsel_cloud(c, xyz, b, o, n, src);
    for (int64_t t = threadIdx.x; t < N; t += 1024) {
        const int64_t i = (int64_t)(uint32_t)sm[t];
        float *dst = out + 3 * ((size_t)b * (size_t)N + (size_t)t);
        dst[0] = src[3 * i]; dst[1] = src[3 * i + 1]; dst[2] = src[3 * i + 2];
        if (index_out) index_out[(size_t)b * (size_t)N + (size_t)t] = (int32_t)i;
    }
}

// PREFIX mode with device counts: slot b = the first min(n, N) rows of cloud b, then zeros
__global__ void __launch_bounds__(256) k_rsel_prefix(const float *xyz, const __grid_constant__ RselClouds c, int64_t N, float *out)
{
    const int b = blockIdx.y;
    int64_t o, n;
    const float *src;
    rsel_cloud(c, xyz, b, o, n, src);
    const int64_t m3 = 3 * (n < N ? n : N);
    float *dst = out + 3 * (size_t)b * (size_t)N;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < 3 * N; e += (int64_t)gridDim.x * blockDim.x)
        dst[e] = e < m3 ? src[e] : 0.0f;
}

__global__ void __launch_bounds__(256) k_resample_gather(const float *xyz, const int32_t *order, int64_t N, float *out,
                                                         int32_t *index_out)
{
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N) return;
    const int64_t i = order[t];
    out[3 * t] = xyz[3 * i]; out[3 * t + 1] = xyz[3 * i + 1]; out[3 * t + 2] = xyz[3 * i + 2];
    if (index_out) index_out[t] = (int32_t)i;
}

// fallback for one cloud: full stable radix sort of (key, index); one 4-byte read validates N <= #valid
int resample_full_sort(kp_ctx *ctx, const float *d_xyz, int64_t n, int64_t N, uint64_t seed, uint64_t stream, float *d_out,
                       int32_t *d_index_out)
{
    uint32_t *keys, *keys_tmp, *keys_sorted;
    int32_t *vals, *vals_tmp, *vals_sorted;
    KP_TRY(kp_ws(ctx, (size_t)n, &keys));
    KP_TRY(kp_ws(ctx, (size_t)n, &keys_tmp));
    KP_TRY(kp_ws(ctx, (size_t)n, &vals));
    KP_TRY(kp_ws(ctx, (size_t)n, &vals_tmp));
    {
        KP_PROFB(ctx, "resample_keys", (double)n * (4.0 + 8.0));
        k_resample_keys<<<kp_blocks(n, 256), 256, 0, ctx->stream>>>(d_xyz, n, seed, stream, keys, vals);
        KP_LAUNCH_CHECK(ctx);
    }
    KP_TRY(kp_prim_sort_pairs_u32(ctx, n, 32, keys, keys_tmp, vals, vals_tmp, &keys_sorted, &vals_sorted));
    {
        KP_PROFB(ctx, "resample_gather", (double)N * (4.0 + 12.0 + 12.0));
        k_resample_gather<<<kp_blocks(N, 256), 256, 0, ctx->stream>>>(d_xyz, vals_sorted, N, d_out, d_index_out);
        KP_LAUNCH_CHECK(ctx);
    }
    // the N-th key is the NaN sentinel <=> fewer than N valid points
    KP_CUDA(ctx, cudaMemcpyAsync(ctx->d_scratch, keys_sorted + (N - 1), sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
    KP_TRY(kp_fetch_scratch(ctx, sizeof(uint32_t)));
    if (*(uint32_t *)ctx->h_scratch == 0xffffffffu)
        return kp_set_err(ctx, KP_E_ARG, "select_points_randomly: fewer than %lld valid (non-NaN) points", (long long)N);
    return KP_OK;
}

// list capacity of the candidate sort (N + the 2048 ties it tolerates) and the power of two its network spans
void rsel_sizes(int64_t N, int &cap, int &cap2)
{
    cap = (int)N + 2048;
    cap2 = 1024;
    while (cap2 < cap) cap2 <<= 1;
}
constexpr size_t RSEL_SORT_SMEM = 160 * 1024;

// the selection launches for B clouds: keys, three histogram + pick passes, collect, sort + gather.
// keys: one uint32 per row, addressed like the points; hist [B][RSEL_BINS] zero on entry (the picks leave it zero);
// st [B] zeroed here; list [B][cap].
int rsel_launch(kp_ctx *ctx, const float *d_xyz, const RselClouds &c, int B, int64_t N, uint64_t seed, unsigned gx, double rows,
                uint32_t *keys, uint32_t *hist, RselState *st, unsigned long long *list, float *d_out, int32_t *d_index_out)
{
    int cap, cap2;
    rsel_sizes(N, cap, cap2);
    KP_CUDA(ctx, cudaMemsetAsync(st, 0, sizeof(RselState) * (size_t)B, ctx->stream));
    const dim3 grid(gx, (unsigned)B);
    {
        KP_PROFB(ctx, "resample_keys", rows * (4.0 + 4.0));
        k_rsel_keys<<<grid, 256, 0, ctx->stream>>>(d_xyz, c, seed, keys, hist, st);
        KP_LAUNCH_CHECK(ctx);
    }
    {
        KP_PROFB(ctx, "resample_select", rows * (2.0 * 4.0 + 4.0) + (double)B * (double)N * 8.0);
        for (int pass = 0; pass < 3; ++pass) {
            if (pass > 0) {
                k_rsel_hist<<<grid, 256, 0, ctx->stream>>>(keys, c, pass, hist, st);
                KP_LAUNCH_CHECK(ctx);
            }
            k_rsel_pick<<<B, 256, 0, ctx->stream>>>(hist, pass, (uint32_t)N, st);
            KP_LAUNCH_CHECK(ctx);
        }
        k_rsel_collect<<<grid, 256, 0, ctx->stream>>>(keys, c, st, list, cap);
        KP_LAUNCH_CHECK(ctx);
    }
    {
        KP_PROFB(ctx, "resample_gather", (double)B * (double)N * (8.0 + 12.0 + 12.0));
        const size_t smem = (size_t)cap * sizeof(unsigned long long);
        if (smem > 48 * 1024)
            KP_CUDA(ctx, cudaFuncSetAttribute(k_rsel_sort_gather, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_rsel_sort_gather<<<B, 1024, smem, ctx->stream>>>(d_xyz, c, st, list, cap, cap2, N, d_out, d_index_out);
        KP_LAUNCH_CHECK(ctx);
    }
    return KP_OK;
}

// random mode for a batch of clouds given by host CSR offsets
int resample_select_batch(kp_ctx *ctx, const float *d_xyz, const int64_t *h_off, int B, int64_t N, uint64_t seed,
                          uint64_t first_stream, float *d_out, int32_t *d_index_out)
{
    int64_t total = h_off[B] - h_off[0], maxn = 0;
    for (int b = 0; b < B; ++b) maxn = h_off[b + 1] - h_off[b] > maxn ? h_off[b + 1] - h_off[b] : maxn;
    int cap, cap2;
    rsel_sizes(N, cap, cap2);
    const bool cta_sort = (size_t)cap * 8 <= RSEL_SORT_SMEM;
    if (!cta_sort || total <= 0) {
        for (int b = 0; b < B; ++b) {
            kp_ws_reset(ctx);
            KP_TRY(resample_full_sort(ctx, d_xyz + 3 * h_off[b], h_off[b + 1] - h_off[b], N, seed, first_stream + (uint64_t)b,
                                      d_out + 3 * (size_t)b * (size_t)N, d_index_out ? d_index_out + (size_t)b * (size_t)N : nullptr));
        }
        return KP_OK;
    }
    int64_t *d_off;
    uint32_t *keys, *hist;
    RselState *st;
    unsigned long long *list;
    KP_TRY(kp_ws(ctx, (size_t)B + 1, &d_off));
    KP_TRY(kp_ws(ctx, (size_t)total, &keys));
    KP_TRY(kp_ws(ctx, (size_t)B * RSEL_BINS, &hist));
    KP_TRY(kp_ws(ctx, (size_t)B, &st));
    KP_TRY(kp_ws(ctx, (size_t)B * (size_t)cap, &list));
    // offsets relative to d_xyz (the caller's rows h_off[0].. are addressed through them directly)
    KP_CUDA(ctx, cudaMemcpyAsync(d_off, h_off, sizeof(int64_t) * ((size_t)B + 1), cudaMemcpyHostToDevice, ctx->stream));
    KP_CUDA(ctx, cudaMemsetAsync(hist, 0, sizeof(uint32_t) * (size_t)B * RSEL_BINS, ctx->stream));
    uint32_t *keys_rel = keys - h_off[0];                     // keys[o + i] with o = absolute offset
    unsigned gx = (unsigned)((maxn + 2047) / 2048);
    if (gx < 1) gx = 1;
    if (gx > 1024) gx = 1024;
    RselClouds c;
    memset(&c, 0, sizeof c);
    c.off = d_off; c.first_stream = first_stream;
    KP_TRY(rsel_launch(ctx, d_xyz, c, B, N, seed, gx, (double)total, keys_rel, hist, st, list, d_out, d_index_out));
    // one read for the whole batch: valid counts (the ValueError of np.random.choice) and list overflows (fallback)
    std::vector<RselState> hs((size_t)B);
    KP_CUDA(ctx, cudaMemcpyAsync(hs.data(), st, sizeof(RselState) * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
    KP_TRY(kp_stream_wait(ctx));
    for (int b = 0; b < B; ++b)
        if ((int64_t)hs[(size_t)b].nvalid < N)
            return kp_set_err(ctx, KP_E_ARG, "select_points_randomly: cloud %d has %u valid (non-NaN) points, fewer than the %lld requested",
                              b, hs[(size_t)b].nvalid, (long long)N);
    for (int b = 0; b < B; ++b)
        if (hs[(size_t)b].count > (uint32_t)cap) {
            kp_ws_reset(ctx);
            KP_TRY(resample_full_sort(ctx, d_xyz + 3 * h_off[b], h_off[b + 1] - h_off[b], N, seed, first_stream + (uint64_t)b,
                                      d_out + 3 * (size_t)b * (size_t)N, d_index_out ? d_index_out + (size_t)b * (size_t)N : nullptr));
        }
    return KP_OK;
}
}  // namespace

extern "C" {

int kp_resample_fixed_n(kp_ctx *ctx, const float *d_xyz, int64_t n, int64_t N, int mode, uint64_t seed, uint64_t stream,
                        float *d_out, int32_t *d_index_out, int64_t *h_count)
{
    if (!ctx || (n > 0 && !d_xyz) || (N > 0 && !d_out)) return kp_set_err(ctx, KP_E_ARG, "kp_resample_fixed_n: NULL argument");
    if (N < 0 || n < 0 || n > 2147483000LL) return kp_set_err(ctx, KP_E_ARG, "kp_resample_fixed_n: bad size");
    if (mode != KP_RESAMPLE_RANDOM && mode != KP_RESAMPLE_PREFIX) return kp_set_err(ctx, KP_E_ARG, "kp_resample_fixed_n: bad mode");
    kp_enter(ctx);
    if (mode == KP_RESAMPLE_PREFIX) {
        const int64_t m = n < N ? n : N;
        if (m > 0) KP_CUDA(ctx, cudaMemcpyAsync(d_out, d_xyz, sizeof(float) * 3 * (size_t)m, cudaMemcpyDeviceToDevice, ctx->stream));
        if (h_count) *h_count = m;
        return KP_OK;
    }
    if (N > n) return kp_set_err(ctx, KP_E_ARG, "select_points_randomly: cannot take a larger sample (%lld) than population (%lld) when replace=False",
                                 (long long)N, (long long)n);
    if (h_count) *h_count = N;
    if (N == 0) return KP_OK;
    const int64_t off[2] = {0, n};
    return resample_select_batch(ctx, d_xyz, off, 1, N, seed, stream, d_out, d_index_out);
}

int kp_resample_batch(kp_ctx *ctx, const float *d_xyz, const int64_t *h_offsets, int B, int64_t N, int mode, uint64_t seed,
                      uint64_t first_stream, float *d_out, int64_t *h_counts)
{
    if (!ctx || !h_offsets || B < 0 || (B > 0 && N > 0 && !d_out)) return kp_set_err(ctx, KP_E_ARG, "kp_resample_batch: NULL argument");
    if (mode != KP_RESAMPLE_RANDOM && mode != KP_RESAMPLE_PREFIX) return kp_set_err(ctx, KP_E_ARG, "kp_resample_batch: bad mode");
    if (N < 0) return kp_set_err(ctx, KP_E_ARG, "kp_resample_batch: N < 0");
    kp_enter(ctx);
    for (int b = 0; b < B; ++b) {
        const int64_t n = h_offsets[b + 1] - h_offsets[b];
        if (n < 0 || n > 2147483000LL) return kp_set_err(ctx, KP_E_ARG, "kp_resample_batch: offsets must be non-decreasing");
        if (mode == KP_RESAMPLE_RANDOM && N > n)
            return kp_set_err(ctx, KP_E_ARG, "select_points_randomly: cloud %d: cannot take a larger sample (%lld) than population (%lld) when replace=False",
                              b, (long long)N, (long long)n);
    }
    if (B == 0 || N == 0) { if (h_counts) for (int b = 0; b < B; ++b) h_counts[b] = 0; return KP_OK; }
    if (mode == KP_RESAMPLE_PREFIX) {
        for (int b = 0; b < B; ++b) {
            const int64_t n = h_offsets[b + 1] - h_offsets[b], m = n < N ? n : N;
            float *o = d_out + 3 * (size_t)b * (size_t)N;
            if (m > 0) KP_CUDA(ctx, cudaMemcpyAsync(o, d_xyz + 3 * h_offsets[b], sizeof(float) * 3 * (size_t)m, cudaMemcpyDeviceToDevice, ctx->stream));
            // a short cloud: the tail of the [N][3] slot is zero-filled (a dense batch tensor)
            if (m < N) KP_CUDA(ctx, cudaMemsetAsync(o + 3 * (size_t)m, 0, sizeof(float) * 3 * (size_t)(N - m), ctx->stream));
            if (h_counts) h_counts[b] = m;
        }
        return KP_OK;
    }
    if (h_counts) for (int b = 0; b < B; ++b) h_counts[b] = N;
    return resample_select_batch(ctx, d_xyz, h_offsets, B, N, seed, first_stream, d_out, nullptr);
}

}  // extern "C"

// frame engine: fixed-N slot of every frame of a batch, without a host round trip.  Cloud b = d_n[b * n_step] rows
// from d_base[b] (keys at b * stride), sample stream h_ids[b]; d_status (int32 at b * status_step) takes KP_E_ARG for a RANDOM
// cloud with fewer than N points and KP_E_RANGE for an overflowing candidate list (a frame that already has a status
// keeps it); such a slot is zero-filled.  Work buffers (allocated by the caller once): keys [B * stride], hist
// [B][kp_resample_engine_hist_elems()] zero, st [B] (kp_resample_engine_state_bytes), list [B][kp_resample_engine_cap(N)].
int kp_resample_engine(kp_ctx *ctx, const float *const *d_base, int64_t stride, const int32_t *d_n, int64_t n_step, int B, int64_t N, int mode,
                       uint64_t seed, const int64_t *h_ids, int32_t *d_status, int64_t status_step, uint32_t *keys, uint32_t *hist,
                       void *st, unsigned long long *list, float *d_out)
{
    if (B <= 0) return KP_OK;
    if (B > RSEL_MAX_IDS) return kp_set_err(ctx, KP_E_ARG, "kp_resample_engine: at most %d clouds per launch", RSEL_MAX_IDS);
    RselClouds c;
    memset(&c, 0, sizeof c);
    c.base = d_base; c.stride = stride; c.n_dev = d_n; c.n_step = n_step; c.use_ids = 1;
    for (int b = 0; b < B; ++b) c.ids[b] = (uint64_t)h_ids[b];
    c.status = d_status; c.status_step = status_step;
    // the final clouds are a fraction of the stride: a few CTAs per SM, grid-stride over the rows
    int64_t gx = ((int64_t)ctx->sm_count * 4 + B - 1) / B;
    const int64_t gmax = (stride + 2047) / 2048;
    if (gx > gmax) gx = gmax;
    if (gx < 1) gx = 1;
    if (mode == KP_RESAMPLE_PREFIX) {
        KP_PROFB(ctx, "resample_prefix", (double)B * (double)N * (12.0 + 12.0));
        k_rsel_prefix<<<dim3((unsigned)gx, (unsigned)B), 256, 0, ctx->stream>>>(nullptr, c, N, d_out);
        KP_LAUNCH_CHECK(ctx);
        return KP_OK;
    }
    return rsel_launch(ctx, nullptr, c, B, N, seed, (unsigned)gx, (double)B * (double)stride, keys, hist, (RselState *)st, list, d_out,
                       nullptr);
}
size_t kp_resample_engine_hist_elems() { return RSEL_BINS; }
size_t kp_resample_engine_state_bytes() { return sizeof(RselState); }
int64_t kp_resample_engine_cap(int64_t N) { int cap, cap2; rsel_sizes(N, cap, cap2); return cap; }
bool kp_resample_engine_fits(int64_t N) { return (size_t)kp_resample_engine_cap(N) * 8 <= RSEL_SORT_SMEM; }

