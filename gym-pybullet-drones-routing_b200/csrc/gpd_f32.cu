// FP32 instantiation of the kernels (throughput mode; FMA contraction on).
#define GPD_REAL float
#include "gpd_launch.inl"

namespace gpd {
// precision-independent helpers live in this translation unit
// ---- episode statistics: reduce the per-block slots ----
__device__ __forceinline__ float ordered_to_float_h(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

__global__ void stats_reduce_kernel(const StatSlot* __restrict__ slots, int64_t nslots, double* __restrict__ out8)
{
    __shared__ double sh[8][32];
    double acc[8] = { 0, 0, 0, 0, 1e300, -1e300, 0, 0 };   // episodes, ret, len, ret^2, min, max, env_steps, terminated
    for (int64_t k = threadIdx.x; k < nslots; k += blockDim.x) {
        const StatSlot& s = slots[k];
        acc[0] += s.s[0]; acc[1] += s.s[1]; acc[2] += s.s[2]; acc[3] += s.s[3];
        if (s.s[0] > 0) { acc[4] = fmin(acc[4], (double)ordered_to_float_h(s.mn)); acc[5] = fmax(acc[5], (double)ordered_to_float_h(s.mx)); }
        acc[6] += s.s[4]; acc[7] += s.s[5];
    }
    for (int off = 16; off > 0; off >>= 1)
        for (int j = 0; j < 8; ++j) {
            double o = __shfl_down_sync(0xffffffffu, acc[j], off);
            if (j == 4) acc[j] = fmin(acc[j], o); else if (j == 5) acc[j] = fmax(acc[j], o); else acc[j] += o;
        }
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) for (int j = 0; j < 8; ++j) sh[j][w] = acc[j];
    __syncthreads();
    if (threadIdx.x == 0) {
        int nw = blockDim.x >> 5;
        for (int j = 0; j < 8; ++j) {
            double v = sh[j][0];
            for (int k = 1; k < nw; ++k) { if (j == 4) v = fmin(v, sh[j][k]); else if (j == 5) v = fmax(v, sh[j][k]); else v += sh[j][k]; }
            out8[j] = v;
        }
    }
}

__global__ void stats_clear_kernel(StatSlot* __restrict__ slots, int64_t nslots)
{
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nslots) return;
    StatSlot& s = slots[k];
    for (int j = 0; j < 6; ++j) s.s[j] = 0.0;
    s.mn = 0x7fffffff; s.mx = (int32_t)0x80000000;
}

// ============================================================================================
// Host mirror support: columns [j0, j1) of a row-major observation [D][W] -> feature-major out[(j - j0) * ld + d].
// Used when the host copy of the observation window is (re)built from the device chain: after a reset, when the
// window reaches the end of the host log (compaction) and when the mirror went stale (tensor-path steps in between).
// 32 x 32 tiles through padded shared memory: both sides coalesced.
// ============================================================================================
__global__ void __launch_bounds__(256)
transpose_cols_kernel(const float* __restrict__ obs, int64_t D, int W, int j0, int j1, float* __restrict__ out, int64_t ld)
{
    __shared__ float tile[32][33];
    const int64_t d0 = (int64_t)blockIdx.x * 32;
    const int c0 = j0 + (int)blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // 32 x 8
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int64_t d = d0 + r;
        const int j = c0 + tx;
        tile[r][tx] = (d < D && j < j1) ? obs[d * W + j] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int j = c0 + r;
        const int64_t d = d0 + tx;
        if (j < j1 && d < D) out[(int64_t)(j - j0) * ld + d] = tile[tx][r];
    }
}

cudaError_t launch_transpose_cols(const float* obs, int64_t D, int W, int j0, int j1, float* out, int64_t ld, cudaStream_t st)
{
    if (j1 <= j0 || D <= 0) return cudaSuccess;
    dim3 grid((unsigned)((D + 31) / 32), (unsigned)((j1 - j0 + 31) / 32));
    transpose_cols_kernel<<<grid, 256, 0, st>>>(obs, D, W, j0, j1, out, ld);
    return cudaGetLastError();
}

// ============================================================================================
// Chained-state handles (SimPtrs, StepArgs::state_in_obs): the state of every tile in chained state back into the arrays
// (position / velocity from the latest observation row, rates / episode return from sR), then the tile's flag cleared.
// One CTA per bulk tile.
// ============================================================================================
__global__ void __launch_bounds__(128) state_sync_kernel(const StepArgs<float> a, const float* __restrict__ obs)
{
    unsigned long long* flag = a.tile_seq + (int64_t)blockIdx.x * 4 + 1;
    if (*flag == 0ull || !obs) return;
    const int64_t d = (int64_t)blockIdx.x * a.DPB + threadIdx.x;
    if ((int)threadIdx.x < a.DPB && d < a.D) {
        const float* k = obs + d * a.W;
        const float4 r = a.sR[d];
        a.p.sP[d] = make_float4(k[0], k[1], k[2], r.x);
        a.p.sV[d] = make_float4(k[6], k[7], k[8], r.y);
        a.p.sWz[d] = r.z;
        if (a.p.ep_ret) a.p.ep_ret[d] = r.w;
    }
    __syncthreads();
    if (threadIdx.x == 0) *flag = 0ull;
}

cudaError_t launch_state_sync(const StepArgs<float>& a, const float* obs_latest, int64_t tiles, cudaStream_t st)
{
    state_sync_kernel<<<(unsigned)tiles, (a.DPB + 31) / 32 * 32, 0, st>>>(a, obs_latest);
    return cudaGetLastError();
}

// job-wide statistics from the all-gathered per-rank vectors {episodes, ret, len, ret^2, min, max, env_steps, terminated}:
// sums in rank order (deterministic), min/max over the ranks that finished at least one episode
__global__ void stats_combine_kernel(const double* __restrict__ g, int nranks, double* __restrict__ out8)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double acc[8] = { 0, 0, 0, 0, 1e300, -1e300, 0, 0 };
    for (int r = 0; r < nranks; ++r) {
        const double* v = g + (size_t)r * 8;
        acc[0] += v[0]; acc[1] += v[1]; acc[2] += v[2]; acc[3] += v[3]; acc[6] += v[6]; acc[7] += v[7];
        if (v[0] > 0) { acc[4] = fmin(acc[4], v[4]); acc[5] = fmax(acc[5], v[5]); }
    }
    for (int j = 0; j < 8; ++j) out8[j] = acc[j];
}

cudaError_t launch_stats_combine(const double* gathered, int nranks, double* out8, cudaStream_t st)
{
    stats_combine_kernel<<<1, 32, 0, st>>>(gathered, nranks, out8);
    return cudaGetLastError();
}

cudaError_t launch_stats(const StatSlot* slots, int64_t nslots, double* out8, int clear, StatSlot* slots_mut, cudaStream_t st)
{
    stats_reduce_kernel<<<1, 256, 0, st>>>(slots, nslots, out8);
    if (clear) stats_clear_kernel<<<(unsigned)((nslots + 127) / 128), 128, 0, st>>>(slots_mut, nslots);
    return cudaGetLastError();
}
}  // namespace gpd
