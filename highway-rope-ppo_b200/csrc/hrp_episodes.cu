// hrp_episodes.cu -- episode returns and lengths of the batched loop (include/hrp.h, hrp_episode_stats).
//
// The reference accumulates `ep_reward += reward` per episode in Python floats (training/routine.py:143) and evaluates
// deterministic episodes one env step at a time (routine.py:14-29).  Here the time-major [T, E] reward and flag buffers
// the step kernel already wrote into the rollout are scanned forward, one thread per env (the mirror image of
// gae_kernel), with each env's running return / length carried across calls in fp64 / int32.  Every finished episode
// goes into per-thread sums, which are reduced in a fixed order (warp tree, warps in order, CTAs in order), so equal
// inputs give the same bits on every run.
#include "hrp_internal.cuh"

namespace {

constexpr int kStats = 6;          // episodes, sum return, sum return^2, sum length, terminated, truncated only
constexpr int kThreads = 256;
constexpr int kMaxCtas = 512;      // the scratch tail holds kStats partials per CTA

__global__ void __launch_bounds__(kThreads)
episode_stats_kernel(const float *__restrict__ reward, const uint8_t *__restrict__ terminated,
                     const uint8_t *__restrict__ truncated, long long T, long long E, uint8_t *__restrict__ active,
                     double *__restrict__ ret, int32_t *__restrict__ len, double *__restrict__ part)
{
    __shared__ double red[kThreads / 32][kStats];
    double acc[kStats] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (long long)gridDim.x * blockDim.x) {
        if (active && !active[e]) continue;
        double r = ret[e];
        int32_t n = len[e];
        for (long long t = 0; t < T; ++t) {
            const size_t o = (size_t)t * E + e;
            r = __dadd_rn(r, (double)reward[o]);   // the reference's Python-float running sum, step by step
            n += 1;
            const bool term = terminated[o] != 0, tr = truncated[o] != 0;
            if (term || tr) {
                acc[0] += 1.0;
                acc[1] += r;
                acc[2] += r * r;
                acc[3] += (double)n;
                acc[4] += term ? 1.0 : 0.0;       // terminated and truncated on one step counts as terminated
                acc[5] += term ? 0.0 : 1.0;
                if (active) {                      // evaluation: the first episode is the one; freeze the env
                    active[e] = 0;
                    break;
                }
                r = 0.0;                           // training: the env has already respawned
                n = 0;
            }
        }
        ret[e] = r;
        len[e] = n;
    }
#pragma unroll
    for (int k = 0; k < kStats; ++k)
        for (int d = 16; d > 0; d >>= 1) acc[k] += __shfl_xor_sync(HRP_FULL, acc[k], d);
    if ((threadIdx.x & 31) == 0)
        for (int k = 0; k < kStats; ++k) red[threadIdx.x >> 5][k] = acc[k];
    __syncthreads();
    if (threadIdx.x < kStats) {
        double s = 0.0;
        for (int w = 0; w < kThreads / 32; ++w) s += red[w][threadIdx.x];
        part[(size_t)blockIdx.x * kStats + threadIdx.x] = s;
    }
}

// stats[k] += sum over CTAs of part[cta][k], CTAs in index order
__global__ void episode_stats_final_kernel(const double *__restrict__ part, int nblocks, double *__restrict__ stats)
{
    if (blockIdx.x == 0 && threadIdx.x < kStats) {
        double s = 0.0;
        for (int i = 0; i < nblocks; ++i) s += part[(size_t)i * kStats + threadIdx.x];
        stats[threadIdx.x] += s;
    }
}

}  // namespace

extern "C" {

int hrp_episode_stats(const float *reward, const uint8_t *terminated, const uint8_t *truncated, int64_t T, int64_t E,
                      uint8_t *active, double *ret, int32_t *len, double *stats, void *stream)
{
    const char *missing = !reward ? "reward_dev" : !terminated ? "terminated_dev" : !truncated ? "truncated_dev"
                        : !ret ? "return_dev" : !len ? "length_dev" : !stats ? "stats_dev" : nullptr;
    if (missing) { hrp_set_error("hrp_episode_stats: %s is null", missing); return -1; }
    if (T < 1) { hrp_set_error("hrp_episode_stats: T = %lld < 1", (long long)T); return -1; }
    if (E < 1) { hrp_set_error("hrp_episode_stats: E = %lld < 1", (long long)E); return -1; }
    long long blocks = (E + kThreads - 1) / kThreads;
    if (blocks > kMaxCtas) blocks = kMaxCtas;
    cudaStream_t s = (cudaStream_t)stream;
    episode_stats_kernel<<<(unsigned)blocks, kThreads, 0, s>>>(reward, terminated, truncated, T, E, active, ret, len,
                                                               stats + kStats);
    episode_stats_final_kernel<<<1, 32, 0, s>>>(stats + kStats, (int)blocks, stats);
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
