// hrp_norm.cu -- running observation / reward normalization of the batched loop (include/hrp.h, hrp_vecnorm_*).
//
// SB3's VecNormalize keeps per-element running mean / variance of the observation and a scalar one of the discounted
// return, both fp64 (RunningMeanStd, Chan's parallel merge).  Here a training step is three launches, so that no CTA
// reads a statistic while another one writes it:
//   moments  the batch moments (n, mean, M2) of every column over the E rows.  A CTA owns 32 columns x one chunk of rows;
//            each thread takes a strided eighth of the chunk two-pass (mean, then squared deviations), the eight are
//            merged in order, and the last CTA of a column tile merges the chunks in chunk order.  With rewards, the
//            return carry is updated here and is one more column.
//   merge    one thread per column combines the moments of R ranks in rank order and merges them into the running
//            statistics; the last CTA advances the counts, once every CTA has read them.
//   apply    normalizes the observation in place, the terminal observation of done envs and the reward, and clears the
//            carry of done envs.
// The per-thread two-pass moments stay accurate for a column far from the current running mean (the first update,
// where that mean is 0), which raw sums of x and x^2 do not.
#include <math.h>

#include "hrp_internal.cuh"

namespace {

constexpr int kCols = 32;           // columns of a CTA (threadIdx.x)
constexpr int kRowThreads = 8;      // threads over the rows of a chunk (threadIdx.y)
constexpr int kMaxChunks = 128;     // HRP_VECNORM_SCRATCH_LEN: 2 C partials per chunk
constexpr int kMinChunkRows = 64;
constexpr int kMergeThreads = 256;
constexpr int kTicketDoubles = 256; // scratch head: uint32 tickets, [0, 145) column tiles, kMergeTicket the merge
constexpr int kMergeTicket = 511;

struct Moments {
    double n, mean, m2;
};

// (n, mean, M2) of a and b together (Chan, Golub & LeVeque); a empty or b empty pass the other through
__device__ __forceinline__ Moments chan(Moments a, Moments b)
{
    if (b.n == 0.0) return a;
    if (a.n == 0.0) return b;
    const double n = a.n + b.n, d = b.mean - a.mean, f = b.n / n;   // one division per merge
    return {n, a.mean + d * f, a.m2 + b.m2 + d * d * a.n * f};
}

__device__ __forceinline__ double carry(double ret, double gamma, float reward)
{
    return __dadd_rn(__dmul_rn(ret, gamma), (double)reward);   // numpy's returns * gamma + reward, not contracted
}

__device__ __forceinline__ float normalize(float x, double mean, double inv_sd, double clip)
{
    const double v = ((double)x - mean) * inv_sd;
    return (float)fmin(fmax(v, -clip), clip);
}

// grid (column tiles, chunks), block (32, 8).  out: [n][mean C][M2 C]; scratch: tickets | partials [chunk][mean C | M2 C]
__global__ void __launch_bounds__(kCols * kRowThreads)
vecnorm_moments_kernel(const float *__restrict__ obs, long long E, int S, const float *__restrict__ reward,
                       double *__restrict__ ret, double gamma, long long chunk_rows, double *__restrict__ out,
                       double *__restrict__ scratch)
{
    __shared__ double sh[3][kRowThreads][kCols];
    __shared__ bool last;
    const int C = S + (reward ? 1 : 0);
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int c = blockIdx.x * kCols + tx;
    const long long r0 = (long long)blockIdx.y * chunk_rows, r1 = min(E, r0 + chunk_rows);
    const int chunks = (int)gridDim.y;
    unsigned *ticket = (unsigned *)scratch;
    double *part = scratch + kTicketDoubles;

    Moments m = {0.0, 0.0, 0.0};
    if (c < C) {
        double s = 0.0;
        for (long long e = r0 + ty; e < r1; e += kRowThreads) {
            double v;
            if (c < S) {
                v = (double)obs[e * S + c];
            } else {
                v = carry(ret[e], gamma, reward[e]);
                ret[e] = v;
            }
            s += v;
            m.n += 1.0;
        }
        if (m.n > 0.0) {
            m.mean = s / m.n;
            double q = 0.0;
            for (long long e = r0 + ty; e < r1; e += kRowThreads) {
                const double d = (c < S ? (double)obs[e * S + c] : ret[e]) - m.mean;
                q += d * d;
            }
            m.m2 = q;
        }
    }
    sh[0][ty][tx] = m.n; sh[1][ty][tx] = m.mean; sh[2][ty][tx] = m.m2;
    __syncthreads();
    if (ty == 0 && c < C) {
        for (int k = 1; k < kRowThreads; ++k) m = chan(m, {sh[0][k][tx], sh[1][k][tx], sh[2][k][tx]});
        part[(size_t)blockIdx.y * 2 * C + c] = m.mean;
        part[(size_t)blockIdx.y * 2 * C + C + c] = m.m2;
    }
    // the last CTA of this column tile merges the chunks, in chunk order
    __threadfence();
    __syncthreads();
    if (tx == 0 && ty == 0) last = atomicAdd(&ticket[blockIdx.x], 1u) == (unsigned)(chunks - 1);
    __syncthreads();
    if (!last) return;
    __threadfence();
    const int per = (chunks + kRowThreads - 1) / kRowThreads;
    m = {0.0, 0.0, 0.0};
    if (c < C) {
        for (int k = ty * per; k < min(chunks, (ty + 1) * per); ++k) {
            const long long k0 = (long long)k * chunk_rows;
            const double nk = (double)(min(E, k0 + chunk_rows) - k0);
            m = chan(m, {nk, __ldcg(&part[(size_t)k * 2 * C + c]), __ldcg(&part[(size_t)k * 2 * C + C + c])});
        }
    }
    sh[0][ty][tx] = m.n; sh[1][ty][tx] = m.mean; sh[2][ty][tx] = m.m2;
    __syncthreads();
    if (ty == 0 && c < C) {
        for (int k = 1; k < kRowThreads; ++k) m = chan(m, {sh[0][k][tx], sh[1][k][tx], sh[2][k][tx]});
        out[1 + c] = m.mean;
        out[1 + C + c] = m.m2;
        if (c == 0) out[0] = (double)E;
    }
    if (tx == 0 && ty == 0) ticket[blockIdx.x] = 0u;
}

// one thread per column: moments of R ranks in rank order, then RunningMeanStd.update_from_moments
__global__ void __launch_bounds__(kMergeThreads)
vecnorm_merge_kernel(const double *__restrict__ mom, int R, int S, int has_ret, double *__restrict__ obs_rms,
                     double *__restrict__ ret_rms, unsigned *__restrict__ ticket)
{
    __shared__ bool last;
    const int C = S + has_ret;
    const size_t stride = 1 + 2 * (size_t)C;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < C) {
        Moments b = {mom[0], mom[1 + c], mom[1 + C + c]};
        for (int r = 1; r < R; ++r) {
            const double *m = mom + r * stride;
            b = chan(b, {m[0], m[1 + c], m[1 + C + c]});
        }
        double *mean = c < S ? obs_rms + c : ret_rms;
        double *var = c < S ? obs_rms + S + c : ret_rms + 1;
        const double count = c < S ? obs_rms[2 * S] : ret_rms[2];
        const double bmean = b.mean, bvar = b.m2 / b.n, bc = b.n;
        const double delta = bmean - *mean, tot = count + bc;
        const double m2 = *var * count + bvar * bc + delta * delta * count * bc / tot;
        *mean = *mean + delta * bc / tot;
        *var = m2 / tot;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last || threadIdx.x != 0) return;
    double n = 0.0;
    for (int r = 0; r < R; ++r) n += mom[r * stride];
    if (S > 0) obs_rms[2 * S] += n;
    if (has_ret) ret_rms[2] += n;
    *ticket = 0u;
}

// grid (column tiles, row chunks), block (32, 8)
__global__ void __launch_bounds__(kCols * kRowThreads)
vecnorm_apply_kernel(float *__restrict__ obs, float *__restrict__ final_obs, const uint8_t *__restrict__ term,
                     const uint8_t *__restrict__ trunc, long long E, int S, const float *__restrict__ reward,
                     float *__restrict__ reward_out, double *__restrict__ ret, const double *__restrict__ obs_rms,
                     const double *__restrict__ ret_rms, double clip_obs, double clip_reward, double eps,
                     long long chunk_rows)
{
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int c = blockIdx.x * kCols + tx;
    const long long r0 = (long long)blockIdx.y * chunk_rows, r1 = min(E, r0 + chunk_rows);
    if (obs && c < S) {
        const double mean = obs_rms[c], inv_sd = 1.0 / sqrt(obs_rms[S + c] + eps);
        for (long long e = r0 + ty; e < r1; e += kRowThreads) {
            obs[e * S + c] = normalize(obs[e * S + c], mean, inv_sd, clip_obs);
            if (final_obs && (term[e] | trunc[e]))
                final_obs[e * S + c] = normalize(final_obs[e * S + c], mean, inv_sd, clip_obs);
        }
    }
    if (blockIdx.x != 0) return;
    const double inv_rsd = reward ? 1.0 / sqrt(ret_rms[1] + eps) : 0.0;
    for (long long e = r0 + tx + kCols * ty; e < r1; e += kCols * kRowThreads) {
        if (reward) reward_out[e] = normalize(reward[e], 0.0, inv_rsd, clip_reward);
        if (ret && term && (term[e] | trunc[e])) ret[e] = 0.0;
    }
}

bool bad_clip(double v) { return !(v > 0.0) || !isfinite(v); }

long long chunk_rows_of(long long E, long long max_chunks)
{
    long long chunks = (E + kMinChunkRows - 1) / kMinChunkRows;
    if (chunks > max_chunks) chunks = max_chunks;
    return (E + chunks - 1) / chunks;
}

int check_shape(const char *fn, int64_t E, int32_t S)
{
    if (E < 1 || E > HRP_VECNORM_MAX_E) {
        hrp_set_error("%s: E = %lld outside [1, %d]", fn, (long long)E, HRP_VECNORM_MAX_E);
        return -1;
    }
    if (S < 0 || S > HRP_VECNORM_MAX_S) {
        hrp_set_error("%s: S = %d outside [0, %d]", fn, (int)S, HRP_VECNORM_MAX_S);
        return -1;
    }
    return 0;
}

}  // namespace

extern "C" {

int hrp_vecnorm_moments(const float *obs, int64_t E, int32_t S, const float *reward, double *ret, double gamma,
                        double *moments, double *scratch, void *stream)
{
    if (check_shape("hrp_vecnorm_moments", E, S)) return -1;
    if (S > 0 && !obs) { hrp_set_error("hrp_vecnorm_moments: obs_dev is null with S = %d", (int)S); return -1; }
    if (S == 0 && !reward) { hrp_set_error("hrp_vecnorm_moments: no column (S = 0 and reward_dev null)"); return -1; }
    if (reward && !ret) { hrp_set_error("hrp_vecnorm_moments: returns_dev is null with reward_dev given"); return -1; }
    if (!moments || !scratch) {
        hrp_set_error("hrp_vecnorm_moments: %s is null", !moments ? "moments_dev" : "scratch_dev");
        return -1;
    }
    if (!(gamma >= 0.0 && gamma <= 1.0)) {
        hrp_set_error("hrp_vecnorm_moments: gamma = %g outside [0, 1]", gamma);
        return -1;
    }
    const int C = S + (reward ? 1 : 0);
    const long long rows = chunk_rows_of(E, kMaxChunks);
    const dim3 grid((unsigned)((C + kCols - 1) / kCols), (unsigned)((E + rows - 1) / rows));
    vecnorm_moments_kernel<<<grid, dim3(kCols, kRowThreads), 0, (cudaStream_t)stream>>>(obs, E, S, reward, ret, gamma,
                                                                                        rows, moments, scratch);
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}

int hrp_vecnorm_merge(const double *mom, int32_t R, int32_t S, int32_t has_ret, double *obs_rms, double *ret_rms,
                      double *scratch, void *stream)
{
    if (check_shape("hrp_vecnorm_merge", 1, S)) return -1;
    if (R < 1) { hrp_set_error("hrp_vecnorm_merge: R = %d < 1", (int)R); return -1; }
    if (has_ret != 0 && has_ret != 1) { hrp_set_error("hrp_vecnorm_merge: has_ret = %d is not 0 or 1", (int)has_ret); return -1; }
    if (S == 0 && !has_ret) { hrp_set_error("hrp_vecnorm_merge: no column (S = 0 and has_ret = 0)"); return -1; }
    const char *missing = !mom ? "moments_dev" : (S > 0 && !obs_rms) ? "obs_rms_dev"
                        : (has_ret && !ret_rms) ? "ret_rms_dev" : !scratch ? "scratch_dev" : nullptr;
    if (missing) { hrp_set_error("hrp_vecnorm_merge: %s is null", missing); return -1; }
    const int C = S + has_ret;
    vecnorm_merge_kernel<<<(C + kMergeThreads - 1) / kMergeThreads, kMergeThreads, 0, (cudaStream_t)stream>>>(
        mom, R, S, has_ret, obs_rms, ret_rms, (unsigned *)scratch + kMergeTicket);
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}

int hrp_vecnorm_apply(float *obs, float *final_obs, const uint8_t *term, const uint8_t *trunc, int64_t E, int32_t S,
                      const float *reward, float *reward_out, double *ret, const double *obs_rms,
                      const double *ret_rms, double clip_obs, double clip_reward, double eps, void *stream)
{
    if (check_shape("hrp_vecnorm_apply", E, S)) return -1;
    if (S > 0 && (!obs || !obs_rms)) {
        hrp_set_error("hrp_vecnorm_apply: %s is null with S = %d", !obs ? "obs_dev" : "obs_rms_dev", (int)S);
        return -1;
    }
    if (S == 0 && !reward) { hrp_set_error("hrp_vecnorm_apply: no column (S = 0 and reward_dev null)"); return -1; }
    if (reward && (!reward_out || !ret_rms)) {
        hrp_set_error("hrp_vecnorm_apply: %s is null with reward_dev given", !reward_out ? "reward_out_dev" : "ret_rms_dev");
        return -1;
    }
    if ((term == nullptr) != (trunc == nullptr)) {
        hrp_set_error("hrp_vecnorm_apply: %s is null and the other flag is not", !term ? "terminated_dev" : "truncated_dev");
        return -1;
    }
    if (final_obs && (!term || S == 0)) {
        hrp_set_error("hrp_vecnorm_apply: final_obs_dev needs terminated_dev / truncated_dev and S > 0");
        return -1;
    }
    if (bad_clip(clip_obs)) { hrp_set_error("hrp_vecnorm_apply: clip_obs = %g is not finite and > 0", clip_obs); return -1; }
    if (bad_clip(clip_reward)) {
        hrp_set_error("hrp_vecnorm_apply: clip_reward = %g is not finite and > 0", clip_reward);
        return -1;
    }
    if (!(eps >= 0.0) || !isfinite(eps)) { hrp_set_error("hrp_vecnorm_apply: epsilon = %g is not finite and >= 0", eps); return -1; }
    const long long rows = chunk_rows_of(E, 65535);
    const dim3 grid((unsigned)(S > 0 ? (S + kCols - 1) / kCols : 1), (unsigned)((E + rows - 1) / rows));
    vecnorm_apply_kernel<<<grid, dim3(kCols, kRowThreads), 0, (cudaStream_t)stream>>>(
        S > 0 ? obs : nullptr, final_obs, term, trunc, E, S, reward, reward_out, ret, obs_rms, ret_rms, clip_obs,
        clip_reward, eps, rows);
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
