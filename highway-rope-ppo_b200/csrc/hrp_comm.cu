// hrp_comm.cu -- the one exchange of the data-parallel PPO path (SURVEY.md 8e), fused with its consumer.
//
// Every rank (one process per GPU, same box) holds the gradient of its shard of the minibatch in a buffer that its
// peers can read through NVLink (cudaIpc).  `hrp_clip_adam_step_p2p` is ONE cooperative kernel per optimizer step:
//
//   1. "my gradient of step e is complete": an epoch word written into every peer's flag block; every CTA polls the
//      W words of its own block (no grid-wide barrier around the cross-GPU wait);
//   2. REDUCE-SCATTER: rank r sums ONLY its 1/W slice of the W gradients, in rank order, with peer loads over NVLink
//      (n (W-1)/W floats read per rank instead of n (W-1));
//   3. ALL-GATHER by push: rank r stores its reduced slice into the `sum` buffer of every rank (its own included) and
//      then raises the per-source epoch word "slice r of step e has arrived" in every peer -- the data flag IS the
//      synchronisation, there is no separate barrier;
//   4. every CTA waits for the W slice words, reads the complete sum (local memory now; the same values in the same
//      order on every rank, hence bit-identical parameters), accumulates its square;
//   5. grid.sync(), fixed-order total -> clip coefficient (clip_grad_norm_, agent.py:249), Adam (agent.py:252).
//
// There is NO "done reading" barrier: the gradient and the sum buffers are DOUBLE-BUFFERED by step parity.  A rank
// overwrites its parity-p buffers at step e + 2, i.e. after its step e + 1 kernel has finished, which waited for every
// peer's "gradient e + 1 complete" word, which a peer raises only after its own step e kernel (the last reader / writer
// of the parity-p buffers of step e) has finished, by stream order.
//
// It replaces all_reduce(grad) + gradnorm + clip + Adam (NCCL launch + 1 kernel) of the NCCL path.  The flags carry
// a monotonically increasing epoch kept in device memory, so the launch can be captured in a CUDA graph and replayed;
// the parity is a launch parameter (the host alternates it; a captured graph keeps the parity it was captured with).
// Kernels of different ranks spin on each other: every rank owns its GPU (never run two ranks on one device).
#include <cooperative_groups.h>
#include <math.h>
#include <string.h>

#include "hrp_internal.cuh"

#define HRP_MAX_RANKS 8

struct hrp_comm {
    int world, rank, device;
    long long n;             // floats per gradient
    long long npad;          // n rounded up to 32 floats
    float *local;            // [grad parity 0 | grad parity 1 | sum parity 0 | sum parity 1 | flags], the IPC-exported allocation
    void *peer_base[HRP_MAX_RANKS];
    unsigned *epoch;         // device: [0] counter of completed steps, [1] timeout bits of the cross-GPU waits
    unsigned long long issued;   // optimizer steps enqueued so far (host): the parity of the next one
    bool connected;
};

namespace {

constexpr int P2P_MAX_CTAS = 120, P2P_THREADS = 512;

// flag block of a rank, [2 kinds][HRP_MAX_RANKS] epoch words: kind 0 = "rank q's gradient is complete", kind 1 = "rank
// q's reduced slice has arrived here"; word q is written by rank q
struct PeerTable {
    float *base[HRP_MAX_RANKS];   // every rank's exported allocation as mapped here
};

__device__ __forceinline__ void st_release_sys(unsigned *p, unsigned v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// wait until the W epoch words of `kind` in this rank's own flag block have reached `epoch`.  Called by a whole CTA:
// thread q < W polls word q.  Bounded (about fifteen seconds of SM clock): a peer that never arrives -- a crashed
// process -- must not leave this GPU spinning; the timeout is recorded in *status (bit `kind`) and the step goes on
// with whatever the buffers hold, for the host to detect (hrp_comm_status).
__device__ __forceinline__ void wait_words(const unsigned *mine, int world, int kind, unsigned epoch, unsigned *status)
{
    if ((int)threadIdx.x < world) {
        const unsigned *w = mine + kind * HRP_MAX_RANKS + threadIdx.x;
        const long long t0 = clock64();
        while ((int)(ld_acquire_sys(w) - epoch) < 0) {
            __nanosleep(32);
            if (clock64() - t0 > 30000000000ll) { atomicOr(status, 1u << kind); break; }
        }
    }
    __syncthreads();
}

// LR_DEV: the learning rate is *lr_dev, as in hrp_ppo.cu's clip_adam_kernel.  KL (target_kl early stopping): the
// exchange covers n = P + 1 floats, the last being every rank's approx-KL share, so the summed KL arrives with the
// gradient (the same bits on every rank); clip and Adam cover the first P.  The step is not taken when *stop is already
// set or the summed KL exceeds kl_limit, and in the second case the kernel raises *stop: both are read before the grid
// barrier, the word is written after it.  The exchange itself (flags, epoch) runs either way, so a rank never waits for
// a peer that skipped it.
template <bool LR_DEV, bool KL>
__global__ void __launch_bounds__(P2P_THREADS)
clip_adam_p2p_kernel(const PeerTable T, int world, int rank, int parity, long long npad, unsigned *__restrict__ epoch_dev,
                     float *__restrict__ p, float *__restrict__ m, float *__restrict__ v, int32_t *__restrict__ step,
                     long long n, double lr, double beta1, double beta2, double eps, float max_norm,
                     float *__restrict__ part, unsigned *__restrict__ arrive, const double *__restrict__ lr_dev,
                     unsigned *__restrict__ stop, double kl_limit)
{
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ float red[P2P_THREADS / 32];
    __shared__ float s_coef, s_step_size, s_bc2_sqrt;
    __shared__ bool s_last;
    // read before anything of this step is written (CTA 0 advances them at the very end, after the grid barrier)
    const unsigned epoch = *epoch_dev + 1u;
    const int k = step[0] + 1;
    const bool stopped = KL && *stop != 0u;
    unsigned *flags_of[HRP_MAX_RANKS];
#pragma unroll
    for (int q = 0; q < HRP_MAX_RANKS; ++q) flags_of[q] = q < world ? (unsigned *)(T.base[q] + 4 * npad) : nullptr;
    unsigned *mine = flags_of[rank];
    // 1. my gradient (written by the kernels before this one in the stream) is complete: tell every rank
    if (blockIdx.x == 0 && (int)threadIdx.x < world) {
        __threadfence_system();
        st_release_sys(flags_of[threadIdx.x] + 0 * HRP_MAX_RANKS + rank, epoch);
    }
    wait_words(mine, world, 0, epoch, epoch_dev + 1);
    // 2. reduce-scatter: my slice [lo, hi) of the W gradients, rank order (identical on every rank)
    const long long chunk = ((n + world - 1) / world + 3) / 4 * 4;
    const long long lo = min(n, chunk * rank), hi = min(n, lo + chunk);
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long i = lo + i0; i < hi; i += stride) {
        float g = 0.f;
#pragma unroll
        for (int q = 0; q < HRP_MAX_RANKS; ++q)
            if (q < world) g += __ldcg(T.base[q] + (size_t)parity * npad + i);
        // 3. all-gather by push: the reduced value goes into every rank's sum buffer
#pragma unroll
        for (int q = 0; q < HRP_MAX_RANKS; ++q)
            if (q < world) __stcg(T.base[q] + (size_t)(2 + parity) * npad + i, g);
    }
    // the last CTA to finish its part of the slice raises "slice `rank` of step `epoch` has arrived" everywhere
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned prev = atomicAdd(arrive, 1u);
        s_last = prev == gridDim.x - 1;
        if (s_last) *arrive = 0u;
    }
    __syncthreads();
    if (s_last && (int)threadIdx.x < world) {
        __threadfence_system();
        st_release_sys(flags_of[threadIdx.x] + 1 * HRP_MAX_RANKS + rank, epoch);
    }
    // 4. the complete sum is local once every slice has arrived
    wait_words(mine, world, 1, epoch, epoch_dev + 1);
    const float *gsum = T.base[rank] + (size_t)(2 + parity) * npad;
    const long long np = KL ? n - 1 : n;   // floats of the parameters
    const bool skip = KL && (stopped || (double)__ldcg(gsum + np) > kl_limit);
    float s = 0.f;
    for (long long i = i0; i < np; i += stride) {
        const float g = __ldcg(gsum + i);
        s = fmaf(g, g, s);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(HRP_FULL, s, d);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < P2P_THREADS / 32; ++i) t += red[i];
        part[blockIdx.x] = t;
    }
    grid.sync();
    // 5. clip coefficient and Adam, as hrp_clip_adam_step
    if (threadIdx.x < 32) {
        float t = 0.f;
        for (int i = threadIdx.x * 4; i < min((int)gridDim.x, threadIdx.x * 4 + 4); ++i) t += __ldcg(part + i);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) t += __shfl_xor_sync(HRP_FULL, t, d);
        if (threadIdx.x == 0) {
            float total_norm = sqrtf(t);
            float c = max_norm / (total_norm + 1e-6f);
            s_coef = max_norm > 0.f ? fminf(c, 1.f) : 1.f;
            double bc1 = 1.0 - pow(beta1, (double)k), bc2 = 1.0 - pow(beta2, (double)k);
            s_step_size = (float)((LR_DEV ? *lr_dev : lr) / bc1);
            s_bc2_sqrt = (float)sqrt(bc2);
        }
    }
    __syncthreads();
    const float w1 = (float)(1.0 - beta1), b2 = (float)beta2, w2 = (float)(1.0 - beta2), ep = (float)eps;
    const float coef = s_coef, step_size = s_step_size, bc2_sqrt = s_bc2_sqrt;
    for (long long i = i0; i < (skip ? 0 : np); i += stride) {
        float gi = __ldcg(gsum + i) * coef;
        float mi = m[i] + w1 * (gi - m[i]);
        float vi = v[i] * b2 + w2 * gi * gi;
        m[i] = mi; v[i] = vi;
        float denom = sqrtf(vi) / bc2_sqrt + ep;
        p[i] = p[i] - step_size * (mi / denom);
    }
    // every CTA read step[0] / *epoch_dev before the grid barrier above
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (!skip) step[0] = k;
        else if (!stopped) *stop = 1u;
        *epoch_dev = epoch;
    }
}

inline size_t comm_floats(long long n) { return (size_t)(4 * ((n + 31) / 32 * 32) + 64); }

}  // namespace

extern "C" {

int hrp_comm_create(int32_t world, int32_t rank, int64_t n, int32_t device, hrp_comm **out, void *handle_out64)
{
    if (!out || !handle_out64 || world < 1 || world > HRP_MAX_RANKS || rank < 0 || rank >= world || n < 1) {
        hrp_set_error("hrp_comm_create: bad arguments (world <= %d)", HRP_MAX_RANKS);
        return -1;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    HRP_CUDA_OK(cudaSetDevice(device));
    hrp_comm *c = new hrp_comm();
    c->world = world; c->rank = rank; c->device = device; c->n = n;
    c->npad = (n + 31) / 32 * 32; c->issued = 0;
    size_t bytes = comm_floats(n) * sizeof(float);
    cudaError_t ce = cudaMalloc(&c->local, bytes);
    if (ce == cudaSuccess) ce = cudaMemset(c->local, 0, bytes);
    if (ce == cudaSuccess) ce = cudaMalloc(&c->epoch, 4 * sizeof(unsigned));   // epoch, timeout bits, CTA arrival counter
    if (ce == cudaSuccess) ce = cudaMemset(c->epoch, 0, 4 * sizeof(unsigned));
    cudaIpcMemHandle_t hd;
    if (ce == cudaSuccess) ce = cudaIpcGetMemHandle(&hd, c->local);
    if (ce != cudaSuccess) {
        hrp_set_error("hrp_comm_create: %s", cudaGetErrorString(ce));
        cudaFree(c->local); cudaFree(c->epoch); delete c;
        return -2;
    }
    memcpy(handle_out64, &hd, 64);
    HRP_CUDA_OK(cudaDeviceSynchronize());
    *out = c;
    return 0;
}

/* handles: world x 64 bytes, rank-major, as gathered from every rank's hrp_comm_create */
int hrp_comm_connect(hrp_comm *c, const void *handles)
{
    if (!c || !handles) { hrp_set_error("hrp_comm_connect: null argument"); return -1; }
    HRP_CUDA_OK(cudaSetDevice(c->device));
    for (int q = 0; q < c->world; ++q) {
        void *base = c->local;
        if (q != c->rank) {
            cudaIpcMemHandle_t hd;
            memcpy(&hd, (const char *)handles + 64 * q, 64);
            HRP_CUDA_OK(cudaIpcOpenMemHandle(&base, hd, cudaIpcMemLazyEnablePeerAccess));
        }
        c->peer_base[q] = base;
    }
    c->connected = true;
    return 0;
}

/* device pointer of the gradient buffer (n floats) the NEXT hrp_clip_adam_step_p2p will exchange: hrp_ppo_loss_grad
 * writes it.  The buffers alternate with the parity of the step. */
float *hrp_comm_grad(hrp_comm *c) { return c ? c->local + (size_t)(c->issued & 1) * c->npad : nullptr; }
/* the same for an explicit parity (0 / 1): callers that capture steps in CUDA graphs keep one graph per parity */
float *hrp_comm_grad_parity(hrp_comm *c, int32_t parity) { return c ? c->local + (size_t)(parity & 1) * c->npad : nullptr; }
int hrp_comm_parity(hrp_comm *c) { return c ? (int)(c->issued & 1) : -1; }

}  // extern "C"

template <bool LR_DEV, bool KL>
static int clip_adam_p2p_launch(hrp_comm *c, float *params, float *exp_avg, float *exp_avg_sq, int32_t *step, double lr,
                                const double *lr_dev, double beta1, double beta2, double eps, float max_grad_norm,
                                float *scratch, void *stream, unsigned *stop = nullptr, double kl_limit = 0.0)
{
    static int max_ctas_dev[HRP_MAX_DEVICES] = {0};
    if (c->device < 0 || c->device >= HRP_MAX_DEVICES) { hrp_set_error("device index %d not supported", c->device); return -1; }
    int &max_ctas = max_ctas_dev[c->device];
    if (max_ctas == 0) {
        int sms = 0, per_sm = 0;
        HRP_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
        HRP_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, clip_adam_p2p_kernel<LR_DEV, KL>, P2P_THREADS, 0));
        max_ctas = sms * per_sm < P2P_MAX_CTAS ? sms * per_sm : P2P_MAX_CTAS;
        if (max_ctas < 1) { hrp_set_error("hrp_clip_adam_step_p2p: kernel does not fit the device"); return -2; }
    }
    PeerTable T;
    for (int q = 0; q < HRP_MAX_RANKS; ++q) T.base[q] = q < c->world ? (float *)c->peer_base[q] : nullptr;
    long long n = c->n, npad = c->npad;
    int ctas = (int)((n + P2P_THREADS - 1) / P2P_THREADS);
    if (ctas > max_ctas) ctas = max_ctas;
    int world = c->world, rank = c->rank, parity = (int)(c->issued & 1);
    unsigned *epoch = c->epoch, *arrive = c->epoch + 2;
    void *args[] = {&T, &world, &rank, &parity, &npad, &epoch, &params, &exp_avg, &exp_avg_sq, &step, &n, &lr, &beta1, &beta2,
                    &eps, &max_grad_norm, &scratch, &arrive, &lr_dev, &stop, &kl_limit};
    HRP_CUDA_OK(cudaLaunchCooperativeKernel((const void *)clip_adam_p2p_kernel<LR_DEV, KL>, dim3(ctas), dim3(P2P_THREADS), args, 0,
                                            (cudaStream_t)stream));
    c->issued += 1;
    return 0;
}

extern "C" {

int hrp_clip_adam_step_p2p(hrp_comm *c, float *params, float *exp_avg, float *exp_avg_sq, int32_t *step, double lr,
                           double beta1, double beta2, double eps, float max_grad_norm, float *scratch, void *stream)
{
    if (!c || !c->connected || !params || !exp_avg || !exp_avg_sq || !step || !scratch) {
        hrp_set_error("hrp_clip_adam_step_p2p: bad arguments (hrp_comm_connect first)");
        return -1;
    }
    return clip_adam_p2p_launch<false, false>(c, params, exp_avg, exp_avg_sq, step, lr, nullptr, beta1, beta2, eps, max_grad_norm,
                                              scratch, stream);
}

int hrp_clip_adam_step_p2p_ex(hrp_comm *c, float *params, float *exp_avg, float *exp_avg_sq, int32_t *step, double lr,
                              const double *lr_dev, double beta1, double beta2, double eps, float max_grad_norm,
                              float *scratch, void *stream)
{
    const char *bad = !c ? "comm" : !c->connected ? "comm (hrp_comm_connect first)" : !params ? "params_dev"
                    : !exp_avg ? "exp_avg_dev" : !exp_avg_sq ? "exp_avg_sq_dev" : !step ? "step_dev"
                    : !scratch ? "scratch_dev" : nullptr;
    if (bad) { hrp_set_error("hrp_clip_adam_step_p2p_ex: bad argument %s", bad); return -1; }
    if (!lr_dev)
        return clip_adam_p2p_launch<false, false>(c, params, exp_avg, exp_avg_sq, step, lr, nullptr, beta1, beta2, eps,
                                                  max_grad_norm, scratch, stream);
    return clip_adam_p2p_launch<true, false>(c, params, exp_avg, exp_avg_sq, step, lr, lr_dev, beta1, beta2, eps, max_grad_norm,
                                             scratch, stream);
}

int hrp_clip_adam_step_p2p_kl(hrp_comm *c, float *params, float *exp_avg, float *exp_avg_sq, int32_t *step, double lr,
                              const double *lr_dev, double beta1, double beta2, double eps, float max_grad_norm,
                              float *scratch, uint32_t *stop, double kl_limit, void *stream)
{
    const char *bad = !c ? "comm" : !c->connected ? "comm (hrp_comm_connect first)" : !params ? "params_dev"
                    : !exp_avg ? "exp_avg_dev" : !exp_avg_sq ? "exp_avg_sq_dev" : !step ? "step_dev"
                    : !scratch ? "scratch_dev" : stop && c->n < 2 ? "comm (created with n_floats = P + 1 >= 2)"
                    : stop && !(isfinite(kl_limit) && kl_limit > 0.0) ? "kl_limit" : nullptr;
    if (bad) { hrp_set_error("hrp_clip_adam_step_p2p_kl: bad argument %s", bad); return -1; }
    if (!stop)
        return lr_dev ? clip_adam_p2p_launch<true, false>(c, params, exp_avg, exp_avg_sq, step, lr, lr_dev, beta1, beta2,
                                                          eps, max_grad_norm, scratch, stream)
                      : clip_adam_p2p_launch<false, false>(c, params, exp_avg, exp_avg_sq, step, lr, nullptr, beta1, beta2,
                                                           eps, max_grad_norm, scratch, stream);
    return lr_dev ? clip_adam_p2p_launch<true, true>(c, params, exp_avg, exp_avg_sq, step, lr, lr_dev, beta1, beta2, eps,
                                                     max_grad_norm, scratch, stream, stop, kl_limit)
                  : clip_adam_p2p_launch<false, true>(c, params, exp_avg, exp_avg_sq, step, lr, nullptr, beta1, beta2, eps,
                                                      max_grad_norm, scratch, stream, stop, kl_limit);
}

/* a captured graph replays the parity it was captured with: the host says which step it is about to replay */
int hrp_comm_note_replay(hrp_comm *c)
{
    if (!c) { hrp_set_error("hrp_comm_note_replay: null argument"); return -1; }
    c->issued += 1;
    return 0;
}

/* synchronises the device; 0 = every cross-GPU wait so far was answered, -4 = a peer did not arrive within the
 * timeout of some step (its results are not to be trusted) */
int hrp_comm_status(hrp_comm *c)
{
    if (!c) { hrp_set_error("hrp_comm_status: null argument"); return -1; }
    HRP_CUDA_OK(cudaSetDevice(c->device));
    unsigned st[2] = {0, 0};
    HRP_CUDA_OK(cudaMemcpy(st, c->epoch, sizeof(st), cudaMemcpyDeviceToHost));
    if (st[1] != 0) { hrp_set_error("hrp_comm: a peer rank did not reach the gradient exchange (wait bits %u) after %u steps", st[1], st[0]); return -4; }
    return 0;
}

int hrp_comm_destroy(hrp_comm *c)
{
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (int q = 0; q < c->world; ++q)
        if (c->connected && q != c->rank && c->peer_base[q]) cudaIpcCloseMemHandle(c->peer_base[q]);
    cudaFree(c->local);
    cudaFree(c->epoch);
    delete c;
    return 0;
}

}  // extern "C"
