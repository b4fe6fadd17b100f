// hrp_ppo.cu -- the PPO half of the hot path (reference: ppo/agent.py).
//
//   ActorCritic.forward / get_action / evaluate      agent.py:46-84
//   PPOMemory.compute_advantages (GAE)               agent.py:126-138
//   advantage normalisation                          agent.py:204
//   clipped surrogate + value MSE + entropy, backward agent.py:218-248
//   clip_grad_norm_ + Adam.step                      agent.py:249-252
//
// Parameters live in one flat fp32 buffer in ActorCritic.parameters() order (the root
// module's own Parameter first): log_std[A], shared.0.{weight[H,S],bias[H]},
// shared.2.{weight[H,H],bias[H]}, actor_mean.0.{weight[H,H],bias[H]},
// actor_mean.2.{weight[A,H],bias[A]}, critic.0.{weight[H,H],bias[H]}, critic.2.{weight[1,H],bias[1]}.
// Gradients, Adam moments use the same layout, so the optimizer (and the multi-GPU
// all-reduce) touch one contiguous range.  The categorical policy (HRP_PPO_CATEGORICAL) has the same layout without
// log_std, A = n logits in actor_mean.2.
#include <cooperative_groups.h>
#include <math.h>

#include <cmath>
#include <stdlib.h>

#include "hrp_internal.cuh"

namespace {

struct Layout {
    int S, A, H;
    long long log_std, w1, b1, w2, b2, wa1, ba1, wa2, ba2, wc1, bc1, wc2, bc2, total;
};
__host__ __device__ inline Layout make_layout(int S, int A, int H, bool categorical = false)
{
    Layout L;
    L.S = S; L.A = A; L.H = H;
    long long o = 0;
    L.log_std = o; o += categorical ? 0 : A;
    L.w1 = o; o += (long long)H * S; L.b1 = o; o += H;
    L.w2 = o; o += (long long)H * H; L.b2 = o; o += H;
    L.wa1 = o; o += (long long)H * H; L.ba1 = o; o += H;
    L.wa2 = o; o += (long long)A * H; L.ba2 = o; o += A;
    L.wc1 = o; o += (long long)H * H; L.bc1 = o; o += H;
    L.wc2 = o; o += H; L.bc2 = o; o += 1;
    L.total = o;
    return L;
}

// ---------------------------------------------------------------------------------------
// Generic fp32 GEMM  C[M,N] (+)= op(A)[M,K] * op(B)[K,N]  with fused epilogues.
//   AT == false: A stored [M,K] (K contiguous);  AT == true: A stored [K,M].
//   BT == false: B stored [K,N] (N contiguous);  BT == true: B stored [N,K].
// Epilogue, in this order: + C (accumulate), + bias[n], ReLU, * (mask[m,n] > 0).  gridDim.z > 1 splits K and
// writes partial tiles to C + z*M*N (summed in split order by final_reduce_kernel, deterministic).
constexpr int GM = 64, GN = 64, GK = 16;

template <bool AT, bool BT>
__global__ void __launch_bounds__(256)
sgemm_kernel(int M, int N, int K, const float *__restrict__ A, int lda, const float *__restrict__ B, int ldb,
             float *__restrict__ C, int ldc, const float *__restrict__ bias, int relu,
             const float *__restrict__ mask, int ldm, int accumulate, int k_chunk)
{
    __shared__ float As[GK][GM + 4];
    __shared__ float Bs[GK][GN + 4];
    const int tid = threadIdx.x;
    const int m0 = blockIdx.y * GM, n0 = blockIdx.x * GN;
    const int kbeg = blockIdx.z * k_chunk, kend = min(K, kbeg + k_chunk);
    const int tx = tid & 15, ty = tid >> 4;  // 16 x 16 threads, 4 x 4 outputs each
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int k0 = kbeg; k0 < kend; k0 += GK) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int m, k;
            if (AT) { k = (tid >> 6) + 4 * i; m = tid & 63; }
            else { m = (tid >> 4) + 16 * i; k = tid & 15; }
            int gm = m0 + m, gk = k0 + k;
            float v = 0.f;
            if (gm < M && gk < kend) v = AT ? A[(size_t)gk * lda + gm] : A[(size_t)gm * lda + gk];
            As[k][m] = v;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int n, k;
            if (BT) { n = (tid >> 4) + 16 * i; k = tid & 15; }
            else { k = (tid >> 6) + 4 * i; n = tid & 63; }
            int gn = n0 + n, gk = k0 + k;
            float v = 0.f;
            if (gn < N && gk < kend) v = BT ? B[(size_t)gn * ldb + gk] : B[(size_t)gk * ldb + gn];
            Bs[k][n] = v;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < GK; ++k) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[k][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
    float *Cz = C + (size_t)blockIdx.z * M * ldc;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int gm = m0 + ty * 4 + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int gn = n0 + tx * 4 + j;
            if (gn >= N) continue;
            size_t o = (size_t)gm * ldc + gn;
            float v = acc[i][j];
            if (accumulate) v += Cz[o];
            if (bias) v += bias[gn];
            if (relu) v = fmaxf(v, 0.f);
            if (mask) v = mask[(size_t)gm * ldm + gn] > 0.f ? v : 0.f;
            Cz[o] = v;
        }
    }
}

// every deterministic second-stage reduction of one backward pass in ONE launch: segment q sums `splits` partial
// arrays of n elements in split order; elements >= n1 go to dst2.
struct ReduceSeg {
    const float *part;
    float *dst, *dst2;
    long long n, n1;
    int splits, block0;
};
struct ReducePlan {
    ReduceSeg seg[8];
    int nseg, blocks;
};
__global__ void __launch_bounds__(256) final_reduce_kernel(const ReducePlan P)
{
    int q = 0;
#pragma unroll
    for (int t = 1; t < 8; ++t)
        if (t < P.nseg && (int)blockIdx.x >= P.seg[t].block0) q = t;
    const ReduceSeg &g = P.seg[q];
    long long i = (long long)(blockIdx.x - g.block0) * blockDim.x + threadIdx.x;
    if (i >= g.n) return;
    // split order, eight loads in flight at a time (the longest segment sets the duration of the launch)
    float s = 0.f;
    int z = 0;
    for (; z + 8 <= g.splits; z += 8) {
        float t[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = __ldcg(g.part + (size_t)(z + j) * g.n + i);
#pragma unroll
        for (int j = 0; j < 8; ++j) s += t[j];
    }
    for (; z < g.splits; ++z) s += __ldcg(g.part + (size_t)z * g.n + i);
    if (i < g.n1) g.dst[i] = s;
    else g.dst2[i - g.n1] = s;
}
static void plan_add(ReducePlan &P, const float *part, long long n, int splits, float *dst, long long n1, float *dst2)
{
    ReduceSeg &g = P.seg[P.nseg++];
    g.part = part; g.n = n; g.splits = splits; g.dst = dst; g.n1 = n1; g.dst2 = dst2;
    g.block0 = P.blocks;
    P.blocks += (int)((n + 255) / 256);
}

// transposed, 16-byte aligned copies of the hidden weight matrices for the input-gradient GEMMs (the flat
// parameter buffer holds W[out, in]; dX = dY W wants W^T K-contiguous).  z = 0: actor_mean.0 -> wt_ac[:, 0:H],
// z = 1: critic.0 -> wt_ac[:, H:2H] (row pitch 2H), z = 2: shared.2 -> wt_2 (row pitch H)
__global__ void __launch_bounds__(256)
transpose_weights_kernel(const float *__restrict__ wa1, const float *__restrict__ wc1, const float *__restrict__ w2,
                         int H, float *__restrict__ wt_ac, float *__restrict__ wt_2)
{
    __shared__ float tile[32][33];
    const float *src = blockIdx.z == 0 ? wa1 : (blockIdx.z == 1 ? wc1 : w2);
    float *dst = blockIdx.z == 2 ? wt_2 : wt_ac + (blockIdx.z == 1 ? H : 0);
    const int ldd = blockIdx.z == 2 ? H : 2 * H;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int r = r0 + ty + 8 * i, c = c0 + tx;
        tile[ty + 8 * i][tx] = (r < H && c < H) ? src[(size_t)r * H + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int r = c0 + ty + 8 * i, c = r0 + tx;   // dst[r, c] = src[c, r]
        if (r < H && c < H) dst[(size_t)r * ldd + c] = tile[tx][ty + 8 * i];
    }
}

// column sums, stage 1: block (x, y) reduces rows [y*rows_per, ...) of 32 columns -> part[y][N]
__global__ void __launch_bounds__(256)
colsum_partial_kernel(const float *__restrict__ G, int ldg, long long B, int N, int rows_per, float *__restrict__ part)
{
    __shared__ float red[8][33];
    const int l = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int col = blockIdx.x * 32 + l;
    const long long r0 = (long long)blockIdx.y * rows_per, r1 = min(B, r0 + rows_per);
    float s = 0.f;
    if (col < N)
        for (long long b = r0 + w; b < r1; b += 8) s += G[(size_t)b * ldg + col];
    red[w][l] = s;
    __syncthreads();
    if (w == 0 && col < N) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += red[i][l];
        part[(size_t)blockIdx.y * N + col] = t;
    }
}

// head weight/bias gradients, stage 1 (agent.py actor_mean.2 / critic.2): for a chunk of rows,
//   dWa2[a,h] = sum_b dmean[b,a] a1[b,h], dba2[a] = sum_b dmean[b,a], dWc2[h] = sum_b dvalue[b] c1[b,h], dbc2 = sum_b dvalue[b]
// part[y] holds [A*H | A | H | 1] floats.  A <= MAXA: 4 (the Gaussian head), or 8 (categorical heads of up to 8 logits).
template <int MAXA>
__global__ void __launch_bounds__(256)
heads_wgrad_partial_kernel(const float *__restrict__ dmean, const float *__restrict__ dvalue,
                           const float *__restrict__ a1, const float *__restrict__ c1, int ld, long long B, int H, int A,
                           int rows_per, float *__restrict__ part)
{
    __shared__ float red[8][MAXA + 2][33];
    const int l = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int h = blockIdx.x * 32 + l;
    const long long r0 = (long long)blockIdx.y * rows_per, r1 = min(B, r0 + rows_per);
    float acc[MAXA] = {}, accc = 0.f, accb = 0.f;
    for (long long b = r0 + w; b < r1; b += 8) {
        float dv = dvalue[b];
        if (h < H) {
            float av = a1[(size_t)b * ld + h];
            for (int a = 0; a < A; ++a) acc[a] = fmaf(dmean[b * A + a], av, acc[a]);
            accc = fmaf(dv, c1[(size_t)b * ld + h], accc);
        }
        if (blockIdx.x == 0 && l <= A) accb += l < A ? dmean[b * A + l] : dv;
    }
    for (int a = 0; a < MAXA; ++a) red[w][a][l] = acc[a];
    red[w][MAXA][l] = accc;
    red[w][MAXA + 1][l] = accb;
    __syncthreads();
    if (w == 0) {
        float *out = part + (size_t)blockIdx.y * ((size_t)A * H + A + H + 1);
        float t[MAXA + 2];
        for (int q = 0; q < MAXA + 2; ++q) {
            t[q] = 0.f;
            for (int i = 0; i < 8; ++i) t[q] += red[i][q][l];
        }
        if (h < H) {
            for (int a = 0; a < A; ++a) out[(size_t)a * H + h] = t[a];
            out[(size_t)A * H + A + h] = t[MAXA];
        }
        if (blockIdx.x == 0 && l <= A) {
            if (l < A) out[(size_t)A * H + l] = t[MAXA + 1];
            else out[(size_t)A * H + A + H] = t[MAXA + 1];
        }
    }
}
// gather the minibatch out of the rollout in one launch: states, pre_tanh, old log-prob, advantage, return, and with
// VOLD the rollout's value (the clipped value loss).  The VOLD arguments come last, so the default instantiation keeps
// the parameter block it had before them.
template <bool VOLD>
__global__ void gather_batch_kernel(const float *__restrict__ states, const float *__restrict__ pre_tanh,
                                    const float *__restrict__ olp, const float *__restrict__ adv,
                                    const float *__restrict__ ret, const long long *__restrict__ idx, long long B, int S,
                                    int A, float *__restrict__ x, float *__restrict__ z,
                                    float *__restrict__ o_olp, float *__restrict__ o_adv, float *__restrict__ o_ret,
                                    const float *__restrict__ vold, float *__restrict__ o_vold)
{
    hrp_pdl_release();   // the first GEMM of the step sets itself up meanwhile (it waits before it reads x)
    const int W = S + A + (VOLD ? 4 : 3);
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * W) return;
    long long b = i / W;
    int c = (int)(i - b * W);
    long long src = idx[b];
    if (c < S) x[b * S + c] = states[(size_t)src * S + c];
    else if (c < S + A) z[b * A + (c - S)] = pre_tanh[(size_t)src * A + (c - S)];
    else if (c == S + A) o_olp[b] = olp[src];
    else if (c == S + A + 1) o_adv[b] = adv[src];
    else if (!VOLD || c == S + A + 2) o_ret[b] = ret[src];
    else o_vold[b] = vold[src];
}

// The clipped value loss (VCLIP of the loss kernels): with v the new value, vo the rollout's, R the return and c the
// clip, the per-sample term is max((v - R)^2, (vo + clamp(v - vo, -c, c) - R)^2).  Returns the term and writes
// d(term)/d(v) / 2 to *half_grad with torch autograd's rules: maximum splits the gradient half and half on a tie, clamp
// passes it where -c <= v - vo <= c.
__device__ __forceinline__ float clipped_value_term(float v, float vo, float R, float c, float *half_grad)
{
    const float d1 = v - R, dvo = v - vo;
    const float d2 = (vo + fminf(fmaxf(dvo, -c), c)) - R;
    const float l1 = d1 * d1, l2 = d2 * d2;
    const float g2 = dvo >= -c && dvo <= c ? d2 : 0.f;
    *half_grad = l1 > l2 ? d1 : (l2 > l1 ? g2 : 0.5f * d1 + 0.5f * g2);
    return fmaxf(l1, l2);
}

// ---------------------------------------------------------------------------------------
// heads: mean[B,A] = a1 Wa2^T + ba2, value[B] = c1 Wc2^T + bc2  (N is 2 and 1: one warp per row)
__global__ void __launch_bounds__(256)
heads_kernel(const float *__restrict__ a1, const float *__restrict__ c1, const float *__restrict__ wa2,
             const float *__restrict__ ba2, const float *__restrict__ wc2, const float *__restrict__ bc2,
             int ld, long long B, int H, int A, float *__restrict__ mean, float *__restrict__ value)
{
    long long b = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (b >= B) return;
    const float *ra = a1 + (size_t)b * ld, *rc = c1 + (size_t)b * ld;
    for (int a = 0; a <= A; ++a) {
        const float *w = a < A ? wa2 + (size_t)a * H : wc2;
        const float *x = a < A ? ra : rc;
        float s = 0.f;
        for (int k = lane; k < H; k += 32) s = fmaf(x[k], w[k], s);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(HRP_FULL, s, d);
        if (lane == 0) {
            if (a < A) mean[b * A + a] = s + ba2[a];
            else value[b] = s + bc2[0];
        }
    }
}

// heads + ActorCritic.get_action (agent.py:56-74) in one pass for the rollout: one warp per row forms mean[A] and
// value from the two hidden activations (all loads of the row in flight together), then lane a < A samples
// z_a = mean_a + std_a * n_a with n ~ N(0,1) from Philox4x32-10(counter = (global row, draw), key = seed) through
// Box-Muller (or takes n from noise[], or n = 0 when deterministic) and writes tanh(z_a), z_a; the log-prob terms of
// the A lanes are added by shuffles.
constexpr int HA_ROWS = 2;   // rows per warp of heads_act_kernel (their loads are in flight together)
__global__ void __launch_bounds__(256)
heads_act_kernel(const float *__restrict__ a1, const float *__restrict__ c1, const float *__restrict__ wa2,
                 const float *__restrict__ ba2, const float *__restrict__ wc2, const float *__restrict__ bc2,
                 const float *__restrict__ log_std, const float *__restrict__ noise, int mode /*0 det, 1 noise[], 2 philox*/,
                 unsigned long long seed, unsigned long long draw, unsigned long long row_base, int ld, long long B,
                 int H, int A, float *__restrict__ action, float *__restrict__ pre_tanh,
                 float *__restrict__ log_prob, float *__restrict__ value, unsigned long long *draw_ctr, int vec)
{
    extern __shared__ __align__(16) float hw[];   // the head weights, [A + 1][H]: read once per CTA, not once per row
    hrp_pdl_release();
    hrp_pdl_wait();
    for (int i = threadIdx.x; i < (A + 1) * H; i += 256) hw[i] = i < A * H ? wa2[i] : wc2[i - A * H];
    if (draw_ctr) {
        // device-resident draw counter (a captured launch cannot take a new `draw` argument per replay): every CTA
        // reads draw_ctr[0], then takes a ticket from draw_ctr[1]; the CTA that takes the last ticket -- by then every
        // CTA has read the counter -- advances it and clears the tickets for the next launch
        __shared__ unsigned long long sdraw;
        if (threadIdx.x == 0) {
            sdraw = *(volatile unsigned long long *)draw_ctr + 1ull;   // the host path pre-increments too
            __threadfence();
            if (atomicAdd(draw_ctr + 1, 1ull) == (unsigned long long)gridDim.x - 1ull) {
                draw_ctr[1] = 0ull;
                draw_ctr[0] = sdraw;
            }
        }
        __syncthreads();
        draw = sdraw;
    } else {
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const long long b0 = ((long long)blockIdx.x * 8 + (threadIdx.x >> 5)) * HA_ROWS;
    if (b0 >= B) return;
    float accs[HA_ROWS][5];
#pragma unroll
    for (int r = 0; r < HA_ROWS; ++r)
#pragma unroll
        for (int a = 0; a < 5; ++a) accs[r][a] = 0.f;
    if (vec) {   // H % 128 == 0, 16-byte aligned rows: lane owns 4 consecutive k per 128
        for (int k = 4 * lane; k < H; k += 128) {
            float4 xa[HA_ROWS], xc[HA_ROWS];
#pragma unroll
            for (int r = 0; r < HA_ROWS; ++r) {
                const long long b = min(b0 + r, B - 1);
                xa[r] = *reinterpret_cast<const float4 *>(a1 + (size_t)b * ld + k);
                xc[r] = *reinterpret_cast<const float4 *>(c1 + (size_t)b * ld + k);
            }
            const float4 wc = *reinterpret_cast<const float4 *>(hw + A * H + k);
#pragma unroll
            for (int a = 0; a < 4; ++a)
                if (a < A) {
                    const float4 w = *reinterpret_cast<const float4 *>(hw + a * H + k);
#pragma unroll
                    for (int r = 0; r < HA_ROWS; ++r)
                        accs[r][a] = fmaf(xa[r].w, w.w, fmaf(xa[r].z, w.z, fmaf(xa[r].y, w.y, fmaf(xa[r].x, w.x, accs[r][a]))));
                }
#pragma unroll
            for (int r = 0; r < HA_ROWS; ++r)
                accs[r][4] = fmaf(xc[r].w, wc.w, fmaf(xc[r].z, wc.z, fmaf(xc[r].y, wc.y, fmaf(xc[r].x, wc.x, accs[r][4]))));
        }
    } else {
        for (int k = lane; k < H; k += 32) {
#pragma unroll
            for (int r = 0; r < HA_ROWS; ++r) {
                const long long b = min(b0 + r, B - 1);
                const float xa = a1[(size_t)b * ld + k], xc = c1[(size_t)b * ld + k];
#pragma unroll
                for (int a = 0; a < 4; ++a)
                    if (a < A) accs[r][a] = fmaf(xa, hw[a * H + k], accs[r][a]);
                accs[r][4] = fmaf(xc, hw[A * H + k], accs[r][4]);
            }
        }
    }
#pragma unroll
    for (int r = 0; r < HA_ROWS; ++r)
#pragma unroll
        for (int a = 0; a < 5; ++a)
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) accs[r][a] += __shfl_xor_sync(HRP_FULL, accs[r][a], d);
#pragma unroll 1
    for (int r = 0; r < HA_ROWS; ++r) {
    const long long b = b0 + r;
    if (b >= B) break;
    float acc[5];
#pragma unroll
    for (int a = 0; a < 5; ++a) acc[a] = r == 0 ? accs[0][a] : accs[HA_ROWS - 1][a];
    // lane a owns action dimension a (lanes >= A compute on dimension 0 and discard)
    const int a = lane < A ? lane : 0;
    float mu = acc[0];
#pragma unroll
    for (int q = 1; q < 4; ++q) mu = a == q ? acc[q] : mu;
    mu += ba2[a];
    float nrm = 0.f;
    if (mode == 2) {
        uint32_t r[4];
        // the counter is the GLOBAL row (row_base = first global env id of this shard): the shards of a sharded
        // rollout draw different noise, and together exactly what one process over all envs would draw
        const unsigned long long gb = row_base + (unsigned long long)b;
        hrp_philox((uint32_t)gb, (uint32_t)(gb >> 32), (uint32_t)draw, (uint32_t)(draw >> 32),
                   (uint32_t)seed, (uint32_t)(seed >> 32) ^ 0x5A5A5A5Au, r);
        const uint32_t r1 = a < 2 ? r[0] : r[2], r2 = a < 2 ? r[1] : r[3];
        float u1 = ((float)(r1 >> 8) + 0.5f) * (1.0f / 16777216.0f);
        float u2 = ((float)(r2 >> 8) + 0.5f) * (1.0f / 16777216.0f);
        float rad = sqrtf(-2.f * logf(u1)), sn, cs;
        sincospif(2.f * u2, &sn, &cs);
        nrm = rad * ((a & 1) ? sn : cs);
    } else if (mode == 1) {
        nrm = noise[b * A + a];
    }
    const float ls = log_std[a], sd = expf(ls);
    const float z = mode ? mu + sd * nrm : mu;
    const float t = tanhf(z);
    const float d = z - mu;
    float lp = -(d * d) / (2.f * sd * sd) - ls - 0.91893853320467274f;
    lp -= log1pf(-(t * t) + 1e-6f);
    lp = lane < A ? lp : 0.f;
    lp += __shfl_xor_sync(HRP_FULL, lp, 1);
    lp += __shfl_xor_sync(HRP_FULL, lp, 2);
    if (lane < A) {
        pre_tanh[b * A + lane] = z;
        action[b * A + lane] = t;
    }
    if (lane == 0) {
        if (log_prob) log_prob[b] = mode ? lp : 0.f;
        value[b] = acc[4] + bc2[0];
    }
    }
}

// heads + PPO loss + the gradient of the hidden head layers in one launch (agent.py:76-84, 223-245): a CTA owns 16
// rows.  Phase 0: a warp per row forms mean[A] and value from a1 | c1 (row pitch ld).  Phase 1: one thread per row
// evaluates the loss terms, writes d(mean), d(value) (the head weight gradients need them) and keeps them in shared
// memory.  Phase 2: the CTA writes d(a1) | d(c1) = (dmean Wa2 | dvalue Wc2) under the ReLU masks for its rows.
// Every CTA leaves 8 partial sums in part[blockIdx.x][8]; the CTA that finishes last adds them in block order
// (deterministic) and writes d(log_std) and the metrics.  `counter` returns to zero.
// KL (target_kl early stopping): the last CTA also writes this shard's approx-KL share, the value it adds to
// metrics[5], to *kl_out, and adds to the metrics only while *stop == 0 (a stopped update's later minibatches do not
// count).  The gradient is the same either way.  The arguments come last, so the default instantiation keeps its
// parameter block.
constexpr int HLB_ROWS = 16;
template <bool VCLIP, bool KL>
__global__ void __launch_bounds__(256)
heads_loss_backward_kernel(const float *__restrict__ a1, const float *__restrict__ c1, int ld, int H,
                           const float *__restrict__ wa2, const float *__restrict__ ba2,
                           const float *__restrict__ wc2, const float *__restrict__ bc2,
                           const float *__restrict__ log_std, const float *__restrict__ pre_tanh,
                           const float *__restrict__ old_lp, const float *__restrict__ adv,
                           const float *__restrict__ ret, long long B, int A, float eps_clip, float value_coef,
                           float entropy_coef, float scale, float *__restrict__ dmean, float *__restrict__ dvalue,
                           float *__restrict__ da1, float *__restrict__ dc1, float *__restrict__ dlog_std,
                           float *__restrict__ metrics, float *__restrict__ part,
                           unsigned *__restrict__ counter, const float *__restrict__ old_value, float value_clip,
                           float *__restrict__ kl_out, const unsigned *__restrict__ stop)
{
    __shared__ float out_s[HLB_ROWS][5], dmean_s[HLB_ROWS][4], dvalue_s[HLB_ROWS];
    __shared__ float red[8][8];
    __shared__ bool last;
    hrp_pdl_release();
    hrp_pdl_wait();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long row0 = (long long)blockIdx.x * HLB_ROWS;
    const int rows = (int)min((long long)HLB_ROWS, B - row0);
    // ---- phase 0: heads.  The loads of a row's dot products are issued together (one memory round trip per row).
    for (int r = w; r < rows; r += 8) {
        const float *ra = a1 + (size_t)(row0 + r) * ld, *rc = c1 + (size_t)(row0 + r) * ld;
        float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        for (int k = lane; k < H; k += 32) {
            const float xa = ra[k], xc = rc[k];
#pragma unroll
            for (int a = 0; a < 4; ++a)
                if (a < A) acc[a] = fmaf(xa, wa2[(size_t)a * H + k], acc[a]);
            acc[4] = fmaf(xc, wc2[k], acc[4]);
        }
#pragma unroll
        for (int a = 0; a < 5; ++a)
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) acc[a] += __shfl_xor_sync(HRP_FULL, acc[a], d);
        if (lane == 0) {
            for (int a = 0; a < A; ++a) out_s[r][a] = acc[a] + ba2[a];
            out_s[r][A] = acc[4] + bc2[0];
        }
    }
    __syncthreads();
    // ---- phase 1: loss terms, one thread per row (warps 0 and 1)
    float vals[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // pol, val, clip, kl, dls[4]
    float ls_[4];
    for (int a = 0; a < A; ++a) ls_[a] = log_std[a];
    if (threadIdx.x < rows) {
        const int r = threadIdx.x;
        const long long b = row0 + r;
        float lp = 0.f;
        float dmu[4], dls[4];
        for (int a = 0; a < A; ++a) {
            float mu = out_s[r][a], ls = ls_[a], sd = expf(ls);
            float z = pre_tanh[b * A + a];
            float t = tanhf(z);
            float d = z - mu, var = sd * sd;
            lp += -(d * d) / (2.f * var) - ls - 0.91893853320467274f;
            lp -= log1pf(-(t * t) + 1e-6f);
            dmu[a] = d / var;
            dls[a] = d * d / var - 1.f;
        }
        float lr = lp - old_lp[b];
        float ratio = expf(lr);
        float ad = adv[b];
        float surr1 = ratio * ad;
        float rc2 = fminf(fmaxf(ratio, 1.f - eps_clip), 1.f + eps_clip);
        float surr2 = rc2 * ad;
        bool inr = ratio >= 1.f - eps_clip && ratio <= 1.f + eps_clip;
        // d min(surr1, surr2) / d ratio with torch's tie rule (half each on equality)
        float g;
        if (surr1 < surr2) g = ad;
        else if (surr1 == surr2) g = 0.5f * ad + (inr ? 0.5f * ad : 0.f);
        else g = inr ? ad : 0.f;
        float dlp = -g * ratio * scale;
        for (int a = 0; a < 4; ++a) dmean_s[r][a] = 0.f;
        for (int a = 0; a < A; ++a) {
            float dm = dlp * dmu[a];
            dmean[b * A + a] = dm;
            dmean_s[r][a] = dm;
            vals[4 + a] = dlp * dls[a];
        }
        float dv = out_s[r][A] - ret[b], vterm = dv * dv;
        if (VCLIP) vterm = clipped_value_term(out_s[r][A], old_value[b], ret[b], value_clip, &dv);
        float dvv = value_coef * 2.f * dv * scale;
        dvalue[b] = dvv;
        dvalue_s[r] = dvv;
        vals[0] = -fminf(surr1, surr2);
        vals[1] = vterm;
        vals[2] = fabsf(ratio - 1.f) > eps_clip ? 1.f : 0.f;
        vals[3] = (ratio - 1.f) - lr;
    }
    if (w < 2) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float x = vals[i];
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(HRP_FULL, x, d);
            if (lane == 0) red[w][i] = x;
        }
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        part[blockIdx.x * 8 + threadIdx.x] = red[0][threadIdx.x] + red[1][threadIdx.x];
        __threadfence();
    }
    // ---- phase 2: d(a1) | d(c1) for the CTA's rows.  A thread owns a column (its head weights stay in registers)
    // and walks the rows with all mask loads in flight.
    for (int k = threadIdx.x; k < H; k += 256) {
        float wk[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) wk[a] = a < A ? wa2[(size_t)a * H + k] : 0.f;
        const float wck = wc2[k];
        float ma[HLB_ROWS], mc[HLB_ROWS];
#pragma unroll
        for (int r = 0; r < HLB_ROWS; ++r) {
            const size_t o = (size_t)(row0 + r) * ld + k;
            ma[r] = r < rows ? a1[o] : 0.f;
            mc[r] = r < rows ? c1[o] : 0.f;
        }
#pragma unroll
        for (int r = 0; r < HLB_ROWS; ++r) {
            if (r >= rows) break;
            const size_t o = (size_t)(row0 + r) * ld + k;
            float sacc = 0.f;
#pragma unroll
            for (int a = 0; a < 4; ++a) sacc = fmaf(dmean_s[r][a], wk[a], sacc);
            const float ga = ma[r] > 0.f ? sacc : 0.f, gc = mc[r] > 0.f ? dvalue_s[r] * wck : 0.f;
            da1[o] = ga;
            dc1[o] = gc;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned prev = atomicAdd(counter, 1u);
        last = prev == gridDim.x - 1;
        if (last) *counter = 0u;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    // thread t adds the sums of CTAs t, t + 256, ... in order; then warps, then the 8 warps, always in index order
    float v8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (unsigned c = threadIdx.x; c < gridDim.x; c += 256)
#pragma unroll
        for (int j = 0; j < 8; ++j) v8[j] += __ldcg(part + c * 8 + j);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        float x = v8[j];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(HRP_FULL, x, d);
        v8[j] = x;
    }
    if (lane == 0)
        for (int j = 0; j < 8; ++j) red[w][j] = v8[j];
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot[8];
        for (int j = 0; j < 8; ++j) {
            float x = 0.f;
            for (int i = 0; i < 8; ++i) x += red[i][j];
            tot[j] = x;
        }
        float ent = 0.f;
        for (int a = 0; a < A; ++a) ent += 0.5f + 0.91893853320467274f + ls_[a];
        float pol = tot[0] * scale, val = tot[1] * scale;
        float frac = (float)B * scale;  // share of the global minibatch held by this shard
        float loss = pol + value_coef * val - entropy_coef * ent * frac;
        for (int a = 0; a < A; ++a) dlog_std[a] = tot[4 + a] - entropy_coef * frac;
        if (KL) *kl_out = tot[3] * scale;
        if (metrics && (!KL || *stop == 0u)) {
            metrics[0] += loss; metrics[1] += pol; metrics[2] += val; metrics[3] += ent * frac;
            metrics[4] += tot[2] * scale; metrics[5] += tot[3] * scale; metrics[6] += frac;
        }
    }
}

// ---------------------------------------------------------------------------------------
// Categorical policy (HRP_PPO_CATEGORICAL): softmax over the n <= CAT_MAX logits of actor_mean.2, same trunk, critic and
// loss formula as the Gaussian head.  The sample conditions the loss through pre_tanh[b] = id.
constexpr int CAT_MAX = 8;

// Softmax, draw and log-prob of one row from its n logits (biases added).  One uniform per row: Philox4x32-10 with the
// Gaussian path's counter (row_base + b, draw) and key, u = ((r0 >> 8) + 0.5) / 2^24 (or noise[b] for mode 1); the id
// is the first j with u < sum_{i <= j} p_i, the sum formed in index order in fp32, and n - 1 if there is none.
// Deterministic mode takes the first maximum (torch.argmax) and reports log-prob 0, as the Gaussian path does.
__device__ __forceinline__ void cat_sample_row(const float (&lg)[CAT_MAX], int n, int mode, const float *__restrict__ noise,
                                               unsigned long long seed, unsigned long long draw, unsigned long long row_base,
                                               long long b, int &id, float &lp)
{
    float m = lg[0];
    int amax = 0;
#pragma unroll
    for (int j = 1; j < CAT_MAX; ++j)
        if (j < n && lg[j] > m) { m = lg[j]; amax = j; }
    float e[CAT_MAX], s = 0.f;
#pragma unroll
    for (int j = 0; j < CAT_MAX; ++j) {
        e[j] = j < n ? expf(lg[j] - m) : 0.f;
        s += e[j];
    }
    if (mode == 0) {
        id = amax;
        lp = 0.f;
        return;
    }
    float u;
    if (mode == 2) {
        uint32_t r[4];
        const unsigned long long gb = row_base + (unsigned long long)b;
        hrp_philox((uint32_t)gb, (uint32_t)(gb >> 32), (uint32_t)draw, (uint32_t)(draw >> 32),
                   (uint32_t)seed, (uint32_t)(seed >> 32) ^ 0x5A5A5A5Au, r);
        u = ((float)(r[0] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    } else {
        u = noise[b];
    }
    id = n - 1;
    float cum = 0.f, lsel = lg[n - 1];
    bool found = false;
#pragma unroll
    for (int j = 0; j < CAT_MAX; ++j) {
        if (j < n && !found) {
            cum += e[j] / s;
            if (u < cum) { id = j; lsel = lg[j]; found = true; }
        }
    }
    lp = (lsel - m) - logf(s);
}

// device-resident draw counter of the capturable sampling path (heads_act_kernel has the same protocol)
__device__ __forceinline__ unsigned long long cat_take_draw(unsigned long long *draw_ctr, unsigned long long draw)
{
    __shared__ unsigned long long sdraw;
    if (draw_ctr) {
        if (threadIdx.x == 0) {
            sdraw = *(volatile unsigned long long *)draw_ctr + 1ull;
            __threadfence();
            if (atomicAdd(draw_ctr + 1, 1ull) == (unsigned long long)gridDim.x - 1ull) {
                draw_ctr[1] = 0ull;
                draw_ctr[0] = sdraw;
            }
        }
    }
    __syncthreads();
    return draw_ctr ? sdraw : draw;
}

// heads + categorical get_action for the rollout (the categorical heads_act_kernel): a warp per HA_ROWS rows forms the
// n logits and the value (n + 1 dot products with the head weights held in shared memory, all loads of the rows in
// flight together, shuffle reductions), then draws as cat_sample_row says.  action[b] = (id, 0) is what hrp_env_step
// reads for the meta-action ego; pre_tanh[b] = id.
__global__ void __launch_bounds__(256)
heads_act_cat_kernel(const float *__restrict__ a1, const float *__restrict__ c1, const float *__restrict__ wa2,
                     const float *__restrict__ ba2, const float *__restrict__ wc2, const float *__restrict__ bc2,
                     const float *__restrict__ noise, int mode /*0 det, 1 noise[], 2 philox*/, unsigned long long seed,
                     unsigned long long draw, unsigned long long row_base, int ld, long long B, int H, int n,
                     float *__restrict__ action, float *__restrict__ pre_tanh, float *__restrict__ log_prob,
                     float *__restrict__ value, unsigned long long *draw_ctr, int vec)
{
    extern __shared__ __align__(16) float hw[];   // [n + 1][H]
    hrp_pdl_release();
    hrp_pdl_wait();
    for (int i = threadIdx.x; i < (n + 1) * H; i += 256) hw[i] = i < n * H ? wa2[i] : wc2[i - n * H];
    draw = cat_take_draw(draw_ctr, draw);
    const int lane = threadIdx.x & 31;
    const long long b0 = ((long long)blockIdx.x * 8 + (threadIdx.x >> 5)) * HA_ROWS;
    if (b0 >= B) return;
    float accs[HA_ROWS][CAT_MAX + 1] = {};
    if (vec) {   // H % 128 == 0, 16-byte aligned rows: lane owns 4 consecutive k per 128
        for (int k = 4 * lane; k < H; k += 128) {
            float4 xa[HA_ROWS], xc[HA_ROWS];
#pragma unroll
            for (int r = 0; r < HA_ROWS; ++r) {
                const long long b = min(b0 + r, B - 1);
                xa[r] = *reinterpret_cast<const float4 *>(a1 + (size_t)b * ld + k);
                xc[r] = *reinterpret_cast<const float4 *>(c1 + (size_t)b * ld + k);
            }
            const float4 wc = *reinterpret_cast<const float4 *>(hw + n * H + k);
#pragma unroll
            for (int a = 0; a < CAT_MAX; ++a)
                if (a < n) {
                    const float4 w = *reinterpret_cast<const float4 *>(hw + a * H + k);
#pragma unroll
                    for (int r = 0; r < HA_ROWS; ++r)
                        accs[r][a] = fmaf(xa[r].w, w.w, fmaf(xa[r].z, w.z, fmaf(xa[r].y, w.y, fmaf(xa[r].x, w.x, accs[r][a]))));
                }
#pragma unroll
            for (int r = 0; r < HA_ROWS; ++r)
                accs[r][CAT_MAX] = fmaf(xc[r].w, wc.w, fmaf(xc[r].z, wc.z, fmaf(xc[r].y, wc.y, fmaf(xc[r].x, wc.x, accs[r][CAT_MAX]))));
        }
    } else {
        for (int k = lane; k < H; k += 32) {
#pragma unroll
            for (int r = 0; r < HA_ROWS; ++r) {
                const long long b = min(b0 + r, B - 1);
                const float xa = a1[(size_t)b * ld + k], xc = c1[(size_t)b * ld + k];
#pragma unroll
                for (int a = 0; a < CAT_MAX; ++a)
                    if (a < n) accs[r][a] = fmaf(xa, hw[a * H + k], accs[r][a]);
                accs[r][CAT_MAX] = fmaf(xc, hw[n * H + k], accs[r][CAT_MAX]);
            }
        }
    }
#pragma unroll
    for (int r = 0; r < HA_ROWS; ++r)
#pragma unroll
        for (int a = 0; a <= CAT_MAX; ++a)
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) accs[r][a] += __shfl_xor_sync(HRP_FULL, accs[r][a], d);
    // every lane holds every sum now; lane r writes row b0 + r
#pragma unroll
    for (int r = 0; r < HA_ROWS; ++r) {
        const long long b = b0 + r;
        if (lane != r || b >= B) continue;
        float lg[CAT_MAX];
#pragma unroll
        for (int j = 0; j < CAT_MAX; ++j) lg[j] = j < n ? accs[r][j] + ba2[j] : 0.f;
        int id;
        float lp;
        cat_sample_row(lg, n, mode, noise, seed, draw, row_base, b, id, lp);
        action[2 * b] = (float)id;
        action[2 * b + 1] = 0.f;
        pre_tanh[b] = (float)id;
        if (log_prob) log_prob[b] = lp;
        value[b] = accs[r][CAT_MAX] + bc2[0];
    }
}

// The categorical act path with the heads fused into the [a1 | c1] GEMM (TcDots, NP partial sums per tile and row): a
// thread per row adds the tiles in tile order, adds the biases and draws exactly as heads_act_cat_kernel does.
template <int NP>
__global__ void __launch_bounds__(128)
heads_finish_cat_kernel(const float *__restrict__ part, int tiles_a, int tiles, const float *__restrict__ ba2,
                        const float *__restrict__ bc2, const float *__restrict__ noise, int mode, unsigned long long seed,
                        unsigned long long draw, unsigned long long row_base, long long B, int n,
                        float *__restrict__ action, float *__restrict__ pre_tanh, float *__restrict__ log_prob,
                        float *__restrict__ value, unsigned long long *draw_ctr)
{
    hrp_pdl_release();
    hrp_pdl_wait();
    draw = cat_take_draw(draw_ctr, draw);
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float lg[CAT_MAX] = {}, val = 0.f;
    for (int t = 0; t < tiles; ++t) {
        const float *p = part + ((size_t)t * B + b) * NP;
        if (t < tiles_a) {
#pragma unroll
            for (int q = 0; q < NP; q += 4) {
                const float4 v = *reinterpret_cast<const float4 *>(p + q);
                lg[q] += v.x; lg[q + 1] += v.y; lg[q + 2] += v.z; lg[q + 3] += v.w;
            }
        } else {
            val += p[0];
        }
    }
#pragma unroll
    for (int j = 0; j < CAT_MAX; ++j) lg[j] = j < n ? lg[j] + ba2[j] : 0.f;
    int id;
    float lp;
    cat_sample_row(lg, n, mode, noise, seed, draw, row_base, b, id, lp);
    action[2 * b] = (float)id;
    action[2 * b + 1] = 0.f;
    pre_tanh[b] = (float)id;
    if (log_prob) log_prob[b] = lp;
    value[b] = val + bc2[0];
}

// heads + categorical PPO loss + the gradient of the hidden head layers in one launch, heads_loss_backward_kernel's
// structure for the softmax head.  Phase 0: a warp per row forms the n logits and the value.  Phase 1: a thread per row
// takes id = pre_tanh[b], log p = log_softmax(logits), the entropy H = -sum p log p, the ratio and the clipped surrogate
// (same tie rule), and writes
//   d(logit_j) = scale [-g ratio (delta_{id,j} - p_j) + c_ent p_j (log p_j + H)]   (g = d min(surr1, surr2) / d ratio)
// and d(value).  Phase 2: d(a1) | d(c1) under the ReLU masks.  Partial sums per CTA: policy loss, value error, clip
// count, approx-KL, entropy; the last CTA adds them in block order and writes the metrics.  No log_std gradient.
// KL: as in heads_loss_backward_kernel.
template <bool VCLIP, bool KL>
__global__ void __launch_bounds__(256)
heads_loss_backward_cat_kernel(const float *__restrict__ a1, const float *__restrict__ c1, int ld, int H,
                               const float *__restrict__ wa2, const float *__restrict__ ba2,
                               const float *__restrict__ wc2, const float *__restrict__ bc2,
                               const float *__restrict__ ids, const float *__restrict__ old_lp,
                               const float *__restrict__ adv, const float *__restrict__ ret, long long B, int n,
                               float eps_clip, float value_coef, float entropy_coef, float scale,
                               float *__restrict__ dlogit, float *__restrict__ dvalue, float *__restrict__ da1,
                               float *__restrict__ dc1, float *__restrict__ metrics, float *__restrict__ part,
                               unsigned *__restrict__ counter, const float *__restrict__ old_value, float value_clip,
                               float *__restrict__ kl_out, const unsigned *__restrict__ stop)
{
    __shared__ float out_s[HLB_ROWS][CAT_MAX + 1], dl_s[HLB_ROWS][CAT_MAX], dvalue_s[HLB_ROWS];
    __shared__ float red[8][8];
    __shared__ bool last;
    hrp_pdl_release();
    hrp_pdl_wait();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long row0 = (long long)blockIdx.x * HLB_ROWS;
    const int rows = (int)min((long long)HLB_ROWS, B - row0);
    // ---- phase 0: logits and value
    for (int r = w; r < rows; r += 8) {
        const float *ra = a1 + (size_t)(row0 + r) * ld, *rc = c1 + (size_t)(row0 + r) * ld;
        float acc[CAT_MAX + 1] = {};
        for (int k = lane; k < H; k += 32) {
            const float xa = ra[k], xc = rc[k];
#pragma unroll
            for (int a = 0; a < CAT_MAX; ++a)
                if (a < n) acc[a] = fmaf(xa, wa2[(size_t)a * H + k], acc[a]);
            acc[CAT_MAX] = fmaf(xc, wc2[k], acc[CAT_MAX]);
        }
#pragma unroll
        for (int a = 0; a <= CAT_MAX; ++a)
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) acc[a] += __shfl_xor_sync(HRP_FULL, acc[a], d);
        if (lane == 0) {
#pragma unroll
            for (int a = 0; a < CAT_MAX; ++a)
                if (a < n) out_s[r][a] = acc[a] + ba2[a];
            out_s[r][CAT_MAX] = acc[CAT_MAX] + bc2[0];
        }
    }
    __syncthreads();
    // ---- phase 1: loss terms, one thread per row (warps 0 and 1)
    float vals[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // pol, val, clip, kl, entropy
    if (threadIdx.x < rows) {
        const int r = threadIdx.x;
        const long long b = row0 + r;
        float m = out_s[r][0];
#pragma unroll
        for (int j = 1; j < CAT_MAX; ++j)
            if (j < n) m = fmaxf(m, out_s[r][j]);
        float e[CAT_MAX], s = 0.f;
#pragma unroll
        for (int j = 0; j < CAT_MAX; ++j) {
            e[j] = j < n ? expf(out_s[r][j] - m) : 0.f;
            s += e[j];
        }
        const float lse = logf(s);
        const int id = min(max((int)ids[b], 0), n - 1);
        float logp[CAT_MAX], p[CAT_MAX], ent = 0.f, lp = 0.f;
#pragma unroll
        for (int j = 0; j < CAT_MAX; ++j) {
            logp[j] = j < n ? (out_s[r][j] - m) - lse : 0.f;
            p[j] = e[j] / s;
            ent -= p[j] * logp[j];
            lp = j == id ? logp[j] : lp;
        }
        float lr = lp - old_lp[b];
        float ratio = expf(lr);
        float ad = adv[b];
        float surr1 = ratio * ad;
        float rc2 = fminf(fmaxf(ratio, 1.f - eps_clip), 1.f + eps_clip);
        float surr2 = rc2 * ad;
        bool inr = ratio >= 1.f - eps_clip && ratio <= 1.f + eps_clip;
        // d min(surr1, surr2) / d ratio with torch's tie rule (half each on equality)
        float g;
        if (surr1 < surr2) g = ad;
        else if (surr1 == surr2) g = 0.5f * ad + (inr ? 0.5f * ad : 0.f);
        else g = inr ? ad : 0.f;
        const float dlp = -g * ratio * scale, ce = entropy_coef * scale;
#pragma unroll
        for (int j = 0; j < CAT_MAX; ++j) {
            const float dl = dlp * ((j == id ? 1.f : 0.f) - p[j]) + ce * p[j] * (logp[j] + ent);
            dl_s[r][j] = j < n ? dl : 0.f;
            if (j < n) dlogit[b * n + j] = dl;
        }
        float dv = out_s[r][CAT_MAX] - ret[b], vterm = dv * dv;
        if (VCLIP) vterm = clipped_value_term(out_s[r][CAT_MAX], old_value[b], ret[b], value_clip, &dv);
        float dvv = value_coef * 2.f * dv * scale;
        dvalue[b] = dvv;
        dvalue_s[r] = dvv;
        vals[0] = -fminf(surr1, surr2);
        vals[1] = vterm;
        vals[2] = fabsf(ratio - 1.f) > eps_clip ? 1.f : 0.f;
        vals[3] = (ratio - 1.f) - lr;
        vals[4] = ent;
    }
    if (w < 2) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float x = vals[i];
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(HRP_FULL, x, d);
            if (lane == 0) red[w][i] = x;
        }
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        part[blockIdx.x * 8 + threadIdx.x] = red[0][threadIdx.x] + red[1][threadIdx.x];
        __threadfence();
    }
    // ---- phase 2: d(a1) | d(c1) for the CTA's rows
    for (int k = threadIdx.x; k < H; k += 256) {
        float wk[CAT_MAX];
#pragma unroll
        for (int a = 0; a < CAT_MAX; ++a) wk[a] = a < n ? wa2[(size_t)a * H + k] : 0.f;
        const float wck = wc2[k];
        float ma[HLB_ROWS], mc[HLB_ROWS];
#pragma unroll
        for (int r = 0; r < HLB_ROWS; ++r) {
            const size_t o = (size_t)(row0 + r) * ld + k;
            ma[r] = r < rows ? a1[o] : 0.f;
            mc[r] = r < rows ? c1[o] : 0.f;
        }
#pragma unroll
        for (int r = 0; r < HLB_ROWS; ++r) {
            if (r >= rows) break;
            const size_t o = (size_t)(row0 + r) * ld + k;
            float sacc = 0.f;
#pragma unroll
            for (int a = 0; a < CAT_MAX; ++a) sacc = fmaf(dl_s[r][a], wk[a], sacc);
            const float ga = ma[r] > 0.f ? sacc : 0.f, gc = mc[r] > 0.f ? dvalue_s[r] * wck : 0.f;
            da1[o] = ga;
            dc1[o] = gc;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned prev = atomicAdd(counter, 1u);
        last = prev == gridDim.x - 1;
        if (last) *counter = 0u;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    // thread t adds the sums of CTAs t, t + 256, ... in order; then warps, then the 8 warps, always in index order
    float v8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (unsigned c = threadIdx.x; c < gridDim.x; c += 256)
#pragma unroll
        for (int j = 0; j < 8; ++j) v8[j] += __ldcg(part + c * 8 + j);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        float x = v8[j];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(HRP_FULL, x, d);
        v8[j] = x;
    }
    if (lane == 0)
        for (int j = 0; j < 8; ++j) red[w][j] = v8[j];
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot[8];
        for (int j = 0; j < 8; ++j) {
            float x = 0.f;
            for (int i = 0; i < 8; ++i) x += red[i][j];
            tot[j] = x;
        }
        float pol = tot[0] * scale, val = tot[1] * scale, ent = tot[4] * scale;   // ent: this shard's share of the mean
        float frac = (float)B * scale;
        float loss = pol + value_coef * val - entropy_coef * ent;
        if (KL) *kl_out = tot[3] * scale;
        if (metrics && (!KL || *stop == 0u)) {
            metrics[0] += loss; metrics[1] += pol; metrics[2] += val; metrics[3] += ent;
            metrics[4] += tot[2] * scale; metrics[5] += tot[3] * scale; metrics[6] += frac;
        }
    }
}

// PPOMemory.compute_advantages (agent.py:126-138): fp64 arithmetic, float32 store of every A_t
__global__ void gae_kernel(const float *__restrict__ reward, const float *__restrict__ value,
                           const uint8_t *__restrict__ done, const float *__restrict__ last_value, long long T,
                           long long E, double gamma, double lam, float *__restrict__ adv,
                           float *__restrict__ ret)
{
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    double next_v = last_value ? (double)last_value[e] : 0.0;
    float last_adv = 0.f;
    for (long long t = T - 1; t >= 0; --t) {
        size_t o = (size_t)t * E + e;
        double nd = 1.0 - (double)(done[o] != 0);
        double v = (double)value[o];
        double delta = (double)reward[o] + gamma * next_v * nd - v;
        float a = (float)(delta + gamma * lam * nd * (double)last_adv);
        adv[o] = a;
        ret[o] = a + value[o];
        last_adv = a;
        next_v = v;
    }
}

// gae_kernel with time-limit bootstrapping (hrp_gae_ex): a truncated step that did not also terminate is bootstrapped
// with V(s_final) instead of 0.  The bootstrap is a select, so final_value rows of other steps are never read into the
// arithmetic (they may hold anything).  Without a truncated step (or final_value == nullptr) every operation is the
// one gae_kernel performs on done = terminated | truncated, so the result is bit-identical.
__global__ void gae_ex_kernel(const float *__restrict__ reward, const float *__restrict__ value,
                              const uint8_t *__restrict__ terminated, const uint8_t *__restrict__ truncated,
                              const float *__restrict__ final_value, const float *__restrict__ last_value, long long T,
                              long long E, double gamma, double lam, float *__restrict__ adv, float *__restrict__ ret)
{
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    double next_v = last_value ? (double)last_value[e] : 0.0;
    float last_adv = 0.f;
    for (long long t = T - 1; t >= 0; --t) {
        size_t o = (size_t)t * E + e;
        const bool term = terminated[o] != 0, tr = truncated[o] != 0;
        const bool boot = final_value && tr && !term;   // a crash on the last step is not bootstrapped
        double nd = 1.0 - (double)(term || tr);
        double v = (double)value[o];
        double bv = boot ? (double)final_value[o] : next_v;
        double bm = boot ? 1.0 : nd;
        double delta = (double)reward[o] + gamma * bv * bm - v;
        float a = (float)(delta + gamma * lam * nd * (double)last_adv);
        adv[o] = a;
        ret[o] = a + value[o];
        last_adv = a;
        next_v = v;
    }
}

// sum, sum of squares, count of the local advantages (fp64), deterministic two-stage
__global__ void __launch_bounds__(256)
adv_stats_kernel(const float *__restrict__ adv, long long n, double *__restrict__ part)
{
    __shared__ double red[2][8];
    double s = 0.0, q = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        double a = adv[i];
        s += a; q += a * a;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) { s += __shfl_xor_sync(HRP_FULL, s, d); q += __shfl_xor_sync(HRP_FULL, q, d); }
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s; red[1][threadIdx.x >> 5] = q; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ts = 0.0, tq = 0.0;
        for (int i = 0; i < 8; ++i) { ts += red[0][i]; tq += red[1][i]; }
        part[2 * blockIdx.x] = ts; part[2 * blockIdx.x + 1] = tq;
    }
}
__global__ void adv_stats_final_kernel(const double *__restrict__ part, int nblocks, long long n,
                                       double *__restrict__ stats)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double s = 0.0, q = 0.0;
        for (int i = 0; i < nblocks; ++i) { s += part[2 * i]; q += part[2 * i + 1]; }
        stats[0] = s; stats[1] = q; stats[2] = (double)n;
    }
}
__global__ void adv_normalize_kernel(float *__restrict__ adv, long long n, const double *__restrict__ stats)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double cnt = stats[2], mean = stats[0] / cnt;
    double var = (stats[1] - cnt * mean * mean) / (cnt - 1.0);  // torch.std: unbiased
    // a cancellation below 0 is clamped; n = 1 gives 0/0 = NaN, as torch.std does (fmax would turn it into 0)
    float m = (float)mean, sd = (float)sqrt(var < 0.0 ? 0.0 : var);
    adv[i] = (adv[i] - m) / (sd + 1e-8f);
}

// clip_grad_norm_ + Adam.step (agent.py:249-252) in ONE cooperative launch: every CTA leaves the sum of squares of
// its slice of the gradient in part[blockIdx.x], the grid synchronises, every CTA adds the partials in the same
// fixed order (so the clip coefficient is identical everywhere and from run to run), then updates its slice and
// CTA 0 advances the step counter.  ADAM_MAX_CTAS partials fit the caller's 128-float scratch buffer.  LR_DEV: the
// learning rate is *lr_dev, read when the step size is formed (a captured launch follows a schedule the host writes
// there); the argument comes last, so the default instantiation keeps its parameter block.
// KL (target_kl early stopping): the step is not taken when *stop is already set or when the minibatch's approx-KL *kl
// exceeds kl_limit (strictly, compared in double); in the second case the kernel raises *stop.  Every CTA reads both
// before the grid barrier and the word is written after it, so all CTAs take the same decision; a step not taken changes
// no parameter, moment or step counter.
constexpr int ADAM_MAX_CTAS = 120, ADAM_THREADS = 512;
template <bool LR_DEV, bool KL>
__global__ void __launch_bounds__(ADAM_THREADS)
clip_adam_kernel(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m,
                 float *__restrict__ v, int32_t *__restrict__ step, long long n, double lr, double beta1,
                 double beta2, double eps, float max_norm, float *__restrict__ part, const double *__restrict__ lr_dev,
                 const float *__restrict__ kl, unsigned *__restrict__ stop, double kl_limit)
{
    __shared__ float red[ADAM_THREADS / 32];
    __shared__ float s_coef, s_step_size, s_bc2_sqrt;
    const bool skip = KL && (*stop != 0u || (double)*kl > kl_limit);
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    float s = 0.f;
    if (!skip)
        for (long long i = i0; i < n; i += stride) s = fmaf(g[i], g[i], s);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(HRP_FULL, s, d);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < ADAM_THREADS / 32; ++i) t += red[i];
        part[blockIdx.x] = t;
    }
    const int k = step[0] + 1;   // read before the barrier, advanced after it
    cooperative_groups::this_grid().sync();
    if (KL && skip) {
        if (blockIdx.x == 0 && threadIdx.x == 0) *stop = 1u;
        return;
    }
    if (threadIdx.x < 32) {
        // partials in index order, four per lane, then a fixed shuffle tree
        float t = 0.f;
        for (int i = threadIdx.x * 4; i < min((int)gridDim.x, threadIdx.x * 4 + 4); ++i) t += __ldcg(part + i);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) t += __shfl_xor_sync(HRP_FULL, t, d);
        if (threadIdx.x == 0) {
            // torch.optim.Adam forms its scalars in Python doubles and hands float32 values to the kernels
            float total_norm = sqrtf(t);
            float c = max_norm / (total_norm + 1e-6f);
            s_coef = max_norm > 0.f ? fminf(c, 1.f) : 1.f;
            double bc1 = 1.0 - pow(beta1, (double)k), bc2 = 1.0 - pow(beta2, (double)k);
            s_step_size = (float)((LR_DEV ? *lr_dev : lr) / bc1);
            s_bc2_sqrt = (float)sqrt(bc2);
            if (blockIdx.x == 0) step[0] = k;
        }
    }
    __syncthreads();
    const float w1 = (float)(1.0 - beta1), b2 = (float)beta2, w2 = (float)(1.0 - beta2), ep = (float)eps;
    const float coef = s_coef, step_size = s_step_size, bc2_sqrt = s_bc2_sqrt;
    for (long long i = i0; i < n; i += stride) {
        float gi = g[i] * coef;
        float mi = m[i] + w1 * (gi - m[i]);  // exp_avg.lerp_(grad, 1 - beta1)
        float vi = v[i] * b2 + w2 * gi * gi;  // mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
        m[i] = mi; v[i] = vi;
        float denom = sqrtf(vi) / bc2_sqrt + ep;
        p[i] = p[i] - step_size * (mi / denom);
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------
struct hrp_ppo {
    Layout L;
    bool cat;                                // HRP_PPO_CATEGORICAL: L.A = n logits, no log_std
    long long max_batch;
    int device;
    float *ws;  // one arena
    float *x, *z, *olp, *adv, *ret;          // gathered minibatch
    float *vold;                             // gathered rollout values (clipped value loss)
    float *h1, *h2;                          // trunk activations [B,H]
    float *ac;                               // actor | critic hidden activations, one [B, 2H] matrix
    float *mean, *value, *dmean, *dvalue;    // heads and their gradients (mean / dmean: logits when categorical)
    float *d12;                              // d(actor hidden) | d(critic hidden), [B, 2H]
    float *dh2, *dh1;                        // trunk activation gradients [B,H]
    float *wt_ac, *wt_2;                     // transposed weights: [H, 2H] (actor_mean.0 | critic.0) and [H, H] (shared.2)
    float *part_w[3];                        // split-K partials of the three weight-gradient GEMMs
    float *part_b[3];                        // column-sum partials of the three bias gradients (<= 64 chunks)
    float *part_h;                           // head-gradient partials (<= 64 chunks)
    float *loss_part;                        // heads_loss_backward_kernel partial sums [CTAs][8]
    unsigned *loss_counter;
    int splits_cap;
    // fork / join inside one backward pass: the weight- and bias-gradient kernels of a layer do not depend on the
    // input-gradient GEMM of the same layer, so they run on two side streams (captured as parallel graph branches)
    cudaStream_t side[2];
    cudaEvent_t ev[8];
};

// tensor-core path (hrp_mlp_tc.cu)
int hrp_tc_gemm(int M, int N, int K, const float *A, long long sam, long long sak, const float *B, long long sbn,
                long long sbk, float *C, int ldc, const float *bias, int relu, const float *mask, int ldm,
                int accumulate, int splits, int nsplit, cudaStream_t s, int nseg = 0, const float *B2 = nullptr,
                const float *bias2 = nullptr, const TcDots *dots = nullptr, int narrow = 0);
int hrp_tc_gemm_bn(int M, int N, int splits, int nseg, int narrow = 0);

// math mode of the hidden-layer GEMMs: 0 = fp32 SIMT, 1 = TF32 tcgen05, 3 = 3xTF32 tcgen05 (default)
static int g_math_mode = 3;

static int gemm(bool AT, bool BT, int M, int N, int K, const float *A, int lda, const float *B, int ldb, float *C,
                int ldc, const float *bias, int relu, const float *mask, int ldm, int accumulate, int splits,
                cudaStream_t s, int narrow = 0)
{
    if (g_math_mode != 0 && N >= 32 && M >= 32)
        return hrp_tc_gemm(M, N, K, A, AT ? 1 : lda, AT ? lda : 1, B, BT ? ldb : 1, BT ? 1 : ldb, C, ldc, bias, relu,
                           mask, ldm, accumulate, splits, g_math_mode == 1 ? 1 : 3, s, 0, nullptr, nullptr, nullptr, narrow);
    int k_chunk = K;
    if (splits > 1) {
        k_chunk = ((K + splits - 1) / splits + GK - 1) / GK * GK;
        splits = (K + k_chunk - 1) / k_chunk;
    }
    dim3 grid((N + GN - 1) / GN, (M + GM - 1) / GM, splits), blk(256);
    if (!AT && BT) sgemm_kernel<false, true><<<grid, blk, 0, s>>>(M, N, K, A, lda, B, ldb, C, ldc, bias, relu, mask, ldm, accumulate, k_chunk);
    else if (!AT && !BT) sgemm_kernel<false, false><<<grid, blk, 0, s>>>(M, N, K, A, lda, B, ldb, C, ldc, bias, relu, mask, ldm, accumulate, k_chunk);
    else if (AT && !BT) sgemm_kernel<true, false><<<grid, blk, 0, s>>>(M, N, K, A, lda, B, ldb, C, ldc, bias, relu, mask, ldm, accumulate, k_chunk);
    else sgemm_kernel<true, true><<<grid, blk, 0, s>>>(M, N, K, A, lda, B, ldb, C, ldc, bias, relu, mask, ldm, accumulate, k_chunk);
    HRP_CUDA_OK(cudaGetLastError());
    return splits;
}

// weight gradient dW[N,K] = dY[B,N]^T X[B,K] (row pitches lddy, ldx), split over B into `part`; the plan's final
// reduction sums the splits in order (deterministic).  Rows >= n1 of dW go to dW2 (two weight matrices fed by
// one [B, N] gradient matrix); n1 = N, dW2 = nullptr for a single one.
static int wgrad(hrp_ppo *h, ReducePlan &plan, float *part, int N, int K, long long B, const float *dY, int lddy,
                 const float *X, int ldx, float *dW, int n1, float *dW2, cudaStream_t s)
{
    int splits = (int)((B + 255) / 256);
    if (splits > h->splits_cap) splits = h->splits_cap;
    if (splits < 1) splits = 1;
    int used = gemm(true, false, N, K, (int)B, dY, lddy, X, ldx, part, K, nullptr, 0, nullptr, 0, 0, splits, s);
    if (used < 0) return used;
    plan_add(plan, part, (long long)N * K, used, dW, (long long)n1 * K, dW2);
    return 0;
}

// bias gradient db[N] = column sums of G[B, N], first stage (<= 64 row chunks); columns >= n1 go to out2
static int colsum(ReducePlan &plan, float *part, const float *G, int ldg, long long B, int N, float *out, int n1,
                  float *out2, cudaStream_t s)
{
    int chunks = (int)((B + 63) / 64);
    if (chunks > 64) chunks = 64;
    if (chunks < 1) chunks = 1;
    int rows_per = (int)((B + chunks - 1) / chunks);
    dim3 grid((N + 31) / 32, chunks);
    colsum_partial_kernel<<<grid, 256, 0, s>>>(G, ldg, B, N, rows_per, part);
    HRP_CUDA_OK(cudaGetLastError());
    plan_add(plan, part, N, chunks, out, n1, out2);
    return 0;
}

// shared trunk and the two hidden head layers; the latter are one GEMM over the row-stacked weights
// [actor_mean.0 ; critic.0] into h->ac = [a1 | c1]
static int forward_impl(hrp_ppo *h, const float *params, const float *x, long long B, float *mean, float *value,
                        cudaStream_t s)
{
    const Layout &L = h->L;
    int H = L.H, S = L.S, A = L.A, Bi = (int)B;
    if (gemm(false, true, Bi, H, S, x, S, params + L.w1, S, h->h1, H, params + L.b1, 1, nullptr, 0, 0, 1, s, 1) < 0) return -2;
    if (gemm(false, true, Bi, H, H, h->h1, H, params + L.w2, H, h->h2, H, params + L.b2, 1, nullptr, 0, 0, 1, s, 1) < 0) return -2;
    if (g_math_mode != 0 && H % 64 == 0 && Bi >= 32) {
        if (hrp_tc_gemm(Bi, 2 * H, H, h->h2, H, 1, params + L.wa1, H, 1, h->ac, 2 * H, params + L.ba1, 1, nullptr, 0, 0, 1,
                        g_math_mode == 1 ? 1 : 3, s, H, params + L.wc1, params + L.bc1) < 0)
            return -2;
    } else {
        if (gemm(false, true, Bi, H, H, h->h2, H, params + L.wa1, H, h->ac, 2 * H, params + L.ba1, 1, nullptr, 0, 0, 1, s) < 0) return -2;
        if (gemm(false, true, Bi, H, H, h->h2, H, params + L.wc1, H, h->ac + H, 2 * H, params + L.bc1, 1, nullptr, 0, 0, 1, s) < 0) return -2;
    }
    if (!mean) return 0;  // trunk + hidden head layers only (the caller fuses the heads)
    heads_kernel<<<(unsigned)((B + 7) / 8), 256, 0, s>>>(h->ac, h->ac + H, params + L.wa2, params + L.ba2, params + L.wc2,
                                                        params + L.bc2, 2 * H, B, H, A, mean, value);
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------
// ActorCritic.get_action (agent.py:56-74) for ONE state each of many INDEPENDENT policies: the sweep's experiments run a
// single env (main.py:50-58), so their rollout forward is a chain of matrix-VECTOR products -- nothing for a tensor core
// (a 128-row tile would be 1/128 full), everything for bandwidth: 0.85 MB of weights per policy at H = 256.  A cluster of
// ACT_CLUSTER CTAs owns one policy: each CTA forms its slice of a layer's outputs (a warp per output row, coalesced
// weight rows, shuffle reduction in a fixed order), writes the slice into the activation vector of every CTA of the
// cluster through distributed shared memory, and the cluster synchronises once per layer.  CTA 0 finishes with the two
// heads, the tanh-Gaussian sample (the same Philox keying and Box-Muller as heads_act_kernel) and the log-prob.
// One launch serves up to ACT_ITEMS policies of different widths (multiplexed experiments, experiments/multiplex.py).
constexpr int ACT_CLUSTER = 4, ACT_THREADS = 512, ACT_ITEMS = 32, ACT_MAX_DIM = HRP_ACT_MAX_DIM;
struct ActBatch { hrp_act_item it[ACT_ITEMS]; };

__device__ __forceinline__ void act_layer(const float *__restrict__ W, const float *__restrict__ bias, const float *in, int K,
                                          int O, float *out_local, int out_off, unsigned rank, bool relu)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = ACT_THREADS / 32;
    const int per = (O + ACT_CLUSTER - 1) / ACT_CLUSTER;
    const int lo = rank * per, hi = min(O, lo + per);
    for (int o = lo + warp; o < hi; o += nw) {
        const float *w = W + (size_t)o * K;
        float acc0 = 0.f, acc1 = 0.f;
        int k = lane;
        for (; k + 32 < K; k += 64) {
            acc0 = fmaf(w[k], in[k], acc0);
            acc1 = fmaf(w[k + 32], in[k + 32], acc1);
        }
        if (k < K) acc0 = fmaf(w[k], in[k], acc0);
        float acc = acc0 + acc1;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(HRP_FULL, acc, d);
        acc += bias[o];
        if (relu) acc = fmaxf(acc, 0.f);
        if (lane < ACT_CLUSTER) *cluster.map_shared_rank(out_local + out_off + o, lane) = acc;   // to every CTA of the cluster
    }
    cluster.sync();
}

__global__ void __cluster_dims__(ACT_CLUSTER, 1, 1) __launch_bounds__(ACT_THREADS)
act_multi_kernel(const __grid_constant__ ActBatch batch)
{
    namespace cg = cooperative_groups;
    __shared__ float xs[ACT_MAX_DIM], h1[ACT_MAX_DIM], h2[ACT_MAX_DIM], ac[2 * ACT_MAX_DIM];
    const hrp_act_item &it = batch.it[blockIdx.y];
    const unsigned rank = cg::this_cluster().block_rank();
    const int S = it.state_dim, A = it.action_dim, H = it.hidden_dim;
    const Layout L = make_layout(S, A, H);
    const float *p = it.params_dev;
    for (int i = threadIdx.x; i < S; i += ACT_THREADS) xs[i] = it.state_dev[i];
    __syncthreads();
    cg::this_cluster().sync();   // every CTA of the cluster is running before anyone writes into its shared memory
    act_layer(p + L.w1, p + L.b1, xs, S, H, h1, 0, rank, true);
    act_layer(p + L.w2, p + L.b2, h1, H, H, h2, 0, rank, true);
    act_layer(p + L.wa1, p + L.ba1, h2, H, H, ac, 0, rank, true);
    act_layer(p + L.wc1, p + L.bc1, h2, H, H, ac, H, rank, true);
    if (rank != 0) return;
    // heads: warp a < A forms mean[a], warp A the value
    __shared__ float head[8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp <= A) {
        const float *w = warp < A ? p + L.wa2 + (size_t)warp * H : p + L.wc2;
        const float *v = warp < A ? ac : ac + H;
        float acc = 0.f;
        for (int k = lane; k < H; k += 32) acc = fmaf(v[k], w[k], acc);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(HRP_FULL, acc, d);
        if (lane == 0) head[warp] = acc + (warp < A ? p[L.ba2 + warp] : p[L.bc2]);
    }
    __syncthreads();
    if (warp != 0) return;
    const int a = lane < A ? lane : 0;
    const float mu = head[a];
    float nrm = 0.f;
    if (!it.deterministic) {
        uint32_t r[4];
        hrp_philox((uint32_t)it.row, (uint32_t)(it.row >> 32), (uint32_t)it.draw, (uint32_t)(it.draw >> 32),
                   (uint32_t)it.seed, (uint32_t)(it.seed >> 32) ^ 0x5A5A5A5Au, r);
        const uint32_t r1 = a < 2 ? r[0] : r[2], r2 = a < 2 ? r[1] : r[3];
        float u1 = ((float)(r1 >> 8) + 0.5f) * (1.0f / 16777216.0f);
        float u2 = ((float)(r2 >> 8) + 0.5f) * (1.0f / 16777216.0f);
        float rad = sqrtf(-2.f * logf(u1)), sn, cs;
        sincospif(2.f * u2, &sn, &cs);
        nrm = rad * ((a & 1) ? sn : cs);
    }
    const float ls = p[L.log_std + a], sd = expf(ls);
    const float z = it.deterministic ? mu : mu + sd * nrm;
    const float t = tanhf(z);
    const float d = z - mu;
    float lp = -(d * d) / (2.f * sd * sd) - ls - 0.91893853320467274f;
    lp -= log1pf(-(t * t) + 1e-6f);
    lp = lane < A ? lp : 0.f;
    lp += __shfl_xor_sync(HRP_FULL, lp, 1);
    lp += __shfl_xor_sync(HRP_FULL, lp, 2);
    if (lane < A) { it.out_dev[lane] = t; it.out_dev[A + lane] = z; }
    if (lane == 0) { it.out_dev[2 * A] = it.deterministic ? 0.f : lp; it.out_dev[2 * A + 1] = head[A]; }
}

// The act path with the heads fused into the last GEMM (TcDots): the [a1 | c1] GEMM left, per N tile and row, the
// partial dot products with the head weights; a thread per row adds the tiles in tile order, adds the biases and
// samples exactly as heads_act_kernel does (same Philox counters, same Box-Muller pairing, same log-prob arithmetic).
__global__ void __launch_bounds__(128)
heads_finish_kernel(const float *__restrict__ part, int tiles_a, int tiles, const float *__restrict__ ba2,
                    const float *__restrict__ bc2, const float *__restrict__ log_std, const float *__restrict__ noise, int mode,
                    unsigned long long seed, unsigned long long draw, unsigned long long row_base, long long B, int A,
                    float *__restrict__ action, float *__restrict__ pre_tanh, float *__restrict__ log_prob,
                    float *__restrict__ value, unsigned long long *draw_ctr)
{
    hrp_pdl_release();
    hrp_pdl_wait();
    if (draw_ctr) {   // device-resident draw counter, as in heads_act_kernel
        __shared__ unsigned long long sdraw;
        if (threadIdx.x == 0) {
            sdraw = *(volatile unsigned long long *)draw_ctr + 1ull;
            __threadfence();
            if (atomicAdd(draw_ctr + 1, 1ull) == (unsigned long long)gridDim.x - 1ull) {
                draw_ctr[1] = 0ull;
                draw_ctr[0] = sdraw;
            }
        }
        __syncthreads();
        draw = sdraw;
    }
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float mu[4] = {0.f, 0.f, 0.f, 0.f}, val = 0.f;
    for (int t = 0; t < tiles; ++t) {
        const float4 p = *reinterpret_cast<const float4 *>(part + ((size_t)t * B + b) * 4);
        if (t < tiles_a) { mu[0] += p.x; mu[1] += p.y; mu[2] += p.z; mu[3] += p.w; }
        else val += p.x;
    }
    uint32_t r[4] = {0u, 0u, 0u, 0u};
    if (mode == 2) {
        const unsigned long long gb = row_base + (unsigned long long)b;
        hrp_philox((uint32_t)gb, (uint32_t)(gb >> 32), (uint32_t)draw, (uint32_t)(draw >> 32),
                   (uint32_t)seed, (uint32_t)(seed >> 32) ^ 0x5A5A5A5Au, r);
    }
    float lp = 0.f;
    for (int a = 0; a < A; ++a) {
        const float m = mu[a] + ba2[a];
        float nrm = 0.f;
        if (mode == 2) {
            const uint32_t r1 = a < 2 ? r[0] : r[2], r2 = a < 2 ? r[1] : r[3];
            float u1 = ((float)(r1 >> 8) + 0.5f) * (1.0f / 16777216.0f);
            float u2 = ((float)(r2 >> 8) + 0.5f) * (1.0f / 16777216.0f);
            float rad = sqrtf(-2.f * logf(u1)), sn, cs;
            sincospif(2.f * u2, &sn, &cs);
            nrm = rad * ((a & 1) ? sn : cs);
        } else if (mode == 1) {
            nrm = noise[b * A + a];
        }
        const float ls = log_std[a], sd = expf(ls);
        const float z = mode ? m + sd * nrm : m;
        const float t = tanhf(z);
        const float d = z - m;
        float l = -(d * d) / (2.f * sd * sd) - ls - 0.91893853320467274f;
        l -= log1pf(-(t * t) + 1e-6f);
        lp += l;
        pre_tanh[b * A + a] = z;
        action[b * A + a] = t;
    }
    if (log_prob) log_prob[b] = mode ? lp : 0.f;
    value[b] = val + bc2[0];
}

static int act_impl(hrp_ppo *h, const float *params, const float *states, const float *noise, int mode,
                    unsigned long long seed, unsigned long long draw, unsigned long long row_base, long long batch,
                    float *action, float *pre_tanh, float *log_prob, float *value, cudaStream_t s,
                    unsigned long long *draw_ctr = nullptr)
{
    const Layout &L = h->L;
    {
        // heads fused into the [a1 | c1] GEMM's epilogue whenever its tiles do not straddle H (HRP_FUSE_HEADS=0: off)
        static const bool fuse_on = !(getenv("HRP_FUSE_HEADS") && getenv("HRP_FUSE_HEADS")[0] == '0');
        const int H = L.H, Bi = (int)batch;
        const int bn = hrp_tc_gemm_bn(Bi, 2 * H, 1, H, 1);
        if (fuse_on && g_math_mode != 0 && H % 64 == 0 && Bi >= 32 && H % bn == 0) {
            if (gemm(false, true, Bi, H, L.S, states, L.S, params + L.w1, L.S, h->h1, H, params + L.b1, 1, nullptr, 0, 0, 1, s, 1) < 0) return -2;
            if (gemm(false, true, Bi, H, H, h->h1, H, params + L.w2, H, h->h2, H, params + L.b2, 1, nullptr, 0, 0, 1, s, 1) < 0) return -2;
            // partial sums in the (idle) backward scratch d12: [2 H / bn tiles][B][4 or 8] <= [B][2 H] floats
            const TcDots dots{params + L.wa2, params + L.wc2, H, L.A, h->d12, 1};
            if (hrp_tc_gemm(Bi, 2 * H, H, h->h2, H, 1, params + L.wa1, H, 1, h->ac, 2 * H, params + L.ba1, 1, nullptr, 0, 0, 1,
                            g_math_mode == 1 ? 1 : 3, s, H, params + L.wc1, params + L.bc1, &dots, 1) < 0)
                return -2;
            if (h->cat) {
                auto kern = L.A <= 4 ? heads_finish_cat_kernel<4> : heads_finish_cat_kernel<8>;
                HRP_CUDA_OK(hrp_launch_pdl(kern, dim3((unsigned)((batch + 127) / 128)), dim3(128), 0, s, (const float *)h->d12,
                                           H / bn, 2 * H / bn, params + L.ba2, params + L.bc2, noise, mode, seed, draw,
                                           row_base, (long long)batch, L.A, action, pre_tanh, log_prob, value, draw_ctr));
                return 0;
            }
            HRP_CUDA_OK(hrp_launch_pdl(heads_finish_kernel, dim3((unsigned)((batch + 127) / 128)), dim3(128), 0, s,
                                       (const float *)h->d12, H / bn, 2 * H / bn, params + L.ba2, params + L.bc2,
                                       params + L.log_std, noise, mode, seed, draw, row_base, (long long)batch, L.A, action,
                                       pre_tanh, log_prob, value, draw_ctr));
            return 0;
        }
    }
    if (int rc = forward_impl(h, params, states, batch, nullptr, nullptr, s)) return rc;
    const float *pa = h->ac, *pc = h->ac + L.H;
    const int vec = L.H % 128 == 0 && (((uintptr_t)pa | (uintptr_t)pc) & 15) == 0 ? 1 : 0;   // row pitch 2 H: a multiple of 4 with H
    const size_t smem = (size_t)(L.A + 1) * L.H * sizeof(float);
    if (h->cat) {
        HRP_CUDA_OK(hrp_launch_pdl(heads_act_cat_kernel, dim3((unsigned)((batch + 8 * HA_ROWS - 1) / (8 * HA_ROWS))), dim3(256),
                                   smem, s, pa, pc, params + L.wa2, params + L.ba2, params + L.wc2, params + L.bc2, noise, mode,
                                   seed, draw, row_base, 2 * L.H, (long long)batch, L.H, L.A, action, pre_tanh, log_prob, value,
                                   draw_ctr, vec));
        return 0;
    }
    HRP_CUDA_OK(hrp_launch_pdl(heads_act_kernel, dim3((unsigned)((batch + 8 * HA_ROWS - 1) / (8 * HA_ROWS))), dim3(256), smem, s,
                               pa, pc, params + L.wa2, params + L.ba2, params + L.wc2, params + L.bc2,
                               params + L.log_std, noise, mode, seed, draw, row_base, 2 * L.H, (long long)batch, L.H, L.A,
                               action, pre_tanh, log_prob, value, draw_ctr, vec));
    return 0;
}

extern "C" {

int hrp_ppo_set_math(int32_t mode)
{
    if (mode != 0 && mode != 1 && mode != 3) { hrp_set_error("hrp_ppo_set_math: mode must be 0, 1 or 3"); return -1; }
    g_math_mode = mode;
    return 0;
}
int hrp_ppo_get_math(void) { return g_math_mode; }

int hrp_gemm_strided(int32_t M, int32_t N, int32_t K, const float *A, int64_t sam, int64_t sak, const float *B,
                     int64_t sbn, int64_t sbk, float *C, int32_t ldc, const float *bias, int32_t relu, int32_t mode,
                     void *stream)
{
    if (!A || !B || !C || M < 1 || N < 1 || K < 1 || ldc < N) { hrp_set_error("hrp_gemm_strided: bad arguments"); return -1; }
    if (mode != 1 && mode != 3) { hrp_set_error("hrp_gemm_strided: mode must be 1 (TF32) or 3 (3xTF32)"); return -1; }
    int rc = hrp_tc_gemm(M, N, K, A, sam, sak, B, sbn, sbk, C, ldc, bias, relu, nullptr, 0, 0, 1, mode,
                         (cudaStream_t)stream);
    return rc < 0 ? rc : 0;
}

int64_t hrp_ppo_param_count(int32_t state_dim, int32_t action_dim, int32_t hidden_dim)
{
    return make_layout(state_dim, action_dim, hidden_dim).total;
}

int64_t hrp_ppo_param_count_ex(int32_t state_dim, int32_t action_dim, int32_t hidden_dim, uint32_t flags)
{
    return make_layout(state_dim, action_dim, hidden_dim, (flags & HRP_PPO_CATEGORICAL) != 0).total;
}

static int ppo_create(int32_t state_dim, int32_t action_dim, int32_t hidden_dim, int64_t max_batch, int32_t device,
                      bool cat, hrp_ppo **out);

int hrp_ppo_create(int32_t state_dim, int32_t action_dim, int32_t hidden_dim, int64_t max_batch, int32_t device,
                   hrp_ppo **out)
{
    if (!out || state_dim < 1 || hidden_dim < 1 || action_dim < 1 || action_dim > 4 || max_batch < 1) {
        hrp_set_error("hrp_ppo_create: bad arguments (action_dim must be 1..4)");
        return -1;
    }
    return ppo_create(state_dim, action_dim, hidden_dim, max_batch, device, false, out);
}

int hrp_ppo_create_ex(int32_t state_dim, int32_t action_dim, int32_t hidden_dim, int64_t max_batch, int32_t device,
                      uint32_t flags, hrp_ppo **out)
{
    if (flags & ~HRP_PPO_CATEGORICAL) { hrp_set_error("hrp_ppo_create_ex: flags 0x%x has unknown bits", (unsigned)flags); return -1; }
    if (!(flags & HRP_PPO_CATEGORICAL)) return hrp_ppo_create(state_dim, action_dim, hidden_dim, max_batch, device, out);
    if (!out) { hrp_set_error("hrp_ppo_create_ex: out is NULL"); return -1; }
    if (state_dim < 1) { hrp_set_error("hrp_ppo_create_ex: state_dim %d must be >= 1", (int)state_dim); return -1; }
    if (hidden_dim < 1) { hrp_set_error("hrp_ppo_create_ex: hidden_dim %d must be >= 1", (int)hidden_dim); return -1; }
    if (max_batch < 1) { hrp_set_error("hrp_ppo_create_ex: max_batch %lld must be >= 1", (long long)max_batch); return -1; }
    if (action_dim < 2 || action_dim > CAT_MAX) {
        hrp_set_error("hrp_ppo_create_ex: action_dim %d (the number of discrete actions) must be in [2, %d]",
                      (int)action_dim, CAT_MAX);
        return -1;
    }
    return ppo_create(state_dim, action_dim, hidden_dim, max_batch, device, true, out);
}

static int ppo_create(int32_t state_dim, int32_t action_dim, int32_t hidden_dim, int64_t max_batch, int32_t device,
                      bool cat, hrp_ppo **out)
{
    int ndev = hrp_device_count();
    if (ndev <= 0) { hrp_set_error("no CUDA device: this library has no CPU path"); return -3; }
    if (device < 0 || device >= ndev) { hrp_set_error("device %d not in [0, %d)", device, ndev); return -1; }
    HRP_CUDA_OK(cudaSetDevice(device));
    {
        // the unfused act kernels keep the A + 1 head rows in shared memory: above 48 KB the launch needs the opt-in.
        // The limit is raised to everything the device allows (not to this policy's need), so that creating a
        // narrower policy later cannot lower it under a wider one's.
        const size_t smem = (size_t)(action_dim + 1) * hidden_dim * sizeof(float);
        if (smem > 48 * 1024) {
            const void *kern = cat ? (const void *)heads_act_cat_kernel : (const void *)heads_act_kernel;
            int optin = 0;
            cudaFuncAttributes fa;
            HRP_CUDA_OK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
            HRP_CUDA_OK(cudaFuncGetAttributes(&fa, kern));
            const size_t room = (size_t)optin - fa.sharedSizeBytes;
            if (smem > room) {
                hrp_set_error("hrp_ppo_create: hidden_dim %d with action_dim %d needs %zu bytes of shared memory for the "
                              "act heads, above the device's %zu", (int)hidden_dim, (int)action_dim, smem, room);
                return -1;
            }
            HRP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)room));
        }
    }
    hrp_ppo *h = new hrp_ppo();
    h->L = make_layout(state_dim, action_dim, hidden_dim, cat);
    h->cat = cat;
    h->max_batch = max_batch; h->device = device;
    h->splits_cap = 32;
    size_t B = (size_t)max_batch, H = hidden_dim, S = state_dim, A = action_dim;
    const size_t cap = (size_t)h->splits_cap;
    // every sub-buffer starts on a 128-byte boundary (float4 / cp.async operand staging)
    auto pad = [](size_t n) { return (n + 31) / 32 * 32; };
    const size_t sizes[] = {B * S, B * A, B, B, B, B * H, B * H, 2 * B * H, B * A, B * A, B, B, 2 * B * H, B * H, B * H,
                            2 * H * H, H * H, cap * 2 * H * H, cap * H * H, cap * H * S, 64 * 2 * H, 64 * H, 64 * H,
                            64 * ((A + 1) * H + A + 1), ((B + HLB_ROWS - 1) / HLB_ROWS) * 8, 32, B};
    size_t n = 0;
    for (size_t q : sizes) n += pad(q);
    cudaError_t ce = cudaMalloc(&h->ws, n * sizeof(float));
    if (ce != cudaSuccess) { hrp_set_error("cudaMalloc(%zu): %s", n * sizeof(float), cudaGetErrorString(ce)); delete h; return -2; }
    float *p = h->ws;
    int qi = 0;
    auto take = [&]() { float *r = p; p += pad(sizes[qi++]); return r; };
    h->x = take(); h->z = take(); h->olp = take(); h->adv = take(); h->ret = take();
    h->h1 = take(); h->h2 = take(); h->ac = take();
    h->mean = take(); h->dmean = take(); h->value = take(); h->dvalue = take();
    h->d12 = take(); h->dh2 = take(); h->dh1 = take();
    h->wt_ac = take(); h->wt_2 = take();
    for (int q = 0; q < 3; ++q) h->part_w[q] = take();
    for (int q = 0; q < 3; ++q) h->part_b[q] = take();
    h->part_h = take(); h->loss_part = take();
    h->loss_counter = (unsigned *)take();
    h->vold = take();
    ce = cudaMemset(h->loss_counter, 0, 32 * sizeof(float));
    for (int q = 0; q < 2 && ce == cudaSuccess; ++q) ce = cudaStreamCreateWithFlags(&h->side[q], cudaStreamNonBlocking);
    for (int q = 0; q < 8 && ce == cudaSuccess; ++q) ce = cudaEventCreateWithFlags(&h->ev[q], cudaEventDisableTiming);
    if (ce != cudaSuccess) { hrp_set_error("hrp_ppo_create: %s", cudaGetErrorString(ce)); cudaFree(h->ws); delete h; return -2; }
    *out = h;
    return 0;
}

int hrp_ppo_destroy(hrp_ppo *h)
{
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaFree(h->ws);
    for (int q = 0; q < 2; ++q) if (h->side[q]) cudaStreamDestroy(h->side[q]);
    for (int q = 0; q < 8; ++q) if (h->ev[q]) cudaEventDestroy(h->ev[q]);
    delete h;
    return 0;
}

int hrp_ppo_forward(hrp_ppo *h, const float *params, const float *states, int64_t batch, float *mean, float *value,
                    void *stream)
{
    if (!h || !params || !states || !mean || !value) { hrp_set_error("hrp_ppo_forward: null argument"); return -1; }
    if (batch < 1 || batch > h->max_batch) { hrp_set_error("batch %lld outside [1, %lld]", (long long)batch, h->max_batch); return -1; }
    return forward_impl(h, params, states, batch, mean, value, (cudaStream_t)stream);
}

int hrp_ppo_act(hrp_ppo *h, const float *params, const float *states, const float *noise, int64_t batch,
                float *action, float *pre_tanh, float *log_prob, float *value, void *stream)
{
    if (!h || !params || !states || !action || !pre_tanh || !value) { hrp_set_error("hrp_ppo_act: null argument"); return -1; }
    if (batch < 1 || batch > h->max_batch) { hrp_set_error("batch %lld outside [1, %lld]", (long long)batch, h->max_batch); return -1; }
    return act_impl(h, params, states, noise, noise ? 1 : 0, 0ull, 0ull, 0ull, batch, action, pre_tanh, log_prob, value,
                    (cudaStream_t)stream);
}

int hrp_ppo_act_sample(hrp_ppo *h, const float *params, const float *states, uint64_t seed, uint64_t draw,
                       uint64_t row_base, int64_t batch, float *action, float *pre_tanh, float *log_prob, float *value,
                       void *stream)
{
    if (!h || !params || !states || !action || !pre_tanh || !value) { hrp_set_error("hrp_ppo_act_sample: null argument"); return -1; }
    if (batch < 1 || batch > h->max_batch) { hrp_set_error("batch %lld outside [1, %lld]", (long long)batch, h->max_batch); return -1; }
    return act_impl(h, params, states, nullptr, 2, seed, draw, row_base, batch, action, pre_tanh, log_prob, value,
                    (cudaStream_t)stream);
}

int hrp_ppo_act_sample_ctr(hrp_ppo *h, const float *params, const float *states, uint64_t seed, uint64_t *draw_ctr_dev,
                           uint64_t row_base, int64_t batch, float *action, float *pre_tanh, float *log_prob,
                           float *value, void *stream)
{
    if (!h || !params || !states || !action || !pre_tanh || !value || !draw_ctr_dev) {
        hrp_set_error("hrp_ppo_act_sample_ctr: null argument");
        return -1;
    }
    if (batch < 1 || batch > h->max_batch) { hrp_set_error("batch %lld outside [1, %lld]", (long long)batch, h->max_batch); return -1; }
    return act_impl(h, params, states, nullptr, 2, seed, 0ull, row_base, batch, action, pre_tanh, log_prob, value,
                    (cudaStream_t)stream, (unsigned long long *)draw_ctr_dev);
}

int hrp_ppo_act_multi(const hrp_act_item *items, int32_t count, void *stream)
{
    if (!items || count < 0) { hrp_set_error("hrp_ppo_act_multi: bad arguments"); return -1; }
    for (int32_t i = 0; i < count; ++i) {
        const hrp_act_item &it = items[i];
        if (!it.params_dev || !it.state_dev || !it.out_dev || it.state_dim < 1 || it.state_dim > ACT_MAX_DIM || it.hidden_dim < 1 ||
            it.hidden_dim > ACT_MAX_DIM || it.action_dim < 1 || it.action_dim > 4) {
            hrp_set_error("hrp_ppo_act_multi: item %d: null pointer, or state_dim / hidden_dim outside [1, %d], or "
                          "action_dim outside [1, 4]", (int)i, ACT_MAX_DIM);
            return -1;
        }
    }
    for (int32_t lo = 0; lo < count; lo += ACT_ITEMS) {
        ActBatch b;
        const int n = count - lo < ACT_ITEMS ? count - lo : ACT_ITEMS;
        for (int i = 0; i < n; ++i) b.it[i] = items[lo + i];
        for (int i = n; i < ACT_ITEMS; ++i) b.it[i] = items[lo];
        act_multi_kernel<<<dim3(ACT_CLUSTER, n), ACT_THREADS, 0, (cudaStream_t)stream>>>(b);
        HRP_CUDA_OK(cudaGetLastError());
    }
    return 0;
}

int hrp_gae(const float *reward, const float *value, const uint8_t *done, const float *last_value, int64_t T,
            int64_t E, double gamma, double lam, float *adv, float *ret, void *stream)
{
    if (!reward || !value || !done || !adv || !ret || T < 1 || E < 1) { hrp_set_error("hrp_gae: bad arguments"); return -1; }
    gae_kernel<<<(unsigned)((E + 127) / 128), 128, 0, (cudaStream_t)stream>>>(reward, value, done, last_value, T, E,
                                                                            gamma, lam, adv, ret);
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}

int hrp_gae_ex(const float *reward, const float *value, const uint8_t *terminated, const uint8_t *truncated,
               const float *final_value, const float *last_value, int64_t T, int64_t E, double gamma, double lam,
               float *adv, float *ret, void *stream)
{
    const char *missing = !reward ? "reward_dev" : !value ? "value_dev" : !terminated ? "terminated_dev"
                        : !truncated ? "truncated_dev" : !adv ? "adv_dev" : !ret ? "ret_dev" : nullptr;
    if (missing) { hrp_set_error("hrp_gae_ex: %s is null", missing); return -1; }
    if (T < 1) { hrp_set_error("hrp_gae_ex: T = %lld < 1", (long long)T); return -1; }
    if (E < 1) { hrp_set_error("hrp_gae_ex: E = %lld < 1", (long long)E); return -1; }
    gae_ex_kernel<<<(unsigned)((E + 127) / 128), 128, 0, (cudaStream_t)stream>>>(reward, value, terminated, truncated,
                                                                               final_value, last_value, T, E, gamma, lam,
                                                                               adv, ret);
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}

int hrp_adv_stats(const float *adv, int64_t n, double *stats, void *stream)
{
    if (!adv || !stats || n < 1) { hrp_set_error("hrp_adv_stats: bad arguments"); return -1; }
    // stats_dev must hold 3 + 2*256 doubles: (sum, sumsq, n) followed by the block partials
    const int nb = 256;
    int blocks = (int)((n + 255) / 256);
    if (blocks > nb) blocks = nb;
    adv_stats_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(adv, n, stats + 3);
    adv_stats_final_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(stats + 3, blocks, n, stats);
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}

int hrp_adv_normalize(float *adv, int64_t n, const double *stats, void *stream)
{
    if (!adv || !stats || n < 1) { hrp_set_error("hrp_adv_normalize: bad arguments"); return -1; }
    adv_normalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(adv, n, stats);
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"

// hrp_ppo_loss_grad, and with old_value non-NULL the clipped value loss of hrp_ppo_loss_grad_ex (the VCLIP kernels)
static int loss_grad_impl(hrp_ppo *h, const float *params, const float *states, const float *pre_tanh,
                          const float *old_log_prob, const float *adv, const float *ret, const int64_t *idx,
                          int64_t batch, float eps_clip, float value_coef, float entropy_coef, float loss_scale,
                          const float *old_value, float value_clip, float *grad, float *metrics, void *stream,
                          float *kl_out = nullptr, const unsigned *stop = nullptr)
{
    if (!h || !params || !states || !pre_tanh || !old_log_prob || !adv || !ret || !grad) {
        hrp_set_error("hrp_ppo_loss_grad: null argument");
        return -1;
    }
    if (batch < 1 || batch > h->max_batch) { hrp_set_error("batch %lld outside [1, %lld]", (long long)batch, h->max_batch); return -1; }
    cudaStream_t s = (cudaStream_t)stream, s0 = h->side[0], s1 = h->side[1];
    const Layout &L = h->L;
    const int H = L.H, S = L.S, A = L.A, Bi = (int)batch, H2 = 2 * H;
    const long long B = batch;
    const float *x = states, *z = pre_tanh, *olp = old_log_prob, *ad = adv, *rt = ret, *vo = old_value;
    const bool vclip = old_value != nullptr;
    // `from` has produced something `to` consumes (also valid while the caller's stream is being captured: the side
    // streams join the capture and are joined back before this function returns)
    auto after = [&](int e, cudaStream_t from, cudaStream_t to) -> cudaError_t {
        cudaError_t ce = cudaEventRecord(h->ev[e], from);
        return ce != cudaSuccess ? ce : cudaStreamWaitEvent(to, h->ev[e], 0);
    };
    const int Az = h->cat ? 1 : A;   // floats per row of pre_tanh: the sampled id of a categorical policy
    auto heads_wgrad = h->cat && A > 4 ? heads_wgrad_partial_kernel<8> : heads_wgrad_partial_kernel<4>;
    // side stream 1: transposed weight copies for the input-gradient GEMMs (needs the parameters only)
    HRP_CUDA_OK(after(0, s, s1));
    {
        dim3 grid((H + 31) / 32, (H + 31) / 32, 3);
        transpose_weights_kernel<<<grid, 256, 0, s1>>>(params + L.wa1, params + L.wc1, params + L.w2, H, h->wt_ac, h->wt_2);
        HRP_CUDA_OK(cudaGetLastError());
        HRP_CUDA_OK(cudaEventRecord(h->ev[3], s1));   // the transposed copies are ready (waited for before d(h2))
    }
    if (idx) {
        const long long *ix = (const long long *)idx;
        long long tot = B * (S + Az + (vclip ? 4 : 3));
        auto gather = vclip ? gather_batch_kernel<true> : gather_batch_kernel<false>;
        gather<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(states, pre_tanh, old_log_prob, adv, ret, ix, B, S, Az, h->x,
                                                              h->z, h->olp, h->adv, h->ret, old_value, h->vold);
        HRP_CUDA_OK(cudaGetLastError());
        x = h->x; z = h->z; olp = h->olp; ad = h->adv; rt = h->ret;
        if (vclip) vo = h->vold;
    }
    if (int rc = forward_impl(h, params, x, B, nullptr, nullptr, s)) return rc;   // trunk + hidden head layers
    const bool kl = kl_out != nullptr;
    auto loss_cat = vclip ? (kl ? heads_loss_backward_cat_kernel<true, true> : heads_loss_backward_cat_kernel<true, false>)
                          : (kl ? heads_loss_backward_cat_kernel<false, true> : heads_loss_backward_cat_kernel<false, false>);
    auto loss_gauss = vclip ? (kl ? heads_loss_backward_kernel<true, true> : heads_loss_backward_kernel<true, false>)
                            : (kl ? heads_loss_backward_kernel<false, true> : heads_loss_backward_kernel<false, false>);
    if (h->cat) HRP_CUDA_OK(hrp_launch_pdl(loss_cat,
                                           dim3((unsigned)((B + HLB_ROWS - 1) / HLB_ROWS)), dim3(256),
                                           0, s, (const float *)h->ac, (const float *)(h->ac + H), H2, H, params + L.wa2,
                                           params + L.ba2, params + L.wc2, params + L.bc2, z, olp, ad, rt, B, A, eps_clip,
                                           value_coef, entropy_coef, loss_scale, h->dmean, h->dvalue, h->d12, h->d12 + H,
                                           metrics, h->loss_part, h->loss_counter, vo, value_clip, kl_out, stop));
    else HRP_CUDA_OK(hrp_launch_pdl(loss_gauss,
                               dim3((unsigned)((B + HLB_ROWS - 1) / HLB_ROWS)), dim3(256), 0, s,
                               (const float *)h->ac, (const float *)(h->ac + H), H2, H, params + L.wa2, params + L.ba2,
                               params + L.wc2, params + L.bc2, params + L.log_std, z, olp, ad, rt, B, A, eps_clip, value_coef,
                               entropy_coef, loss_scale, h->dmean, h->dvalue, h->d12, h->d12 + H, grad + L.log_std, metrics,
                               h->loss_part, h->loss_counter, vo, value_clip, kl_out, stop));
    const float *a1 = h->ac, *c1 = h->ac + H;
    ReducePlan plan;
    plan.nseg = 0; plan.blocks = 0;
    // side stream 0 -- heads: dWa2 = dmean^T a1, dba2 = colsum(dmean); dWc2 = dvalue^T c1, dbc2 = sum(dvalue).  The
    // chunk sums are laid out [A*H + A | H + 1]: the first part lands on grad + wa2 (ba2 follows wa2), the second on
    // grad + wc2.
    HRP_CUDA_OK(after(1, s, s0));
    {
        int chunks = (int)((B + 63) / 64);
        if (chunks > 64) chunks = 64;
        int rows_per = (int)((B + chunks - 1) / chunks);
        dim3 grid((H + 31) / 32, chunks);
        heads_wgrad<<<grid, 256, 0, s0>>>(h->dmean, h->dvalue, a1, c1, H2, B, H, A, rows_per, h->part_h);
        HRP_CUDA_OK(cudaGetLastError());
        plan_add(plan, h->part_h, (long long)A * H + A + H + 1, chunks, grad + L.wa2, (long long)A * H + A, grad + L.wc2);
    }
    // side 1: [dWa1 ; dWc1] = [d(a1) | d(c1)]^T h2 in one GEMM, [dba1 | dbc1] in one column sum
    HRP_CUDA_OK(after(2, s, s1));
    if (wgrad(h, plan, h->part_w[0], H2, H, B, h->d12, H2, h->h2, H, grad + L.wa1, H, grad + L.wc1, s1)) return -2;
    if (colsum(plan, h->part_b[0], h->d12, H2, B, H2, grad + L.ba1, H, grad + L.bc1, s1)) return -2;
    // main: d(h2) = [d(a1) | d(c1)] [Wa1 ; Wc1] (.) (h2>0): K = 2H against the transposed copies
    HRP_CUDA_OK(cudaStreamWaitEvent(s, h->ev[3], 0));
    if (gemm(false, true, Bi, H, H2, h->d12, H2, h->wt_ac, H2, h->dh2, H, nullptr, 0, h->h2, H, 0, 1, s) < 0) return -2;
    // side 0 (behind the short heads kernel; side 1 is still busy with [dWa1 ; dWc1]): dW2, db2 start as soon as d(h2)
    // exists, beside d(h1), so that dW1 at the end of the chain does not have to share the machine with them
    HRP_CUDA_OK(after(4, s, s0));
    if (wgrad(h, plan, h->part_w[1], H, H, B, h->dh2, H, h->h1, H, grad + L.w2, H, nullptr, s0)) return -2;
    if (colsum(plan, h->part_b[1], h->dh2, H, B, H, grad + L.b2, H, nullptr, s0)) return -2;
    // main: d(h1) = d(h2) W2 (.) (h1>0), dW1; side 0: db1
    if (gemm(false, true, Bi, H, H, h->dh2, H, h->wt_2, H, h->dh1, H, nullptr, 0, h->h1, H, 0, 1, s) < 0) return -2;
    HRP_CUDA_OK(after(5, s, s0));
    if (colsum(plan, h->part_b[2], h->dh1, H, B, H, grad + L.b1, H, nullptr, s0)) return -2;
    if (wgrad(h, plan, h->part_w[2], H, S, B, h->dh1, H, x, S, grad + L.w1, H, nullptr, s)) return -2;
    // join, then every second-stage reduction in one launch
    HRP_CUDA_OK(after(6, s0, s));
    HRP_CUDA_OK(after(7, s1, s));
    final_reduce_kernel<<<plan.blocks, 256, 0, s>>>(plan);
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}

template <bool LR_DEV, bool KL>
static int clip_adam_launch(float *params, const float *grad, float *exp_avg, float *exp_avg_sq, int32_t *step, int64_t n,
                            double lr, const double *lr_dev, double beta1, double beta2, double eps, float max_grad_norm,
                            float *scratch, void *stream, const float *kl = nullptr, unsigned *stop = nullptr,
                            double kl_limit = 0.0)
{
    cudaStream_t s = (cudaStream_t)stream;
    // per device: a process may drive several GPUs (ExperimentRunner with a device pool)
    static int max_ctas_dev[HRP_MAX_DEVICES] = {0};
    int dev = 0;
    HRP_CUDA_OK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= HRP_MAX_DEVICES) { hrp_set_error("device index %d not supported", dev); return -1; }
    int &max_ctas = max_ctas_dev[dev];
    if (max_ctas == 0) {
        int sms = 0, per_sm = 0;
        HRP_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        HRP_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, clip_adam_kernel<LR_DEV, KL>, ADAM_THREADS, 0));
        max_ctas = sms * per_sm < ADAM_MAX_CTAS ? sms * per_sm : ADAM_MAX_CTAS;
        if (max_ctas < 1) { hrp_set_error("hrp_clip_adam_step: kernel does not fit the device"); return -2; }
    }
    int ctas = (int)((n + ADAM_THREADS - 1) / ADAM_THREADS);
    if (ctas > max_ctas) ctas = max_ctas;
    long long n_ = n;
    void *args[] = {&params, &grad, &exp_avg, &exp_avg_sq, &step, &n_, &lr, &beta1, &beta2, &eps, &max_grad_norm, &scratch,
                    &lr_dev, &kl, &stop, &kl_limit};
    HRP_CUDA_OK(cudaLaunchCooperativeKernel((const void *)clip_adam_kernel<LR_DEV, KL>, dim3(ctas), dim3(ADAM_THREADS), args, 0, s));
    return 0;
}

extern "C" {

int hrp_ppo_loss_grad(hrp_ppo *h, const float *params, const float *states, const float *pre_tanh,
                      const float *old_log_prob, const float *adv, const float *ret, const int64_t *idx, int64_t batch,
                      float eps_clip, float value_coef, float entropy_coef, float loss_scale, float *grad,
                      float *metrics, void *stream)
{
    return loss_grad_impl(h, params, states, pre_tanh, old_log_prob, adv, ret, idx, batch, eps_clip, value_coef,
                          entropy_coef, loss_scale, nullptr, 0.f, grad, metrics, stream);
}

int hrp_ppo_loss_grad_ex(hrp_ppo *h, const float *params, const float *states, const float *pre_tanh,
                         const float *old_log_prob, const float *adv, const float *ret, const int64_t *idx,
                         int64_t batch, float eps_clip, float value_coef, float entropy_coef, float loss_scale,
                         const float *old_value, float value_clip, float *grad, float *metrics, void *stream)
{
    // checked first: the other arguments are then validated exactly as hrp_ppo_loss_grad validates them
    if (old_value && !(std::isfinite(value_clip) && value_clip > 0.f)) {
        hrp_set_error("hrp_ppo_loss_grad_ex: value_clip must be finite and > 0 with old_value_dev, got %g", (double)value_clip);
        return -1;
    }
    return loss_grad_impl(h, params, states, pre_tanh, old_log_prob, adv, ret, idx, batch, eps_clip, value_coef,
                          entropy_coef, loss_scale, old_value, value_clip, grad, metrics, stream);
}

int hrp_clip_adam_step(float *params, const float *grad, float *exp_avg, float *exp_avg_sq, int32_t *step, int64_t n,
                       double lr, double beta1, double beta2, double eps, float max_grad_norm, float *scratch,
                       void *stream)
{
    if (!params || !grad || !exp_avg || !exp_avg_sq || !step || !scratch || n < 1) {
        hrp_set_error("hrp_clip_adam_step: bad arguments");
        return -1;
    }
    return clip_adam_launch<false, false>(params, grad, exp_avg, exp_avg_sq, step, n, lr, nullptr, beta1, beta2, eps,
                                          max_grad_norm, scratch, stream);
}

int hrp_clip_adam_step_ex(float *params, const float *grad, float *exp_avg, float *exp_avg_sq, int32_t *step, int64_t n,
                          double lr, const double *lr_dev, double beta1, double beta2, double eps, float max_grad_norm,
                          float *scratch, void *stream)
{
    const char *bad = !params ? "params_dev" : !grad ? "grad_dev" : !exp_avg ? "exp_avg_dev" : !exp_avg_sq ? "exp_avg_sq_dev"
                    : !step ? "step_dev" : !scratch ? "scratch_dev" : n < 1 ? "n" : nullptr;
    if (bad) { hrp_set_error("hrp_clip_adam_step_ex: bad argument %s", bad); return -1; }
    if (!lr_dev)
        return clip_adam_launch<false, false>(params, grad, exp_avg, exp_avg_sq, step, n, lr, nullptr, beta1, beta2, eps,
                                              max_grad_norm, scratch, stream);
    return clip_adam_launch<true, false>(params, grad, exp_avg, exp_avg_sq, step, n, lr, lr_dev, beta1, beta2, eps,
                                         max_grad_norm, scratch, stream);
}

int hrp_ppo_loss_grad_kl(hrp_ppo *h, const float *params, const float *states, const float *pre_tanh,
                         const float *old_log_prob, const float *adv, const float *ret, const int64_t *idx,
                         int64_t batch, float eps_clip, float value_coef, float entropy_coef, float loss_scale,
                         const float *old_value, float value_clip, float *kl_out, const uint32_t *stop, float *grad,
                         float *metrics, void *stream)
{
    if ((kl_out == nullptr) != (stop == nullptr)) {
        hrp_set_error("hrp_ppo_loss_grad_kl: bad argument %s (kl_out_dev and stop_dev go together)",
                      kl_out ? "stop_dev" : "kl_out_dev");
        return -1;
    }
    if (old_value && !(std::isfinite(value_clip) && value_clip > 0.f)) {
        hrp_set_error("hrp_ppo_loss_grad_kl: value_clip must be finite and > 0 with old_value_dev, got %g", (double)value_clip);
        return -1;
    }
    return loss_grad_impl(h, params, states, pre_tanh, old_log_prob, adv, ret, idx, batch, eps_clip, value_coef,
                          entropy_coef, loss_scale, old_value, value_clip, grad, metrics, stream, kl_out, stop);
}

int hrp_clip_adam_step_kl(float *params, const float *grad, float *exp_avg, float *exp_avg_sq, int32_t *step, int64_t n,
                          double lr, const double *lr_dev, double beta1, double beta2, double eps, float max_grad_norm,
                          float *scratch, const float *kl, uint32_t *stop, double kl_limit, void *stream)
{
    const char *bad = !params ? "params_dev" : !grad ? "grad_dev" : !exp_avg ? "exp_avg_dev" : !exp_avg_sq ? "exp_avg_sq_dev"
                    : !step ? "step_dev" : !scratch ? "scratch_dev" : n < 1 ? "n"
                    : (kl == nullptr) != (stop == nullptr) ? (kl ? "stop_dev" : "kl_dev")
                    : kl && !(std::isfinite(kl_limit) && kl_limit > 0.0) ? "kl_limit" : nullptr;
    if (bad) { hrp_set_error("hrp_clip_adam_step_kl: bad argument %s", bad); return -1; }
    if (!kl)
        return lr_dev ? clip_adam_launch<true, false>(params, grad, exp_avg, exp_avg_sq, step, n, lr, lr_dev, beta1, beta2,
                                                      eps, max_grad_norm, scratch, stream)
                      : clip_adam_launch<false, false>(params, grad, exp_avg, exp_avg_sq, step, n, lr, nullptr, beta1,
                                                       beta2, eps, max_grad_norm, scratch, stream);
    return lr_dev ? clip_adam_launch<true, true>(params, grad, exp_avg, exp_avg_sq, step, n, lr, lr_dev, beta1, beta2, eps,
                                                 max_grad_norm, scratch, stream, kl, stop, kl_limit)
                  : clip_adam_launch<false, true>(params, grad, exp_avg, exp_avg_sq, step, n, lr, nullptr, beta1, beta2,
                                                  eps, max_grad_norm, scratch, stream, kl, stop, kl_limit);
}

}  // extern "C"
