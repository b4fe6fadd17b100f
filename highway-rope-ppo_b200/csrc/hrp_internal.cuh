// hrp_internal.cuh -- device-side parameter block and helpers shared by the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "hrp.h"

#define HRP_VS 64            // vehicle slots per env in every SoA array (two per lane)
#define HRP_WARPS_PER_CTA 4  // envs per CTA (one warp each)
#define HRP_STEP_CTAS_PER_SM 7  // 28 envs per SM: 4096 envs fill 148 SMs in one wave (<= 72 registers)
#define HRP_WARPS_PER_CTA_F64 2  // the fp64 validation instantiation: its per-warp shared-memory block is twice as large
#define HRP_FULL 0xffffffffu
#define HRP_MAX_DEVICES 64  // per-device caches of launch configuration

typedef unsigned long long ull;

// Everything a kernel needs, passed by value (lives in the constant bank).
struct EnvDev {
    int E, V, lanes, frames;
    int ego_mode, autoreset, normalize_reward, offroad_terminal;
    int real64;      // 0: product arithmetic (fp32 + fp64 x / timer); 1: fp64 validation instantiation (fp64 state arrays)
    double dt64;     // 1/simulation_frequency (IDM timer is advanced in fp64, SURVEY A.6)
    double coll_window;  // rank-order x gap beyond which no pair can pass collide_pair's pre-check (hrp_env_create_ex)
    double dtime;    // 1/policy_frequency
    double duration;
    double collision_reward, right_lane_reward, high_speed_reward, rs_lo, rs_hi;
    // Kinematics observation
    int N, F, Fout;
    int feat[HRP_MAX_FEATURES];
    int has_range[HRP_MAX_FEATURES];
    double lo[HRP_MAX_FEATURES], hi[HRP_MAX_FEATURES];
    int normalize, clip, absolute, sorted, see_behind;
    // embedding
    int embed_kind, embed_dim, use_euclid, ego_idx;
    float max_dist;
    const float *table;
    // spawn
    double ego_spacing, inv_density, gap_factor;
    int initial_lane;
    ull env_id_base, seed;
    // multiplexed independent experiments (hrp_env_set_seeds): when non-null, env e draws from (seed_env[e], global env
    // id 0), i.e. it is bit-for-bit the single-env handle an experiment with that seed would own
    const ull *seed_env;
    const uint8_t *step_mask;   // multiplexed experiments: when non-null, hrp_env_step leaves env e untouched unless step_mask[e]
    // SoA simulator state in HBM: [E][HRP_VS] per vehicle field, [E] per env field
    double *x, *timer, *time;
    void *y, *heading, *speed, *tspeed, *delta, *impx, *impy;   // float arrays, double arrays when real64
    uint32_t *flags;  // lane | target_lane<<8 | crashed<<16 | has_impact<<17
    uint32_t *episode, *obs_draw;
    // validation aid (hrp_env_set_trace): when non-null, [E][frames][HRP_VS][HRP_TRACE_FIELDS] doubles receive every
    // vehicle's state at the end of every simulation frame of a step (x, y, speed, heading, impact_x, impact_y, flags)
    double *trace;
};
#define HRP_TRACE_FIELDS 7

// Philox4x32-10 (Salmon et al. SC'11), the counter-based generator behind spawn and shuffle.
__host__ __device__ __forceinline__ void hrp_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                    uint32_t k0, uint32_t k1, uint32_t out[4])
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        unsigned long long p0 = (unsigned long long)0xD2511F53u * c0;
        unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// library-internal error plumbing (hrp_api.cu)
void hrp_set_error(const char *fmt, ...);
#define HRP_CUDA_OK(expr)                                                                   \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            hrp_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                          __LINE__);                                                        \
            return -2;                                                                      \
        }                                                                                   \
    } while (0)

// Programmatic dependent launch (PDL): a kernel launched through hrp_launch_pdl may be scheduled while its
// predecessor in the stream is still running -- its prologue (barrier init, TMEM allocation, index arithmetic) then
// overlaps the predecessor's tail.  Such a kernel MUST call hrp_pdl_wait() before it reads or writes anything the
// predecessor touches; hrp_pdl_release() at its top lets ITS successor be scheduled early in turn.  Both are no-ops
// in a kernel that was launched the ordinary way.  HRP_PDL=0 disables the attribute.
__device__ __forceinline__ void hrp_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void hrp_pdl_release() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
bool hrp_pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t hrp_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = hrp_pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// fused consumer of the tcgen05 GEMM's epilogue (hrp_mlp_tc.cu: tc_epilogue): per-row dot products of the output tile
// with the head weights.  out == nullptr: off.
struct TcDots {
    const float *wa;   // actor head weights [A][H]   (columns [0, H) of the output)
    const float *wc;   // critic head weights [H]     (columns [H, 2 H))
    int H, A;          // A: head rows, 1..8
    float *out;        // [N / BN tiles][M][A <= 4 ? 4 : 8] partial sums
    int skip_store;    // do not write the activation itself
};

// launchers implemented in hrp_env.cu
int hrp_launch_step(const EnvDev &P, const float *actions, float *obs, float *reward, uint8_t *term,
                    uint8_t *trunc, const int32_t *perm, int32_t *row_vehicle, cudaStream_t s);
int hrp_launch_observe(const EnvDev &P, float *obs, const int32_t *perm, int32_t *row_vehicle,
                       cudaStream_t s);
int hrp_launch_reset(const EnvDev &P, const uint8_t *mask, float *obs, cudaStream_t s);
int hrp_launch_embed(int kind, int embed_dim, int use_euclid, int ego_idx, float max_dist,
                     const float *table, const float *obs, float *out, long long batch, int rows,
                     int cols, const float *dist_override, cudaStream_t s);
