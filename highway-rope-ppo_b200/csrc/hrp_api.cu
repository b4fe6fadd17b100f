// hrp_api.cu -- the extern "C" boundary of the simulator half (include/hrp.h).
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "hrp_internal.cuh"

static thread_local char g_err[512] = "";

bool hrp_pdl_enabled()
{
    static const bool on = !(getenv("HRP_PDL") && getenv("HRP_PDL")[0] == '0');
    return on;
}

void hrp_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

struct hrp_env {
    hrp_cfg cfg;
    EnvDev P;
    GridDev G;
    int device;
    void *arena;  // one allocation behind every state array
    size_t arena_bytes;
    float *table_dev;
    // pinned staging + device buffers of the host-buffer entry points
    float *h_actions, *h_obs, *h_reward;
    uint8_t *h_term, *h_trunc;
    float *d_actions, *d_obs, *d_reward;
    uint8_t *d_term, *d_trunc;
    cudaStream_t host_stream;
};

// ---- state injection / extraction (synchronous, host SoA <-> padded device SoA) ----
template <typename T>
static int pull(std::vector<T> &dst, const T *src_dev, size_t n)
{
    dst.resize(n);
    HRP_CUDA_OK(cudaMemcpy(dst.data(), src_dev, n * sizeof(T), cudaMemcpyDeviceToHost));
    return 0;
}
template <typename T>
static int push(T *dst_dev, const std::vector<T> &src)
{
    HRP_CUDA_OK(cudaMemcpy(dst_dev, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
}
// a vehicle field of the working type (float, or double for the fp64 validation instantiation) <-> host doubles
static int pull_real(std::vector<double> &dst, const void *src_dev, size_t n, bool real64)
{
    if (real64) return pull(dst, (const double *)src_dev, n);
    std::vector<float> t;
    if (pull(t, (const float *)src_dev, n)) return -2;
    dst.assign(t.begin(), t.end());
    return 0;
}
static int push_real(void *dst_dev, const std::vector<double> &src, bool real64)
{
    if (real64) return push((double *)dst_dev, src);
    std::vector<float> t(src.size());
    for (size_t i = 0; i < src.size(); ++i) t[i] = (float)src[i];
    return push((float *)dst_dev, t);
}

// Host-to-device copy of a page-locked buffer done by SMs instead of the copy engine: the kernel reads the mapped host
// memory (cache-volatile 16-byte loads, every one of them in flight at once) and stores to device memory.  Same PCIe
// time as cudaMemcpyAsync, but it is a KERNEL in the stream: the policy's first GEMM follows it with programmatic
// dependent launch after ~1 us, where a copy-engine transfer costs ~14 us before a dependent kernel starts
// (profiles/r02_timeline_pipeline_g1.txt).
__global__ void __launch_bounds__(256) fetch_host_kernel(const uint4 *__restrict__ src, uint4 *__restrict__ dst, size_t n16,
                                                         const unsigned char *__restrict__ src8, unsigned char *__restrict__ dst8,
                                                         size_t tail)
{
    hrp_pdl_release();
    hrp_pdl_wait();
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) dst[i] = __ldcv(src + i);
    if (blockIdx.x == 0 && threadIdx.x < tail) dst8[threadIdx.x] = *((const volatile unsigned char *)src8 + threadIdx.x);
}

extern "C" {

const char *hrp_last_error(void) { return g_err; }
int hrp_version(void) { return 3; }   // 2: OccupancyGrid fields of hrp_cfg, hrp_env_grid_shape; 3: ego_collisions_only
int hrp_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        hrp_set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
        cudaGetLastError();
        return -2;
    }
    return n;
}

int hrp_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    hrp_philox(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1], out);
    return 0;
}

// W (axis 0) or H (axis 1) of an OccupancyGrid config: floor((hi - lo) / step) in fp64, 0 when it is not a count >= 1
static int grid_extent(const hrp_cfg *c, int axis)
{
    const double n = floor((c->grid_hi[axis] - c->grid_lo[axis]) / c->grid_step[axis]);
    return (c->grid_step[axis] > 0.0 && n >= 1.0 && n <= HRP_MAX_GRID_VALUES) ? (int)n : 0;
}

static int validate_grid(const hrp_cfg *c)
{
    if (c->obs_nfeat < 1 || c->obs_nfeat > HRP_MAX_FEATURES) {
        hrp_set_error("feature count %d outside [1, %d]", c->obs_nfeat, HRP_MAX_FEATURES);
        return -1;
    }
    for (int f = 0; f < c->obs_nfeat; ++f)
        if (c->obs_feat[f] < HRP_F_PRESENCE || c->obs_feat[f] > HRP_F_ON_ROAD) {
            hrp_set_error("unsupported feature code %d", c->obs_feat[f]);
            return -1;
        }
    for (int a = 0; a < 2; ++a) {
        if (!(c->grid_step[a] > 0.0) || !isfinite(c->grid_step[a]) || !isfinite(c->grid_lo[a]) || !isfinite(c->grid_hi[a])) {
            hrp_set_error("grid_step[%d] = %g must be > 0 and grid_size[%d] = [%g, %g] finite", a, c->grid_step[a], a,
                          c->grid_lo[a], c->grid_hi[a]);
            return -1;
        }
        if (!grid_extent(c, a)) {
            hrp_set_error("grid_size[%d] = [%g, %g] with grid_step %g holds no cell", a, c->grid_lo[a], c->grid_hi[a],
                          c->grid_step[a]);
            return -1;
        }
    }
    const int W = grid_extent(c, 0), H = grid_extent(c, 1);
    if ((long long)c->obs_nfeat * W * H > HRP_MAX_GRID_VALUES) {
        hrp_set_error("grid features x W x H = %d x %d x %d exceeds %d", c->obs_nfeat, W, H, HRP_MAX_GRID_VALUES);
        return -1;
    }
    if (c->embed_kind != HRP_EMBED_NONE) {
        hrp_set_error("embed_kind %d: an OccupancyGrid observation takes no embedding", c->embed_kind);
        return -1;
    }
    if (c->policy_frequency < 1 || c->simulation_frequency < c->policy_frequency) {
        hrp_set_error("bad simulation/policy frequency %d/%d", c->simulation_frequency, c->policy_frequency);
        return -1;
    }
    if (c->ego_mode != 0 && c->ego_mode != 1) {
        hrp_set_error("ego_mode %d not in {0,1}", c->ego_mode);
        return -1;
    }
    return 0;
}

static int validate_cfg(const hrp_cfg *c, int64_t table_len)
{
    if (c->ego_collisions_only != 0 && c->ego_collisions_only != 1) {
        hrp_set_error("ego_collisions_only %d not in {0 (highway-v0), 1 (highway-fast-v0)}", c->ego_collisions_only);
        return -1;
    }
    if (c->vehicles_count < 0 || c->vehicles_count + 1 > HRP_MAX_VEHICLES) {
        hrp_set_error("vehicles_count %d outside [0, %d]", c->vehicles_count, HRP_MAX_VEHICLES - 1);
        return -1;
    }
    if (c->lanes_count < 1 || c->lanes_count > HRP_MAX_LANES) {
        hrp_set_error("lanes_count %d outside [1, %d]", c->lanes_count, HRP_MAX_LANES);
        return -1;
    }
    if (c->obs_type != HRP_OBS_KINEMATICS && c->obs_type != HRP_OBS_OCCUPANCY_GRID) {
        hrp_set_error("obs_type %d not in {0 (Kinematics), 1 (OccupancyGrid)}", c->obs_type);
        return -1;
    }
    if (c->obs_type == HRP_OBS_OCCUPANCY_GRID) return validate_grid(c);
    if (c->obs_vehicles < 1 || c->obs_vehicles > HRP_MAX_OBS_ROWS) {
        hrp_set_error("observation vehicles_count %d outside [1, %d]", c->obs_vehicles, HRP_MAX_OBS_ROWS);
        return -1;
    }
    if (c->obs_nfeat < 1 || c->obs_nfeat > HRP_MAX_FEATURES) {
        hrp_set_error("feature count %d outside [1, %d]", c->obs_nfeat, HRP_MAX_FEATURES);
        return -1;
    }
    for (int f = 0; f < c->obs_nfeat; ++f)
        if (c->obs_feat[f] < HRP_F_PRESENCE || c->obs_feat[f] > HRP_F_SIN_H) {
            hrp_set_error("unsupported feature code %d", c->obs_feat[f]);
            return -1;
        }
    if (c->policy_frequency < 1 || c->simulation_frequency < c->policy_frequency) {
        hrp_set_error("bad simulation/policy frequency %d/%d", c->simulation_frequency, c->policy_frequency);
        return -1;
    }
    if (c->ego_mode != 0 && c->ego_mode != 1) {
        hrp_set_error("ego_mode %d not in {0,1}", c->ego_mode);
        return -1;
    }
    int F = c->obs_nfeat, N = c->obs_vehicles, d = c->embed_dim;
    switch (c->embed_kind) {
    case HRP_EMBED_NONE: break;
    case HRP_EMBED_ROPE:
        if (d % 2 != 0 || d > F || d < 0) { hrp_set_error("rotate_dim must be even and <= %d; got %d", F, d); return -1; }
        if (F < 2) { hrp_set_error("RoPE needs at least 2 features"); return -1; }
        if (table_len != d / 2) { hrp_set_error("RoPE table must hold rotate_dim/2 = %d floats", d / 2); return -1; }
        break;
    case HRP_EMBED_DIST:
        if (d % 2 != 0 || d <= 0 || d > HRP_MAX_EMBED) { hrp_set_error("DistPE d_embed must be even and <= %d; got %d", HRP_MAX_EMBED, d); return -1; }
        if (F < (c->embed_use_euclidean ? 2 : 1)) { hrp_set_error("DistPE needs more features"); return -1; }
        if (table_len != d / 2) { hrp_set_error("DistPE table must hold d_embed/2 = %d floats", d / 2); return -1; }
        break;
    case HRP_EMBED_RANK:
        if (d <= 0 || d > HRP_MAX_EMBED) { hrp_set_error("RankPE d_embed outside [1, %d]", HRP_MAX_EMBED); return -1; }
        if (table_len != (int64_t)N * d) { hrp_set_error("RankPE table must hold N*d = %d floats", N * d); return -1; }
        break;
    default: hrp_set_error("unknown embed_kind %d", c->embed_kind); return -1;
    }
    if (c->embed_ego_idx < 0 || c->embed_ego_idx >= N) { hrp_set_error("ego_idx outside the observation"); return -1; }
    return 0;
}

int hrp_env_create(const hrp_cfg *cfg, const float *embed_table_host, int64_t embed_table_len,
                   int32_t num_envs, uint64_t env_id_base, int32_t device, hrp_env **out)
{
    return hrp_env_create_ex(cfg, embed_table_host, embed_table_len, num_envs, env_id_base, device, 0u, out);
}

int hrp_env_create_ex(const hrp_cfg *cfg, const float *embed_table_host, int64_t embed_table_len,
                      int32_t num_envs, uint64_t env_id_base, int32_t device, uint32_t flags, hrp_env **out)
{
    if (!cfg || !out || num_envs < 1) { hrp_set_error("hrp_env_create: bad arguments"); return -1; }
    if (flags & ~(uint32_t)HRP_ENV_REAL64) { hrp_set_error("hrp_env_create_ex: unknown flags 0x%x", flags); return -1; }
    if (cfg->embed_kind != HRP_EMBED_NONE && !embed_table_host) { hrp_set_error("embedding table missing"); return -1; }
    if (int rc = validate_cfg(cfg, cfg->embed_kind == HRP_EMBED_NONE ? 0 : embed_table_len)) return rc;
    int ndev = hrp_device_count();
    if (ndev <= 0) { hrp_set_error("no CUDA device: this library has no CPU path"); return -3; }
    if (device < 0 || device >= ndev) { hrp_set_error("device %d not in [0, %d)", device, ndev); return -1; }
    HRP_CUDA_OK(cudaSetDevice(device));

    hrp_env *h = new hrp_env();
    memset(h, 0, sizeof(*h));
    h->cfg = *cfg;
    h->device = device;
    EnvDev &P = h->P;
    P.E = num_envs; P.V = cfg->vehicles_count + 1; P.lanes = cfg->lanes_count;
    P.frames = cfg->simulation_frequency / cfg->policy_frequency;
    P.ego_mode = cfg->ego_mode; P.autoreset = cfg->autoreset;
    P.normalize_reward = cfg->normalize_reward; P.offroad_terminal = cfg->offroad_terminal;
    P.real64 = (flags & HRP_ENV_REAL64) ? 1 : 0;
    P.dt64 = 1.0 / cfg->simulation_frequency;
    // collide_pair's pre-check radius is sqrt(5^2 + 2^2) + v dt.  Above 40 m/s the speed only decays (the clip of
    // Vehicle.clip_actions), so |v| <= 40 + 10 dt (10 m/s^2: the largest acceleration, the ego's continuous action);
    // 1e-2 m covers the fp32 working copies of x.  8.8 m is the window of 15 Hz and above.  The bound holds for the
    // speeds a simulation reaches; a state injected with |speed| > 40 + 10 dt (hrp_env_set_state) can miss a pair.
    P.coll_window = fmax(8.8, sqrt(29.0) + (40.0 + 10.0 * P.dt64) * P.dt64 + 1e-2);
    P.dtime = 1.0 / cfg->policy_frequency; P.duration = cfg->duration;
    P.collision_reward = cfg->collision_reward; P.right_lane_reward = cfg->right_lane_reward;
    P.high_speed_reward = cfg->high_speed_reward;
    P.rs_lo = cfg->reward_speed_lo; P.rs_hi = cfg->reward_speed_hi;
    P.N = cfg->obs_vehicles; P.F = cfg->obs_nfeat;
    P.Fout = (cfg->embed_kind == HRP_EMBED_DIST || cfg->embed_kind == HRP_EMBED_RANK) ? P.F + cfg->embed_dim : P.F;
    for (int f = 0; f < HRP_MAX_FEATURES; ++f) {
        P.feat[f] = cfg->obs_feat[f]; P.has_range[f] = cfg->obs_has_range[f];
        P.lo[f] = cfg->obs_lo[f]; P.hi[f] = cfg->obs_hi[f];
    }
    P.normalize = cfg->obs_normalize; P.clip = cfg->obs_clip; P.absolute = cfg->obs_absolute;
    P.sorted = cfg->obs_sorted; P.see_behind = cfg->obs_see_behind;
    P.embed_kind = cfg->embed_kind; P.embed_dim = cfg->embed_dim; P.use_euclid = cfg->embed_use_euclidean;
    P.ego_idx = cfg->embed_ego_idx; P.max_dist = (float)cfg->embed_max_dist;
    P.ego_spacing = cfg->ego_spacing; P.inv_density = 1.0 / cfg->vehicles_density;
    P.gap_factor = exp(-5.0 / 40.0 * cfg->lanes_count);
    P.initial_lane = cfg->initial_lane_id;
    P.env_id_base = env_id_base; P.seed = 0;
    GridDev &G = h->G;
    G.obs_type = cfg->obs_type;
    G.gx = G.gy = -1;
    if (cfg->obs_type == HRP_OBS_OCCUPANCY_GRID) {
        // the observation is [F][W][H]: rows F and columns W*H for every N * F_out consumer
        G.gw = grid_extent(cfg, 0); G.gh = grid_extent(cfg, 1);
        G.galign = cfg->grid_align ? 1 : 0;
        for (int a = 0; a < 2; ++a) { G.glo[a] = cfg->grid_lo[a]; G.gstep[a] = cfg->grid_step[a]; }
        for (int f = cfg->obs_nfeat - 1; f >= 0; --f) {
            if (!cfg->obs_has_range[f]) continue;
            if (cfg->obs_feat[f] == HRP_F_X) G.gx = f;
            if (cfg->obs_feat[f] == HRP_F_Y) G.gy = f;
        }
        P.N = cfg->obs_nfeat; P.Fout = G.gw * G.gh;
        P.normalize = 1; P.absolute = 0; P.sorted = 1; P.see_behind = 0;
        P.embed_kind = HRP_EMBED_NONE; P.embed_dim = 0; P.ego_idx = 0;
    }

    size_t n = (size_t)num_envs * HRP_VS, ne = (size_t)num_envs;
    const size_t rsz = P.real64 ? sizeof(double) : sizeof(float);
    size_t bytes = n * (2 * sizeof(double) + 7 * rsz + sizeof(uint32_t)) +
                   ne * (sizeof(double) + 2 * sizeof(uint32_t));
    h->arena_bytes = bytes;
    cudaError_t ce = cudaMalloc(&h->arena, bytes);
    if (ce != cudaSuccess) { hrp_set_error("cudaMalloc(%zu): %s", bytes, cudaGetErrorString(ce)); delete h; return -2; }
    cudaMemset(h->arena, 0, bytes);
    char *p = (char *)h->arena;
    P.x = (double *)p; p += n * sizeof(double);
    P.timer = (double *)p; p += n * sizeof(double);
    P.time = (double *)p; p += ne * sizeof(double);
    P.y = p; p += n * rsz;
    P.heading = p; p += n * rsz;
    P.speed = p; p += n * rsz;
    P.tspeed = p; p += n * rsz;
    P.delta = p; p += n * rsz;
    P.impx = p; p += n * rsz;
    P.impy = p; p += n * rsz;
    P.flags = (uint32_t *)p; p += n * sizeof(uint32_t);
    P.episode = (uint32_t *)p; p += ne * sizeof(uint32_t);
    P.obs_draw = (uint32_t *)p; p += ne * sizeof(uint32_t);
    if (cfg->embed_kind != HRP_EMBED_NONE && embed_table_len > 0) {
        HRP_CUDA_OK(cudaMalloc(&h->table_dev, embed_table_len * sizeof(float)));
        HRP_CUDA_OK(cudaMemcpy(h->table_dev, embed_table_host, embed_table_len * sizeof(float),
                               cudaMemcpyHostToDevice));
    }
    P.table = h->table_dev;
    // spawn episode 0 with seed 0 so that a handle is always in a valid state
    if (int rc = hrp_launch_reset(P, G, nullptr, nullptr, 0)) { return rc; }
    HRP_CUDA_OK(cudaDeviceSynchronize());
    *out = h;
    return 0;
}

int hrp_env_destroy(hrp_env *h)
{
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaFree(h->arena);
    cudaFree(h->table_dev);
    if (h->h_actions) {
        cudaFreeHost(h->h_actions); cudaFreeHost(h->h_obs); cudaFreeHost(h->h_reward);
        cudaFreeHost(h->h_term); cudaFreeHost(h->h_trunc);
        cudaFree(h->d_actions); cudaFree(h->d_obs); cudaFree(h->d_reward);
        cudaFree(h->d_term); cudaFree(h->d_trunc);
        cudaStreamDestroy(h->host_stream);
    }
    delete h;
    return 0;
}

int hrp_env_obs_dim(const hrp_env *h, int32_t *rows, int32_t *cols)
{
    if (!h) { hrp_set_error("null handle"); return -1; }
    if (rows) *rows = h->P.N;
    if (cols) *cols = h->P.Fout;
    return 0;
}
int hrp_env_grid_shape(const hrp_env *h, int32_t *features, int32_t *width, int32_t *height)
{
    if (!h) { hrp_set_error("null handle"); return -1; }
    if (h->G.obs_type != HRP_OBS_OCCUPANCY_GRID) { hrp_set_error("hrp_env_grid_shape: not an OccupancyGrid handle"); return -1; }
    if (features) *features = h->P.F;
    if (width) *width = h->G.gw;
    if (height) *height = h->G.gh;
    return 0;
}
int hrp_env_num_vehicles(const hrp_env *h) { return h ? h->P.V : -1; }

int hrp_env_reset(hrp_env *h, uint64_t seed, const uint8_t *mask_dev, float *obs_dev, void *stream)
{
    if (!h) { hrp_set_error("null handle"); return -1; }
    h->P.seed = seed;
    return hrp_launch_reset(h->P, h->G, mask_dev, obs_dev, (cudaStream_t)stream);
}

int hrp_env_step(hrp_env *h, const float *actions_dev, float *obs_dev, float *reward_dev,
                 uint8_t *terminated_dev, uint8_t *truncated_dev, const int32_t *perm_dev,
                 int32_t *row_vehicle_dev, void *stream)
{
    if (!h || !actions_dev || !obs_dev || !reward_dev || !terminated_dev || !truncated_dev) {
        hrp_set_error("hrp_env_step: null argument");
        return -1;
    }
    if (perm_dev && h->G.obs_type == HRP_OBS_OCCUPANCY_GRID) {
        hrp_set_error("hrp_env_step: perm_dev must be NULL for an OccupancyGrid handle (a grid has no row order)");
        return -1;
    }
    return hrp_launch_step(h->P, h->G, h->cfg.ego_collisions_only != 0, actions_dev, obs_dev, reward_dev, terminated_dev,
                           truncated_dev, perm_dev, row_vehicle_dev, (cudaStream_t)stream);
}

int hrp_env_step_final(hrp_env *h, const float *actions_dev, float *obs_dev, float *reward_dev,
                       uint8_t *terminated_dev, uint8_t *truncated_dev, float *final_obs_dev, const int32_t *perm_dev,
                       int32_t *row_vehicle_dev, void *stream)
{
    if (final_obs_dev && final_obs_dev == obs_dev) {
        hrp_set_error("hrp_env_step_final: final_obs_dev must not be obs_dev (a respawned env writes both)");
        return -1;
    }
    if (!h || !actions_dev || !obs_dev || !reward_dev || !terminated_dev || !truncated_dev) {
        hrp_set_error("hrp_env_step_final: null argument");
        return -1;
    }
    if (perm_dev && h->G.obs_type == HRP_OBS_OCCUPANCY_GRID) {
        hrp_set_error("hrp_env_step_final: perm_dev must be NULL for an OccupancyGrid handle (a grid has no row order)");
        return -1;
    }
    return hrp_launch_step(h->P, h->G, h->cfg.ego_collisions_only != 0, actions_dev, obs_dev, reward_dev, terminated_dev,
                           truncated_dev, perm_dev, row_vehicle_dev, (cudaStream_t)stream, final_obs_dev);
}

int hrp_env_observe(hrp_env *h, float *obs_dev, const int32_t *perm_dev, int32_t *row_vehicle_dev,
                    void *stream)
{
    if (!h || !obs_dev) { hrp_set_error("hrp_env_observe: null argument"); return -1; }
    if (perm_dev && h->G.obs_type == HRP_OBS_OCCUPANCY_GRID) {
        hrp_set_error("hrp_env_observe: perm_dev must be NULL for an OccupancyGrid handle (a grid has no row order)");
        return -1;
    }
    return hrp_launch_observe(h->P, h->G, obs_dev, perm_dev, row_vehicle_dev, (cudaStream_t)stream);
}

static int ensure_host_path(hrp_env *h)
{
    if (h->h_actions) return 0;
    HRP_CUDA_OK(cudaSetDevice(h->device));
    size_t E = h->P.E, no = E * h->P.N * h->P.Fout;
    HRP_CUDA_OK(cudaMallocHost(&h->h_actions, E * 2 * sizeof(float)));
    HRP_CUDA_OK(cudaMallocHost(&h->h_obs, no * sizeof(float)));
    HRP_CUDA_OK(cudaMallocHost(&h->h_reward, E * sizeof(float)));
    HRP_CUDA_OK(cudaMallocHost(&h->h_term, E));
    HRP_CUDA_OK(cudaMallocHost(&h->h_trunc, E));
    HRP_CUDA_OK(cudaMalloc(&h->d_actions, E * 2 * sizeof(float)));
    HRP_CUDA_OK(cudaMalloc(&h->d_obs, no * sizeof(float)));
    HRP_CUDA_OK(cudaMalloc(&h->d_reward, E * sizeof(float)));
    HRP_CUDA_OK(cudaMalloc(&h->d_term, E));
    HRP_CUDA_OK(cudaMalloc(&h->d_trunc, E));
    HRP_CUDA_OK(cudaStreamCreateWithFlags(&h->host_stream, cudaStreamNonBlocking));
    return 0;
}

// page-locked caller memory (cudaMallocHost / cudaHostRegister / torch pin_memory) is copied to and from directly;
// pageable memory goes through the handle's own pinned staging buffers
static bool is_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// `actions` may be pageable host, page-locked host or device memory (a device action, e.g. the policy kernel's
// output on `s`, is used in place: no H2D copy and no synchronisation between the policy and the step)
static int step_host_impl(hrp_env *h, const float *actions, float *obs_host, float *reward_host,
                          uint8_t *terminated_host, uint8_t *truncated_host, cudaStream_t s, bool sync = true)
{
    if (!h || !actions || !obs_host || !reward_host || !terminated_host || !truncated_host) {
        hrp_set_error("hrp_env_step_host: null argument");
        return -1;
    }
    if (int rc = ensure_host_path(h)) return rc;
    size_t E = h->P.E, no = E * h->P.N * h->P.Fout;
    cudaPointerAttributes pa;
    bool dev_a = false, pin_a = false;
    if (cudaPointerGetAttributes(&pa, actions) == cudaSuccess) {
        dev_a = pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged;
        pin_a = pa.type == cudaMemoryTypeHost;
    } else {
        cudaGetLastError();
    }
    const bool pin_o = is_pinned(obs_host);
    const bool pin_r = is_pinned(reward_host) && is_pinned(terminated_host) && is_pinned(truncated_host);
    if (!sync && (!pin_o || !pin_r || !(dev_a || pin_a))) {
        hrp_set_error("hrp_env_step_host_async: every host buffer must be page-locked (the copies complete after the call returns)");
        return -1;
    }
    const float *d_act = actions;
    if (!dev_a) {
        if (!pin_a) memcpy(h->h_actions, actions, E * 2 * sizeof(float));
        HRP_CUDA_OK(cudaMemcpyAsync(h->d_actions, pin_a ? actions : h->h_actions, E * 2 * sizeof(float),
                                    cudaMemcpyHostToDevice, s));
        d_act = h->d_actions;
    }
    // Page-locked result buffers are mapped into the device's address space (unified addressing): the step kernel
    // writes observation, reward and flags STRAIGHT into them -- coalesced posted writes over PCIe that drain while the
    // kernel is still simulating other envs -- instead of into device buffers followed by device-to-host copies.
    // HRP_ZERO_COPY=0 keeps the copies.
    static const bool zero_copy = !(getenv("HRP_ZERO_COPY") && getenv("HRP_ZERO_COPY")[0] == '0');
    if (zero_copy && pin_o && pin_r) {
        float *o_dev = nullptr, *r_dev = nullptr;
        uint8_t *te_dev = nullptr, *tr_dev = nullptr;
        if (cudaHostGetDevicePointer((void **)&o_dev, obs_host, 0) == cudaSuccess &&
            cudaHostGetDevicePointer((void **)&r_dev, reward_host, 0) == cudaSuccess &&
            cudaHostGetDevicePointer((void **)&te_dev, terminated_host, 0) == cudaSuccess &&
            cudaHostGetDevicePointer((void **)&tr_dev, truncated_host, 0) == cudaSuccess) {
            if (int rc = hrp_launch_step(h->P, h->G, h->cfg.ego_collisions_only != 0, d_act, o_dev, r_dev, te_dev, tr_dev,
                                         nullptr, nullptr, s))
                return rc;
            if (!sync) return 0;
            HRP_CUDA_OK(cudaStreamSynchronize(s));
            return 0;
        }
        cudaGetLastError();   // not mapped: fall through to the copies
    }
    if (int rc = hrp_launch_step(h->P, h->G, h->cfg.ego_collisions_only != 0, d_act, h->d_obs, h->d_reward, h->d_term,
                                 h->d_trunc, nullptr, nullptr, s))
        return rc;
    HRP_CUDA_OK(cudaMemcpyAsync(pin_o ? obs_host : h->h_obs, h->d_obs, no * sizeof(float), cudaMemcpyDeviceToHost, s));
    HRP_CUDA_OK(cudaMemcpyAsync(pin_r ? reward_host : h->h_reward, h->d_reward, E * sizeof(float), cudaMemcpyDeviceToHost, s));
    HRP_CUDA_OK(cudaMemcpyAsync(pin_r ? terminated_host : h->h_term, h->d_term, E, cudaMemcpyDeviceToHost, s));
    HRP_CUDA_OK(cudaMemcpyAsync(pin_r ? truncated_host : h->h_trunc, h->d_trunc, E, cudaMemcpyDeviceToHost, s));
    if (!sync) return 0;   // the caller synchronises with the stream (an event after this call) before it reads the results
    HRP_CUDA_OK(cudaStreamSynchronize(s));
    if (!pin_o) memcpy(obs_host, h->h_obs, no * sizeof(float));
    if (!pin_r) {
        memcpy(reward_host, h->h_reward, E * sizeof(float));
        memcpy(terminated_host, h->h_term, E);
        memcpy(truncated_host, h->h_trunc, E);
    }
    return 0;
}

int hrp_env_step_host(hrp_env *h, const float *actions_host, float *obs_host, float *reward_host,
                      uint8_t *terminated_host, uint8_t *truncated_host)
{
    if (!h) { hrp_set_error("hrp_env_step_host: null argument"); return -1; }
    if (int rc = ensure_host_path(h)) return rc;
    return step_host_impl(h, actions_host, obs_host, reward_host, terminated_host, truncated_host, h->host_stream);
}

int hrp_env_step_host_on(hrp_env *h, const float *actions, float *obs_host, float *reward_host,
                         uint8_t *terminated_host, uint8_t *truncated_host, void *stream)
{
    return step_host_impl(h, actions, obs_host, reward_host, terminated_host, truncated_host, (cudaStream_t)stream);
}

int hrp_env_step_host_async(hrp_env *h, const float *actions, float *obs_host, float *reward_host,
                            uint8_t *terminated_host, uint8_t *truncated_host, void *stream)
{
    return step_host_impl(h, actions, obs_host, reward_host, terminated_host, truncated_host, (cudaStream_t)stream, false);
}

int hrp_env_reset_host(hrp_env *h, uint64_t seed, float *obs_host)
{
    if (!h || !obs_host) { hrp_set_error("hrp_env_reset_host: null argument"); return -1; }
    if (int rc = ensure_host_path(h)) return rc;
    size_t no = (size_t)h->P.E * h->P.N * h->P.Fout;
    h->P.seed = seed;
    const bool pin_o = is_pinned(obs_host);
    if (int rc = hrp_launch_reset(h->P, h->G, nullptr, h->d_obs, h->host_stream)) return rc;
    HRP_CUDA_OK(cudaMemcpyAsync(pin_o ? obs_host : h->h_obs, h->d_obs, no * sizeof(float), cudaMemcpyDeviceToHost,
                                h->host_stream));
    HRP_CUDA_OK(cudaStreamSynchronize(h->host_stream));
    if (!pin_o) memcpy(obs_host, h->h_obs, no * sizeof(float));
    return 0;
}

int hrp_env_set_seeds(hrp_env *h, const uint64_t *seeds_dev)
{
    if (!h) { hrp_set_error("hrp_env_set_seeds: null handle"); return -1; }
    h->P.seed_env = (const ull *)seeds_dev;
    return 0;
}

int hrp_env_set_step_mask(hrp_env *h, const uint8_t *mask_dev)
{
    if (!h) { hrp_set_error("hrp_env_set_step_mask: null handle"); return -1; }
    h->P.step_mask = mask_dev;
    return 0;
}

int hrp_env_set_trace(hrp_env *h, double *trace_dev)
{
    if (!h) { hrp_set_error("hrp_env_set_trace: null handle"); return -1; }
    h->P.trace = trace_dev;
    return 0;
}
int hrp_env_trace_shape(const hrp_env *h, int32_t *frames, int32_t *slots, int32_t *fields)
{
    if (!h) { hrp_set_error("hrp_env_trace_shape: null handle"); return -1; }
    if (frames) *frames = h->P.frames;
    if (slots) *slots = HRP_VS;
    if (fields) *fields = HRP_TRACE_FIELDS;
    return 0;
}

int hrp_env_get_state(hrp_env *h, hrp_state *d)
{
    if (!h || !d) { hrp_set_error("hrp_env_get_state: null argument"); return -1; }
    HRP_CUDA_OK(cudaSetDevice(h->device));
    HRP_CUDA_OK(cudaDeviceSynchronize());
    const EnvDev &P = h->P;
    size_t E = P.E, V = P.V, n = E * HRP_VS;
    std::vector<double> x, timer, time, y, hd, sp, ts, de, ix, iy;
    std::vector<uint32_t> fl, ep, dr;
    const bool r64 = P.real64 != 0;
    if (pull(x, P.x, n) || pull(timer, P.timer, n) || pull(time, P.time, E) || pull_real(y, P.y, n, r64) ||
        pull_real(hd, P.heading, n, r64) || pull_real(sp, P.speed, n, r64) || pull_real(ts, P.tspeed, n, r64) ||
        pull_real(de, P.delta, n, r64) || pull_real(ix, P.impx, n, r64) || pull_real(iy, P.impy, n, r64) ||
        pull(fl, P.flags, n) || pull(ep, P.episode, E) || pull(dr, P.obs_draw, E))
        return -2;
    for (size_t e = 0; e < E; ++e) {
        for (size_t k = 0; k < V; ++k) {
            size_t s = e * HRP_VS + k, o = e * V + k;
            if (d->x) d->x[o] = x[s];
            if (d->y) d->y[o] = y[s];
            if (d->heading) d->heading[o] = hd[s];
            if (d->speed) d->speed[o] = sp[s];
            if (d->target_speed) d->target_speed[o] = ts[s];
            if (d->delta) d->delta[o] = de[s];
            if (d->timer) d->timer[o] = timer[s];
            if (d->impact_x) d->impact_x[o] = ix[s];
            if (d->impact_y) d->impact_y[o] = iy[s];
            if (d->lane) d->lane[o] = fl[s] & 0xff;
            if (d->target_lane) d->target_lane[o] = (fl[s] >> 8) & 0xff;
            if (d->crashed) d->crashed[o] = (fl[s] >> 16) & 1;
            if (d->has_impact) d->has_impact[o] = (fl[s] >> 17) & 1;
        }
        if (d->time) d->time[e] = time[e];
        if (d->episode) d->episode[e] = ep[e];
        if (d->obs_draw) d->obs_draw[e] = dr[e];
    }
    return 0;
}

int hrp_env_set_state(hrp_env *h, const hrp_state *s)
{
    if (!h || !s) { hrp_set_error("hrp_env_set_state: null argument"); return -1; }
    if (!s->x || !s->y || !s->heading || !s->speed || !s->target_speed || !s->delta || !s->timer ||
        !s->impact_x || !s->impact_y || !s->lane || !s->target_lane || !s->crashed || !s->has_impact ||
        !s->time) {
        hrp_set_error("hrp_env_set_state: every vehicle field and time must be given");
        return -1;
    }
    HRP_CUDA_OK(cudaSetDevice(h->device));
    HRP_CUDA_OK(cudaDeviceSynchronize());
    const EnvDev &P = h->P;
    size_t E = P.E, V = P.V, n = E * HRP_VS;
    std::vector<double> x(n, 0.0), timer(n, 0.0), time(E, 0.0);
    std::vector<double> y(n, 0.0), hd(n, 0.0), sp(n, 0.0), ts(n, 0.0), de(n, 0.0), ix(n, 0.0), iy(n, 0.0);
    std::vector<uint32_t> fl(n, 0u);
    const bool r64 = P.real64 != 0;
    for (size_t e = 0; e < E; ++e) {
        for (size_t k = 0; k < V; ++k) {
            size_t d = e * HRP_VS + k, o = e * V + k;
            if (s->lane[o] < 0 || s->lane[o] >= P.lanes || s->target_lane[o] < 0 || s->target_lane[o] >= P.lanes) {
                hrp_set_error("set_state: lane index out of range at env %zu vehicle %zu", e, k);
                return -1;
            }
            x[d] = s->x[o]; timer[d] = s->timer[o];
            y[d] = s->y[o]; hd[d] = s->heading[o]; sp[d] = s->speed[o];
            ts[d] = s->target_speed[o]; de[d] = s->delta[o];
            ix[d] = s->impact_x[o]; iy[d] = s->impact_y[o];
            fl[d] = (uint32_t)s->lane[o] | ((uint32_t)s->target_lane[o] << 8) |
                    ((uint32_t)(s->crashed[o] != 0) << 16) | ((uint32_t)(s->has_impact[o] != 0) << 17);
        }
        time[e] = s->time[e];
    }
    if (push(P.x, x) || push(P.timer, timer) || push(P.time, time) || push_real(P.y, y, r64) ||
        push_real(P.heading, hd, r64) || push_real(P.speed, sp, r64) || push_real(P.tspeed, ts, r64) ||
        push_real(P.delta, de, r64) || push_real(P.impx, ix, r64) || push_real(P.impy, iy, r64) || push(P.flags, fl))
        return -2;
    if (s->episode) HRP_CUDA_OK(cudaMemcpy(P.episode, s->episode, E * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if (s->obs_draw) HRP_CUDA_OK(cudaMemcpy(P.obs_draw, s->obs_draw, E * sizeof(uint32_t), cudaMemcpyHostToDevice));
    return 0;
}

int hrp_embed_apply(int32_t kind, int32_t embed_dim, int32_t use_euclidean, int32_t ego_idx, float max_dist,
                    const float *table_dev, const float *obs_dev, float *out_dev, int64_t batch, int32_t rows,
                    int32_t cols, const float *dist_override_dev, void *stream)
{
    if (!obs_dev || !out_dev || batch < 0) { hrp_set_error("hrp_embed_apply: bad arguments"); return -1; }
    if (rows < 1 || rows > HRP_MAX_OBS_ROWS || cols < 1 || cols > HRP_MAX_EMBED_COLS) {
        hrp_set_error("hrp_embed_apply: observation shape (%d, %d) unsupported (max %d x %d)", rows, cols,
                      HRP_MAX_OBS_ROWS, HRP_MAX_EMBED_COLS);
        return -1;
    }
    if ((kind == HRP_EMBED_ROPE || (kind == HRP_EMBED_DIST && use_euclidean)) && cols < 2) {
        hrp_set_error("hrp_embed_apply: the distance needs the first two features");
        return -1;
    }
    if (kind != HRP_EMBED_NONE && !table_dev) { hrp_set_error("hrp_embed_apply: table missing"); return -1; }
    if (kind == HRP_EMBED_ROPE && (embed_dim % 2 != 0 || embed_dim > cols)) {
        hrp_set_error("rotate_dim must be even and <= %d; got %d", cols, embed_dim);
        return -1;
    }
    if (kind == HRP_EMBED_DIST && (embed_dim % 2 != 0 || embed_dim > HRP_MAX_EMBED)) {
        hrp_set_error("DistPE d_embed must be even and <= %d; got %d", HRP_MAX_EMBED, embed_dim);
        return -1;
    }
    if (ego_idx < 0 || ego_idx >= rows) { hrp_set_error("ego_idx outside the observation"); return -1; }
    if (batch == 0) return 0;
    return hrp_launch_embed(kind, embed_dim, use_euclidean, ego_idx, max_dist, table_dev, obs_dev, out_dev, batch,
                            rows, cols, dist_override_dev, (cudaStream_t)stream);
}

int hrp_fetch_host(void *dst_dev, const void *src_host, uint64_t bytes, void *stream)
{
    if (!dst_dev || !src_host) { hrp_set_error("hrp_fetch_host: null argument"); return -1; }
    if (bytes == 0) return 0;
    if (((uintptr_t)dst_dev | (uintptr_t)src_host) & 15) { hrp_set_error("hrp_fetch_host: both pointers must be 16-byte aligned"); return -1; }
    void *src_dev = nullptr;
    if (cudaHostGetDevicePointer(&src_dev, const_cast<void *>(src_host), 0) != cudaSuccess) {
        cudaGetLastError();
        hrp_set_error("hrp_fetch_host: src_host is not page-locked, mapped host memory");
        return -1;
    }
    const size_t n16 = bytes / 16, tail = bytes % 16;
    const unsigned grid = (unsigned)((n16 + 255) / 256 < 1 ? 1 : ((n16 + 255) / 256 > 1184 ? 1184 : (n16 + 255) / 256));
    HRP_CUDA_OK(hrp_launch_pdl(fetch_host_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, (const uint4 *)src_dev,
                               (uint4 *)dst_dev, n16, (const unsigned char *)src_dev + 16 * n16,
                               (unsigned char *)dst_dev + 16 * n16, tail));
    return 0;
}

}  // extern "C"
