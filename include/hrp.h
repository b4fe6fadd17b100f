/*
 * hrp.h -- C ABI of the B200-native hot path of highway-rope-ppo.
 *
 * The reference (DhruvDh/highway-rope-ppo) is pure Python and has no FFI of its
 * own; the boundary it exposes for this path is two Python protocols:
 *   - the gymnasium env produced by experiments/wrappers.py:14-104 (make_env) and
 *     stepped at training/routine.py:18,24,127,134, with the observation wrappers
 *     experiments/rope_embed.py:64-74, dist_embed.py:76-96, rank_embed.py:45-51;
 *   - ppo/agent.py:157-327 (PPOAgent.select_action / memory / update).
 * Each entry point below names the reference interface it replaces.  The Python
 * host (highway-rope-ppo_b200/) binds this library with ctypes and mirrors the
 * reference classes on top; INTEGRATION.md shows the stub a maintainer would add.
 *
 * Conventions: plain pointers and sizes only.  "_dev" pointers are device memory
 * owned by the caller (e.g. torch allocations), contiguous; "_host" pointers are
 * host memory.  Every call returns 0 on success, <0 on error
 * (hrp_last_error() gives the thread-local message).  Work is enqueued on the
 * caller's stream (a cudaStream_t passed as void*), with no hidden
 * synchronisation unless the entry point says "synchronous".  A handle is bound to
 * one device and is not thread-safe.  There is no CPU fallback: without a CUDA
 * device every compute entry point fails.
 */
#ifndef HRP_H
#define HRP_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HRP_MAX_VEHICLES 64   /* vehicles per env incl. ego (one warp, two per lane) */
#define HRP_MAX_OBS_ROWS 64
#define HRP_MAX_FEATURES 8
#define HRP_MAX_LANES 8
#define HRP_MAX_EMBED 64
#define HRP_MAX_EMBED_COLS 1024 /* F of hrp_embed_apply on caller-provided observations */

#define HRP_MAX_GRID_VALUES (HRP_MAX_OBS_ROWS * HRP_MAX_FEATURES) /* F*W*H of an OccupancyGrid observation */

/* Kinematics feature codes (highway-env Vehicle.to_dict keys used by
 * config/base_config.py:9,11-19); HRP_F_ON_ROAD is the OccupancyGrid road layer and is valid in a grid only */
enum { HRP_F_PRESENCE = 0, HRP_F_X, HRP_F_Y, HRP_F_VX, HRP_F_VY, HRP_F_HEADING, HRP_F_COS_H, HRP_F_SIN_H, HRP_F_ON_ROAD };
/* observation types */
enum { HRP_OBS_KINEMATICS = 0, HRP_OBS_OCCUPANCY_GRID = 1 };
/* observation embedding fused behind the Kinematics observation */
enum { HRP_EMBED_NONE = 0, HRP_EMBED_ROPE = 1, HRP_EMBED_DIST = 2, HRP_EMBED_RANK = 3 };

/* highway-v0 / highway-fast-v0 config (config/base_config.py:5-39 over HighwayEnv.default_config) */
typedef struct hrp_cfg {
    int32_t lanes_count;
    int32_t vehicles_count;        /* other vehicles; V = vehicles_count + 1 */
    int32_t simulation_frequency;
    int32_t policy_frequency;
    int32_t initial_lane_id;       /* -1 == None */
    int32_t ego_mode;              /* 0 ContinuousAction (base_config.py:23-27), 1 DiscreteMetaAction */
    int32_t normalize_reward;
    int32_t offroad_terminal;
    double  duration;
    double  ego_spacing;
    double  vehicles_density;
    double  collision_reward;
    double  right_lane_reward;
    double  high_speed_reward;
    double  reward_speed_lo;
    double  reward_speed_hi;
    /* KinematicObservation */
    int32_t obs_vehicles;          /* N rows */
    int32_t obs_nfeat;             /* F */
    int32_t obs_feat[HRP_MAX_FEATURES];
    int32_t obs_has_range[HRP_MAX_FEATURES];
    double  obs_lo[HRP_MAX_FEATURES];
    double  obs_hi[HRP_MAX_FEATURES];
    int32_t obs_normalize;
    int32_t obs_clip;
    int32_t obs_absolute;
    int32_t obs_sorted;            /* 1 "sorted", 0 "shuffled" (wrappers.py:47-57) */
    int32_t obs_see_behind;
    /* embedding wrapper (rope_embed.py:14-42, dist_embed.py:10-66, rank_embed.py:10-37) */
    int32_t embed_kind;            /* HRP_EMBED_* */
    int32_t embed_dim;             /* rotate_dim (RoPE) or d_embed (Dist/Rank) */
    int32_t embed_use_euclidean;   /* DistanceEmbedWrapper(use_euclidean=) */
    double  embed_max_dist;        /* max_dist, utils/defaults.py:10-13 */
    /* vec-env behaviour */
    int32_t autoreset;             /* respawn inside the step that ended the episode */
    int32_t embed_ego_idx;         /* ego_idx of the embed wrappers (row the distance refers to) */
    /* OccupancyGridObservation (absolute=False, as_image=False).  obs_type 0 (all of this zero) is Kinematics.  A grid
     * uses obs_nfeat / obs_feat (HRP_F_ON_ROAD allowed), obs_has_range / obs_lo / obs_hi as features_range and obs_clip
     * as clip; obs_vehicles, obs_normalize, obs_absolute, obs_sorted and obs_see_behind are ignored, and embed_kind
     * must be HRP_EMBED_NONE.  W = floor((grid_hi[0] - grid_lo[0]) / grid_step[0]), H likewise (fp64), 1 <= W, H and
     * F*W*H <= HRP_MAX_GRID_VALUES.  The observation is float32 [F][W][H]; DESIGN.md §3.1 states its semantics. */
    int32_t obs_type;              /* HRP_OBS_* */
    int32_t grid_align;            /* align_to_vehicle_axes */
    double  grid_lo[2];            /* grid_size[0][0], grid_size[1][0] */
    double  grid_hi[2];            /* grid_size[0][1], grid_size[1][1] */
    double  grid_step[2];
    /* the env id's collision rule: 0 is highway-v0 (every pair of vehicles is tested), 1 is highway-fast-v0
     * (HighwayEnvFast: the uncontrolled vehicles do not check collisions, so only the ego's pairs (0, k) are tested;
     * DESIGN.md Appendix C).  Any other value is an error (-1). */
    int32_t ego_collisions_only;
} hrp_cfg;

/* Host-side SoA view of the simulator state, [num_envs * V] per vehicle field
 * (ego = index 0 of every env), [num_envs] per env field.  Used for state
 * injection (parity tests) and checkpointing. */
typedef struct hrp_state {
    double  *x, *y, *heading, *speed, *target_speed, *delta, *timer, *impact_x, *impact_y;
    int32_t *lane, *target_lane, *crashed, *has_impact;
    double  *time;      /* env.time */
    uint32_t *episode;  /* spawn counter of every env */
    uint32_t *obs_draw; /* shuffle counter of every env */
} hrp_state;

typedef struct hrp_env hrp_env;

const char *hrp_last_error(void);
int hrp_version(void);
/* number of CUDA devices visible; <0 on driver error */
int hrp_device_count(void);

/* ---- simulator: replaces gym.make("highway-v0", config=cfg) + wrapper construction
 *      (experiments/wrappers.py:80,100-104).  embed_table_host: RoPE inv_freq[rotate_dim/2]
 *      (rope_embed.py:37-39), DistPE freqs[d/2] (dist_embed.py:48-52) or tanh(rank table)[N*d]
 *      (rank_embed.py:21-22,48); copied.  env_id_base offsets the Philox counter so that
 *      a shard owns envs [env_id_base, env_id_base+num_envs). */
int hrp_env_create(const hrp_cfg *cfg, const float *embed_table_host, int64_t embed_table_len,
                   int32_t num_envs, uint64_t env_id_base, int32_t device, hrp_env **out);
/* the same with flags.  HRP_ENV_REAL64 selects the VALIDATION instantiation of the simulator kernels: fp64 state
 * arrays and IEEE fp64 arithmetic throughout (the product keeps x and the lane-change timer in fp64 and everything
 * else in fp32).  Same code path, same entry points, several times slower; the parity tests use it to compare the
 * kernel's logic bit-exactly with the fp64 oracle, and the fp32 kernel with the fp64 kernel. */
#define HRP_ENV_REAL64 1u
int hrp_env_create_ex(const hrp_cfg *cfg, const float *embed_table_host, int64_t embed_table_len,
                      int32_t num_envs, uint64_t env_id_base, int32_t device, uint32_t flags, hrp_env **out);
int hrp_env_destroy(hrp_env *env);
/* observation extent per env: rows = N and cols = F_out for Kinematics, rows = F and cols = W*H for a grid */
int hrp_env_obs_dim(const hrp_env *env, int32_t *rows, int32_t *cols);
/* F, W, H of an OccupancyGrid handle; -1 for a Kinematics handle */
int hrp_env_grid_shape(const hrp_env *env, int32_t *features, int32_t *width, int32_t *height);
int hrp_env_num_vehicles(const hrp_env *env);

/* env.reset(seed=...) (training/routine.py:18,127): counter-based spawn of every env whose
 * mask byte is non-zero (mask_dev NULL: all), then the observation into obs_dev[E,N,F_out]. */
int hrp_env_reset(hrp_env *env, uint64_t seed, const uint8_t *mask_dev, float *obs_dev, void *stream);

/* env.step(action) (training/routine.py:24,134): 15 fused sub-steps + observation + embedding.
 * actions_dev[E,2] float32 (ContinuousAction) or [E,2] with the meta-action id in column 0.
 * perm_dev (nullable) [E,N-1] int32 injects the row shuffle; row_vehicle_dev (nullable)
 * [E,N] int32 receives the vehicle index shown in each row (-1 padding).
 * OccupancyGrid handle: obs_dev is [E,F,W,H]; perm_dev must be NULL (-1 otherwise); row_vehicle_dev is [E,W*H] and
 * receives the vehicle whose values fill each cell, -1 for a cell no vehicle is in. */
int hrp_env_step(hrp_env *env, const float *actions_dev, float *obs_dev, float *reward_dev,
                 uint8_t *terminated_dev, uint8_t *truncated_dev, const int32_t *perm_dev,
                 int32_t *row_vehicle_dev, void *stream);

/* hrp_env_step that also returns the observation each finished episode ended in -- what a vectorised env with autoreset
 * hands back as the final observation, so that a time-limit truncation can be bootstrapped with V(s_final).
 * final_obs_dev (nullable) [E,N,F_out]: an env whose episode ended on this step (terminated or truncated) writes the
 * observation of its terminal state there, BEFORE the respawn overwrites that state, with the normalisation, clipping,
 * row order and embedding of obs_dev.  It uses the step's own shuffle draw and advances no counter: it is bit for bit
 * the observation an autoreset = 0 handle returns from the same state and actions, and the new episode's first
 * observation in obs_dev is unchanged.  In shuffled mode both observations therefore share one row permutation; an
 * injected perm_dev applies to both.  row_vehicle_dev describes obs_dev only.  Rows of envs that did not finish, and of
 * envs the step mask skips, are not written.  With autoreset = 0, final_obs[e] == obs[e] for every finished env.
 * final_obs_dev NULL launches exactly what hrp_env_step launches; final_obs_dev == obs_dev is an error.  The default
 * kernels carry none of this code: it is a separate instantiation of the step kernel (fp32 and HRP_ENV_REAL64). */
int hrp_env_step_final(hrp_env *env, const float *actions_dev, float *obs_dev, float *reward_dev,
                       uint8_t *terminated_dev, uint8_t *truncated_dev, float *final_obs_dev,
                       const int32_t *perm_dev, int32_t *row_vehicle_dev, void *stream);

/* observation_type.observe() + wrapper.observation() of the current state */
int hrp_env_observe(hrp_env *env, float *obs_dev, const int32_t *perm_dev, int32_t *row_vehicle_dev,
                    void *stream);

/* the same step for callers with HOST buffers (what the reference's CPU loop would bind):
 * pinned staging, H2D actions, kernel, D2H results; synchronous. */
int hrp_env_step_host(hrp_env *env, const float *actions_host, float *obs_host, float *reward_host,
                      uint8_t *terminated_host, uint8_t *truncated_host);
int hrp_env_reset_host(hrp_env *env, uint64_t seed, float *obs_host);
/* the same on the caller's stream (synchronised before returning); `actions` may also be DEVICE memory produced
 * earlier on that stream -- the policy's output goes into the step without a host round trip while the host still
 * receives every result.  Page-locked host buffers are copied to and from directly, pageable ones are staged. */
int hrp_env_step_host_on(hrp_env *env, const float *actions, float *obs_host, float *reward_host,
                         uint8_t *terminated_host, uint8_t *truncated_host, void *stream);

/* Host-to-device copy of a page-locked (mapped) host buffer by a kernel instead of the copy engine -- the first link of
 * the host-buffer policy step (the observation the reference loop holds on the host, training/routine.py:133-135): a
 * dependent kernel (the policy's first GEMM) starts ~1 us after it, not ~14 us as after a cudaMemcpyAsync.  Both
 * pointers 16-byte aligned. */
int hrp_fetch_host(void *dst_dev, const void *src_host, uint64_t bytes, void *stream);

/* Multiplexed independent experiments (the replacement of utils/device_pool.py:45-72 + main.py:234-242: many single-env
 * runs of the sweep share ONE handle instead of time-sharing the GPU as processes).  While seeds_dev[E] (device, owned by
 * the caller, read at every reset / shuffle draw) is non-NULL, env e draws its spawn and shuffle randoms from
 * (seeds_dev[e], global env id 0) instead of (seed, env_id_base + e): it is bit for bit the single-env handle that an
 * experiment calling env.reset(seed=seeds[e]) would own.  The training loop rewrites seeds_dev[e] = exp_seed + episode
 * before it resets env e through hrp_env_reset's mask (training/routine.py:132-133).  NULL switches it off. */
int hrp_env_set_seeds(hrp_env *env, const uint64_t *seeds_dev);
/* while mask_dev[E] (device, owned by the caller, read by every hrp_env_step) is non-NULL, a step leaves env e
 * untouched -- state, counters, outputs -- unless mask_dev[e] != 0: multiplexed experiments are not in lock step (one
 * is evaluating, one is in its PPO update, one has finished).  NULL: every env steps. */
int hrp_env_set_step_mask(hrp_env *env, const uint8_t *mask_dev);

/* validation aid: while trace_dev is non-NULL every hrp_env_step also writes the state of every vehicle at the end
 * of every simulation frame -- trace_dev[E][frames][slots][fields] doubles (x, y, speed, heading, impact_x, impact_y,
 * flags = lane | target_lane<<8 | crashed<<16 | has_impact<<17); hrp_env_trace_shape gives the three inner extents.
 * The parity tests use it to compare a step with the oracle frame by frame.  NULL switches it off. */
int hrp_env_set_trace(hrp_env *env, double *trace_dev);
int hrp_env_trace_shape(const hrp_env *env, int32_t *frames, int32_t *slots, int32_t *fields);

/* the same WITHOUT the final synchronisation: kernel and device-to-host copies are enqueued on `stream` and the call
 * returns; the results are in the host buffers once the stream has reached this point (record an event after the
 * call and wait for it).  Every host buffer must be page-locked.  With two env handles on two streams one group's
 * PCIe copies run under the other group's kernels (bench.py e2e). */
int hrp_env_step_host_async(hrp_env *env, const float *actions, float *obs_host, float *reward_host,
                            uint8_t *terminated_host, uint8_t *truncated_host, void *stream);

/* state injection / extraction; synchronous */
int hrp_env_get_state(hrp_env *env, hrp_state *dst_host);
int hrp_env_set_state(hrp_env *env, const hrp_state *src_host);

/* the generator behind spawn and shuffle (known-answer test) */
int hrp_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

/* ---- wrappers on caller-provided observations: RotaryEmbedWrapper.observation
 *      (rope_embed.py:64-74), DistanceEmbedWrapper.observation (dist_embed.py:76-96),
 *      RankEmbedWrapper.observation (rank_embed.py:45-51).  obs_dev[B,N,F] -> out_dev[B,N,F_out].
 *      dist_override_dev (nullable) [B,N] replaces the computed normalised distance, which is
 *      RotaryEmbedWrapper._apply_rope(obs, dist_norm) (rope_embed.py:44-62). */
int hrp_embed_apply(int32_t kind, int32_t embed_dim, int32_t use_euclidean, int32_t ego_idx,
                    float max_dist, const float *table_dev, const float *obs_dev, float *out_dev,
                    int64_t batch, int32_t rows, int32_t cols, const float *dist_override_dev,
                    void *stream);

/* ---- PPO (ppo/agent.py).  Parameters live in ONE flat fp32 buffer, laid out in
 *      ActorCritic.parameters() order (agent.py:12-44; the root module's own Parameter comes
 *      first): log_std, shared.0.{weight,bias}, shared.2.{weight,bias}, actor_mean.0.*,
 *      actor_mean.2.*, critic.0.*, critic.2.*; nn.Linear weights row-major [out,in].
 *      hrp_ppo_param_count gives P. */
int64_t hrp_ppo_param_count(int32_t state_dim, int32_t action_dim, int32_t hidden_dim);
/* Categorical policy (flag HRP_PPO_CATEGORICAL): a softmax over action_dim = n discrete actions, 2 <= n <= 8 (n = 5 for
 * the DiscreteMetaAction ego, hrp_cfg.ego_mode = 1), on the same trunk and critic with the same loss formula: log-prob
 * log_softmax(logits)[a], state-dependent entropy -sum p log p, clipped surrogate, value MSE, entropy bonus.  Its flat
 * buffer is the layout above WITHOUT log_std: shared.0.*, shared.2.*, actor_mean.0.*, actor_mean.2.{weight[n,H],
 * bias[n]} (the logits), critic.0.*, critic.2.*.  hrp_ppo_param_count_ex(S, n, H, flags) gives its P; flags 0 is
 * hrp_ppo_param_count. */
#define HRP_PPO_CATEGORICAL 1u
int64_t hrp_ppo_param_count_ex(int32_t state_dim, int32_t action_dim, int32_t hidden_dim, uint32_t flags);
/* arithmetic of the hidden-layer GEMMs (process-wide): 3 = tcgen05 tensor cores, 3xTF32 split (fp32-grade
 * accuracy; default), 1 = tcgen05 single-pass TF32, 0 = fp32 CUDA-core GEMM.  torch's nn.Linear in the
 * reference is fp32 (ppo/agent.py:22-42). */
int hrp_ppo_set_math(int32_t mode);
int hrp_ppo_get_math(void);
/* the dense contraction behind every nn.Linear of the path, on the tcgen05 tensor cores:
 * C[M,N] = act(sum_k A[m*sam + k*sak] * B[n*sbn + k*sbk] + bias[n]); mode 1 = TF32, 3 = 3xTF32. */
int hrp_gemm_strided(int32_t M, int32_t N, int32_t K, const float *A_dev, int64_t sam, int64_t sak,
                     const float *B_dev, int64_t sbn, int64_t sbk, float *C_dev, int32_t ldc,
                     const float *bias_dev, int32_t relu, int32_t mode, void *stream);

typedef struct hrp_ppo hrp_ppo;
/* workspace for batches up to max_batch rows */
int hrp_ppo_create(int32_t state_dim, int32_t action_dim, int32_t hidden_dim, int64_t max_batch,
                   int32_t device, hrp_ppo **out);
/* the same with flags: HRP_PPO_CATEGORICAL makes a categorical handle (action_dim = n in [2, 8]); flags 0 is exactly
 * hrp_ppo_create.  The arguments are validated before any device query (-1, with a message naming the field).
 * A categorical handle goes through the entry points below unchanged:
 *   hrp_ppo_forward          mean_dev[B, n] receives the logits;
 *   hrp_ppo_act, _act_sample, _act_sample_ctr
 *                            action_dev[B, 2] = (id, 0.0f) -- what hrp_env_step reads for ego_mode = 1 --,
 *                            pre_tanh_dev[B] = id as float (the sample the loss conditions on), log_prob, value.
 *                            Deterministic: the argmax, first maximum on ties, log-prob 0.  noise_dev (nullable) holds
 *                            ONE uniform in (0, 1) per row.  Sampling draws one uniform per row from Philox4x32-10 with
 *                            the Gaussian path's counter (row_base + row, draw) and key, u = ((r0 >> 8) + 0.5) / 2^24,
 *                            and takes the first id j with u < sum_{i <= j} p_i (summed in index order in fp32), n - 1
 *                            if there is none;
 *   hrp_ppo_loss_grad        reads the ids from pre_tanh_dev[B]; same metrics layout, with the state-dependent
 *                            entropy; there is no log_std gradient.
 * hrp_ppo_act_multi is Gaussian-only. */
int hrp_ppo_create_ex(int32_t state_dim, int32_t action_dim, int32_t hidden_dim, int64_t max_batch,
                      int32_t device, uint32_t flags, hrp_ppo **out);
int hrp_ppo_destroy(hrp_ppo *h);

/* ActorCritic.forward (agent.py:46-54): states[B,S] -> mean[B,A], value[B] */
int hrp_ppo_forward(hrp_ppo *h, const float *params_dev, const float *states_dev, int64_t batch,
                    float *mean_dev, float *value_dev, void *stream);
/* ActorCritic.get_action (agent.py:56-74) for a batch: noise_dev[B,A] standard normals
 * (nullable => deterministic).  Outputs action=tanh(z), pre_tanh=z, log_prob[B], value[B]. */
int hrp_ppo_act(hrp_ppo *h, const float *params_dev, const float *states_dev, const float *noise_dev,
                int64_t batch, float *action_dev, float *pre_tanh_dev, float *log_prob_dev,
                float *value_dev, void *stream);
/* the same with the standard normals drawn inside the kernel: Philox4x32-10 keyed by seed, counter =
 * (row_base + row, draw), Box-Muller.  row_base is the global index of this batch's first row (the shard's first
 * global env id): a rollout sharded over ranks draws exactly the noise one process over all envs would draw.  The
 * reference samples with torch's generator (Normal.sample, agent.py:64); the stream differs, the distribution does
 * not. */
int hrp_ppo_act_sample(hrp_ppo *h, const float *params_dev, const float *states_dev, uint64_t seed, uint64_t draw,
                       uint64_t row_base, int64_t batch, float *action_dev, float *pre_tanh_dev,
                       float *log_prob_dev, float *value_dev, void *stream);
/* hrp_ppo_act_sample with the draw counter resident on the device, for CUDA-graph capture (a captured launch cannot take
 * a new scalar per replay): draw_ctr_dev[2] = {counter, 0}; a launch draws with counter + 1 -- the value a host loop that
 * pre-increments `draw` (PPOAgent.act) would pass -- and leaves counter + 1 behind.  Everything else as above. */
int hrp_ppo_act_sample_ctr(hrp_ppo *h, const float *params_dev, const float *states_dev, uint64_t seed,
                           uint64_t *draw_ctr_dev, uint64_t row_base, int64_t batch, float *action_dev,
                           float *pre_tanh_dev, float *log_prob_dev, float *value_dev, void *stream);
/* ActorCritic.get_action (agent.py:56-74) for ONE state each of `count` independent policies in one launch: the rollout
 * forward of the sweep's single-env experiments (main.py:50-58, E = 1), which utils/device_pool.py:45-72 time-shares
 * as processes and experiments/multiplex.py batches.  Matrix-vector products in fp32 FMA arithmetic (a cluster of CTAs per
 * policy, weights streamed once); the policies may differ in every dimension.  out_dev[2 * action_dim + 2] receives
 * action = tanh(z), pre_tanh = z, log_prob (0 when deterministic), value.  Sampling: Philox4x32-10 keyed by seed,
 * counter (row, draw), as hrp_ppo_act_sample with row_base + row = `row`.  items is a HOST array. */
typedef struct hrp_act_item {
    const float *params_dev;   /* flat parameter buffer of this policy, ActorCritic.parameters() order */
    const float *state_dev;    /* [state_dim] */
    float *out_dev;            /* [2 * action_dim + 2] */
    uint64_t seed, draw, row;
    int32_t state_dim, action_dim, hidden_dim, deterministic;
} hrp_act_item;
int hrp_ppo_act_multi(const hrp_act_item *items, int32_t count, void *stream);
/* PPOMemory.compute_advantages (agent.py:126-138) over [T,E] (time-major), reverse scan.
 * last_value_dev[E]; done as uint8.  Outputs advantages[T,E] (float32), returns[T,E]. */
int hrp_gae(const float *reward_dev, const float *value_dev, const uint8_t *done_dev,
            const float *last_value_dev, int64_t T, int64_t E, double gamma, double lam,
            float *adv_dev, float *ret_dev, void *stream);
/* GAE with time-limit bootstrapping (the standard treatment of truncation; the reference treats it as termination,
 * which hrp_gae keeps).  terminated_dev / truncated_dev [T,E] uint8 as the step wrote them, final_value_dev (nullable)
 * [T,E] = V(final observation) of the step.  Per (t, e), fp64 arithmetic, float32 store of every A_t:
 *   term = terminated; trunc = truncated && !terminated (a crash on the last step is not bootstrapped); done = term|trunc
 *   boot = trunc ? final_value : (done ? 0 : V_{t+1});  delta = r + gamma boot - V_t;  A = delta + gamma lam (1-done) A_{t+1}
 * boot is a select: final_value rows of steps that were not truncated are never read into the arithmetic and may hold
 * anything, NaN included.  final_value_dev NULL, or no truncated step: bit-identical to hrp_gae with
 * done = terminated | truncated.  Bad arguments return -1 with a message naming the field, before any launch. */
int hrp_gae_ex(const float *reward_dev, const float *value_dev, const uint8_t *terminated_dev,
               const uint8_t *truncated_dev, const float *final_value_dev, const float *last_value_dev, int64_t T,
               int64_t E, double gamma, double lam, float *adv_dev, float *ret_dev, void *stream);
/* advantage normalisation (agent.py:204): (a-mean)/(std_unbiased+1e-8), in place.
 * hrp_adv_stats writes (sum, sum of squares, n) of the local shard to stats_dev[0..2] (fp64;
 * stats_dev must hold 3 + 512 doubles, the tail is scratch); a sharded run all-reduces those
 * three numbers before hrp_adv_normalize consumes them. */
int hrp_adv_stats(const float *adv_dev, int64_t n, double *stats_dev, void *stream);
int hrp_adv_normalize(float *adv_dev, int64_t n, const double *stats_dev, void *stream);
/* episode returns and lengths (the reference's ep_reward / evaluate bookkeeping, training/routine.py:14-29,143) over the
 * time-major [T,E] reward / terminated / truncated buffers the step wrote, forward scan, one thread per env.
 * return_dev[E] (fp64) and length_dev[E] (int32) carry each env's running episode across calls, so an episode may span
 * two rollouts; the caller zeroes them when it resets the envs.  For each step t, in order, of an env that takes part:
 * ret += (double)reward[t,e] (a sequential fp64 sum, bit-exact against Python's ep_reward += reward) and len += 1; if
 * terminated | truncated, the episode is counted.  A step both terminated and truncated counts as terminated (the rule
 * of hrp_gae_ex).
 *   active_dev NULL (training): after an episode is counted ret and len restart at 0 (the env has autoreset).
 *   active_dev[E] uint8 (evaluation): only envs with active[e] != 0 take part; when an env's first episode ends,
 *     active[e] = 0 and ret / len keep that episode.  The same buffer serves as the handle's step mask
 *     (hrp_env_set_step_mask), so a finished env stops stepping and its return stays on the device.
 * stats_dev is accumulated into (+=), fp64: [0] episodes finished, [1] sum of returns, [2] sum of squared returns,
 * [3] sum of lengths, [4] episodes that ended by termination, [5] episodes that ended by truncation only.  It must hold
 * 6 + 6 * 512 doubles: the tail is scratch for per-CTA partials, which are added in a fixed order, so equal inputs give
 * the same bits on every run; a sharded run all-reduces the six sums.  Bad arguments (a null pointer other than
 * active_dev, T < 1, E < 1) return -1 with a message naming the field, before any launch. */
#define HRP_EPISODE_STATS_LEN (6 + 6 * 512)
int hrp_episode_stats(const float *reward_dev, const uint8_t *terminated_dev, const uint8_t *truncated_dev, int64_t T,
                      int64_t E, uint8_t *active_dev, double *return_dev, int32_t *length_dev, double *stats_dev,
                      void *stream);
/* one minibatch of PPOAgent.update (agent.py:218-245 + backward): evaluate, clipped surrogate,
 * value MSE, entropy; writes d(loss)/d(params) into grad_dev[P] (overwritten) and
 * metrics_dev[8] += (loss, policy_loss, value_loss, entropy, clip_fraction, approx_kl, 1, 0).
 * idx_dev (nullable) [B] int64 gathers the minibatch rows out of the rollout tensors.
 * loss_scale multiplies every per-sample term (1/B_global for sharded minibatches). */
int hrp_ppo_loss_grad(hrp_ppo *h, const float *params_dev, const float *states_dev,
                      const float *pre_tanh_dev, const float *old_log_prob_dev, const float *adv_dev,
                      const float *ret_dev, const int64_t *idx_dev, int64_t batch, float eps_clip,
                      float value_coef, float entropy_coef, float loss_scale, float *grad_dev,
                      float *metrics_dev, void *stream);
/* hrp_ppo_loss_grad with the clipped value loss (PPO's clip_range_vf).  old_value_dev NULL: exactly hrp_ppo_loss_grad
 * (value_clip is not read).  old_value_dev non-NULL: [rollout rows] float32, the value the rollout stored for each sample,
 * gathered through idx_dev like the other per-sample inputs (read as [B] when idx_dev is NULL); value_clip = c must be
 * finite and > 0.  With v the new value, vo the old one and R the return, the value term of every sample becomes
 *   max((v - R)^2, (vo + clamp(v - vo, -c, c) - R)^2)
 * weighted as before (value_coef * the minibatch mean), and metrics_dev[2] accumulates it.  Its gradient follows torch
 * autograd on that expression: maximum splits it half and half on a tie, clamp passes it where -c <= v - vo <= c.
 * Gaussian and categorical handles; capturable and launched with programmatic dependent launch like hrp_ppo_loss_grad.
 * Bad arguments return -1 with a message naming the field, before any launch. */
int hrp_ppo_loss_grad_ex(hrp_ppo *h, const float *params_dev, const float *states_dev,
                         const float *pre_tanh_dev, const float *old_log_prob_dev, const float *adv_dev,
                         const float *ret_dev, const int64_t *idx_dev, int64_t batch, float eps_clip,
                         float value_coef, float entropy_coef, float loss_scale, const float *old_value_dev,
                         float value_clip, float *grad_dev, float *metrics_dev, void *stream);
/* clip_grad_norm_ + Adam.step (agent.py:247-252) fused over the flat buffers: ONE cooperative launch (per-CTA
 * sums of squares, grid synchronisation, clip coefficient, Adam).  step_dev[1] int32 is incremented on device
 * (bias correction).  The launch is capturable in a CUDA graph. */
int hrp_clip_adam_step(float *params_dev, const float *grad_dev, float *exp_avg_dev,
                       float *exp_avg_sq_dev, int32_t *step_dev, int64_t n, double lr, double beta1,
                       double beta2, double eps, float max_grad_norm, float *scratch_dev /* >=128 floats */,
                       void *stream);
/* hrp_clip_adam_step with the learning rate in device memory, so that a captured step follows a schedule.  lr_dev NULL:
 * exactly what hrp_clip_adam_step launches.  lr_dev non-NULL: one double, read by the kernel when it runs, in place of lr
 * (which is then not read) and in the same arithmetic, so *lr_dev == lr gives the same bits.  The caller writes it in
 * stream order before the launch, or before the replay of a graph that holds the launch.  Bad arguments return -1 with
 * a message naming the field, before any launch. */
int hrp_clip_adam_step_ex(float *params_dev, const float *grad_dev, float *exp_avg_dev, float *exp_avg_sq_dev,
                          int32_t *step_dev, int64_t n, double lr, const double *lr_dev, double beta1, double beta2,
                          double eps, float max_grad_norm, float *scratch_dev /* >=128 floats */, void *stream);

/* ---- target_kl early stopping (SB3's PPO(target_kl=...)) -------------------------------------------------------------
 * A minibatch's approx-KL mean((ratio - 1) - log ratio) is reduced by the loss kernel; when it exceeds 1.5 target_kl the
 * optimizer step is not taken and no later step of the update is either.  The decision is taken on the device through a
 * 32-bit stop word (0 = running), which the caller clears before the update.
 *
 * hrp_ppo_loss_grad_kl: hrp_ppo_loss_grad_ex, plus, with kl_out_dev / stop_dev non-NULL (both or neither): the last CTA
 * writes this shard's approx-KL share (the value it adds to metrics_dev[5]) to *kl_out_dev, and metrics_dev is added to
 * only while *stop_dev == 0.  The gradient is unchanged.  The caller places kl_out_dev at grad_dev + P, so that a
 * gradient exchange over P + 1 floats also sums the KL in rank order.  Both NULL: exactly hrp_ppo_loss_grad_ex.
 * hrp_clip_adam_step_kl: hrp_clip_adam_step_ex over the n = P parameters, plus, with kl_dev / stop_dev non-NULL (both or
 * neither): a no-op when *stop_dev != 0; otherwise when (double)*kl_dev > kl_limit (finite, > 0) it sets *stop_dev = 1
 * and takes no step (no parameter, moment or step_dev change).  Both NULL: exactly hrp_clip_adam_step_ex.
 * Bad arguments return -1 with a message naming the field, before any launch. */
int hrp_ppo_loss_grad_kl(hrp_ppo *h, const float *params_dev, const float *states_dev,
                         const float *pre_tanh_dev, const float *old_log_prob_dev, const float *adv_dev,
                         const float *ret_dev, const int64_t *idx_dev, int64_t batch, float eps_clip,
                         float value_coef, float entropy_coef, float loss_scale, const float *old_value_dev,
                         float value_clip, float *kl_out_dev, const uint32_t *stop_dev, float *grad_dev,
                         float *metrics_dev, void *stream);
int hrp_clip_adam_step_kl(float *params_dev, const float *grad_dev, float *exp_avg_dev, float *exp_avg_sq_dev,
                          int32_t *step_dev, int64_t n, double lr, const double *lr_dev, double beta1, double beta2,
                          double eps, float max_grad_norm, float *scratch_dev /* >=128 floats */, const float *kl_dev,
                          uint32_t *stop_dev, double kl_limit, void *stream);

/* ---- a captured graph behind a device-side gate (csrc/hrp_graph.cu) ---------------------------------------------------
 * hrp_graph_if_create builds [gate kernel] -> IF { child graph body_graph } (a conditional node; body_graph is a
 * cudaGraph_t, which is cloned, e.g. torch.cuda.CUDAGraph(keep_graph=True).raw_cuda_graph()) and instantiates it on the
 * current device.  Each hrp_graph_if_launch runs the gate, which opens the body iff *stop_dev == 0 and then adds one to
 * *opened_dev; a closed body costs the gate kernel only.  Bad arguments return -1 with a message naming the field, and so
 * does a graph CUDA refuses to build or instantiate, with the CUDA error text.  hrp_graph_if_destroy: after the launches
 * have completed. */
typedef struct hrp_graph_if hrp_graph_if;
int hrp_graph_if_create(void *body_graph, const uint32_t *stop_dev, uint32_t *opened_dev, hrp_graph_if **out);
int hrp_graph_if_launch(hrp_graph_if *wrapped, void *stream);
int hrp_graph_if_destroy(hrp_graph_if *wrapped);

/* ---- the gradient exchange of the sharded PPO update, fused with clip + Adam (csrc/hrp_comm.cu) --------------
 * One process per GPU on one box.  hrp_comm_create allocates this rank's peer-visible buffers and returns their
 * 64-byte cudaIpc handle; the caller gathers the handles of all ranks (rank-major) and passes them to
 * hrp_comm_connect.  hrp_ppo_loss_grad then writes hrp_comm_grad(), and hrp_clip_adam_step_p2p replaces
 * all_reduce(grad) + hrp_clip_adam_step: ONE cooperative kernel that waits for every rank's gradient, reduces this
 * rank's 1/W slice over NVLink in rank order, pushes the reduced slice to every rank (reduce-scatter + all-gather,
 * the arrival flags are the only synchronisation), clips and applies Adam -- bit-identical parameters on every
 * rank.  Gradient and sum buffers are double-buffered by step parity, so there is no "done reading" barrier:
 * hrp_comm_grad() is the buffer of the NEXT step and alternates.  Every rank must call the step once per optimizer
 * step; ranks must own different devices.  A caller that replays a captured step keeps one graph per parity and
 * announces every replay with hrp_comm_note_replay. */
typedef struct hrp_comm hrp_comm;
int hrp_comm_create(int32_t world, int32_t rank, int64_t n_floats, int32_t device, hrp_comm **out,
                    void *ipc_handle_out64);
int hrp_comm_connect(hrp_comm *comm, const void *ipc_handles /* world x 64 bytes */);
float *hrp_comm_grad(hrp_comm *comm);
float *hrp_comm_grad_parity(hrp_comm *comm, int32_t parity);
int hrp_comm_parity(hrp_comm *comm);          /* parity of the next step (0 / 1) */
int hrp_comm_note_replay(hrp_comm *comm);     /* a captured step is about to be replayed */
int hrp_clip_adam_step_p2p(hrp_comm *comm, float *params_dev, float *exp_avg_dev, float *exp_avg_sq_dev,
                           int32_t *step_dev, double lr, double beta1, double beta2, double eps,
                           float max_grad_norm, float *scratch_dev /* >=128 floats */, void *stream);
/* hrp_clip_adam_step_p2p with the learning rate in device memory: lr_dev as in hrp_clip_adam_step_ex (NULL: exactly
 * hrp_clip_adam_step_p2p).  Bad arguments return -1 with a message naming the field, before any launch. */
int hrp_clip_adam_step_p2p_ex(hrp_comm *comm, float *params_dev, float *exp_avg_dev, float *exp_avg_sq_dev,
                              int32_t *step_dev, double lr, const double *lr_dev, double beta1, double beta2, double eps,
                              float max_grad_norm, float *scratch_dev /* >=128 floats */, void *stream);
/* hrp_clip_adam_step_p2p_ex with target_kl early stopping: with stop_dev non-NULL the comm must have been created with
 * n_floats = P + 1, the last float of each rank's gradient buffer holding its approx-KL share (hrp_ppo_loss_grad_kl's
 * kl_out_dev); the exchange sums all P + 1, clip and Adam cover P, and the step is decided on the summed KL as in
 * hrp_clip_adam_step_kl -- the same bits on every rank, so every rank takes the same decision.  The exchange runs either
 * way.  stop_dev NULL: exactly hrp_clip_adam_step_p2p_ex. */
int hrp_clip_adam_step_p2p_kl(hrp_comm *comm, float *params_dev, float *exp_avg_dev, float *exp_avg_sq_dev,
                              int32_t *step_dev, double lr, const double *lr_dev, double beta1, double beta2, double eps,
                              float max_grad_norm, float *scratch_dev /* >=128 floats */, uint32_t *stop_dev,
                              double kl_limit, void *stream);
/* synchronous: 0, or -4 when some cross-GPU wait timed out (a peer never arrived; ~15 s bound per wait) */
int hrp_comm_status(hrp_comm *comm);
int hrp_comm_destroy(hrp_comm *comm);

/* ---- running observation / reward normalization (SB3 VecNormalize; csrc/hrp_norm.cu) ------------------------------
 * Running statistics are fp64: obs_rms_dev = [mean S][var S][count], ret_rms_dev = [mean, var, count].  A training step
 * is three launches on one stream: hrp_vecnorm_moments -> hrp_vecnorm_merge -> hrp_vecnorm_apply.  Every reduction
 * runs in a fixed order, so equal inputs give the same bits.
 *
 * hrp_vecnorm_moments: batch moments of the C = S (+1 with reward_dev) columns of obs_dev [E][S] (NULL with S = 0).
 * With reward_dev non-NULL, column S is the return carry, updated in place first:
 * returns_dev[e] = returns_dev[e] * gamma + reward_dev[e] (fp64, no FMA).  The result goes to moments_dev:
 * [n][mean C][M2 C] (HRP_VECNORM_MOMENTS_LEN(C) doubles, M2 = sum of squared deviations).  A sharded caller gathers
 * these blocks of every rank, rank-major, and passes them to hrp_vecnorm_merge.  scratch_dev holds
 * HRP_VECNORM_SCRATCH_LEN(C) doubles, zero-filled before its first use; every call leaves it reusable, for any C.
 *
 * hrp_vecnorm_merge: combines the R moment blocks of moments_dev [R][HRP_VECNORM_MOMENTS_LEN(S + has_ret)] in rank
 * order (Chan et al.) and merges them into the running statistics as RunningMeanStd.update does; counts grow by the
 * summed n.  obs_rms_dev is NULL with S = 0, ret_rms_dev with has_ret = 0.  scratch_dev: as above.
 *
 * hrp_vecnorm_apply: obs_dev (in place) and, where terminated_dev[e] | truncated_dev[e], row e of final_obs_dev become
 * clip((x - mean) / sqrt(var + epsilon), +-clip_obs), computed in fp64 and rounded once.  reward_out_dev[e] =
 * clip(reward_dev[e] / sqrt(ret var + epsilon), +-clip_reward).  returns_dev[e] = 0 where the env is done.  Every
 * pointer but the flags is nullable by part: obs_dev with obs_rms_dev (S = 0 when absent), final_obs_dev needs the
 * flags, reward_dev with reward_out_dev and ret_rms_dev.
 *
 * Bad arguments (E outside [1, 2^24], S outside [0, 4608], no column at all, non-finite or non-positive clips,
 * epsilon < 0, gamma outside [0, 1], R < 1, a required NULL) return -1 with a message naming the field, before any
 * launch. */
#define HRP_VECNORM_MAX_S 4608
#define HRP_VECNORM_MAX_E (1 << 24)
#define HRP_VECNORM_MOMENTS_LEN(C) (1 + 2 * (C))
#define HRP_VECNORM_SCRATCH_LEN(C) (256 + 256 * (C))
int hrp_vecnorm_moments(const float *obs_dev, int64_t E, int32_t S, const float *reward_dev, double *returns_dev,
                        double gamma, double *moments_dev, double *scratch_dev, void *stream);
int hrp_vecnorm_merge(const double *moments_dev, int32_t R, int32_t S, int32_t has_ret, double *obs_rms_dev,
                      double *ret_rms_dev, double *scratch_dev, void *stream);
int hrp_vecnorm_apply(float *obs_dev, float *final_obs_dev, const uint8_t *terminated_dev,
                      const uint8_t *truncated_dev, int64_t E, int32_t S, const float *reward_dev, float *reward_out_dev,
                      double *returns_dev, const double *obs_rms_dev, const double *ret_rms_dev, double clip_obs,
                      double clip_reward, double epsilon, void *stream);

#ifdef __cplusplus
}
#endif
#endif
