"""GPU parity of the simulator kernel across the configuration space hrp_env_create_ex accepts (tests/test_abi_cpu.py
test_env_config_limits), against the CPU oracle (oracle/highway_oracle.c), with the rules of tests/test_env_gpu.py:

* every case runs the fp64 validation instantiation (discrete state exact on every injected step, only separating-axis
  ties flipped) and the fp32 product kernel (either-branch rule, no `neither`), each on >= 500 env-steps;
* the fused embedding epilogue is compared with oracle/embed.py applied to a plain handle's observation of the same
  injected states (2e-6 for RoPE / DistPE, exact for RankPE, as tests/test_embed_gpu.py);
* captured launches (the rollout graph of training/routine.py, the group graphs of training/host_pipeline.py) respawn
  from the seed of the latest reset, like the eager launches.
"""
import numpy as np
import pytest
import torch

from oracle import embed as oe
from oracle import highway as oh

from test_env_gpu import _cfg, _injected_parity, _random_actions, _gentle_actions, _report, _vec

pytestmark = pytest.mark.gpu

_F8 = ["presence", "x", "y", "vx", "vy", "heading", "cos_h", "sin_h"]


def _steering_actions(rng, E, t):
    a = rng.uniform(-1, 1, (E, 2))
    a[:, 1] = np.sign(a[:, 1]) * rng.uniform(0.6, 1.0, E)   # hard steering: the ego leaves the road within a step
    return a


# name -> (config overrides, actions, sorted observation)
CASES = {
    "sim 5 / policy 1": (dict(simulation_frequency=5), _random_actions, True),
    "sim 10 / policy 1": (dict(simulation_frequency=10), _random_actions, True),
    "sim 30 / policy 2": (dict(simulation_frequency=30, policy_frequency=2), _random_actions, True),
    "sim 20 / policy 3": (dict(simulation_frequency=20, policy_frequency=3), _random_actions, True),
    "sim 15 / policy 2": (dict(policy_frequency=2), _random_actions, True),
    "duration 3 at 15 / 2": (dict(policy_frequency=2, duration=3), _gentle_actions, True),
    "duration 2.5 at 15 / 2": (dict(policy_frequency=2, duration=2.5), _gentle_actions, True),
    "1 lane": (dict(lanes_count=1), _random_actions, True),
    "8 lanes": (dict(lanes_count=8), _gentle_actions, True),
    "V 31": (dict(vehicles_count=30, observation=dict(vehicles_count=30)), _random_actions, True),
    "V 32": (dict(vehicles_count=31), _gentle_actions, True),
    "V 33": (dict(vehicles_count=32), _random_actions, True),
    "road 5 km": (dict(vehicles_count=63, vehicles_density=0.25), _gentle_actions, True),
    "road 38 km": (dict(vehicles_count=63, vehicles_density=0.05, lanes_count=1), _gentle_actions, True),
    "initial lane 0, spacing 1": (dict(initial_lane_id=0, ego_spacing=1), _random_actions, True),
    "initial lane 3, spacing 4": (dict(initial_lane_id=3, ego_spacing=4), _random_actions, True),
    "raw reward": (dict(normalize_reward=False), _random_actions, True),
    "offroad terminal": (dict(offroad_terminal=True), _steering_actions, True),
    "reward weights": (dict(collision_reward=-2.5, right_lane_reward=0.3, high_speed_reward=0.7,
                            reward_speed_range=[15, 35]), _random_actions, True),
    "N 1": (dict(observation=dict(vehicles_count=1)), _random_actions, True),
    "N 2 shuffled": (dict(observation=dict(vehicles_count=2, order="shuffled")), _random_actions, False),
    "N 31": (dict(observation=dict(vehicles_count=31)), _random_actions, True),
    "N 31 shuffled": (dict(observation=dict(vehicles_count=31, order="shuffled")), _random_actions, False),
    "N 32": (dict(observation=dict(vehicles_count=32)), _random_actions, True),
    "N 32 shuffled": (dict(observation=dict(vehicles_count=32, order="shuffled")), _random_actions, False),
    "N 33": (dict(observation=dict(vehicles_count=33)), _random_actions, True),
    "N 33 shuffled": (dict(observation=dict(vehicles_count=33, order="shuffled")), _random_actions, False),
    "N 64": (dict(vehicles_count=63, observation=dict(vehicles_count=64)), _random_actions, True),
    "N 64 shuffled": (dict(vehicles_count=63, observation=dict(vehicles_count=64, order="shuffled")), _random_actions,
                      False),
    "F 1": (dict(observation=dict(features=["presence"])), _random_actions, True),
    "F 8": (dict(observation=dict(features=_F8)), _random_actions, True),
    "absolute": (dict(observation=dict(absolute=True, features=_F8)), _random_actions, True),
    # fp64 kernel only (FP64_ONLY): unnormalised x / y / vx / vy are metres and m/s, and the fp32 kernel's state error
    # (TOL: 1e-3 m) reaches them unscaled, beyond the observation rule (2e-5, normalised units)
    "not normalised": (dict(observation=dict(normalize=False)), _random_actions, True),
    "not clipped": (dict(observation=dict(clip=False)), _random_actions, True),
    # x clipped beyond 20 m; vy is not narrowed below the default: a range of +-2 m/s scales vy's fp32 error
    # (speed x heading, up to 1.5e-4 m/s) past the observation rule
    "narrow range": (dict(observation=dict(features_range=dict(x=[-20, 20], y=[-12, 12], vx=[-10, 10], vy=[-30, 30]))),
                     _random_actions, True),
    "see behind shuffled": (dict(observation=dict(order="shuffled", see_behind=True)), _random_actions, False),
}
FP64_ONLY = {"not normalised"}
E, STEPS = 24, 21   # 504 env-steps per case and precision


@pytest.mark.parametrize("name,real64", [pytest.param(n, r, id=f"{n}-{'fp64' if r else 'fp32'}") for n in CASES
                                         for r in (True, False) if r or n not in FP64_ONLY])
def test_step_parity_across_configs(highway_config, name, real64):
    over, fn, sorted_obs = CASES[name]
    cfg = _cfg(highway_config, **{k: dict(v) if isinstance(v, dict) else v for k, v in over.items()})
    seed = 100 + list(CASES).index(name)
    if name.startswith("road"):
        # the roads these cases spawn put vehicles beyond 4096 m (and, at 0.05, beyond 2^15 m) from the ego, where
        # the fp32 working copies of x lose the precision of the default road
        o = oh.OracleEnv(cfg)
        o.reset(seed, env_id=0, episode=0)
        x = o.get_state()["x"]
        assert np.abs(x - x[0]).max() > (32768 if "38" in name else 4096)
    s = _injected_parity(cfg, E=E, steps=STEPS, seed=seed, action_fn=fn, sorted_obs=sorted_obs, real64=real64)
    n = _report(f"{'fp64' if real64 else 'fp32'} kernel, {name}", s)
    assert n == E * STEPS
    if real64:
        assert s["flipped"] <= 0.002 * n and set(s["kinds"]) <= {"sat_will", "sat_now", "sat_axis"}
    else:
        assert s["flipped"] <= 0.3 * s["agree"]


def test_collision_window_at_5hz_registers_the_impact(highway_config):
    """An ego at 40 m/s, 19 m behind a crashed vehicle of its lane, at 5 Hz.  After the first frame's move the x gap is
    11 m: beyond the 8.8 m candidate window of 15 Hz, inside the pre-check radius sqrt(29) + 40.5 / 5, and the oracle
    registers the will-intersect impact there (the ego is crashed from the second frame on).  The kernel must find the
    pair in the same frame."""
    cfg = _cfg(highway_config, vehicles_count=1, simulation_frequency=5)
    for real64 in (True, False):
        env = _vec(cfg, 1, autoreset=False, real64=real64)
        o = oh.OracleEnv(cfg)
        o.reset(1, env_id=0, episode=0)
        st = o.get_state()
        st["x"][:] = [100.0, 119.0]
        st["y"][:] = [4.0, 4.0]
        st["lane"][:] = st["target_lane"][:] = [1, 1]
        st["speed"][:] = [40.0, 0.0]
        st["target_speed"][:] = [40.0, 0.0]
        st["heading"][:] = 0.0
        st["crashed"][:] = [0, 1]
        st["has_impact"][:] = 0
        o.set_state(st)
        full = {k: np.asarray(st[k])[None] for k in oh.STATE_F64 + oh.STATE_I32}
        full["time"] = np.array([st["time"]])
        env.set_state(full)
        r, te, tr = o.step(np.zeros(2, np.float32))
        _, rk, tk, _ = env.step(torch.zeros((1, 2), device="cuda:0"))
        got, want = env.get_state(), o.get_state()
        assert te and bool(tk[0]), "the oracle's and the kernel's ego must both crash"
        assert np.array_equal(got["crashed"][0], want["crashed"]) and np.array_equal(got["has_impact"][0], want["has_impact"])
        np.testing.assert_allclose(got["x"][0], want["x"], atol=1e-3)
        np.testing.assert_allclose(got["speed"][0], want["speed"], atol=2e-4)
        env.close()


# ---- the fused embedding epilogue on injected states ----------------------------------------------------------------
def _spec(kind, d, N, ego_idx=0, use_euclidean=True, seed=0):
    from highway_rope_ppo_b200._lib import EMBED_DIST, EMBED_RANK, EMBED_ROPE
    from highway_rope_ppo_b200.envs.highway_vec import EmbedSpec

    if kind == "rope":
        return EmbedSpec(EMBED_ROPE, d, oe.rope_inv_freq(d, 100.0), 100.0, True, ego_idx)
    if kind == "dist":
        return EmbedSpec(EMBED_DIST, d, oe.dist_freqs(d, 100.0), 100.0, use_euclidean, ego_idx)
    table = np.tanh(np.random.default_rng(seed).normal(0, 0.05, (N, d))).astype(np.float32)
    return EmbedSpec(EMBED_RANK, d, table, 100.0, True, ego_idx)


def _want(kind, obs, spec, N):
    if kind == "rope":
        return oe.rope(obs, spec.dim, 100.0, ego_idx=spec.ego_idx)
    if kind == "dist":
        return oe.distpe(obs, spec.dim, 100.0, use_euclidean=spec.use_euclidean, ego_idx=spec.ego_idx)
    return oe.rankpe(obs, spec.table.reshape(N, spec.dim))


_N30 = dict(vehicles_count=30, observation=dict(vehicles_count=30, order="shuffled"))
_N64 = dict(vehicles_count=63, observation=dict(vehicles_count=64, order="shuffled"))
# name -> (config overrides, kind, d, ego_idx, use_euclidean); RankPE d = 1 is the one odd F_out (F + 1 = 5)
EMBED_CASES = {
    "N30 rank 4": (_N30, "rank", 4, 0, True),
    "N30 rank 8": (_N30, "rank", 8, 0, True),
    "N30 rank 16": (_N30, "rank", 16, 0, True),
    "N30 dist 4": (_N30, "dist", 4, 0, True),
    "N30 dist 8": (_N30, "dist", 8, 0, True),
    "N30 dist 16": (_N30, "dist", 16, 0, True),
    "N30 rope 4": (_N30, "rope", 4, 0, True),
    "dist 64 |dx|": (dict(observation=dict(order="shuffled")), "dist", 64, 0, False),
    "rope ego 3": (dict(observation=dict(order="shuffled")), "rope", 4, 3, True),
    "dist ego 3": (dict(observation=dict(order="shuffled")), "dist", 8, 3, True),
    "rope all 8 features": (dict(observation=dict(features=_F8)), "rope", 8, 0, True),
    "N64 rope": (_N64, "rope", 4, 0, True),
    "N64 dist": (_N64, "dist", 16, 0, True),
    "N64 rank": (_N64, "rank", 8, 0, True),
    "rank 1": (dict(observation=dict(order="shuffled")), "rank", 1, 0, True),
}


@pytest.mark.parametrize("name", list(EMBED_CASES))
def test_fused_embedding_on_injected_states(highway_config, name):
    over, kind, d, ego_idx, eu = EMBED_CASES[name]
    cfg = _cfg(highway_config, **{k: dict(v) if isinstance(v, dict) else v for k, v in over.items()})
    N = cfg["observation"]["vehicles_count"]
    spec = _spec(kind, d, N, ego_idx, eu)
    sorted_obs = cfg["observation"].get("order", "sorted") == "sorted"
    s = _injected_parity(cfg, E=16, steps=12, seed=300 + list(EMBED_CASES).index(name), action_fn=_random_actions,
                         sorted_obs=sorted_obs, embed=spec)
    # the fused output against the plain handle's own observation first: it does not depend on the plain parity
    assert len(s["embedded"]) == 12
    for plain, fused in s["embedded"]:
        assert fused.shape == (16, N, spec.out_features(len(cfg["observation"]["features"])))
        for e in range(16):
            want = _want(kind, plain[e], spec, N)
            if kind == "rank":
                assert np.array_equal(fused[e], want), (name, e)
            else:
                np.testing.assert_allclose(fused[e], want, atol=2e-6, err_msg=name)
    _report(f"plain observation, {name}", s)


@pytest.mark.xfail(strict=True, reason="fp32 heading error 1.33e-4 rad > TOL 1e-4 (step 9, env 12, vehicle 16), "
                                       "not explained by a marginal decision")
def test_fp32_heading_finding_default_config_shuffled_seed_214(highway_config):
    """An open parity finding: on the default config with shuffled rows, seed 214, the fp32 kernel ends one injected
    env-step with a heading error above TOL and no marginal decision of the oracle to explain it.  Strict: the test
    reports when a change of the kernel or of the oracle makes it pass."""
    cfg = _cfg(highway_config, observation=dict(order="shuffled"))
    s = _injected_parity(cfg, E=16, steps=12, seed=214, action_fn=_random_actions, sorted_obs=False)
    _report("default config, shuffled, seed 214", s)


# ---- extended draws and respawns --------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [2, 33, 64])
def test_shuffle_draw_at_more_rows(highway_config, N):
    """The in-kernel Philox permutation (test_env_gpu.test_shuffle_draw_matches_oracle_permutation) at row counts whose
    draw loop spans one block, two warps' worth of rows and several lanes."""
    cfg = _cfg(highway_config, vehicles_count=max(50, N - 1), observation=dict(order="shuffled", vehicles_count=N))
    E, seed, base = 24, 99, 500
    env = _vec(cfg, E, env_id_base=base, autoreset=False)
    env.reset(seed)
    rows = torch.zeros((E, N), dtype=torch.int32, device="cuda:0")
    st0 = env.get_state()
    env.observe(row_vehicle=rows)
    rv = rows.cpu().numpy()
    o = oh.OracleEnv(cfg)
    for e in range(E):
        o.reset(seed, env_id=base + e, episode=0)
        perm = oh.shuffle_perm(seed, base + e, int(st0["obs_draw"][e]), N - 1)
        _, want = o.observe(perm=perm, with_rows=True)
        assert np.array_equal(rv[e], want), e
    assert np.all(env.get_state()["obs_draw"] == st0["obs_draw"] + 1)
    env.close()


@pytest.mark.parametrize("sim,policy", [(5, 1), (30, 2)])
def test_autoreset_after_other_step_lengths(highway_config, sim, policy):
    """test_env_gpu.test_autoreset_respawns_inside_the_step at other frame counts and step lengths: envs whose time
    reaches the duration on this step respawn inside it, equal to the oracle's reset."""
    cfg = _cfg(highway_config, simulation_frequency=sim, policy_frequency=policy)
    E, seed, dtime = 64, 7, 1.0 / policy
    env = _vec(cfg, E, autoreset=True)
    env.reset(seed)
    st = env.get_state()
    st["time"][::2] = 40.0 - dtime
    env.set_state(st)
    obs, rew, term, trunc = env.step(torch.zeros((E, 2), device="cuda:0"))
    trunc = trunc.cpu().numpy().astype(bool)
    assert trunc[::2].all() and not trunc[1::2].any()
    got = env.get_state()
    o = oh.OracleEnv(cfg)
    for e in range(0, E, 2):
        o.reset(seed, env_id=e, episode=1)
        ref = o.get_state()
        assert got["episode"][e] == 1 and got["time"][e] == 0.0
        np.testing.assert_allclose(got["x"][e], ref["x"], atol=1e-9)
        assert np.array_equal(got["lane"][e], ref["lane"])
        np.testing.assert_allclose(obs[e].cpu().numpy(), o.observe(), atol=2e-6)
    alive = ~(trunc | term.cpu().numpy().astype(bool))
    assert alive[1::2].sum() > E // 4
    assert np.all(got["episode"][alive] == 0) and np.allclose(got["time"][alive], dtime)
    env.close()


# ---- captured launches after a reseed ---------------------------------------------------------------------------------
def _short_episodes(highway_config):
    return _cfg(highway_config, duration=3)


def test_graph_rollout_respawns_from_the_new_seed(highway_config):
    """collect_rollout replays a captured rollout; after vec_env.reset(seed=s2) its in-kernel respawns must draw from
    s2 -- equal to the oracle's reset(s2) -- and the rollout must equal the launch-by-launch one."""
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.routine import collect_rollout

    cfg = _short_episodes(highway_config)
    E, T, s1, s2 = 64, 8, 5, 6
    runs = []
    for use_graph in (False, True):
        torch.manual_seed(4)
        env = HighwayVecEnv(cfg, E, device="cuda:0")
        agent = PPOAgent(60, 2, hidden_dim=64, batch_size=E, epochs=1)
        got = []
        for seed in (s1, s2):
            obs = env.reset(seed=seed).clone()
            for _ in range(2):   # the first rollout of a key runs eagerly, the second is captured and replayed
                r = collect_rollout(env, agent, T, obs, use_graph=use_graph)
                got.append({k: v.clone() for k, v in r.items()})
                obs = r["states"][T].clone()
        runs.append(got)
        env.close()
    for i, (a, b) in enumerate(zip(*runs)):
        for k in a:
            assert torch.equal(a[k], b[k]), (i, k)
    after = runs[1][2:]
    done = np.concatenate([r["done"].cpu().numpy().astype(bool) for r in after])
    states = np.concatenate([r["states"][1:].cpu().numpy().reshape(T, E, 15, 4) for r in after])
    assert done.sum() >= 2 * E   # duration 3: every env respawns inside each rollout
    o = oh.OracleEnv(cfg)
    for e in range(E):
        ep = 0
        for t in range(2 * T):
            if done[t, e]:
                ep += 1
                o.reset(s2, env_id=e, episode=ep)
                np.testing.assert_allclose(states[t, e], o.observe(), atol=2e-6, err_msg=f"t {t} env {e}")


def test_host_pipeline_graphs_respawn_from_the_new_seed(highway_config):
    """HostBufferPipeline with group graphs: pipe.reset(s2) after graphs were captured under s1 reproduces the eager
    pipeline (test_api_gpu.test_host_buffer_pipeline_equals_the_device_loop) step for step, respawns included."""
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.host_pipeline import HostBufferPipeline

    cfg = _short_episodes(highway_config)
    E, groups = 128, 2
    Eg = E // groups
    runs = []
    for graphs in (False, True):
        torch.manual_seed(1)
        agent = PPOAgent(60, 2, hidden_dim=64, batch_size=E)
        pipe = HostBufferPipeline(agent, [HighwayVecEnv(cfg, Eg, device="cuda:0", env_id_base=g * Eg)
                                          for g in range(groups)], use_graphs=graphs)
        got = []
        for seed, steps in ((42, 4), (43, 8)):
            pipe.reset(seed)
            for _ in range(steps):
                for g in range(groups):
                    pipe.launch(g)
                for g in range(groups):
                    b = pipe.wait(g)
                    got.append({k: v.copy() for k, v in b.items()})
        pipe.close()
        for env in pipe.envs:
            env.close()
        runs.append(got)
    assert sum(int(b["truncated"].sum()) for b in runs[0][8:]) >= E
    for i, (a, b) in enumerate(zip(*runs)):
        for k in a:
            assert np.array_equal(a[k], b[k]), (i, k)
