"""OccupancyGrid observation on the GPU, through the C ABI: the grid epilogue of the step / observe / reset kernels
against the fp64 restatement (tests/grid_oracle.py), its independence of the simulation, and every training path on a
grid env.

- HRP_ENV_REAL64 kernel: bit-exact grid values and cell vehicles, on states the kernel stepped to (free running with
  in-kernel respawn) and on injected states (random headings, vehicles on cell boundaries).  The oracle reads the
  handle's own state, so these tests check the epilogue; the simulation's parity is tests/test_env_gpu.py's.
- fp32 kernel: the same comparison under the either-branch rule -- a cell whose floor the oracle takes within 1e-3 m
  of a boundary may fall either way (the fp32 kernel's headings differ in the last bits), values within 2e-5.  Every
  observation is compared: 0 "neither", 0 skipped.
"""
import copy

import numpy as np
import pytest
import torch

import grid_oracle as go

pytestmark = pytest.mark.gpu

GRID = {"type": "OccupancyGrid"}
ALL8 = ["presence", "x", "y", "vx", "vy", "heading", "cos_h", "sin_h"]
CONFIGS = {
    "default": ({}, {}),
    "aligned": ({"align_to_vehicle_axes": True}, {}),
    "non_square": ({"grid_size": [[-40, 24], [-9, 13]], "grid_step": [4, 2.5]}, {}),
    "one_lane_v31": ({"features": ["presence", "vy", "on_road"]}, {"lanes_count": 1, "vehicles_count": 30}),
    "eight_lanes_v64": ({"grid_step": [6, 8], "grid_size": [[-30, 30], [-30, 34]]}, {"lanes_count": 8, "vehicles_count": 63}),
    "all_ranged": ({"features": ALL8, "grid_size": [[-32, 32], [-16, 16]], "grid_step": [8, 4],
                    "features_range": {"x": [-50, 50], "y": [-20, 20], "vx": [-30, 30], "vy": [-10, 10],
                                       "heading": [-1, 1], "cos_h": [-1, 1], "sin_h": [-1, 1], "presence": [0, 1]},
                    "align_to_vehicle_axes": True}, {}),
    "all_raw": ({"features": ["x", "y", "vx", "vy", "heading", "cos_h", "sin_h", "on_road"], "features_range": {},
                 "grid_size": [[-32, 32], [-16, 16]], "grid_step": [8, 4], "clip": False}, {}),
}


def _cfg(highway_config, name, meta=False, **env):
    obs, over = CONFIGS[name]
    c = copy.deepcopy(highway_config)
    c["observation"] = dict(GRID, **obs)
    c.update(over)
    c.update(env)
    if meta:
        c["action"] = {"type": "DiscreteMetaAction"}
    return c


def _vec(cfg, E, **kw):
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv

    return HighwayVecEnv(cfg, E, device="cuda:0", **kw)


def _oracle(env):
    return go.oracle_for(env.config["observation"], int(env.config["lanes_count"]))


def _actions(rng, E, meta):
    if meta:
        return torch.tensor(np.stack([rng.integers(0, 5, E), np.zeros(E)], 1), dtype=torch.float32, device="cuda:0")
    return torch.tensor(rng.uniform(-0.4, 0.4, (E, 2)), dtype=torch.float32, device="cuda:0")


class _Judge:
    def __init__(self, real64):
        self.real64 = real64
        self.counts = {"agree": 0, "flipped": 0, "neither": 0}

    def check(self, o, st, obs, cells, e, where):
        state = (st["x"][e], st["y"][e], st["heading"][e], st["speed"][e])
        grid, cv = obs[e], cells[e]
        if self.real64:
            want, want_cells = o.observe(*state)
            assert np.array_equal(cv, want_cells), where
            assert np.array_equal(grid, want), (where, np.abs(grid - want).max())
            self.counts["agree"] += 1
            return
        r = go.either_branch(o, state, grid, cv, tol=2e-5)
        self.counts["agree" if r is None else ("neither" if r is False else "flipped")] += 1
        assert r is not False, where


def _inject(env, rng, st):
    """perturb a stepped state: random headings, and a few vehicles moved onto cell boundaries of the ego's grid"""
    st = {k: v.copy() for k, v in st.items()}
    st["heading"] = st["heading"] + rng.uniform(-0.6, 0.6, st["heading"].shape)
    obs = env.config["observation"]
    (x0, _), (y0, _) = obs["grid_size"]
    sx, sy = obs["grid_step"]
    E, V = st["x"].shape
    for e in range(E):
        for k in rng.choice(np.arange(1, V), size=min(4, V - 1), replace=False):
            st["x"][e, k] = st["x"][e, 0] + x0 + sx * rng.integers(0, 8)
            st["y"][e, k] = st["y"][e, 0] + y0 + sy * rng.integers(0, 8)
    return st


@pytest.mark.parametrize("real64", [True, False], ids=["fp64", "fp32"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_grid_matches_oracle(highway_config, name, real64):
    E, steps = 32, 12
    meta = name == "one_lane_v31"
    env = _vec(_cfg(highway_config, name, meta=meta), E, real64=real64, seed=7)
    o = _oracle(env)
    F, W, H = env.obs_shape
    assert o.shape == (F, W, H) and env.obs.shape == (E, F, W, H) and (env.N, env.F_out) == (F, W * H)
    judge = _Judge(real64)
    rng = np.random.default_rng(3)
    cells = torch.full((E, W * H), -7, dtype=torch.int32, device="cuda:0")
    env.reset(seed=5)
    for t in range(steps):
        obs, *_ = env.step(_actions(rng, E, meta), row_vehicle=cells)
        o_np, c_np, st = obs.cpu().numpy(), cells.cpu().numpy(), env.get_state()
        for e in range(E):
            judge.check(o, st, o_np, c_np, e, (name, "step", t, e))
        if t % 4 == 3:   # injected states through the observe kernel
            inj = _inject(env, rng, st)
            env.set_state(inj)
            out = env.observe(row_vehicle=cells)
            o_np, c_np, st2 = out.cpu().numpy(), cells.cpu().numpy(), env.get_state()
            for e in range(E):
                judge.check(o, st2, o_np, c_np, e, (name, "injected", t, e))
    print(name, "fp64" if real64 else "fp32", judge.counts)
    assert judge.counts["neither"] == 0
    assert sum(judge.counts.values()) == E * (steps + steps // 4)
    env.close()


def test_reset_observation_matches_oracle(highway_config):
    env = _vec(_cfg(highway_config, "default"), 16, real64=True)
    o = _oracle(env)
    obs = env.reset(seed=11).cpu().numpy()
    st = env.get_state()
    for e in range(16):
        want, _ = o.observe(st["x"][e], st["y"][e], st["heading"][e], st["speed"][e])
        assert np.array_equal(obs[e], want)
    env.close()


@pytest.mark.parametrize("real64", [False, True], ids=["fp32", "fp64"])
def test_grid_handle_simulates_like_a_kinematics_twin(highway_config, real64):
    E = 64
    rng = np.random.default_rng(1)
    g = _vec(_cfg(highway_config, "default"), E, real64=real64, seed=3)
    k = _vec(copy.deepcopy(highway_config), E, real64=real64, seed=3)
    g.reset(seed=9)
    k.reset(seed=9)
    for t in range(30):
        a = _actions(rng, E, False)
        _, rg, teg, trg = g.step(a)
        _, rk, tek, trk = k.step(a)
        assert torch.equal(rg, rk) and torch.equal(teg, tek) and torch.equal(trg, trk), t
    sg, sk = g.get_state(), k.get_state()
    for key in sg:
        assert np.array_equal(sg[key], sk[key]), key
    g.close()
    k.close()


@pytest.mark.parametrize("real64", [False, True], ids=["fp32", "fp64"])
def test_final_observation_equals_an_autoreset_0_twin(highway_config, real64):
    E = 64
    rng = np.random.default_rng(2)
    cfg = _cfg(highway_config, "default", duration=5)
    a_env = _vec(cfg, E, real64=real64, seed=1)
    b_env = _vec(cfg, E, real64=real64, seed=1, autoreset=False)
    a_env.reset(seed=4)
    fin = torch.full_like(a_env.obs, 7.0)
    finished = 0
    for t in range(12):
        b_env.set_state(a_env.get_state())
        fin.fill_(7.0)
        act = _actions(rng, E, False)
        obs_a, _, te, tr = a_env.step(act, final_obs_out=fin)
        obs_b, _, te_b, tr_b = b_env.step(act)
        assert torch.equal(te, te_b) and torch.equal(tr, tr_b)
        done = (te | tr) != 0
        finished += int(done.sum())
        assert torch.equal(fin[done], obs_b[done]), t
        assert (fin[~done] == 7.0).all()
        assert torch.equal(obs_a[~done], obs_b[~done])
    assert finished > 0
    a_env.close()
    b_env.close()


def test_step_mask_and_per_env_seeds(highway_config):
    E = 8
    cfg = _cfg(highway_config, "default")
    env = _vec(cfg, E)
    seeds = torch.arange(100, 100 + E, dtype=torch.int64, device="cuda:0")
    env.set_env_seeds(seeds)
    obs = env.reset().clone()
    for e in (0, 5):
        one = _vec(cfg, 1)
        want = one.reset(seed=100 + e)
        assert torch.equal(obs[e], want[0])
        one.close()
    mask = torch.zeros(E, dtype=torch.uint8, device="cuda:0")
    mask[::2] = 1
    env.set_step_mask(mask)
    before = env.get_state()
    out = env.obs.clone()
    env.step(torch.zeros(E, 2, device="cuda:0"), out=out)
    after = env.get_state()
    for e in range(E):
        moved = not np.array_equal(before["x"][e], after["x"][e])
        assert moved == bool(e % 2 == 0), e
        if e % 2:
            assert torch.equal(out[e], obs[e])
    env.close()


def test_perm_is_refused_on_a_grid(highway_config):
    import ctypes as C

    from highway_rope_ppo_b200 import _lib

    env = _vec(_cfg(highway_config, "default"), 2)
    with pytest.raises(ValueError, match="row order"):
        env.step(torch.zeros(2, 2, device="cuda:0"), perm=torch.zeros(2, 3, dtype=torch.int32))
    lib = _lib.load()
    perm = torch.zeros(8, dtype=torch.int32, device="cuda:0")
    a = torch.zeros(2, 2, device="cuda:0")
    r = torch.zeros(2, device="cuda:0")
    f = torch.zeros(2, dtype=torch.uint8, device="cuda:0")
    rc = lib.hrp_env_step(env._h, a.data_ptr(), env.obs.data_ptr(), r.data_ptr(), f.data_ptr(), f.data_ptr(),
                          perm.data_ptr(), None, None)
    assert rc == -1 and "perm_dev" in _lib.last_error()
    fw, ww, hh = C.c_int32(), C.c_int32(), C.c_int32()
    assert lib.hrp_env_grid_shape(env._h, C.byref(fw), C.byref(ww), C.byref(hh)) == 0
    assert (fw.value, ww.value, hh.value) == (4, 11, 11)
    k = _vec(copy.deepcopy(highway_config), 2)
    assert lib.hrp_env_grid_shape(k._h, C.byref(fw), C.byref(ww), C.byref(hh)) == -1
    env.close()
    k.close()


@pytest.mark.parametrize("meta", [False, True], ids=["gaussian", "categorical-meta"])
def test_rollout_graph_equals_eager_and_training_runs(highway_config, meta):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.routine import collect_rollout, evaluate_vectorized, train_vectorized

    E, T = 128, 8
    cfg = _cfg(highway_config, "default", meta=meta, duration=6)
    runs = []
    for use_graph in (False, True):
        torch.manual_seed(0)
        env = _vec(cfg, E, seed=2)
        S = env.N * env.F_out
        assert S == 484
        agent = PPOAgent(S, 5 if meta else 2, hidden_dim=64, batch_size=256, epochs=1, discrete=meta)
        obs = env.reset(seed=2).clone()
        r = collect_rollout(env, agent, T, obs, use_graph=use_graph, bootstrap_truncated=True)
        runs.append({k: v.clone() for k, v in r.items()})
        env.close()
    for k in ("states", "action", "reward", "terminated", "truncated", "value"):
        if k in runs[0]:
            assert torch.equal(runs[0][k], runs[1][k]), k
    env = _vec(cfg, E, seed=2)
    torch.manual_seed(0)
    agent = PPOAgent(env.N * env.F_out, 5 if meta else 2, hidden_dim=64, batch_size=256, epochs=1, discrete=meta)
    hist = train_vectorized(env, agent, 3, T, seed=2, bootstrap_truncated=True, eval_episodes=32, eval_interval=2)
    assert len(hist) == 3 and all(np.isfinite(m["loss"]) for m in hist)
    assert sum(m["episodes"] for m in hist) > 0
    ev_env = _vec(cfg, 32, seed=2, autoreset=False)
    ev = evaluate_vectorized(ev_env, agent, exp_seed=1)
    assert ev["episodes"] == 32 and np.isfinite(ev["mean"])
    env.close()
    ev_env.close()


def test_grid_experiments_multiplexed_equal_sequential(highway_config, tmp_path):
    from highway_rope_ppo_b200.experiments.config import Condition, ConditionHP, Experiment
    from highway_rope_ppo_b200.experiments.multiplex import MultiplexedRunner
    from highway_rope_ppo_b200.experiments.runner import ExperimentRunner

    over = {"observation": {"type": "OccupancyGrid", "features": ["presence", "vx", "vy", "on_road"]}}
    exps = []
    for i, cond in enumerate((Condition.SORTED, Condition.SHUFFLED, Condition.SORTED)):
        hp = ConditionHP(lr=3e-4, hidden_dim=64, batch_size=32, epochs=2, steps_per_update=48)
        exps.append(Experiment(Experiment.make_name(cond, hp, 42 + i) + f"_grid{i}", cond, hp, seed=42 + i, max_episodes=3,
                               env_config_overrides=over, extra={"eval_interval": 3, "log_interval": 1}))
    seq = [ExperimentRunner(highway_config, artifacts_dir=str(tmp_path / "seq")).launch(e) for e in exps]
    mux = MultiplexedRunner(highway_config, artifacts_dir=str(tmp_path / "mux"), max_concurrent=4).launch_many(exps)
    for a, b in zip(seq, mux):
        assert a["status"] == b["status"] == "COMPLETED", (a.get("error_traceback"), b.get("error_traceback"))
        assert a["rewards"] == b["rewards"] and a["avg_rewards"] == b["avg_rewards"]
        ua, ub = a["metrics_history"]["policy_updates"], b["metrics_history"]["policy_updates"]
        assert len(ua) == len(ub)
        for x, y in zip(ua, ub):
            assert {k: v for k, v in x.items() if k != "time"} == {k: v for k, v in y.items() if k != "time"}


def test_gym_view_of_a_grid(highway_config):
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_env

    env = make_env(Condition.SHUFFLED, highway_config, env_overrides={"observation": dict(GRID, features=["presence", "on_road"])})
    assert env.observation_space.shape == (2, 11, 11)
    obs, _ = env.reset(seed=3)
    assert obs.shape == (2, 11, 11) and obs[0, 5, 5] == 1.0 and obs[1].sum() > 0
    obs, r, te, tr, _ = env.step(np.zeros(2, np.float32))
    assert obs.shape == (2, 11, 11) and obs[0, 5, 5] == 1.0
    env.close()
