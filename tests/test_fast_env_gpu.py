"""highway-fast-v0 on the GPU: the ego-only collision pass of the step kernels against the fp64 oracle, with the rules
of tests/test_env_gpu.py (fp64 kernel exact in the discrete state on every injected step, only separating-axis ties
flipped; fp32 kernel by the either-branch rule, 0 `neither`, 0 skipped), the hand-built collision cases of
tests/test_fast_env_cpu.py, and every path that builds a twin handle from the resolved config.  The oracle of a fast env
is tests/fast_oracle.py's."""
import copy

import numpy as np
import pytest
import torch

import fast_oracle
import test_env_gpu
from fast_oracle import FAST, oracle_module
from oracle import highway as oh
from test_env_gpu import _cfg, _injected_parity, _meta_actions, _random_actions, _report, _vec
from test_fast_env_cpu import HAND_CASES, KINEMATICS, _hand_cfg, _hand_state

pytestmark = pytest.mark.gpu


def _fast(meta=False, **over):
    """fast defaults, with the observation block spelled out for the parity harness"""
    c = {"gym_id": FAST, "observation": dict(KINEMATICS),
         "action": {"type": "DiscreteMetaAction"} if meta else {"type": "ContinuousAction"}}
    c.update(over)
    return c


# name -> (config, actions, sorted observation, E, steps): >= 500 env-steps each
CASES = {
    "fast defaults, continuous": (lambda hc: _fast(), _random_actions, True, 20, 26),
    "fast defaults, meta-action": (lambda hc: _fast(meta=True), _meta_actions, True, 20, 26),
    "reference config, sorted": (lambda hc: _cfg(hc, gym_id=FAST), _random_actions, True, 20, 26),
    "reference config, shuffled": (lambda hc: _cfg(hc, gym_id=FAST, observation=dict(order="shuffled")), _random_actions,
                                   False, 20, 26),
}


@pytest.mark.parametrize("real64", [True, False], ids=["fp64", "fp32"])
@pytest.mark.parametrize("name", list(CASES))
def test_injected_parity(highway_config, name, real64, monkeypatch):
    monkeypatch.setattr(test_env_gpu, "oh", fast_oracle.highway)   # the harness's oracle: the ego-only one
    make, fn, sorted_obs, E, steps = CASES[name]
    cfg = make(highway_config)
    s = _injected_parity(cfg, E=E, steps=steps, seed=21, action_fn=fn, sorted_obs=sorted_obs, real64=real64)
    n = _report(f"{FAST} {name}, {'fp64' if real64 else 'fp32'}", s)
    assert n == E * steps >= 500
    if real64:
        assert s["flipped"] <= 0.002 * n and set(s["kinds"]) <= {"sat_will", "sat_now", "sat_axis"}


class _FinalStepEnv:
    """A handle that steps through hrp_env_step_final and checks its final observation on the way (autoreset = 0:
    final_obs[e] == obs[e] for every finished env, untouched rows elsewhere)."""

    def __init__(self, cfg, E, **kw):
        self.env = _vec(cfg, E, **kw)
        self.finished = 0

    def __getattr__(self, name):
        return getattr(self.env, name)

    def step(self, actions, **kw):
        fin = torch.full_like(self.env.obs, 7.0)
        obs, r, te, tr = self.env.step(actions, final_obs_out=fin, **kw)
        done = (te | tr) != 0
        assert torch.equal(fin[done], obs[done]) and bool((fin[~done] == 7.0).all())
        self.finished += int(done.sum())
        _FinalStepEnv.total += int(done.sum())
        return obs, r, te, tr


@pytest.mark.parametrize("real64", [True, False], ids=["fp64", "fp32"])
def test_injected_parity_through_step_final(highway_config, real64, monkeypatch):
    _FinalStepEnv.total = 0
    monkeypatch.setattr(test_env_gpu, "oh", fast_oracle.highway)
    monkeypatch.setattr(test_env_gpu, "_vec", lambda cfg, E, **kw: _FinalStepEnv(cfg, E, **kw))
    # an 8 s episode: every env is truncated at least twice, so final observations are written and checked
    s = _injected_parity(_fast(duration=8), E=20, steps=26, seed=22, action_fn=_random_actions, real64=real64)
    assert _report(f"{FAST} through hrp_env_step_final", s) == 520
    assert _FinalStepEnv.total > 0


# ---- the hand-built cases (a), (c), (d) --------------------------------------------------------------------------------
@pytest.mark.parametrize("real64", [True, False], ids=["fp64", "fp32"])
@pytest.mark.parametrize("gym_id", ["highway-v0", FAST])
def test_directed_collision_cases(gym_id, real64):
    cases = ("a", "c", "d")
    cfg = _hand_cfg(gym_id)
    E = len(cases)
    env = _vec(cfg, E, autoreset=False, real64=real64)
    trace = env.enable_trace()
    states = [_hand_state(HAND_CASES[c]) for c in cases]
    st = {k: np.stack([s[k] for s in states]) for k in oh.STATE_F64 + oh.STATE_I32}
    st["time"] = np.zeros(E)
    env.set_state(st)
    env.step(torch.zeros(E, 2, device="cuda:0"))
    got = trace.cpu().numpy()
    tol = 1e-9 if real64 else 2e-3
    # frame 0 sets the flags and impacts, frame 1 applies the impacts.  Later frames are left out: vehicles pushed
    # apart rest exactly against each other there, and such separating-axis ties may fall either way
    for e, c in enumerate(cases):
        o = oracle_module(cfg).OracleEnv(cfg)
        o.set_state(states[e])
        want = o.trace()
        o.step(np.zeros(2, np.float32))
        g, w = got[e, 0], want[0]
        assert np.array_equal(g[:, 6], w[:, 6]), (c, g[:, 6], w[:, 6])   # lane, target lane, crashed, has_impact
        np.testing.assert_allclose(g[:, [0, 1, 4, 5]], w[:, [0, 1, 4, 5]], atol=tol, err_msg=c)
        np.testing.assert_allclose(got[e, 1][:, :2], want[1][:, :2], atol=tol, err_msg=f"{c}, frame 1")
    env.close()


# ---- the fast step kernels next to the other ones ---------------------------------------------------------------------
@pytest.mark.parametrize("real64", [False, True], ids=["fp32", "fp64"])
def test_final_observation_equals_an_autoreset_0_twin(real64):
    E = 64
    rng = np.random.default_rng(2)
    cfg = _fast(duration=6)
    a_env = _vec(cfg, E, real64=real64, seed=1)
    b_env = _vec(cfg, E, real64=real64, seed=1, autoreset=False)
    a_env.reset(seed=4)
    fin = torch.full_like(a_env.obs, 7.0)
    finished = 0
    for t in range(14):
        b_env.set_state(a_env.get_state())
        fin.fill_(7.0)
        act = torch.tensor(rng.uniform(-1, 1, (E, 2)), dtype=torch.float32, device="cuda:0")
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


@pytest.mark.parametrize("real64", [False, True], ids=["fp32", "fp64"])
def test_fast_grid_handle_simulates_like_a_kinematics_twin(real64):
    E = 64
    rng = np.random.default_rng(1)
    g = _vec(_fast(observation={"type": "OccupancyGrid"}), E, real64=real64, seed=3)
    k = _vec(_fast(), E, real64=real64, seed=3)
    assert g.cfg.ego_collisions_only == k.cfg.ego_collisions_only == 1
    g.reset(seed=9)
    k.reset(seed=9)
    for t in range(30):
        a = torch.tensor(rng.uniform(-1, 1, (E, 2)), dtype=torch.float32, device="cuda:0")
        _, rg, teg, trg = g.step(a)
        _, rk, tek, trk = k.step(a)
        assert torch.equal(rg, rk) and torch.equal(teg, tek) and torch.equal(trg, trk), t
    sg, sk = g.get_state(), k.get_state()
    for key in sg:
        assert np.array_equal(sg[key], sk[key]), key
    g.close()
    k.close()


def test_captured_rollout_equals_eager():
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.routine import collect_rollout

    E, T = 128, 8
    runs = []
    for use_graph in (False, True):
        torch.manual_seed(0)
        env = _vec(_fast(meta=True), E, seed=2)
        agent = PPOAgent(env.N * env.F_out, 5, hidden_dim=64, batch_size=256, epochs=1, discrete=True)
        obs = env.reset(seed=2).clone()
        r = collect_rollout(env, agent, T, obs, use_graph=use_graph, bootstrap_truncated=True)
        runs.append({k: v.clone() for k, v in r.items()})
        env.close()
    for k in ("states", "action", "reward", "terminated", "truncated", "value"):
        if k in runs[0]:
            assert torch.equal(runs[0][k], runs[1][k]), k


def test_train_vectorized_categorical_with_evaluation(monkeypatch):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training import routine
    from highway_rope_ppo_b200.training.episodes import policy_steps

    handles = []
    make = routine.eval_env_for
    monkeypatch.setattr(routine, "eval_env_for", lambda vec_env, n: handles.append(make(vec_env, n)) or handles[-1])
    E, T = 256, 16
    env = _vec(_fast(meta=True), E, seed=5)
    torch.manual_seed(0)
    agent = PPOAgent(env.N * env.F_out, 5, hidden_dim=64, batch_size=512, epochs=2, discrete=True)
    hist = routine.train_vectorized(env, agent, 3, T, seed=5, bootstrap_truncated=True, eval_episodes=64,
                                    eval_interval=10)
    assert len(hist) == 3
    for m in hist:
        assert all(np.isfinite(m[k]) for k in ("loss", "policy_loss", "value_loss", "entropy"))
    assert np.isfinite(hist[0]["eval_return_mean"]) and 1 <= hist[0]["eval_length_mean"] <= 30
    (ev,) = handles
    assert ev.config["gym_id"] == FAST and ev.cfg.ego_collisions_only == 1
    steps = policy_steps(ev.config["duration"], ev.config["policy_frequency"])
    assert steps == policy_steps(30, 1) == 30
    assert ev.launches == 1 + steps   # one eager evaluation: a reset and 30 steps
    env.close()


def test_multiplexed_sweep_equals_sequential_and_groups_by_id(highway_config, tmp_path, monkeypatch):
    from highway_rope_ppo_b200.experiments import multiplex
    from highway_rope_ppo_b200.experiments.config import Condition, ConditionHP, Experiment
    from highway_rope_ppo_b200.experiments.runner import ExperimentRunner

    groups = []
    build = multiplex._Group.build
    monkeypatch.setattr(multiplex._Group, "build",
                        lambda self: groups.append((self.cfg.get("gym_id", "highway-v0"), len(self.slots))) or build(self))
    exps = []
    for i, (cond, over) in enumerate(((Condition.SORTED, {"gym_id": FAST}), (Condition.SORTED, {}),
                                      (Condition.SORTED, {"gym_id": FAST}))):
        hp = ConditionHP(lr=3e-4, hidden_dim=64, batch_size=32, epochs=2, steps_per_update=48)
        exps.append(Experiment(Experiment.make_name(cond, hp, 42 + i) + f"_fast{i}", cond, hp, seed=42 + i,
                               max_episodes=3, env_config_overrides=over, extra={"eval_interval": 3, "log_interval": 1}))
    seq = [ExperimentRunner(copy.deepcopy(highway_config), artifacts_dir=str(tmp_path / "seq")).launch(e) for e in exps]
    mux = multiplex.MultiplexedRunner(copy.deepcopy(highway_config), artifacts_dir=str(tmp_path / "mux"),
                                      max_concurrent=4).launch_many(exps)
    for a, b in zip(seq, mux):
        assert a["status"] == b["status"] == "COMPLETED", (a.get("error_traceback"), b.get("error_traceback"))
        assert a["rewards"] == b["rewards"] and a["avg_rewards"] == b["avg_rewards"]
        ua, ub = a["metrics_history"]["policy_updates"], b["metrics_history"]["policy_updates"]
        assert len(ua) == len(ub)
        for x, y in zip(ua, ub):
            assert {k: v for k, v in x.items() if k != "time"} == {k: v for k, v in y.items() if k != "time"}
    assert sorted(groups) == [("highway-fast-v0", 2), ("highway-v0", 1)]
