"""GPU checks of the episode statistics (hrp_episode_stats), the training statistics of train_vectorized, the batched
deterministic evaluation (evaluate_vectorized) and the best checkpoint.

* The kernel equals the fp64 oracle (oracle/episode_stats.py): per-env carries bit for bit, counts exact, sums within
  1e-12; repeated calls give the same bits, a rollout split in two calls gives the same carries and counts, evaluation
  mode likewise, and a captured-graph replay equals the eager call.
* train_vectorized's statistics do not perturb training (parameters and Adam moments bit-identical to a plain
  rollout_and_update loop) and equal the oracle over the rollouts it collected.
* evaluate_vectorized: every env finishes within the time limit; per-episode returns and lengths are bit-identical to an
  eager loop on an unmasked autoreset = 0 twin; sorted first observations equal single-env reset(seed=exp_seed+1000+e);
  two half-size shards reproduce one handle; graph replay equals eager; the training handle is not touched; a RankPE
  evaluation handle uses the training table.
"""
import copy

import numpy as np
import pytest
import torch

from oracle import episode_stats as es

pytestmark = pytest.mark.gpu


def _launch(r, te, tr, ret, ln, stats, active=None):
    from highway_rope_ppo_b200.training.episodes import episode_stats

    episode_stats(r, te, tr, ret, ln, stats, active=active)


def _inputs(T, E, density, seed):
    rng = np.random.default_rng(seed)
    r = rng.normal(size=(T, E)).astype(np.float32)
    if density >= 1.0:
        te = rng.random((T, E)) < 0.5
        tr = ~te | (rng.random((T, E)) < 0.3)         # every step ends an episode, some both ways
    else:
        te = rng.random((T, E)) < density * 0.5
        tr = rng.random((T, E)) < density * 0.6
    ret0 = rng.normal(size=E) * 3.0
    len0 = rng.integers(0, 30, E).astype(np.int32)
    return r, te.astype(np.uint8), tr.astype(np.uint8), ret0, len0


def _dev(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _check_sums(got, want):
    np.testing.assert_array_equal(got[[0, 3, 4, 5]], want[[0, 3, 4, 5]])
    np.testing.assert_allclose(got[[1, 2]], want[[1, 2]], rtol=1e-12, atol=1e-12 * max(1.0, float(want[0])))


SHAPES = [(1, 1), (1, 4096), (32, 4096), (50, 17), (2048, 33), (7, 65536)]


@pytest.mark.parametrize("T,E", SHAPES, ids=[f"T{t}-E{e}" for t, e in SHAPES])
@pytest.mark.parametrize("density", [0.0, 0.03, 1.0], ids=["none", "3pct", "all"])
@pytest.mark.parametrize("evaluation", [False, True], ids=["train", "eval"])
def test_kernel_matches_oracle(T, E, density, evaluation):
    from highway_rope_ppo_b200.training.episodes import new_stats

    r, te, tr, ret0, len0 = _inputs(T, E, density, seed=T * 7 + E + int(density * 100))
    act0 = (np.random.default_rng(E).random(E) < 0.8).astype(np.uint8) if evaluation else None
    want_ret, want_len, want_act, want = es.episode_stats(r, te, tr, ret0, len0, act0)
    dr, dte, dtr = _dev(r, te, tr)

    def run(splits=(T,)):
        ret, ln = _dev(ret0.copy(), len0.copy())
        act = None if act0 is None else _dev(act0.copy())[0]
        stats = new_stats("cuda:0")
        t0 = 0
        for n in splits:
            _launch(dr[t0:t0 + n], dte[t0:t0 + n], dtr[t0:t0 + n], ret, ln, stats, act)
            t0 += n
        torch.cuda.synchronize()
        return ret.cpu().numpy(), ln.cpu().numpy(), None if act is None else act.cpu().numpy(), stats[:6].cpu().numpy()

    got_ret, got_len, got_act, got = run()
    assert np.array_equal(got_ret.view(np.uint64), want_ret.view(np.uint64))   # bit for bit, -0.0 included
    np.testing.assert_array_equal(got_len, want_len)
    if evaluation:
        np.testing.assert_array_equal(got_act, want_act)
    _check_sums(got, want)
    again = run()
    for a, b in zip(again, (got_ret, got_len, got_act, got)):
        assert (a is None and b is None) or a.tobytes() == b.tobytes()
    if T > 1:
        half = run((T // 2, T - T // 2))
        assert half[0].tobytes() == got_ret.tobytes() and np.array_equal(half[1], got_len)
        if evaluation:
            np.testing.assert_array_equal(half[2], got_act)
        _check_sums(half[3], want)


@pytest.mark.parametrize("evaluation", [False, True], ids=["train", "eval"])
def test_graph_replay_equals_eager(evaluation):
    from highway_rope_ppo_b200.training.episodes import new_stats

    T, E = 32, 4096
    r, te, tr, ret0, len0 = _inputs(T, E, 0.03, seed=3)
    dr, dte, dtr = _dev(r, te, tr)
    act0 = np.ones(E, dtype=np.uint8)
    res = []
    for graphed in (False, True):
        ret, ln, act = _dev(ret0.copy(), len0.copy(), act0.copy())
        act = act if evaluation else None
        stats = new_stats("cuda:0")
        if graphed:
            g = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                g.capture_begin()
                _launch(dr, dte, dtr, ret, ln, stats, act)
                g.capture_end()
            torch.cuda.current_stream().wait_stream(side)
            g.replay()
        else:
            _launch(dr, dte, dtr, ret, ln, stats, act)
        torch.cuda.synchronize()
        res.append([x.cpu().numpy().tobytes() for x in (ret, ln, stats[:6])])
    assert res[0] == res[1]


# ------------------------------------------------------------------------------------------------ training statistics
def _train_setup(highway_config, discrete, E, seed=7):
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_vec_env
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    torch.manual_seed(4)
    np.random.seed(4)
    cfg = copy.deepcopy(highway_config)
    cfg["duration"] = 6
    if discrete:
        cfg["action"] = {"type": "DiscreteMetaAction"}
    env = make_vec_env(Condition.SORTED, cfg, num_envs=E, seed=seed)
    agent = PPOAgent(env.N * env.F_out, 5 if discrete else 2, hidden_dim=64, batch_size=256, epochs=2,
                     discrete=discrete)
    return env, agent


@pytest.mark.parametrize("discrete", [False, True], ids=["gaussian", "categorical-meta"])
def test_training_statistics_do_not_perturb_training_and_match_oracle(highway_config, discrete, monkeypatch):
    from highway_rope_ppo_b200.training import routine
    from highway_rope_ppo_b200.training.episodes import summarize

    E, T, iters, seed = 512, 8, 3, 7
    env, agent = _train_setup(highway_config, discrete, E, seed)
    obs = env.reset(seed=seed)
    for _ in range(iters):
        _, obs = routine.rollout_and_update(env, agent, T, obs=obs)
    want = [agent.actor_critic.flat.clone(), agent.optimizer.exp_avg.clone(), agent.optimizer.exp_avg_sq.clone()]
    env.close()

    env, agent = _train_setup(highway_config, discrete, E, seed)
    recorded = []
    real = routine.collect_rollout

    def recording(*a, **kw):
        r = real(*a, **kw)
        recorded.append([r[k].cpu().numpy() for k in ("reward", "terminated", "truncated")])
        return r

    monkeypatch.setattr(routine, "collect_rollout", recording)
    hist = routine.train_vectorized(env, agent, iters, T, seed=seed)
    got = [agent.actor_critic.flat, agent.optimizer.exp_avg, agent.optimizer.exp_avg_sq]
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    ret, ln = np.zeros(E), np.zeros(E, dtype=np.int32)
    total = 0
    for m, (r, te, tr) in zip(hist, recorded):
        ret, ln, _, st = es.episode_stats(r, te, tr, ret, ln)
        s = summarize(st)
        assert m["episodes"] == s["episodes"] and s["episodes"] > 0
        for k, mk in (("return_mean", "episode_return_mean"), ("return_std", "episode_return_std"),
                      ("length_mean", "episode_length_mean"), ("terminated_fraction", "terminated_fraction")):
            assert abs(m[mk] - s[k]) <= 1e-12 * max(1.0, abs(s[k])), (mk, m[mk], s[k])
        total += s["episodes"]
    assert len(hist) == iters and "loss" in hist[0] and "samples_per_s" in hist[0] and "eval_return_mean" not in hist[0]
    print("training episodes", total)
    env.close()


# ------------------------------------------------------------------------------------------------ evaluation
def _eval_cfg(highway_config, kind):
    cfg = copy.deepcopy(highway_config)
    if kind == "meta":
        cfg["action"] = {"type": "DiscreteMetaAction"}
    elif kind == "short":
        cfg.update(duration=3, policy_frequency=2, offroad_terminal=True)
    return cfg


def _agent_for(env, discrete, hidden=64):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    torch.manual_seed(9)
    return PPOAgent(env.N * env.F_out, 5 if discrete else 2, hidden_dim=hidden, batch_size=256, discrete=discrete)


def _twin_reference(cfg, agent, K, exp_seed, env_id_base, embed=None):
    """Eager loop on an unmasked autoreset = 0 handle with the same per-env seeds and the same deterministic actions;
    the first episode of every env is booked in numpy (the reference's `total += reward` in Python floats)."""
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.training.episodes import policy_steps

    twin = HighwayVecEnv(cfg, K, device="cuda:0", embed=embed, autoreset=False, env_id_base=env_id_base)
    seeds = torch.arange(K, dtype=torch.int64, device="cuda:0") + exp_seed + 1000 + env_id_base
    twin.set_env_seeds(seeds)
    obs = twin.reset().clone()
    steps = policy_steps(twin.config["duration"], twin.config["policy_frequency"])
    ret, ln, live = [0.0] * K, np.zeros(K, dtype=np.int32), np.ones(K, dtype=bool)
    for _ in range(steps):
        out = agent.act(obs.view(K, -1), deterministic=True)
        o, r, te, tr = twin.step(out["action"])
        obs = o.clone()
        r, done = r.cpu().numpy(), ((te | tr) != 0).cpu().numpy()
        for e in np.flatnonzero(live):
            ret[e] += float(r[e])
            ln[e] += 1
            if done[e]:
                live[e] = False
    assert not live.any()
    twin.close()
    return np.array(ret), ln


@pytest.mark.parametrize("kind,K", [("default", 1), ("default", 17), ("default", 4096), ("meta", 4096),
                                    ("short", 4096), ("meta", 17)])
def test_evaluation_matches_eager_twin(highway_config, kind, K):
    from highway_rope_ppo_b200.envs.highway_env import HighwayEnv
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.training.episodes import policy_steps
    from highway_rope_ppo_b200.training.routine import evaluate_vectorized

    cfg = _eval_cfg(highway_config, kind)
    env = HighwayVecEnv(cfg, K, device="cuda:0", autoreset=False)
    agent = _agent_for(env, kind == "meta")
    exp_seed = 3
    steps = policy_steps(env.config["duration"], env.config["policy_frequency"])
    assert steps == {"default": 40, "meta": 40, "short": 6}[kind]
    runs = [evaluate_vectorized(env, agent, exp_seed=exp_seed) for _ in range(3)]   # eager, capture + replay, replay
    runs.append(evaluate_vectorized(env, agent, exp_seed=exp_seed, use_graph=False))
    ev = runs[0]
    assert ev["episodes"] == K and (ev["lengths"] >= 1).all() and (ev["lengths"] <= steps).all()
    for other in runs[1:]:
        assert other["returns"].tobytes() == ev["returns"].tobytes()
        assert np.array_equal(other["lengths"], ev["lengths"]) and other["mean"] == ev["mean"]
    want_ret, want_len = _twin_reference(cfg, agent, K, exp_seed, 0)
    assert ev["returns"].tobytes() == want_ret.tobytes()
    np.testing.assert_array_equal(ev["lengths"], want_len)
    assert abs(ev["mean"] - want_ret.mean()) <= 1e-12 * max(1.0, abs(want_ret.mean()))
    assert abs(ev["std"] - want_ret.std()) <= 1e-9 * max(1.0, want_ret.std())
    assert ev["min"] == want_ret.min() and ev["max"] == want_ret.max()
    assert abs(ev["length_mean"] - want_len.mean()) < 1e-12
    if kind == "short":
        assert ev["terminated_fraction"] > 0   # crashes and off-road episodes end by termination
    # sorted order: the first observations are those of single-env reset(seed=exp_seed + 1000 + e)
    first = env.reset().cpu().numpy()
    single = HighwayEnv(cfg)
    for e in sorted({0, min(1, K - 1), K // 2, K - 1}):
        o, _ = single.reset(seed=exp_seed + 1000 + e)
        assert np.array_equal(np.asarray(o, dtype=np.float32), first[e]), e
    single.close()
    print(kind, K, "eval return", ev["mean"], "+-", ev["std"], "length", ev["length_mean"],
          "terminated", ev["terminated_fraction"])
    env.close()


def test_half_shards_reproduce_one_handle(highway_config):
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.training.routine import evaluate_vectorized

    K = 4096
    whole = HighwayVecEnv(highway_config, K, device="cuda:0", autoreset=False)
    agent = _agent_for(whole, False)
    want = evaluate_vectorized(whole, agent, exp_seed=5)
    parts = []
    for base in (0, K // 2):
        h = HighwayVecEnv(highway_config, K // 2, device="cuda:0", autoreset=False, env_id_base=base)
        parts.append(evaluate_vectorized(h, agent, exp_seed=5))
        h.close()
    got = np.concatenate([p["returns"] for p in parts])
    assert got.tobytes() == want["returns"].tobytes()
    np.testing.assert_array_equal(np.concatenate([p["lengths"] for p in parts]), want["lengths"])
    whole.close()


def test_evaluation_leaves_training_handle_alone_and_rankpe_shares_the_table(highway_config):
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_vec_env
    from highway_rope_ppo_b200.training.routine import eval_env_for, evaluate_vectorized

    torch.manual_seed(2)
    over = {"observation": {"order": "shuffled"}}
    train = make_vec_env(Condition.SHUFFLED_RANKPE, highway_config, 4, over, num_envs=256, seed=1, env_id_base=256)
    train.reset(seed=1)
    before = train.get_state()
    rng_before = torch.get_rng_state()
    ev_env = eval_env_for(train, 128)
    assert torch.equal(torch.get_rng_state(), rng_before)   # no new RankPE table drawn
    assert ev_env.embed is train.embed and ev_env.embed.table is train.embed.table
    assert ev_env.env_id_base == 128 and ev_env.num_envs == 128 and ev_env.config == train.config
    agent = _agent_for(train, False)
    ev = evaluate_vectorized(ev_env, agent, exp_seed=0)
    assert ev["episodes"] == 128
    after = train.get_state()
    for k in before:
        assert np.array_equal(before[k], after[k]), k
    # the evaluation handle observes through the training table: same state, same observation
    probe = make_vec_env(Condition.SHUFFLED_RANKPE, highway_config, 4, over, num_envs=128, seed=1)
    assert not np.array_equal(probe.embed.table, train.embed.table)
    ev_env.close()
    probe.close()
    train.close()


def test_best_checkpoint_written_only_on_improvement(highway_config, tmp_path, monkeypatch):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.routine import train_vectorized

    env, agent = _train_setup(highway_config, False, 256)
    path = str(tmp_path / "best.pth")
    saves = []
    real = agent.save

    def save(p):
        saves.append((p, agent.actor_critic.flat.clone()))
        real(p)

    monkeypatch.setattr(agent, "save", save)
    hist = train_vectorized(env, agent, 6, 8, seed=7, eval_episodes=64, eval_interval=2, best_checkpoint=path)
    means = [m.get("eval_return_mean") for m in hist]
    assert [m is not None for m in means] == [True, False, True, False, True, False]
    evals = [m for m in means if m is not None]
    improved = [i for i, m in enumerate(evals) if m > max(evals[:i], default=-np.inf)]
    assert len(saves) == len(improved) >= 1 and all(p == path for p, _ in saves)
    for m in hist[::2]:
        assert m["eval_length_mean"] <= 6 and 0 <= m["eval_terminated_fraction"] <= 1 and m["eval_return_std"] >= 0
    fresh = PPOAgent(env.N * env.F_out, 2, hidden_dim=64, batch_size=256)
    fresh.load(path)
    assert torch.equal(fresh.actor_critic.flat, saves[-1][1])
    env.close()
