"""GPU checks of running observation / reward normalization (``VecNormalize``, csrc/hrp_norm.cu):

* the kernels against the numpy restatement of SB3 (tests/vecnormalize_oracle.py) over step sequences with random dones,
  from one env and 60 columns to 16 384 envs and to the largest Kinematics output (4608 columns), with a column offset
  by 1e4 of its spread at the first update: running mean / var within 1e-12 relative, counts within 1e-12, the return
  carry bit for bit, normalized values within 2 float32 ulps and exactly +-clip where clipped;
* on real handles (Kinematics, OccupancyGrid, highway-fast-v0): the wrapper does not touch the simulation, and its
  observations, rewards and terminal observations follow the oracle;
* a captured rollout equals an eager one bit for bit, frozen evaluation, and train_vectorized with the wrapper.
"""
import copy
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import episode_stats as es
from test_env_gpu import _cfg, _vec
from test_fast_env_cpu import FAST
from vecnormalize_oracle import VecNormOracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _ulps(got, want):
    """|got - want| in float32 ulps of want"""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    return np.abs(got.astype(np.float64) - want.astype(np.float64)) / np.spacing(np.abs(want)).astype(np.float64)


def _check_normalized(got, want, clip):
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    clipped = np.abs(want) == np.float32(clip)
    assert np.array_equal(got[clipped], want[clipped]), "clipped values must be exactly +-clip"
    u = _ulps(got[~clipped], want[~clipped])
    assert u.size == 0 or u.max() <= 2, u.max()


def _check_stats(w, o):
    mean, var = w.obs_rms.mean.cpu().numpy(), w.obs_rms.var.cpu().numpy()
    np.testing.assert_allclose(mean, o.obs_rms.mean, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(var, o.obs_rms.var, rtol=1e-12, atol=1e-15)
    assert abs(float(w.obs_rms.count) - o.obs_rms.count) <= 1e-12 * o.obs_rms.count
    np.testing.assert_allclose(float(w.ret_rms.mean), o.ret_rms.mean, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(float(w.ret_rms.var), o.ret_rms.var, rtol=1e-12, atol=1e-15)
    assert abs(float(w.ret_rms.count) - o.ret_rms.count) <= 1e-12 * o.ret_rms.count
    assert np.array_equal(w.returns.cpu().numpy(), o.returns), "return carry"


class _ScriptedEnv:
    """A stand-in for a HighwayVecEnv whose steps return prepared observations, rewards and flags."""

    def __init__(self, E, S):
        self.num_envs, self.N, self.F_out, self.obs_shape, self.device = E, 1, S, (1, S), DEV
        self.obs = torch.zeros((E, 1, S), dtype=torch.float32, device=DEV)
        self.reward = torch.zeros(E, dtype=torch.float32, device=DEV)
        self.terminated = torch.zeros(E, dtype=torch.uint8, device=DEV)
        self.truncated = torch.zeros(E, dtype=torch.uint8, device=DEV)
        self.next = None

    def reset(self, seed=None, mask=None, out=None):
        o = self.obs if out is None else out
        o.copy_(self.next["obs"])
        return o

    def observe(self, perm=None, row_vehicle=None, out=None):
        return self.obs if out is None else out

    def step(self, actions, perm=None, row_vehicle=None, out=None, reward_out=None, terminated_out=None,
             truncated_out=None, final_obs_out=None):
        n = self.next
        o = self.obs if out is None else out
        r = self.reward if reward_out is None else reward_out
        te = self.terminated if terminated_out is None else terminated_out
        tr = self.truncated if truncated_out is None else truncated_out
        o.copy_(n["obs"]); r.copy_(n["reward"]); te.copy_(n["terminated"]); tr.copy_(n["truncated"])
        if final_obs_out is not None:
            d = (n["terminated"] | n["truncated"]).bool()
            final_obs_out.view(self.num_envs, -1)[d] = n["final"].view(self.num_envs, -1)[d]
        return o, r, te, tr


def _draw(rng, E, S, first):
    spread = rng.uniform(0.1, 3.0, S)
    centre = rng.normal(0, 2, S)
    if first:
        centre[0] = 1e4 * spread[0]      # a column far from the running mean 0 at the first update
    obs = (centre + spread * rng.standard_normal((E, S))).astype(np.float32)
    obs[:, 1] = rng.choice([0.0, 1.0, 50.0], E)   # values that clip
    p = 0.1
    return {"obs": obs, "reward": (rng.uniform(-1, 1, E) * rng.choice([1, 30], E)).astype(np.float32),
            "terminated": (rng.random(E) < p).astype(np.uint8), "truncated": (rng.random(E) < p).astype(np.uint8),
            "final": (centre + spread * rng.standard_normal((E, S))).astype(np.float32)}


FLAGS = {"obs+reward": (True, True), "reward only": (False, True), "obs only": (True, False), "off": (False, False)}


@pytest.mark.parametrize("flags", list(FLAGS))
@pytest.mark.parametrize("E,S", [(1, 60), (33, 60), (4096, 60), (4097, 484), (16384, 600), (256, 4608)])
def test_kernels_match_the_oracle(E, S, flags):
    """Also with either part switched off: the S = 0 launches (reward only), the merge without a return column (obs
    only) and the pass-through with both off."""
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize

    norm_obs, norm_reward = FLAGS[flags]
    rng = np.random.default_rng(E * 7919 + S)
    env = _ScriptedEnv(E, S)
    kw = dict(norm_obs=norm_obs, norm_reward=norm_reward, clip_obs=5.0, clip_reward=3.0, gamma=0.97)
    w = VecNormalize(env, **kw)
    o = VecNormOracle(E, (1, S), **kw)
    d = _draw(rng, E, S, True)
    env.next = {"obs": torch.from_numpy(d["obs"]).view(E, 1, S).to(DEV)}
    got = w.reset().cpu().numpy()
    want = o.reset(d["obs"].reshape(E, 1, S))
    _check_normalized(got, want, 5.0)
    _check_stats(w, o)
    final = torch.full((E, 1, S), 7.0, dtype=torch.float32, device=DEV)
    acts = torch.zeros((E, 2), dtype=torch.float32, device=DEV)
    raw = torch.empty(E, dtype=torch.float32, device=DEV)
    rout = torch.empty(E, dtype=torch.float32, device=DEV)
    for t in range(5):
        d = _draw(rng, E, S, False)
        env.next = {k: torch.from_numpy(v).to(DEV) for k, v in d.items()}
        env.next["obs"] = env.next["obs"].view(E, 1, S)
        before = final.cpu().numpy()
        obs, rew, te, tr = w.step(acts, final_obs_out=final, raw_reward_out=raw, reward_out=rout)
        assert rew is rout
        want_obs, want_rew, want_fin = o.step(d["obs"].reshape(E, 1, S), d["reward"], d["terminated"], d["truncated"],
                                              final_obs=np.where((d["terminated"] | d["truncated"])[:, None, None],
                                                                 d["final"].reshape(E, 1, S), before))
        _check_normalized(obs.cpu().numpy(), want_obs, 5.0)
        _check_normalized(rew.cpu().numpy(), want_rew, 3.0)
        _check_normalized(final.cpu().numpy(), want_fin, 5.0)
        assert np.array_equal(raw.cpu().numpy(), d["reward"])
        _check_stats(w, o)


@pytest.mark.parametrize("E0,E1,S", [(1, 33, 60), (4096, 4096, 484), (4097, 1024, 4608)])
def test_merge_of_two_shards_matches_one_batch(E0, E1, S):
    """hrp_vecnorm_moments on two shards, their moment blocks in rank order into hrp_vecnorm_merge (R = 2, as a sharded
    run all-gathers them): the statistics of one batch over both shards, within the oracle's tolerances, over two
    steps."""
    from highway_rope_ppo_b200 import _lib
    from vecnormalize_oracle import RunningMeanStd

    lib, st = _lib.load(), torch.cuda.current_stream(DEV).cuda_stream
    C = S + 1
    rng = np.random.default_rng(E0 + E1 + S)
    rets = [torch.zeros(E, dtype=torch.float64, device=DEV) for E in (E0, E1)]
    moms = [torch.zeros(_lib.vecnorm_moments_len(C), dtype=torch.float64, device=DEV) for _ in range(2)]
    scratch = [torch.zeros(_lib.vecnorm_scratch_len(C), dtype=torch.float64, device=DEV) for _ in range(2)]
    obs_rms = torch.zeros(2 * S + 1, dtype=torch.float64, device=DEV)
    obs_rms[S:2 * S] = 1.0
    obs_rms[2 * S] = 1e-4
    ret_rms = torch.tensor([0.0, 1.0, 1e-4], dtype=torch.float64, device=DEV)
    o_obs, o_ret, o_returns = RunningMeanStd(shape=(S,)), RunningMeanStd(shape=()), np.zeros(E0 + E1)
    for step in range(2):
        d = _draw(rng, E0 + E1, S, step == 0)
        obs, rew = torch.from_numpy(d["obs"]).to(DEV), torch.from_numpy(d["reward"]).to(DEV)
        for k, (lo, hi) in enumerate(((0, E0), (E0, E0 + E1))):
            _lib.check(lib.hrp_vecnorm_moments(obs[lo:hi].data_ptr(), hi - lo, S, rew[lo:hi].data_ptr(),
                                               rets[k].data_ptr(), 0.99, moms[k].data_ptr(), scratch[k].data_ptr(), st))
        gathered = torch.cat(moms)
        _lib.check(lib.hrp_vecnorm_merge(gathered.data_ptr(), 2, S, 1, obs_rms.data_ptr(), ret_rms.data_ptr(),
                                         scratch[0].data_ptr(), st))
        o_obs.update(d["obs"])
        o_returns = o_returns * 0.99 + d["reward"].astype(np.float64)
        o_ret.update(o_returns)
        got = obs_rms.cpu().numpy()
        np.testing.assert_allclose(got[:S], o_obs.mean, rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(got[S:2 * S], o_obs.var, rtol=1e-12, atol=1e-15)
        assert abs(got[2 * S] - o_obs.count) <= 1e-12 * o_obs.count
        r = ret_rms.cpu().numpy()
        np.testing.assert_allclose(r[:2], [o_ret.mean, o_ret.var], rtol=1e-12, atol=1e-15)
        assert abs(r[2] - o_ret.count) <= 1e-12 * o_ret.count
        assert np.array_equal(torch.cat(rets).cpu().numpy(), o_returns)


def _configs(highway_config):
    short = _cfg(highway_config, duration=3)   # truncations within the test's steps
    grid = copy.deepcopy(short)
    grid["observation"] = {"type": "OccupancyGrid"}
    fast = {"gym_id": FAST, "duration": 4, "action": {"type": "ContinuousAction"}}
    return {"kinematics": short, "grid": grid, "fast": fast}


@pytest.mark.parametrize("kind", ["kinematics", "grid", "fast"])
def test_real_handles_simulation_untouched_and_oracle(highway_config, kind):
    """A wrapped and an unwrapped twin stepped with the same actions hold bit-identical states, raw rewards and flags;
    the wrapper's observations, rewards and terminal observations follow the oracle fed with the twin's raw outputs."""
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize

    cfg = _configs(highway_config)[kind]
    E, seed = 512, 3
    plain, inner = _vec(cfg, E, seed=seed), _vec(cfg, E, seed=seed)
    w = VecNormalize(inner)
    o = VecNormOracle(E, plain.obs_shape)
    raw_obs = plain.reset(seed=seed).cpu().numpy()
    _check_normalized(w.reset(seed=seed).cpu().numpy(), o.reset(raw_obs), 10.0)
    shape = (E,) + tuple(plain.obs_shape)
    fin_p = torch.zeros(shape, dtype=torch.float32, device=DEV)
    fin_w = torch.zeros(shape, dtype=torch.float32, device=DEV)
    raw = torch.empty(E, dtype=torch.float32, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(1)
    dones = 0
    for t in range(8):
        a = torch.rand((E, 2), generator=g, device=DEV) * 2 - 1
        before = fin_w.cpu().numpy()
        po, pr, pte, ptr = plain.step(a, final_obs_out=fin_p)
        wo, wr, wte, wtr = w.step(a, final_obs_out=fin_w, raw_reward_out=raw)
        sw = inner.get_state()
        for k, v in plain.get_state().items():
            assert np.array_equal(v, sw[k]), (t, k)
        assert torch.equal(raw, pr) and torch.equal(wte, pte) and torch.equal(wtr, ptr)
        te, tr = pte.cpu().numpy(), ptr.cpu().numpy()
        done = (te | tr).astype(bool)
        dones += int(done.sum())
        fin = np.where(done.reshape((E,) + (1,) * len(plain.obs_shape)), fin_p.cpu().numpy(), before)
        want_obs, want_rew, want_fin = o.step(po.cpu().numpy(), pr.cpu().numpy(), te, tr, final_obs=fin)
        _check_normalized(wo.cpu().numpy(), want_obs, 10.0)
        _check_normalized(wr.cpu().numpy(), want_rew, 10.0)
        _check_normalized(fin_w.cpu().numpy(), want_fin, 10.0)
        _check_stats(w, o)
    assert dones > 0
    plain.close()
    w.close()


def _wrapped_setup(cfg, E, seed, discrete, hidden=64, **wkw):
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    w = VecNormalize(_vec(cfg, E, seed=seed), **wkw)
    torch.manual_seed(seed)
    agent = PPOAgent(w.N * w.F_out, 5 if discrete else 2, lr=3e-4, hidden_dim=hidden, batch_size=512, epochs=2,
                     discrete=discrete)
    return w, agent


@pytest.mark.parametrize("boot", [False, True], ids=["plain", "bootstrap_truncated"])
def test_captured_rollout_equals_eager(highway_config, boot):
    from highway_rope_ppo_b200.training.routine import collect_rollout

    cfg = _configs(highway_config)["kinematics"]
    E, T, seed = 256, 6, 4
    runs = []
    for use_graph in (False, True):
        w, agent = _wrapped_setup(cfg, E, seed, False)
        obs = w.reset(seed=seed).clone()
        out = []
        for _ in range(3):   # eager, captured + replayed, replayed
            r = collect_rollout(w, agent, T, obs, use_graph=use_graph, bootstrap_truncated=boot)
            out.append({k: v.clone() for k, v in r.items()})
            obs = r["states"][T].clone()
        out.append({"obs_rms": w.obs_rms.buf.clone(), "ret_rms": w.ret_rms.buf.clone(), "returns": w.returns.clone()})
        runs.append(out)
        if use_graph:
            assert agent._rollout_graph["graph"] is not None
        w.close()
    for a, b in zip(*runs):
        for k in a:
            assert torch.equal(a[k], b[k]), k
    assert "reward_raw" in runs[0][0] and not torch.equal(runs[0][0]["reward"], runs[0][0]["reward_raw"])


def test_bootstrapped_rollout_matches_the_oracle(highway_config):
    """collect_rollout(bootstrap_truncated=True) on a wrapper: replaying the rollout's actions on an unwrapped twin and
    feeding its raw outputs to the oracle gives the rollout's normalized states, rewards and, at the rows of envs done
    at step t, final_states[t]."""
    from highway_rope_ppo_b200.training.routine import collect_rollout

    cfg = _configs(highway_config)["kinematics"]
    E, T, seed = 256, 7, 6
    w, agent = _wrapped_setup(cfg, E, seed, False)
    plain = _vec(cfg, E, seed=seed)
    o = VecNormOracle(E, plain.obs_shape)
    obs = w.reset(seed=seed).clone()
    _check_normalized(obs.cpu().numpy(), o.reset(plain.reset(seed=seed).cpu().numpy()), 10.0)
    r = collect_rollout(w, agent, T, obs, bootstrap_truncated=True)
    shape = (E,) + tuple(plain.obs_shape)
    fin = torch.zeros(shape, dtype=torch.float32, device=DEV)
    dones = 0
    for t in range(T):
        po, pr, pte, ptr = plain.step(r["action"][t], final_obs_out=fin)
        te, tr = pte.cpu().numpy(), ptr.cpu().numpy()
        done = (te | tr).astype(bool)
        dones += int(done.sum())
        want_obs, want_rew, want_fin = o.step(po.cpu().numpy(), pr.cpu().numpy(), te, tr, final_obs=fin.cpu().numpy())
        _check_normalized(r["states"][t + 1].view(shape).cpu().numpy(), want_obs, 10.0)
        _check_normalized(r["reward"][t].cpu().numpy(), want_rew, 10.0)
        assert torch.equal(r["reward_raw"][t], pr)
        _check_normalized(r["final_states"][t].view(shape).cpu().numpy()[done], want_fin[done], 10.0)
    assert dones > 0
    plain.close()
    w.close()


def test_frozen_evaluation(highway_config):
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize
    from highway_rope_ppo_b200.training import routine
    from highway_rope_ppo_b200.training.episodes import policy_steps

    cfg = _cfg(highway_config, duration=6)
    E, T, K, seed = 256, 4, 128, 11
    w, agent = _wrapped_setup(cfg, E, seed, False)
    obs = w.reset(seed=seed)
    for _ in range(2):
        r = routine.collect_rollout(w, agent, T, obs)
        obs = r["states"][T].clone()
    ev = routine.eval_env_for(w, K)
    assert isinstance(ev, VecNormalize) and not ev.training and not ev.norm_reward and ev.obs_rms is w.obs_rms
    stats = (w.obs_rms.buf.clone(), w.ret_rms.buf.clone())
    res = [routine.evaluate_vectorized(ev, agent, exp_seed=seed) for _ in range(3)]   # eager, captured, replayed
    assert torch.equal(stats[0], w.obs_rms.buf) and torch.equal(stats[1], w.ret_rms.buf)
    for x in res[1:]:
        assert np.array_equal(x["returns"], res[0]["returns"])
    # an eager loop on an unmasked autoreset=0 twin wrapped with the same statistics
    twin = VecNormalize(_vec(cfg, K, seed=seed, autoreset=False, env_id_base=ev.env_id_base), training=False,
                        norm_reward=False)
    twin.share_statistics(w)
    base = seed + 1000 + ev.env_id_base
    twin.set_env_seeds(torch.arange(base, base + K, dtype=torch.int64, device=DEV))
    o = twin.reset()
    ret, active = np.zeros(K), np.ones(K, bool)
    for _ in range(policy_steps(ev.config["duration"], ev.config["policy_frequency"])):
        a = agent.act(o.view(K, -1).contiguous(), deterministic=True)["action"]
        o, rew, te, tr = twin.step(a)
        rew, done = rew.cpu().numpy(), (te | tr).cpu().numpy().astype(bool)
        ret[active] += rew[active].astype(np.float64)
        active &= ~done
        o = o.clone()
    assert not active.any()
    assert np.array_equal(ret, res[0]["returns"])
    ev.close()
    twin.close()
    w.close()


@pytest.mark.parametrize("kind", ["gaussian-reference", "categorical-fast"])
def test_train_vectorized_with_the_wrapper(highway_config, kind, tmp_path, monkeypatch):
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize
    from highway_rope_ppo_b200.training import routine
    from highway_rope_ppo_b200.training.episodes import summarize

    discrete = kind.startswith("categorical")
    cfg = {"gym_id": FAST, "action": {"type": "DiscreteMetaAction"}} if discrete else copy.deepcopy(highway_config)
    E, T, iters, seed = 256, 8, 3, 5
    real = routine.collect_rollout
    runs = []
    for run in range(2):
        recorded = []

        def recording(*a, **kw):
            r = real(*a, **kw)
            recorded.append([r[k].cpu().numpy() for k in ("reward_raw", "terminated", "truncated")])
            return r

        monkeypatch.setattr(routine, "collect_rollout", recording)
        w, agent = _wrapped_setup(cfg, E, seed, discrete)
        ckpt = str(tmp_path / f"best{run}.pth")
        np.random.seed(0)
        hist = routine.train_vectorized(w, agent, iters, T, seed=seed, eval_episodes=64, eval_interval=2,
                                        best_checkpoint=ckpt)
        ret, ln = np.zeros(E), np.zeros(E, dtype=np.int32)
        for m, (r, te, tr) in zip(hist, recorded):
            ret, ln, _, st = es.episode_stats(r, te, tr, ret, ln)
            s = summarize(st)
            assert m["episodes"] == s["episodes"]
            if s["episodes"]:
                for k, mk in (("return_mean", "episode_return_mean"), ("return_std", "episode_return_std"),
                              ("length_mean", "episode_length_mean")):
                    assert abs(m[mk] - s[k]) <= 1e-12 * max(1.0, abs(s[k])), (mk, m[mk], s[k])
        assert sorted(torch.load(ckpt, map_location="cpu")) == ["model", "optimizer"]
        loaded = VecNormalize.load(ckpt + ".vecnormalize", _vec(cfg, E, seed=seed))
        saved = torch.load(ckpt + ".vecnormalize", map_location="cpu")
        assert torch.equal(loaded.obs_rms.mean.cpu(), saved["obs_mean"]) and float(loaded.ret_rms.var) == saved["ret_var"]
        runs.append((hist, agent.actor_critic.flat.clone(), w.obs_rms.buf.clone(), w.ret_rms.buf.clone()))
        loaded.close()
        w.close()
    (h0, f0, o0, r0), (h1, f1, o1, r1) = runs
    assert torch.equal(f0, f1) and torch.equal(o0, o1) and torch.equal(r0, r1)
    for a, b in zip(h0, h1):
        assert all(a[k] == b[k] or (a[k] != a[k] and b[k] != b[k]) for k in a if k != "samples_per_s")


def test_state_dict_round_trip_in_place(highway_config):
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize

    cfg = _configs(highway_config)["kinematics"]
    a = VecNormalize(_vec(cfg, 64, seed=1))
    a.reset(seed=1)
    a.step(torch.zeros((64, 2), device=DEV))
    b = VecNormalize(_vec(cfg, 64, seed=1), clip_obs=3.0)
    ptr = b.obs_rms.buf.data_ptr()
    b.load_state_dict(a.state_dict())
    assert b.obs_rms.buf.data_ptr() == ptr and torch.equal(a.obs_rms.buf, b.obs_rms.buf)
    assert torch.equal(a.ret_rms.buf, b.ret_rms.buf) and b.clip_obs == 10.0
    a.close()
    b.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_statistics_are_identical_and_match_one_process():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29651", os.path.join(root, "tools", "p2p_check.py"), "--vecnormalize"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "vecnormalize: ranks bit-identical: True" in res.stdout and "matches one process: True" in res.stdout
