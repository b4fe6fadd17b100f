"""GPU checks of the categorical policy (HRP_PPO_CATEGORICAL, PPOAgent(discrete=True)) against the fp64 torch oracle
(oracle/ppo_categorical_ref.py), the in-kernel sampling against Philox4x32-10 on the CPU, and the policy on the
DiscreteMetaAction env through the batched and the single-env loops.

Tolerances are those tests/test_ppo_gpu.py uses for the corresponding Gaussian quantities: logits and value 2e-5;
log-prob 5e-5 + 1e-5 relative; gradients 1e-4 of the gradient's max-abs + 2e-6; parameters after one Adam step 5e-6.
"""
import copy
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from oracle import ppo_categorical_ref as cref
from oracle import ppo_ref

pytestmark = pytest.mark.gpu


def _agent(S, n, H, B, **kw):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    return PPOAgent(S, n, lr=3e-4, hidden_dim=H, batch_size=B, device="cuda:0", discrete=True, **kw)


def _lib():
    from highway_rope_ppo_b200 import _lib

    return _lib, _lib.load()


def _uniforms(lib, seed, draw, rows):
    """The kernels' per-row uniform: Philox4x32-10(counter = (row, draw), key = (seed lo, seed hi ^ 0x5A5A5A5A)), word 0,
    u = ((r0 >> 8) + 0.5) / 2^24 in float32 arithmetic."""
    m = 0xFFFFFFFF
    key = (C.c_uint32 * 2)(seed & m, ((seed >> 32) & m) ^ 0x5A5A5A5A)
    out = (C.c_uint32 * 4)()
    r0 = np.empty(len(rows), dtype=np.uint32)
    for i, r in enumerate(rows):
        assert lib.hrp_philox4x32_10((C.c_uint32 * 4)(r & m, r >> 32, draw & m, draw >> 32), key, out) == 0
        r0[i] = out[0]
    return ((r0 >> 8).astype(np.float32) + np.float32(0.5)) * np.float32(1.0 / 16777216.0)


def _ref_logits(ac, x):
    S, n, H = ac.state_dim, ac.action_dim, ac.hidden_dim
    logits, value = cref.forward(ac.flat.cpu().double(), torch.as_tensor(x).double(), S, n, H)
    return logits.numpy(), value.numpy()[:, 0]


def _softmax(lg):
    e = np.exp(lg - lg.max(1, keepdims=True))
    return e / e.sum(1, keepdims=True)


SIZES = [(60, 5, 256, 64), (60, 5, 256, 4096), (20, 3, 32, 17), (600, 8, 512, 64), (60, 4, 128, 256)]


@pytest.mark.parametrize("mode", [3, 0])
@pytest.mark.parametrize("S,n,H,B", SIZES)
def test_forward_act_loss_grad_adam_match_oracle(S, n, H, B, mode):
    """(60, 5, 256, B >= 32) and (600, 8, 512, 64) act through the fused eight-wide GEMM epilogue in math mode 3,
    (60, 4, 128, 256) through the four-wide one; (20, 3, 32, 17) and math mode 0 through heads_act_cat_kernel."""
    _l, lib = _lib()
    prev = lib.hrp_ppo_get_math()
    _l.check(lib.hrp_ppo_set_math(mode))
    try:
        torch.manual_seed(S + n + H + B)
        agent = _agent(S, n, H, B)
        ac = agent.actor_critic
        g = torch.Generator().manual_seed(1)
        x = torch.randn(B, S, generator=g) * 0.5
        lg_ref, v_ref = _ref_logits(ac, x)
        logits, none, value = ac.forward(x.cuda())
        assert none is None and logits.shape == (B, n)
        np.testing.assert_allclose(logits.cpu().numpy(), lg_ref, atol=2e-5)
        np.testing.assert_allclose(value.cpu().numpy()[:, 0], v_ref, atol=2e-5)
        logp_ref = lg_ref - lg_ref.max(1, keepdims=True)
        logp_ref = logp_ref - np.log(np.exp(logp_ref).sum(1, keepdims=True))
        p_ref = np.exp(logp_ref)
        rows = np.arange(B)

        # deterministic: the argmax (rows whose two largest logits lie within 1e-4 could go either way)
        out = ac.act(x.cuda(), deterministic=True)
        a = out["action"].cpu().numpy()
        top = np.sort(lg_ref, 1)
        clear = top[:, -1] - top[:, -2] > 1e-4
        assert np.array_equal(a[clear, 0], lg_ref.argmax(1)[clear]) and (a[:, 1] == 0).all()
        assert np.array_equal(out["pre_tanh"].cpu().numpy()[:, 0], a[:, 0])
        np.testing.assert_allclose(out["value"].cpu().numpy(), v_ref, atol=2e-5)

        # one uniform per row from noise[]: the inverse-CDF draw
        u = torch.rand(B, generator=g).clamp(1e-6, 1 - 1e-6)
        out = ac.act(x.cuda(), noise=u.cuda())
        ids = out["action"].cpu().numpy()[:, 0].astype(np.int64)
        want, margin = cref.sample(p_ref, u.numpy().astype(np.float64))
        sure = margin > 1e-5
        assert np.array_equal(ids[sure], want[sure])
        lp = out["log_prob"].cpu().numpy()
        np.testing.assert_allclose(lp, logp_ref[rows, ids], atol=5e-5, rtol=1e-5)

        # one minibatch: loss, gradient, clip + Adam against the fp64 oracle
        old = torch.from_numpy(logp_ref[rows, ids]) + 0.2 * torch.randn(B, generator=g, dtype=torch.float64)
        adv, ret = torch.randn(B, generator=g, dtype=torch.float64), torch.randn(B, generator=g, dtype=torch.float64)
        flat64 = ac.flat.cpu().double()
        r = cref.loss_and_grad(flat64, x.double(), torch.from_numpy(ids), old, adv, ret, S, n, H)
        dev = {"states": x.cuda(), "pre_tanh": torch.from_numpy(ids).float().view(B, 1).cuda(),
               "log_prob": old.float().cuda(), "adv": adv.float().cuda(), "ret": ret.float().cuda()}
        agent._metrics.zero_()
        agent._minibatch_step(dev, None, B, 1)
        m = agent._metrics.cpu().numpy()
        assert abs(m[0] - r["loss"]) < 2e-5 * max(1.0, abs(r["loss"])) and abs(m[1] - r["actor"]) < 2e-5
        assert abs(m[2] - r["critic"]) < 2e-5 * max(1.0, r["critic"]) and abs(m[3] - r["entropy"]) < 2e-5
        assert abs(m[4] - r["clip_fraction"]) <= 1.0 / B + 1e-6 and abs(m[5] - r["approx_kl"]) < 2e-5
        assert m[6] == 1.0
        want_g = r["grad"].numpy()
        np.testing.assert_allclose(agent.grad.cpu().numpy(), want_g, atol=1e-4 * np.abs(want_g).max() + 2e-6)
        zeros = torch.zeros_like(flat64)
        p1_ref, _, _, total = cref.clip_adam(flat64, r["grad"], zeros, zeros, 1)
        p1 = ac.flat.cpu().numpy()
        solid = np.abs(want_g) * min(1.0, 0.5 / total) > 1e-5   # Adam's first step is well-conditioned only there
        assert solid.sum() > 0
        np.testing.assert_allclose(p1[solid], p1_ref.numpy()[solid], atol=5e-6)
        assert np.abs(p1 - p1_ref.numpy()).max() <= 3.1e-4
    finally:
        lib.hrp_ppo_set_math(prev)


@pytest.mark.parametrize("S,n,H,E", [(60, 5, 256, 4096), (20, 3, 32, 17)])
def test_sampling_reproduces_philox_inverse_cdf(S, n, H, E):
    """Every sampled id is the one the CPU computes from hrp_philox4x32_10 and fp64 softmax probabilities, except rows
    whose uniform lies within 1e-5 of a cumulative boundary (at most 0.1 % of them, or one row)."""
    _l, lib = _lib()
    torch.manual_seed(9)
    agent = _agent(S, n, H, E)
    ac = agent.actor_critic
    ac._views["actor_mean.2.weight"].mul_(10.0)   # spread the probabilities
    x = torch.randn(E, S, generator=torch.Generator().manual_seed(3)) * 0.5
    for _ in range(2):
        out = ac.act(x.cuda())
        u = _uniforms(lib, ac._noise_seed, ac._draw, range(E))
        lg, _ = _ref_logits(ac, x)
        want, margin = cref.sample(_softmax(lg), u.astype(np.float64))
        ids = out["action"].cpu().numpy()[:, 0].astype(np.int64)
        near = margin < 1e-5
        assert near.sum() <= max(1, 0.001 * E), near.sum()
        assert np.array_equal(ids[~near], want[~near])
        assert np.array_equal(out["pre_tanh"].cpu().numpy()[:, 0], ids)


def test_sampling_frequencies_chi_square():
    """2^20 draws from one state: the id frequencies against the softmax probabilities."""
    from scipy.stats import chisquare

    S, n, H, E = 8, 5, 64, 1 << 16
    torch.manual_seed(2)
    agent = _agent(S, n, H, E)
    ac = agent.actor_critic
    ac._views["actor_mean.2.weight"].mul_(10.0)
    x = (torch.randn(1, S) * 0.5).repeat(E, 1).cuda()
    logits, _, _ = ac.forward(x[:1])
    p = torch.softmax(logits.double(), -1).cpu().numpy()[0]
    counts = np.zeros(n)
    for _ in range(16):
        out = ac.act(x)
        counts += torch.bincount(out["action"][:, 0].long(), minlength=n).cpu().numpy()
    N = counts.sum()
    assert N == 1 << 20 and p.min() * N > 100, p
    stat, pv = chisquare(counts, p * N)
    print("chi-square", stat, "p-value", pv, "probabilities", p)
    assert pv > 1e-4


def test_two_row_shards_equal_one_batch():
    """A 2E-row batch samples what two E-row calls with row_base 0 and E sample."""
    _l, lib = _lib()
    S, n, H, E = 60, 5, 256, 2048
    torch.manual_seed(6)
    agent = _agent(S, n, H, 2 * E)
    ac = agent.actor_critic
    x = (torch.randn(2 * E, S) * 0.5).cuda()
    st = torch.cuda.current_stream().cuda_stream

    def sample(xs, row_base):
        o = ac._new_act_out(xs.shape[0])
        _l.check(lib.hrp_ppo_act_sample(ac._h, ac.flat.data_ptr(), xs.data_ptr(), 1234, 7, row_base, xs.shape[0],
                                        o["action"].data_ptr(), o["pre_tanh"].data_ptr(), o["log_prob"].data_ptr(),
                                        o["value"].data_ptr(), st))
        return o

    whole = sample(x, 0)
    halves = [sample(x[:E].contiguous(), 0), sample(x[E:].contiguous(), E)]
    for k in ("action", "pre_tanh"):
        assert torch.equal(whole[k], torch.cat([h[k] for h in halves])), k
    for k in ("log_prob", "value"):   # (the GEMM's tile width depends on the batch: last-bit differences)
        np.testing.assert_allclose(whole[k].cpu().numpy(), torch.cat([h[k] for h in halves]).cpu().numpy(), atol=1e-5)


def test_act_sample_ctr_graph_replay_equals_host_counter():
    """hrp_ppo_act_sample_ctr captured in a CUDA graph: replay k draws what the host path draws with draw d0 + k."""
    _l, lib = _lib()
    S, n, H, E = 60, 5, 256, 512
    torch.manual_seed(8)
    agent = _agent(S, n, H, E)
    ac = agent.actor_critic
    x = (torch.randn(E, S) * 0.5).cuda()
    ac.act(x, draw_counter=ac.new_draw_counter())   # warm every kernel before the capture
    torch.cuda.synchronize()
    d0 = ac._draw
    ctr = torch.tensor([d0, 0], dtype=torch.int64, device="cuda:0")
    out = ac._new_act_out(E)
    graph = torch.cuda.CUDAGraph()
    cur, side = torch.cuda.current_stream(), torch.cuda.Stream()
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        graph.capture_begin()
        ac.act(x, out=out, draw_counter=ctr)
        graph.capture_end()
    cur.wait_stream(side)
    st = cur.cuda_stream
    for k in (1, 2, 3):
        graph.replay()
        ref = ac._new_act_out(E)
        _l.check(lib.hrp_ppo_act_sample(ac._h, ac.flat.data_ptr(), x.data_ptr(), ac._noise_seed, d0 + k, 0, E,
                                        ref["action"].data_ptr(), ref["pre_tanh"].data_ptr(), ref["log_prob"].data_ptr(),
                                        ref["value"].data_ptr(), st))
        for key in out:
            assert torch.equal(out[key], ref[key]), (k, key)
    assert ctr.tolist() == [d0 + 3, 0]


def test_full_update_matches_oracle():
    """PPOAgent(discrete=True).update on a [T, E] rollout equals the oracle's update (GAE, normalisation, the same
    minibatch permutation, clip + Adam per minibatch) at test_full_update_matches_reference's tolerances."""
    S, n, H, T, E, bs, epochs = 12, 5, 16, 10, 10, 25, 3
    torch.manual_seed(5)
    agent = _agent(S, n, H, bs, epochs=epochs)
    ac = agent.actor_critic
    flat0 = ac.flat.cpu().double()
    rng = np.random.default_rng(0)
    N = T * E
    states = (rng.standard_normal((T + 1, E, S)) * 0.5).astype(np.float32)
    X = torch.from_numpy(states[:T].reshape(N, S)).double()
    lg, _ = cref.forward(flat0, X, S, n, H)
    p = torch.softmax(lg, -1).numpy()
    ids = np.array([rng.choice(n, p=pr / pr.sum()) for pr in p])
    logp = torch.log_softmax(lg, -1).numpy()[np.arange(N), ids]
    old = (logp + 0.1 * rng.standard_normal(N)).astype(np.float32)
    value = rng.standard_normal((T, E)).astype(np.float32)
    reward = rng.standard_normal((T, E)).astype(np.float32)
    done = rng.random((T, E)) < 0.1
    last = rng.standard_normal(E).astype(np.float32)
    r = agent.memory.begin_rollout(T, E, S, 2, 1)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    r["states"].copy_(cu(states))
    r["action"].copy_(cu(np.stack([ids.reshape(T, E), np.zeros((T, E))], -1).astype(np.float32)))
    r["pre_tanh"].copy_(cu(ids.reshape(T, E, 1).astype(np.float32)))
    r["log_prob"].copy_(cu(old.reshape(T, E)))
    r["value"].copy_(cu(value))
    r["reward"].copy_(cu(reward))
    r["done"].copy_(cu(done.astype(np.uint8)))
    np.random.seed(11)
    metrics = agent.update(last_value=cu(last))
    # the oracle
    adv = np.zeros((T, E), dtype=np.float32)
    for e in range(E):
        adv[:, e], _ = ppo_ref.gae(reward[:, e], value[:, e], done[:, e], last[e])
    ret = torch.from_numpy((adv + value).reshape(N)).double()
    advn = torch.from_numpy(adv.reshape(N)).double()
    advn = (advn - advn.mean()) / (advn.std() + 1e-8)
    np.random.seed(11)
    perm = np.arange(N, dtype=np.int64)
    np.random.shuffle(perm)
    flat, m, v, step, mets = flat0.clone(), torch.zeros_like(flat0), torch.zeros_like(flat0), 0, []
    idt, oldt = torch.from_numpy(ids), torch.from_numpy(old).double()
    for _ in range(epochs):
        for start in range(0, N, bs):
            i = torch.from_numpy(perm[start:start + bs])
            rr = cref.loss_and_grad(flat, X[i], idt[i], oldt[i], advn[i], ret[i], S, n, H)
            step += 1
            flat, m, v, _ = cref.clip_adam(flat, rr["grad"], m, v, step)
            mets.append(rr)
    want = {k: float(np.mean([q[src] for q in mets])) for k, src in
            (("loss", "loss"), ("policy_loss", "actor"), ("value_loss", "critic"), ("entropy", "entropy"))}
    for k in want:
        assert abs(metrics[k] - want[k]) <= 2e-3 * max(1.0, abs(want[k])), (k, metrics[k], want[k])
    p1 = ac.flat.cpu().numpy()
    moved = np.abs(flat.numpy() - flat0.numpy()).max()
    err = np.abs(p1 - flat.numpy()).max()
    print(f"discrete update: max parameter motion {moved:.3e}, max error {err:.3e} = {err / moved:.2e} of it")
    assert err <= 1e-4 * moved
    assert len(agent.memory) == 0


def _meta_cfg(highway_config):
    cfg = copy.deepcopy(highway_config)
    cfg["action"] = {"type": "DiscreteMetaAction"}
    return cfg


def _meta_vec_env(highway_config, E, seed):
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_vec_env

    return make_vec_env(Condition.SORTED, _meta_cfg(highway_config), num_envs=E, seed=seed)


def test_meta_action_rollout_graph_equals_eager_and_replays_on_the_env(highway_config):
    """collect_rollout of a discrete agent on a DiscreteMetaAction vec env: the captured-graph rollout is bit-identical
    to the eager one, and a second handle with the same seed, stepped on the recorded ids, reproduces the
    observations, rewards and flags."""
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.routine import collect_rollout

    E, T, R = 128, 6, 3
    runs = []
    for use_graph in (False, True):
        torch.manual_seed(4)
        np.random.seed(4)
        env = _meta_vec_env(highway_config, E, 7)
        S = env.N * env.F_out
        agent = PPOAgent(S, 5, hidden_dim=64, batch_size=256, epochs=1, discrete=True)
        obs = env.reset(7).clone()
        got = []
        for it in range(R):
            r = collect_rollout(env, agent, T, obs, use_graph=use_graph)
            assert r["action"].shape == (T, E, 2) and r["pre_tanh"].shape == (T, E, 1)
            got.append({k: v.clone() for k, v in r.items()})
            obs = r["states"][T].clone()
            _, _, v = agent.actor_critic.forward(obs.view(E, -1))
            agent.update(last_value=v.view(-1))
        runs.append(got)
        env.close()
    for a, b in zip(*runs):
        for k in a:
            assert torch.equal(a[k], b[k]), k
    env2 = _meta_vec_env(highway_config, E, 7)
    o = env2.reset(7)
    assert torch.equal(o.reshape(E, -1), runs[1][0]["states"][0])
    for g in runs[1]:
        a = g["action"]
        assert ((a[..., 0] >= 0) & (a[..., 0] <= 4) & (a[..., 0] == a[..., 0].round()) & (a[..., 1] == 0)).all()
        assert torch.equal(a[..., 0], g["pre_tanh"][..., 0])
        for t in range(T):
            o, rew, term, trunc = env2.step(a[t].contiguous())
            assert torch.equal(o.reshape(E, -1), g["states"][t + 1]), t
            assert torch.equal(rew, g["reward"][t]) and torch.equal(term, g["terminated"][t])
            assert torch.equal(trunc, g["truncated"][t])
    env2.close()


def test_discrete_agent_env_mismatch_raises(highway_config):
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_vec_env
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.routine import collect_rollout, rollout_and_update, train_vectorized

    cont = make_vec_env(Condition.SORTED, highway_config, num_envs=8, seed=0)
    meta = _meta_vec_env(highway_config, 8, 0)
    S = cont.N * cont.F_out
    five = PPOAgent(S, 5, hidden_dim=32, batch_size=32, discrete=True)
    three = PPOAgent(S, 3, hidden_dim=32, batch_size=32, discrete=True)
    launches = (cont.launches, meta.launches)
    for fn in (lambda e, a: collect_rollout(e, a, 4), lambda e, a: rollout_and_update(e, a, 4),
               lambda e, a: train_vectorized(e, a, 1, 4)):
        with pytest.raises(ValueError, match="DiscreteMetaAction"):
            fn(cont, five)
        with pytest.raises(ValueError, match="has 3 actions"):
            fn(meta, three)
    assert (cont.launches, meta.launches) == launches and five.launches == three.launches == 0
    cont.close()
    meta.close()


def test_checkpoint_roundtrip_and_gaussian_checkpoint_rejected(tmp_path):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    torch.manual_seed(0)
    a = _agent(60, 5, 64, 32)
    flat = {"states": torch.randn(32, 60).cuda(), "pre_tanh": torch.randint(0, 5, (32, 1)).float().cuda(),
            "log_prob": torch.randn(32).cuda() - 2, "adv": torch.randn(32).cuda(), "ret": torch.randn(32).cuda()}
    a._minibatch_step(flat, None, 32, 1)
    path = str(tmp_path / "cat.pth")
    a.save(path)
    ck = torch.load(path, map_location="cpu")
    assert list(ck["model"]) == ["shared.0.weight", "shared.0.bias", "shared.2.weight", "shared.2.bias",
                                 "actor_mean.0.weight", "actor_mean.0.bias", "actor_mean.2.weight",
                                 "actor_mean.2.bias", "critic.0.weight", "critic.0.bias", "critic.2.weight",
                                 "critic.2.bias"]
    assert tuple(ck["model"]["actor_mean.2.weight"].shape) == (5, 64)
    torch.manual_seed(1)
    b = _agent(60, 5, 64, 32)
    b.load(path)
    assert torch.equal(b.actor_critic.flat, a.actor_critic.flat)
    assert int(b.optimizer.step_dev.item()) == 1
    assert torch.equal(b.optimizer.exp_avg_sq, a.optimizer.exp_avg_sq)
    gauss = PPOAgent(60, 2, hidden_dim=64, batch_size=32, device="cuda:0")
    gpath = str(tmp_path / "gauss.pth")
    gauss.save(gpath)
    with pytest.raises(RuntimeError, match="log_std"):
        b.load(gpath)


def test_single_env_loop_on_meta_action_env(highway_config, tmp_path):
    """train_with_experiment_name on make_env(DiscreteMetaAction) with a discrete agent: the reference loop as it is,
    deterministic (argmax) evaluation, the metrics JSON and summary CSV of tests/golden/result_schema.json."""
    import re

    from highway_rope_ppo_b200.experiments.config import Condition, ConditionHP
    from highway_rope_ppo_b200.experiments.runner import experiment_name
    from highway_rope_ppo_b200.experiments.wrappers import make_env
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.routine import train_with_experiment_name

    env = make_env(Condition.SORTED, _meta_cfg(highway_config))
    S, n = int(np.prod(env.observation_space.shape)), int(env.action_space.n)
    torch.manual_seed(0)
    np.random.seed(0)
    agent = PPOAgent(S, n, lr=3e-4, hidden_dim=64, batch_size=32, epochs=2, discrete=True)
    obs, _ = env.reset(seed=1)
    flat = obs.reshape(-1)
    idx, pre, lp, val = agent.select_action(flat, deterministic=True)
    logits, _, _ = agent.actor_critic.forward(flat)
    assert isinstance(idx, int) and idx == int(torch.argmax(logits)) and lp is None
    assert pre.dtype == np.float32 and pre.tolist() == [float(idx)]
    idx, pre, lp, val = agent.select_action(flat)
    assert 0 <= idx < n and np.isfinite(lp) and np.isfinite(val)
    name = experiment_name("SORTED", ConditionHP(lr=3e-4, hidden_dim=64, batch_size=32, epochs=2, d_embed=4), 42)
    rewards, avg, hist = train_with_experiment_name(env, agent, max_episodes=3, eval_interval=3, log_interval=1,
                                                    steps_per_update=48, experiment_name=name, exp_seed=42,
                                                    artifacts_dir=str(tmp_path))
    env.close()
    assert len(rewards) == 2 and all(np.isfinite(rewards)) and hist["policy_updates"]
    assert all(np.isfinite(u["loss"]) and u["entropy"] > 0 for u in hist["policy_updates"])
    schema = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "result_schema.json")))
    data = json.load(open(tmp_path / f"training_metrics_{name}.json"))
    assert list(data) == schema["metrics_keys"]
    assert re.match(schema["exp_rx"], data["experiment_name"])
    lines = (tmp_path / f"summary_{name}.csv").read_text().splitlines()
    assert lines[0] == schema["summary_header"] and lines[1].split(",")[0] == name and len(lines[1].split(",")) == 6
