"""GPU parity of the PPO kernels against the reference agent (tests/golden/ppo_*.npz, produced by
/root/reference/ppo/agent.py through tools/gen_golden.py) and the torch fp32 oracle (oracle/ppo_ref.py).

Tolerances (fp32 kernels, different summation order than ATen):
  forward mean/value 2e-5 abs;  log-prob 5e-5;  loss terms 2e-5;  gradients 1e-4 relative to the gradient's
  max-abs (plus 2e-6 abs);  parameters after Adam 5e-6 abs for one step (Adam's first steps move every weight
  by ~lr = 3e-4 regardless of the gradient's size, so sign-level agreement of tiny gradients is what matters);
  GAE: advantages 2e-6 abs (fp64 scan, fp32 store, same as the reference).
"""
import numpy as np
import pytest
import torch

from conftest import golden
from oracle import ppo_ref

pytestmark = pytest.mark.gpu


def _agent(S, A, H, B, **kw):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    return PPOAgent(S, A, lr=3e-4, hidden_dim=H, batch_size=B, device="cuda:0", **kw)


def _load_flat(agent, flat):
    agent.actor_critic.flat.copy_(torch.from_numpy(flat).cuda())


@pytest.mark.parametrize("name", ["s60_h256_b64", "s20_h32_b17", "s300_h64_b256"])
def test_init_matches_reference_for_the_same_seed(name):
    """Same torch seed -> same nn.Linear initialisation stream as the reference's ActorCritic."""
    g = golden(f"ppo_step_{name}.npz")
    S, A, H, B, seed = (int(v) for v in g["dims"])
    torch.manual_seed(seed)
    agent = _agent(S, A, H, B)
    assert [n for n, _ in agent.actor_critic.named_parameters()] == [str(n) for n in g["names"]]
    assert np.array_equal(agent.actor_critic.flat.cpu().numpy(), g["params0"])


@pytest.mark.parametrize("name", ["s60_h256_b64", "s20_h32_b17", "s300_h64_b256"])
def test_forward_loss_grad_adam_match_reference(name):
    from highway_rope_ppo_b200 import _lib

    g = golden(f"ppo_step_{name}.npz")
    S, A, H, B, _ = (int(v) for v in g["dims"])
    agent = _agent(S, A, H, B)
    _load_flat(agent, g["params0"])
    ac = agent.actor_critic
    cu = lambda k: torch.from_numpy(g[k]).cuda()
    mean, std, value = ac.forward(cu("states"))
    np.testing.assert_allclose(mean.cpu().numpy(), g["mean"], atol=2e-5)
    np.testing.assert_allclose(value.cpu().numpy(), g["value"], atol=2e-5)
    logp, v, ent = ac.evaluate(cu("states"), None, cu("pre_tanh"))
    np.testing.assert_allclose(logp.cpu().numpy(), g["logp"], atol=5e-5, rtol=1e-5)
    np.testing.assert_allclose(ent.cpu().numpy(), g["entropy"], atol=1e-6)
    # act kernel: deterministic noise reproduces pre_tanh -> log-prob of the reference's evaluate()
    noise = (cu("pre_tanh") - mean) / std
    out = ac.act(cu("states"), noise=noise.contiguous())
    np.testing.assert_allclose(out["pre_tanh"].cpu().numpy(), g["pre_tanh"], atol=1e-5)
    np.testing.assert_allclose(out["log_prob"].cpu().numpy(), g["logp"], atol=1e-4, rtol=1e-5)
    np.testing.assert_allclose(out["action"].cpu().numpy(), np.tanh(g["pre_tanh"]), atol=1e-6)
    np.testing.assert_allclose(out["value"].cpu().numpy(), g["value"][:, 0], atol=2e-5)
    # one minibatch: loss, gradient, clip + Adam
    flat = {"states": cu("states"), "pre_tanh": cu("pre_tanh"), "log_prob": cu("old_logp"), "adv": cu("adv"),
            "ret": cu("ret")}
    agent._metrics.zero_()
    agent._minibatch_step(flat, None, B, 1)
    m = agent._metrics.cpu().numpy()
    assert abs(m[0] - float(g["loss"])) < 2e-5 and abs(m[1] - float(g["actor_loss"])) < 2e-5
    assert abs(m[2] - float(g["critic_loss"])) < 2e-5 * max(1.0, float(g["critic_loss"]))
    assert abs(m[4] - float(g["clip_fraction"])) < 1e-6 and abs(m[5] - float(g["approx_kl"])) < 2e-5
    assert m[6] == 1.0
    grad = agent.grad.cpu().numpy()
    scale = np.abs(g["grads"]).max()
    np.testing.assert_allclose(grad, g["grads"], atol=1e-4 * scale + 2e-6)
    # Adam's first step moves every weight by lr * g / (|g| + 1e-8): it is only well-conditioned where |g| >> eps
    p1 = ac.flat.cpu().numpy()
    solid = np.abs(g["grads"]) * min(1.0, 0.5 / float(g["total_norm"])) > 1e-5
    assert solid.mean() > 0.5
    np.testing.assert_allclose(p1[solid], g["params1"][solid], atol=5e-6)
    assert np.abs(p1 - g["params1"]).max() <= 3.1e-4  # never more than one lr-sized step apart
    # gathered minibatch (idx) gives the same step: run step 2 through an identity-permuted gather
    idx = torch.arange(B, device="cuda:0", dtype=torch.int64)
    agent._minibatch_step(flat, idx, B, 1)
    np.testing.assert_allclose(ac.flat.cpu().numpy()[solid], g["params2"][solid], atol=2e-5)
    assert int(agent.optimizer.step_dev.item()) == 2


@pytest.mark.parametrize("name", ["t50", "t2048"])
def test_gae_matches_reference(name):
    from highway_rope_ppo_b200.ppo.agent import gae

    g = golden(f"ppo_gae_{name}.npz")
    T = len(g["reward"])
    adv, ret = gae(torch.from_numpy(g["reward"].astype(np.float32)).cuda().view(T, 1),
                   torch.from_numpy(g["value"]).cuda().view(T, 1),
                   torch.from_numpy(g["done"].astype(np.uint8)).cuda().view(T, 1), float(g["last_value"]), 0.99, 0.95)
    # rewards are float32 on the device (float64 python floats in the reference): 2e-6 covers the input rounding
    np.testing.assert_allclose(adv.cpu().numpy()[:, 0], g["adv"], atol=2e-6, rtol=2e-6)
    np.testing.assert_allclose(ret.cpu().numpy()[:, 0], g["ret"], atol=2e-6, rtol=2e-6)


def test_gae_batched_matches_oracle():
    from highway_rope_ppo_b200.ppo.agent import gae

    rng = np.random.default_rng(0)
    T, E = 64, 300
    rew = rng.random((T, E)).astype(np.float32)
    val = rng.standard_normal((T, E)).astype(np.float32)
    done = (rng.random((T, E)) < 0.1)
    last = rng.standard_normal(E).astype(np.float32)
    adv, ret = gae(torch.from_numpy(rew).cuda(), torch.from_numpy(val).cuda(),
                   torch.from_numpy(done.astype(np.uint8)).cuda(), torch.from_numpy(last).cuda(), 0.99, 0.95)
    adv, ret = adv.cpu().numpy(), ret.cpu().numpy()
    for e in range(0, E, 17):
        a, r = ppo_ref.gae(rew[:, e], val[:, e], done[:, e], last[e])
        assert np.array_equal(adv[:, e], a) and np.array_equal(ret[:, e], r)


def test_adv_normalize_matches_torch():
    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    a = torch.randn(100_003, device="cuda:0") * 3 + 1.5
    want = ((a - a.mean()) / (a.std() + 1e-8)).cpu().numpy()
    stats = torch.zeros(3 + 512, dtype=torch.float64, device="cuda:0")
    s = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.hrp_adv_stats(a.data_ptr(), a.numel(), stats.data_ptr(), s))
    _lib.check(lib.hrp_adv_normalize(a.data_ptr(), a.numel(), stats.data_ptr(), s))
    np.testing.assert_allclose(a.cpu().numpy(), want, atol=2e-6, rtol=1e-5)


@pytest.mark.parametrize("name", ["s12_h16_n100", "s60_h256_n2048"])
def test_full_update_matches_reference(name):
    """PPOAgent.update on the reference's stored rollout with the reference's minibatch permutation."""
    g = golden(f"ppo_update_{name}.npz")
    S, A, H, n, bs, epochs, np_seed = (int(v) for v in g["dims"])
    agent = _agent(S, A, H, bs, epochs=epochs)
    _load_flat(agent, g["params0"])
    for t in range(n):
        agent.memory.store(g["states"][t], g["action"][t], g["pre_tanh"][t], float(g["reward"][t]), None,
                           float(g["logp"][t]), bool(g["done"][t]), np.float32(g["value"][t]))
    np.random.seed(np_seed)
    metrics = agent.update(last_value=float(g["last_value"]))
    want = dict(zip((str(k) for k in g["metric_names"]), g["metric_values"]))
    print({k: (metrics[k], float(want[k])) for k in want})
    # hundreds of optimizer steps amplify fp32 summation-order differences: compare at 2e-3 relative
    for k in ("loss", "policy_loss", "value_loss", "entropy", "explained_variance"):
        assert abs(metrics[k] - want[k]) <= 2e-3 * max(1.0, abs(want[k])), (k, metrics[k], want[k])
    assert abs(metrics["clip_fraction"] - want["clip_fraction"]) <= 0.01
    assert abs(metrics["approx_kl"] - want["approx_kl"]) <= 2e-3 * max(1e-2, abs(want["approx_kl"]))
    p1 = agent.actor_critic.flat.cpu().numpy()
    moved = np.abs(g["params1"] - g["params0"]).max()
    err = np.abs(p1 - g["params1"]).max()
    print(f"update {name}: max parameter motion {moved:.3e}, max error {err:.3e} = {err / moved:.2e} of it")
    # measured on B200 (3xTF32 GEMMs): 8e-6 of the largest parameter motion after the 12 optimizer steps of the small
    # fixture, 1.6e-2 after the 64 steps of the H = 256 one (Adam divides every gradient entry by its running RMS, so an
    # entry whose gradient is at rounding level still moves by ~lr per step, in a direction rounding decides); bounds at
    # about twice / ten times the measured figures
    assert err <= {"s12_h16_n100": 1e-4, "s60_h256_n2048": 0.03}[name] * moved
    assert len(agent.memory) == 0


def _check_large_batch_loss_grad(gather):
    S, A, H, B = 60, 2, 256, 4096
    torch.manual_seed(1)
    agent = _agent(S, A, H, B)
    g = torch.Generator().manual_seed(2)
    x = torch.randn(B, S, generator=g) * 0.5
    flat = agent.actor_critic.flat.cpu()
    mean, log_std, _ = ppo_ref.forward(flat, x, S, A, H)
    z = mean + torch.randn(B, A, generator=g)
    logp, _, _ = ppo_ref.evaluate(flat, x, z, S, A, H)
    old = logp + 0.2 * torch.randn(B, generator=g)
    adv, ret = torch.randn(B, generator=g), torch.randn(B, generator=g)
    r = ppo_ref.loss_and_grad(flat, x, z, old, adv, ret, S, A, H)
    dev = {"states": x.cuda(), "pre_tanh": z.cuda(), "log_prob": old.cuda(), "adv": adv.cuda(), "ret": ret.cuda()}
    agent._metrics.zero_()
    agent._minibatch_step(dev, torch.arange(B, device="cuda:0") if gather else None, B, 1)
    m = agent._metrics.cpu().numpy()
    assert abs(m[0] - r["loss"]) < 5e-5 and abs(m[4] - r["clip_fraction"]) < 1e-3
    want = r["grad"].numpy()
    np.testing.assert_allclose(agent.grad.cpu().numpy(), want, atol=2e-4 * np.abs(want).max() + 1e-6)


def test_loss_grad_large_batch_matches_oracle():
    """BASELINE-size minibatch (4096 x S=60, H=256): gradient vs the torch fp32 oracle (split-K wgrad path)."""
    _check_large_batch_loss_grad(gather=False)


def test_loss_grad_large_batch_through_gather_matches_oracle():
    """The same minibatch taken from the rollout by the gather kernel (idx = arange(B)), same tolerances."""
    _check_large_batch_loss_grad(gather=True)


def test_checkpoint_roundtrip_and_reference_key_names(tmp_path):
    torch.manual_seed(0)
    a = _agent(60, 2, 64, 32)
    flat = {"states": torch.randn(32, 60).cuda(), "pre_tanh": torch.randn(32, 2).cuda(),
            "log_prob": torch.randn(32).cuda() - 2, "adv": torch.randn(32).cuda(), "ret": torch.randn(32).cuda()}
    a._minibatch_step(flat, None, 32, 1)
    path = str(tmp_path / "ck.pth")
    a.save(path)
    ck = torch.load(path, map_location="cpu")
    assert list(ck["model"]) == ["log_std", "shared.0.weight", "shared.0.bias", "shared.2.weight", "shared.2.bias",
                                 "actor_mean.0.weight", "actor_mean.0.bias", "actor_mean.2.weight",
                                 "actor_mean.2.bias", "critic.0.weight", "critic.0.bias", "critic.2.weight",
                                 "critic.2.bias"]
    # visualize.py:54-57 infers the dimensions from these two tensors
    assert ck["model"]["shared.0.weight"].shape == (64, 60) and ck["model"]["actor_mean.2.weight"].shape == (2, 64)
    assert set(ck["optimizer"]) == {"state", "param_groups"} and len(ck["optimizer"]["state"]) == 13
    b = _agent(60, 2, 64, 32)
    b.load(path)
    assert torch.equal(a.actor_critic.flat, b.actor_critic.flat)
    assert torch.equal(a.optimizer.exp_avg, b.optimizer.exp_avg) and int(b.optimizer.step_dev.item()) == 1
    # the checkpoint loads into a plain torch module with the reference's layout
    import torch.nn as nn

    class Ref(nn.Module):
        def __init__(s):
            super().__init__()
            s.shared = nn.Sequential(nn.Linear(60, 64), nn.ReLU(), nn.Linear(64, 64), nn.ReLU())
            s.actor_mean = nn.Sequential(nn.Linear(64, 64), nn.ReLU(), nn.Linear(64, 2))
            s.log_std = nn.Parameter(torch.zeros(2))
            s.critic = nn.Sequential(nn.Linear(64, 64), nn.ReLU(), nn.Linear(64, 1))

    Ref().load_state_dict(ck["model"])
    opt = torch.optim.Adam(Ref().parameters(), lr=1e-4)
    opt.load_state_dict(ck["optimizer"])


def test_select_action_protocol():
    a = _agent(60, 2, 64, 32)
    s = np.random.randn(60).astype(np.float32)
    action, pre, lp, v = a.select_action(s)
    assert action.shape == (2,) and pre.shape == (2,) and isinstance(lp, float) and v.dtype == np.float32
    assert np.allclose(action, np.tanh(pre), atol=1e-6) and np.all(np.abs(action) <= 1)
    action, pre, lp, v = a.select_action(s, deterministic=True)
    assert lp is None
    mean, std, value = a.actor_critic.forward(s)
    assert mean.shape == (2,) and std.shape == (2,) and value.shape == (1,)
    assert np.allclose(pre, mean.cpu().numpy(), atol=1e-6)


def test_in_kernel_sampling_is_standard_normal_and_self_consistent():
    """hrp_ppo_act_sample: z = mean + std * n with n from Philox + Box-Muller; the log-prob it returns is the
    one evaluate() assigns to the same pre-tanh action (what PPO's ratio at epoch 0 relies on)."""
    torch.manual_seed(3)
    a = _agent(60, 2, 64, 8192)
    x = torch.randn(8192, 60, device="cuda:0") * 0.3
    out1 = {k: v.clone() for k, v in a.act(x).items()}
    out2 = a.act(x)
    mean, std, value = a.actor_critic.forward(x)
    n1 = ((out1["pre_tanh"] - mean) / std).flatten()
    n2 = ((out2["pre_tanh"] - mean) / std).flatten()
    assert abs(float(n1.mean())) < 0.03 and abs(float(n1.std()) - 1) < 0.03
    assert abs(float((n1 ** 3).mean())) < 0.1 and abs(float((n1 ** 4).mean()) - 3) < 0.25
    assert abs(float((n1 * n2).mean())) < 0.03                       # successive draws are independent
    assert abs(float((n1[0::2] * n1[1::2]).mean())) < 0.03           # so are the two action components
    logp, v, _ = a.actor_critic.evaluate(x, None, out1["pre_tanh"])
    np.testing.assert_allclose(out1["log_prob"].cpu().numpy(), logp.cpu().numpy(), atol=2e-5, rtol=1e-5)
    np.testing.assert_allclose(out1["value"].cpu().numpy(), value[:, 0].cpu().numpy(), atol=1e-6)
    np.testing.assert_allclose(out1["action"].cpu().numpy(), np.tanh(out1["pre_tanh"].cpu().numpy()), atol=1e-6)
    # same seed, same draw counter -> same sample
    torch.manual_seed(3)
    b = _agent(60, 2, 64, 8192)
    assert torch.equal(b.act(x)["pre_tanh"], out1["pre_tanh"])


def test_sharded_sampling_equals_single_process_sampling():
    """The exploration noise is keyed by (seed, GLOBAL row, draw): two shards acting on rows [0, B/2) and [B/2, B)
    with their row_base draw exactly what one process draws for rows [0, B), and NOT the same noise as each other."""
    torch.manual_seed(5)
    whole = _agent(60, 2, 64, 4096)
    x = torch.randn(4096, 60, device="cuda:0") * 0.3
    want = {k: v.clone() for k, v in whole.act(x).items()}
    parts = []
    for r in range(2):
        torch.manual_seed(5)                       # every rank seeds identically (set_random_seeds)
        shard = _agent(60, 2, 64, 2048)
        shard.actor_critic.row_base = 2048 * r
        parts.append({k: v.clone() for k, v in shard.act(x[2048 * r:2048 * (r + 1)]).items()})
    for k in ("pre_tanh", "action", "log_prob"):
        assert torch.equal(torch.cat([parts[0][k], parts[1][k]]), want[k]), k
    mean, std, _ = whole.actor_critic.forward(x)
    n = (want["pre_tanh"] - mean) / std
    assert abs(float((n[:2048] * n[2048:]).mean())) < 0.05      # the two shards' noise is independent
    # a graph captured against one workspace must not survive its re-creation
    g0 = whole.actor_critic.workspace_generation
    whole.actor_critic._ensure_workspace(8192)
    assert whole.actor_critic.workspace_generation == g0 + 1


def test_loads_a_checkpoint_written_by_the_reference_agent(tmp_path):
    """tests/golden/checkpoint_ref_s12_h16.pth was written by the reference's PPOAgent.save (agent.py:310-318) after
    one update; dims are inferred the way visualize.py:53-58 does.  Outputs must match the reference network's, the
    Adam state must land in the flat moment buffers."""
    import os

    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    here = os.path.join(os.path.dirname(__file__), "golden")
    g = golden("checkpoint_ref_s12_h16_outputs.npz")
    chk = torch.load(os.path.join(here, "checkpoint_ref_s12_h16.pth"), map_location="cpu")
    assert set(chk) >= {"model", "optimizer"}
    sd = chk["model"]
    hidden_dim, state_dim = sd["shared.0.weight"].shape
    action_dim = sd["actor_mean.2.weight"].shape[0]
    agent = PPOAgent(state_dim, action_dim, hidden_dim=hidden_dim, device="cuda:0")
    cfg = agent.load(os.path.join(here, "checkpoint_ref_s12_h16.pth"))
    assert cfg == {}
    mean, std, value = agent.actor_critic.forward(torch.from_numpy(g["states"]).cuda())
    np.testing.assert_allclose(mean.cpu().numpy(), g["mean"], atol=2e-5)
    np.testing.assert_allclose(value.cpu().numpy().reshape(g["value"].shape), g["value"], atol=2e-5)
    np.testing.assert_allclose(std.cpu().numpy().reshape(-1)[:action_dim], g["std"].reshape(-1)[:action_dim], rtol=1e-6)
    opt = agent.optimizer
    assert int(opt.step_dev.item()) == int(g["step"]) and opt.lr == pytest.approx(float(g["lr"]))
    n0 = action_dim  # log_std comes first in the flat layout, shared.0.weight second
    w1 = opt.exp_avg[n0:n0 + hidden_dim * state_dim].cpu().numpy().reshape(hidden_dim, state_dim)
    np.testing.assert_array_equal(w1, g["exp_avg_w1"])
    # and the round trip: what this agent saves, torch loads back with the reference's key names and shapes
    out = str(tmp_path / "ckpt_roundtrip.pth")
    agent.save(out)
    back = torch.load(out, map_location="cpu")
    assert list(back["model"]) == list(sd)
    for k in sd:
        assert torch.equal(back["model"][k], sd[k]), k
    assert back["optimizer"]["param_groups"][0]["lr"] == chk["optimizer"]["param_groups"][0]["lr"]
    os.remove(out)


def test_peer_memory_adam_step_with_one_rank_equals_the_plain_step():
    """hrp_clip_adam_step_p2p (csrc/hrp_comm.cu) with a world of one rank: the cross-GPU barriers see only their own
    flags and the rank-ordered sum has one term, so parameters and moments must equal hrp_clip_adam_step bit for bit,
    step after step (epoch counter, flag reuse)."""
    import ctypes as C

    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    n = 213765
    g = torch.Generator(device="cuda:0").manual_seed(3)
    comm, handle = C.c_void_p(), (C.c_ubyte * 64)()
    _lib.check(lib.hrp_comm_create(1, 0, n, 0, C.byref(comm), handle))
    _lib.check(lib.hrp_comm_connect(comm, bytes(handle)))
    views = []
    for parity in (0, 1):   # the exchange alternates two gradient buffers with the parity of the step
        ptr = lib.hrp_comm_grad_parity(comm, parity)

        class _Raw:
            __cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (int(ptr), False), "version": 2}

        views.append((_Raw(),))
        views[-1] = (views[-1][0], torch.as_tensor(views[-1][0], device="cuda:0"))
    st = torch.cuda.current_stream().cuda_stream
    pa = torch.randn(n, generator=g, device="cuda:0") * 0.1
    pb = pa.clone()
    ma, va, mb, vb = (torch.zeros(n, device="cuda:0") for _ in range(4))
    sa, sb = torch.zeros(1, dtype=torch.int32, device="cuda:0"), torch.zeros(1, dtype=torch.int32, device="cuda:0")
    scr_a, scr_b = torch.zeros(128, device="cuda:0"), torch.zeros(128, device="cuda:0")
    try:
        for it in range(5):
            grad = torch.randn(n, generator=g, device="cuda:0") * (0.5 if it % 2 else 5e-4)  # clipped and unclipped steps
            assert lib.hrp_comm_parity(comm) == it % 2 and lib.hrp_comm_grad(comm) == views[it % 2][1].data_ptr()
            views[it % 2][1].copy_(grad)
            _lib.check(lib.hrp_clip_adam_step_p2p(comm, pa.data_ptr(), ma.data_ptr(), va.data_ptr(), sa.data_ptr(), 3e-4, 0.9,
                                                  0.999, 1e-8, 0.5, scr_a.data_ptr(), st))
            _lib.check(lib.hrp_clip_adam_step(pb.data_ptr(), grad.data_ptr(), mb.data_ptr(), vb.data_ptr(), sb.data_ptr(), n,
                                              3e-4, 0.9, 0.999, 1e-8, 0.5, scr_b.data_ptr(), st))
            torch.cuda.synchronize()
            assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb), it
            assert int(sa.item()) == int(sb.item()) == it + 1
    finally:
        torch.cuda.synchronize()
        del views
        lib.hrp_comm_destroy(comm)
    # error paths
    assert lib.hrp_comm_create(9, 0, n, 0, C.byref(comm), handle) == -1      # more ranks than one box holds
    assert lib.hrp_clip_adam_step_p2p(None, pa.data_ptr(), ma.data_ptr(), va.data_ptr(), sa.data_ptr(), 3e-4, 0.9, 0.999,
                                      1e-8, 0.5, scr_a.data_ptr(), st) == -1


# ---- the swept and benchmarked widths (main.py:50-58: hidden_dim 128 / 256 / 384, batch 32 / 64; BASELINE configs[2..3]:
# ---- hidden_dim 512, state_dim 240 / 360 / 600), pinned to fixtures the reference's own agent produced
def _compact_of(vec, sizes):
    v = np.asarray(vec, dtype=np.float64)
    rng = np.random.default_rng(1234)
    proj = np.array([float(rng.standard_normal(v.size) @ v) for _ in range(8)])
    norms, off = [], 0
    for n in sizes:
        norms.append(float(np.sqrt((v[off:off + n] ** 2).sum())))
        off += int(n)
    return {"norms": np.array(norms), "proj": proj, "samples": np.asarray(vec, dtype=np.float32)[::257].copy()}


def _check_compact(vec, g, tag, atol, sizes):
    c = _compact_of(vec, sizes)
    np.testing.assert_allclose(c["samples"], g[f"{tag}_samples"], atol=atol, rtol=0)
    lim = atol * np.sqrt(np.maximum(np.asarray(sizes, dtype=np.float64), 1.0)) + 1e-4 * np.abs(g[f"{tag}_norms"])
    assert np.all(np.abs(c["norms"] - g[f"{tag}_norms"]) <= lim), (tag, c["norms"], g[f"{tag}_norms"])
    np.testing.assert_allclose(c["proj"], g[f"{tag}_proj"], atol=4 * atol * np.sqrt(len(vec)), rtol=1e-4)


import glob  # noqa: E402
import os  # noqa: E402

from conftest import GOLDEN  # noqa: E402

_WIDE = sorted(os.path.basename(p)[len("ppo_wide_"):-4] for p in glob.glob(os.path.join(GOLDEN, "ppo_wide_*.npz")))


@pytest.mark.parametrize("name", _WIDE)
def test_swept_widths_match_reference(name):
    g = golden(f"ppo_wide_{name}.npz")
    S, A, H, B, seed = (int(v) for v in g["dims"])
    sizes = g["sizes"]
    torch.manual_seed(seed)
    agent = _agent(S, A, H, B)
    ac = agent.actor_critic
    flat0 = ac.flat.cpu().numpy()
    assert np.array_equal(flat0[::257], g["params0_samples"])            # same initialisation stream as the reference
    assert abs(float(flat0.astype(np.float64).sum()) - float(g["params0_sum"])) < 1e-9
    cu = lambda k: torch.from_numpy(g[k]).cuda()
    mean, std, value = ac.forward(cu("states"))
    np.testing.assert_allclose(mean.cpu().numpy(), g["mean"], atol=2e-5)
    np.testing.assert_allclose(value.cpu().numpy(), g["value"], atol=2e-5)
    logp, _, _ = ac.evaluate(cu("states"), None, cu("pre_tanh"))
    np.testing.assert_allclose(logp.cpu().numpy(), g["logp"], atol=5e-5, rtol=1e-5)
    flat = {"states": cu("states"), "pre_tanh": cu("pre_tanh"), "log_prob": cu("old_logp"), "adv": cu("adv"),
            "ret": cu("ret")}
    agent._metrics.zero_()
    agent._minibatch_step(flat, None, B, 1)
    m = agent._metrics.cpu().numpy()
    assert abs(m[0] - float(g["loss"])) < 2e-5 and abs(m[1] - float(g["actor_loss"])) < 2e-5
    assert abs(m[2] - float(g["critic_loss"])) < 2e-5 * max(1.0, float(g["critic_loss"]))
    assert abs(m[4] - float(g["clip_fraction"])) < 1e-6
    _check_compact(agent.grad.cpu().numpy(), g, "grads", 1e-4 * float(g["grad_absmax"]) + 2e-6, sizes)
    # Adam's first step: lr * g_clipped / (|g_clipped| + eps), ~ +-lr wherever |g| >> eps
    step1 = ac.flat.cpu().numpy() - flat0
    want = g["step1_samples"]
    # entries whose clipped gradient is far above Adam's eps = 1e-8 (the step is lr * g / (|g| + eps): below that a
    # 1e-9 difference of the gradient moves it visibly; dead ReLU units have no gradient at all)
    solid = np.abs(g["grads_samples"]) * min(1.0, 0.5 / float(g["total_norm"])) > 3e-6
    assert solid.mean() > 0.3
    np.testing.assert_allclose(step1[::257][solid], want[solid], atol=3e-6)


def test_full_update_at_hidden_512_matches_reference():
    """PPOAgent.update at BASELINE configs[3]'s hidden_dim (512 stored transitions, bs 64, 2 epochs = 16 optimizer steps)."""
    g = golden("ppo_wideupdate_s60_h512_n512.npz")
    S, A, H, n, bs, epochs, np_seed, seed = (int(v) for v in g["dims"])
    torch.manual_seed(seed)
    agent = _agent(S, A, H, bs, epochs=epochs)
    flat0 = agent.actor_critic.flat.cpu().numpy()
    assert np.array_equal(flat0[::257], g["params0_samples"])
    for t in range(n):
        agent.memory.store(g["states"][t], g["action"][t], g["pre_tanh"][t], float(g["reward"][t]), None,
                           float(g["logp"][t]), bool(g["done"][t]), np.float32(g["value"][t]))
    np.random.seed(np_seed)
    metrics = agent.update(last_value=float(g["last_value"]))
    want = dict(zip((str(k) for k in g["metric_names"]), g["metric_values"]))
    for k in ("loss", "policy_loss", "value_loss", "entropy", "explained_variance"):
        assert abs(metrics[k] - want[k]) <= 2e-3 * max(1.0, abs(want[k])), (k, metrics[k], want[k])
    motion = agent.actor_critic.flat.cpu().numpy() - flat0
    moved = float(np.abs(g["motion_samples"]).max())
    err = float(np.abs(motion[::257] - g["motion_samples"]).max())
    print("H=512 update: max parameter motion", moved, "max error of the sampled entries", err)
    assert err <= 5e-4 * moved   # measured 3.3e-5 of the motion after these 16 optimizer steps


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_update_keeps_ranks_bit_identical(tmp_path):
    """Two ranks (one process per GPU, NCCL rendezvous, the peer-memory exchange of csrc/hrp_comm.cu inside CUDA
    graphs): after two sharded PPO updates every rank holds bit-identical parameters, and they agree with the NCCL
    all-reduce path to summation-order accuracy (tools/p2p_check.py)."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29641", os.path.join(root, "tools", "p2p_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "identical on every rank: True" in res.stdout, res.stdout[-3000:]


def test_workspace_lanes_share_the_parameters():
    """act(lane=k) runs on its own native workspace (two streams may act at once) with the same parameters, seed and
    global-row keyed noise: the same call on lane 0 and on lane 1 gives the same sample."""
    torch.manual_seed(8)
    a = _agent(60, 2, 64, 512)
    torch.manual_seed(8)
    b = _agent(60, 2, 64, 512)
    x = torch.randn(512, 60, device="cuda:0") * 0.3
    s1 = torch.cuda.Stream()
    want = a.act(x)
    with torch.cuda.stream(s1):
        s1.wait_stream(torch.cuda.current_stream())
        got = b.act(x, lane=1)
    s1.synchronize()
    for k in ("action", "pre_tanh", "log_prob", "value"):
        assert torch.equal(got[k], want[k]), k


def test_device_resident_draw_counter_equals_host_counter_and_replays_in_a_graph():
    """hrp_ppo_act_sample_ctr: the sampling path with its draw counter in device memory draws exactly what the host
    counter path draws, call after call, eagerly and as a replayed CUDA graph (the host-buffer pipeline relies on it)."""
    torch.manual_seed(9)
    a = _agent(60, 2, 64, 1024)
    torch.manual_seed(9)
    b = _agent(60, 2, 64, 1024)
    x = torch.randn(1000, 60, device="cuda:0") * 0.3
    want = [{k: v.clone() for k, v in a.act(x).items()} for _ in range(5)]
    ctr = b.actor_critic.new_draw_counter()
    out = {k: torch.empty_like(v) for k, v in want[0].items()}
    for i in range(2):   # eager
        b.act(x, out=out, draw_counter=ctr)
        for k in out:
            assert torch.equal(out[k], want[i][k]), (i, k)
    assert ctr.tolist() == [2, 0]
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.graph(g, stream=s):
        b.act(x, out=out, draw_counter=ctr)
    for i in range(2, 5):   # replays advance the counter themselves
        g.replay()
        torch.cuda.synchronize()
        for k in out:
            assert torch.equal(out[k], want[i][k]), (i, k)
    assert ctr.tolist() == [5, 0]


def test_multi_policy_act_matches_the_batched_forward_and_the_reference():
    """hrp_ppo_act_multi: one state each of several policies of different widths in ONE launch (the sweep's single-env
    rollout forward) == each policy's own batched forward (3xTF32 tensor-core path) to fp32 rounding, deterministic and
    sampled, and the B = 1 call of ActorCritic.act goes through it."""
    import ctypes as C

    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    dims = [(60, 128), (60, 256), (120, 384), (300, 512), (60, 64), (12, 16)]
    agents, states = [], []
    for i, (S, H) in enumerate(dims):
        torch.manual_seed(20 + i)
        agents.append(_agent(S, 2, H, 8))
        states.append(torch.randn(1, S, device="cuda:0") * 0.5)
    for det in (True, False):
        res = torch.zeros((len(dims), 6), device="cuda:0")
        items = (_lib.HrpActItem * len(dims))()
        for i, a in enumerate(agents):
            items[i] = a.actor_critic.act_item(states[i], res[i], det)
        assert lib.hrp_ppo_act_multi(items, len(dims), torch.cuda.current_stream().cuda_stream) == 0
        torch.cuda.synchronize()
        for i, a in enumerate(agents):
            ac = a.actor_critic
            mean, std, value = ac.forward(states[i])
            got = res[i].cpu().numpy()
            np.testing.assert_allclose(got[5], value.cpu().numpy().reshape(()), atol=2e-6, rtol=2e-6)
            if det:
                np.testing.assert_allclose(got[2:4], mean.cpu().numpy().reshape(-1), atol=2e-6, rtol=2e-6)
                assert got[4] == 0.0
            else:
                # the same noise as the batched sampling path with the same (seed, row, draw)
                want = ac.act(torch.cat([states[i], states[i]]), out=None)   # B = 2 -> tensor-core path, draw + 1
                z = got[2:4]
                n_multi = (z - mean.cpu().numpy().reshape(-1)) / std.cpu().numpy()
                n_batch = ((want["pre_tanh"][0] - mean.view(-1)) / std).cpu().numpy()
                assert np.all(np.isfinite(n_multi)) and np.abs(n_multi).max() < 6 and np.abs(n_batch).max() < 6
                logp, _, _ = ac.evaluate(states[i], None, torch.from_numpy(z).to("cuda:0").view(1, 2))
                np.testing.assert_allclose(got[4], logp.cpu().numpy().reshape(()), atol=3e-5, rtol=1e-5)
            np.testing.assert_allclose(got[0:2], np.tanh(got[2:4]), atol=1e-6)
    # ActorCritic.act with one state == the item path, bit for bit
    torch.manual_seed(31)
    a = _agent(60, 2, 256, 8)
    torch.manual_seed(31)
    b = _agent(60, 2, 256, 8)
    x = torch.randn(1, 60, device="cuda:0")
    o1 = a.act(x)
    row = torch.zeros(6, device="cuda:0")
    it = b.actor_critic.act_item(x, row, False)
    assert lib.hrp_ppo_act_multi(C.byref(it), 1, torch.cuda.current_stream().cuda_stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(o1["action"].view(-1), row[0:2]) and torch.equal(o1["pre_tanh"].view(-1), row[2:4])
    assert torch.equal(o1["log_prob"].view(-1), row[4:5]) and torch.equal(o1["value"].view(-1), row[5:6])


@pytest.mark.parametrize("A,H,B", [(1, 128, 256), (2, 256, 4096), (4, 384, 1000), (3, 64, 64), (2, 512, 130)])
def test_fused_heads_act_path_matches_the_unfused_forward(A, H, B):
    """The act path with the heads fused into the [a1 | c1] GEMM's epilogue (TcDots + heads_finish_kernel; taken whenever
    the N tiles do not straddle H) against forward() (separate heads kernel): deterministic actions are the means,
    values agree, for 1 to 4 action dimensions, whole and ragged M tiles, 64- and 128-wide N tiles; and the sampled
    path's log-prob is the one evaluate() assigns to its own pre-tanh sample."""
    torch.manual_seed(40 + A)
    agent = _agent(60, A, H, B)
    ac = agent.actor_critic
    x = torch.randn(B, 60, device="cuda:0") * 0.4
    mean, std, value = ac.forward(x)
    det = ac.act(x, deterministic=True)
    scale = float(mean.abs().max()) + 1e-3
    np.testing.assert_allclose(det["pre_tanh"].cpu().numpy(), mean.cpu().numpy(), atol=3e-6 * max(1.0, scale))
    np.testing.assert_allclose(det["value"].cpu().numpy(), value[:, 0].cpu().numpy(), atol=3e-6 * max(1.0, float(value.abs().max())))
    np.testing.assert_allclose(det["action"].cpu().numpy(), np.tanh(det["pre_tanh"].cpu().numpy()), atol=1e-6)
    out = ac.act(x)
    logp, _, _ = ac.evaluate(x, None, out["pre_tanh"])
    # log(1 - tanh(z)^2 + 1e-6) is ill-conditioned for a saturated action (|z| > 4: 1 - t^2 ~ 1e-4, one ulp of t moves it
    # by 1e-3 relative), per action dimension
    np.testing.assert_allclose(out["log_prob"].cpu().numpy(), logp.cpu().numpy(), atol=1e-4 * A, rtol=3e-5)
    n = ((out["pre_tanh"] - mean) / std).flatten()
    assert abs(float(n.mean())) < 0.2 and 0.7 < float(n.std()) < 1.3
