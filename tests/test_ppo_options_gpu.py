"""GPU checks of the PPO update options: the clipped value loss (``hrp_ppo_loss_grad_ex``, ``PPOAgent(clip_value=...)``)
against the fp64 oracle (tests/ppo_options_oracle.py), the learning rate read from device memory
(``hrp_clip_adam_step_ex``, ``hrp_clip_adam_step_p2p_ex``, ``PPOAgent.set_lr``) against the by-value kernels bit for bit,
captured minibatch graphs that survive ``set_lr``, ``train_vectorized(anneal_lr=True)`` and checkpoints.

Tolerances are those of tests/test_ppo_gpu.py and tests/test_categorical_gpu.py: loss terms 2e-5, gradients 1e-4 of
the gradient's max-abs + 2e-6, parameters after a full update 1e-4 of their largest motion.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import ppo_categorical_ref as cref
from oracle import ppo_ref
from ppo_options_oracle import loss_and_grad, loss_and_grad_cat
from test_env_gpu import _cfg, _vec
from test_fast_env_cpu import FAST
from test_fast_env_gpu import _fast

pytestmark = pytest.mark.gpu


def _lib():
    from highway_rope_ppo_b200 import _lib

    return _lib, _lib.load()


def _agent(S, A, H, B, discrete, **kw):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    return PPOAgent(S, A, lr=3e-4, hidden_dim=H, batch_size=B, device="cuda:0", discrete=discrete, **kw)


def _relu_margin(flat, x, S, A, H, discrete):
    """Per row, the smallest |pre-activation| of the four hidden ReLU layers (fp64)."""
    p = (cref if discrete else ppo_ref).unflatten(flat, S, A, H)
    z1 = x @ p["shared.0.weight"].T + p["shared.0.bias"]
    z2 = torch.relu(z1) @ p["shared.2.weight"].T + p["shared.2.bias"]
    h2 = torch.relu(z2)
    za = h2 @ p["actor_mean.0.weight"].T + p["actor_mean.0.bias"]
    zc = h2 @ p["critic.0.weight"].T + p["critic.0.bias"]
    return torch.cat([z1, z2, za, zc], 1).abs().min(1).values


def _minibatch(agent, B, seed):
    """Random states, samples, old log-probs, advantages and returns of one minibatch (fp64, CPU) and the oracle's
    fp64 value of every row.

    The states are drawn away from the ReLU kinks: a row with a hidden pre-activation within fp32 rounding of 0 is
    masked differently by the fp32 kernels and the fp64 oracle, which moves bias and weight gradients by far more than
    the tolerance whether or not the value loss is clipped (hrp_ppo_loss_grad against the unclipped oracle shows it on
    the same states).  Such rows are redrawn, so the comparison measures the loss arithmetic, not mask flips."""
    ac = agent.actor_critic
    S, A, H = ac.state_dim, ac.action_dim, ac.hidden_dim
    g = torch.Generator().manual_seed(seed)
    flat = ac.flat.cpu().double()
    rows = []
    while sum(len(r) for r in rows) < B:
        cand = (torch.randn(B, S, generator=g) * 0.5).double()
        rows.append(cand[_relu_margin(flat, cand, S, A, H, agent.discrete) > 1e-4])
    x = torch.cat(rows)[:B]
    if agent.discrete:
        act = torch.randint(0, A, (B,), generator=g)
        logp, value, _ = cref.evaluate(flat, x, act, S, A, H)
        pre = act.float().view(B, 1)
    else:
        mean, _, _ = ppo_ref.forward(flat, x, S, A, H)
        act = mean + torch.randn(B, A, generator=g, dtype=torch.float64)
        act = act.float().double()
        logp, value, _ = ppo_ref.evaluate(flat, x, act, S, A, H)
        pre = act.float()
    old = logp.detach() + 0.2 * torch.randn(B, generator=g, dtype=torch.float64)
    # likewise rows on the surrogate's clip kink (ratio = 1 +- eps), where fp32 and fp64 may take different branches:
    # move them 1 % away
    ratio = torch.exp(logp.detach() - old)
    old = torch.where(((ratio - 0.8).abs() < 2e-3) | ((ratio - 1.2).abs() < 2e-3), old - 0.01, old).float().double()
    adv = torch.randn(B, generator=g, dtype=torch.float64).float().double()
    return g, x.float().double(), act, pre, old, adv, value.detach().squeeze(-1)


def _old_values(v, c, g):
    """Old values and returns that make every case of the clipped term occur, each with a margin to the kinks that the
    fp32 kernel's value (within 2e-5 of the fp64 one) cannot cross: v - v_old = +-2c or +-3c (outside the clamp) with a
    return that makes the clipped branch win or lose by 0.6 c^2, and |v - v_old| <= c/2 (inside: v_old + (v - v_old)
    rounds to v, a tie whose halves both pass)."""
    B = v.numel()
    kind = torch.arange(B) % 5
    s = torch.where(torch.rand(B, generator=g) < 0.5, 1.0, -1.0).double()
    mag = torch.where(torch.rand(B, generator=g) < 0.5, 2.0, 3.0).double()
    vo = torch.where(kind < 4, v - s * mag * c, v - s * c * 0.5 * torch.rand(B, generator=g, dtype=torch.float64))
    # outside: the clipped value is v - s c; it wins iff s (v - R) < c / 2
    d = s * torch.where(kind % 2 == 0, 0.2 * c, 0.8 * c)
    R = torch.where(kind < 4, v - d, v + torch.randn(B, generator=g, dtype=torch.float64))
    return vo.float().double(), R.float().double(), kind


def _ex(lib, agent, dev, idx, B, old_value, clip):
    ac = agent.actor_critic
    agent._metrics.zero_()
    return lib.hrp_ppo_loss_grad_ex(ac._h, ac.flat.data_ptr(), dev["states"].data_ptr(), dev["pre_tanh"].data_ptr(),
                                    dev["log_prob"].data_ptr(), dev["adv"].data_ptr(), dev["ret"].data_ptr(),
                                    None if idx is None else idx.data_ptr(), B, 0.2, 0.5, 0.005, 1.0 / B,
                                    None if old_value is None else old_value.data_ptr(), clip, agent.grad.data_ptr(),
                                    agent._metrics.data_ptr(), torch.cuda.current_stream().cuda_stream)


SIZES = [(60, 256, 64), (60, 256, 4096), (20, 32, 17), (600, 512, 64), (60, 128, 256)]
POLICIES = [(False, 2), (True, 5), (True, 8)]


@pytest.mark.parametrize("mode", [3, 0])
@pytest.mark.parametrize("S,H,B", SIZES)
@pytest.mark.parametrize("discrete,A", POLICIES, ids=["gaussian-2", "categorical-5", "categorical-8"])
def test_loss_grad_ex_matches_oracle(discrete, A, S, H, B, mode):
    _l, lib = _lib()
    prev = lib.hrp_ppo_get_math()
    _l.check(lib.hrp_ppo_set_math(mode))
    try:
        torch.manual_seed(S + A + H + B)
        agent = _agent(S, A, H, B, discrete)
        c = 1.0   # value residuals of the size the existing tests have, so the gradient tolerance means the same
        g, x, act, pre, old, adv, v = _minibatch(agent, B, 3)
        vo, R, kind = _old_values(v, c, g)
        fn = loss_and_grad_cat if discrete else loss_and_grad
        flat64 = agent.actor_critic.flat.cpu().double()
        r = fn(flat64, x, act, old, adv, R, S, A, H, old_value=vo, clip_value=c)
        # the cases, as the fp64 oracle decides them
        l1 = (v - R) ** 2
        l2 = (vo + torch.clamp(v - vo, -c, c) - R) ** 2
        if B >= 64:
            assert (l2[kind < 4] > l1[kind < 4]).any() and (l1[kind < 4] > l2[kind < 4]).any()
            assert ((v - vo).abs()[kind == 4] <= c).all()
        dev = {"states": x.float().cuda(), "pre_tanh": pre.cuda(), "log_prob": old.float().cuda(),
               "adv": adv.float().cuda(), "ret": R.float().cuda()}
        vo_dev = vo.float().cuda()
        # direct rows and rows gathered out of a larger rollout through idx
        perm = torch.randperm(B, generator=g)
        big = {k: torch.zeros((2 * B,) + t.shape[1:], dtype=t.dtype, device="cuda:0") for k, t in dev.items()}
        big_vo = torch.zeros(2 * B, device="cuda:0")
        src = (2 * perm).cuda()
        for k in dev:
            big[k][src] = dev[k]
        big_vo[src] = vo_dev
        for d, vv, idx in ((dev, vo_dev, None), (big, big_vo, src)):
            _l.check(_ex(lib, agent, d, idx, B, vv, c), "hrp_ppo_loss_grad_ex")
            m = agent._metrics.cpu().numpy()
            assert abs(m[0] - r["loss"]) < 2e-5 * max(1.0, abs(r["loss"])) and abs(m[1] - r["actor"]) < 2e-5
            assert abs(m[2] - r["critic"]) < 2e-5 * max(1.0, r["critic"])
            assert abs(m[3] - r["entropy"]) < 2e-5 and abs(m[5] - r["approx_kl"]) < 2e-5 and m[6] == 1.0
            want = r["grad"].numpy()
            np.testing.assert_allclose(agent.grad.cpu().numpy(), want, atol=1e-4 * np.abs(want).max() + 2e-6)
    finally:
        lib.hrp_ppo_set_math(prev)


# (v_old - v, R - v) for v = 0.25 exactly, c = 0.5 -> d(term)/dv, worked out by hand (tests/test_ppo_options_cpu.py)
EXACT_CASES = {
    "boundary +c": (-0.5, 1.75, 2 * -1.75),     # v - v_old = c: v_clip = v, a tie whose halves both pass
    "boundary -c": (0.5, -1.75, 2 * 1.75),
    "tie outside": (-1.0, -0.25, 0.5 * 2 * 0.25),   # (v - R)^2 = (v_old + c - R)^2, the clamp blocks its half
    "clipped wins": (-1.0, 0.75, 0.0),
    "unclipped wins": (-1.0, -1.25, 2 * 1.25),
    "inside": (0.125, 1.0, 2 * -1.0),
}


@pytest.mark.parametrize("case", list(EXACT_CASES))
@pytest.mark.parametrize("discrete,A", [(False, 2), (True, 5)], ids=["gaussian", "categorical"])
def test_loss_grad_ex_boundary_and_tie_rows(discrete, A, case):
    """critic.2.weight = 0 makes every value exactly critic.2.bias = 0.25 in the kernel and in the oracle, so the old
    values and returns can put every row exactly on a clamp boundary or a tie.  d(loss)/d(critic.2.bias) is then
    value_coef * the hand-worked derivative, and the whole gradient matches the oracle."""
    _l, lib = _lib()
    S, H, B, c = 20, 32, 17, 0.5
    torch.manual_seed(4)
    agent = _agent(S, A, H, B, discrete)
    sd = agent.actor_critic.state_dict()
    sd["critic.2.weight"].zero_()
    sd["critic.2.bias"].fill_(0.25)
    agent.actor_critic.load_state_dict(sd)
    g, x, act, pre, old, adv, v = _minibatch(agent, B, 5)
    assert (v == 0.25).all()
    dvo, dR, dv = EXACT_CASES[case]
    vo, R = torch.full((B,), 0.25 + dvo, dtype=torch.float64), torch.full((B,), 0.25 + dR, dtype=torch.float64)
    fn = loss_and_grad_cat if discrete else loss_and_grad
    r = fn(agent.actor_critic.flat.cpu().double(), x, act, old, adv, R, S, A, H, old_value=vo, clip_value=c)
    dev = {"states": x.float().cuda(), "pre_tanh": pre.cuda(), "log_prob": old.float().cuda(), "adv": adv.float().cuda(),
           "ret": R.float().cuda()}
    _l.check(_ex(lib, agent, dev, None, B, vo.float().cuda(), c), "hrp_ppo_loss_grad_ex")
    grad = agent.grad.cpu()
    assert float(grad[-1]) == pytest.approx(0.5 * dv, rel=1e-6, abs=1e-7)
    assert float(r["grad"][-1]) == pytest.approx(0.5 * dv, rel=1e-12, abs=1e-12)
    want = r["grad"].numpy()
    np.testing.assert_allclose(grad.numpy(), want, atol=1e-4 * np.abs(want).max() + 2e-6)
    assert abs(agent._metrics[2].item() - r["critic"]) < 2e-5 * max(1.0, r["critic"])


@pytest.mark.parametrize("gather", [False, True])
@pytest.mark.parametrize("discrete,A", [(False, 2), (True, 5)], ids=["gaussian", "categorical"])
def test_loss_grad_ex_without_old_values_is_loss_grad_bit_for_bit(discrete, A, gather):
    _l, lib = _lib()
    S, H, B = 60, 256, 4096
    torch.manual_seed(9)
    agent = _agent(S, A, H, B, discrete)
    ac = agent.actor_critic
    g, x, act, pre, old, adv, v = _minibatch(agent, B, 6)
    dev = {"states": x.float().cuda(), "pre_tanh": pre.cuda(), "log_prob": old.float().cuda(), "adv": adv.float().cuda(),
           "ret": (v + torch.randn(B, generator=g, dtype=torch.float64)).float().cuda()}
    idx = torch.randperm(B, generator=g).cuda() if gather else None
    st = torch.cuda.current_stream().cuda_stream
    agent._metrics.zero_()
    _l.check(lib.hrp_ppo_loss_grad(ac._h, ac.flat.data_ptr(), dev["states"].data_ptr(), dev["pre_tanh"].data_ptr(),
                                   dev["log_prob"].data_ptr(), dev["adv"].data_ptr(), dev["ret"].data_ptr(),
                                   None if idx is None else idx.data_ptr(), B, 0.2, 0.5, 0.005, 1.0 / B,
                                   agent.grad.data_ptr(), agent._metrics.data_ptr(), st))
    g0, m0 = agent.grad.clone(), agent._metrics.clone()
    _l.check(_ex(lib, agent, dev, idx, B, None, float("nan")), "hrp_ppo_loss_grad_ex")
    assert torch.equal(agent.grad, g0) and torch.equal(agent._metrics, m0)


def test_clip_adam_step_ex_with_device_lr_is_bit_identical():
    """hrp_clip_adam_step_ex with *lr_dev == lr against hrp_clip_adam_step, and hrp_clip_adam_step_p2p_ex against
    hrp_clip_adam_step_p2p with a world of one rank: parameters, both moments and the step counter, step after step,
    at several learning rates (clipped and unclipped steps)."""
    _l, lib = _lib()
    n = 213765
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device="cuda:0").manual_seed(3)
    comm, handle = C.c_void_p(), (C.c_ubyte * 64)()
    _l.check(lib.hrp_comm_create(1, 0, n, 0, C.byref(comm), handle))
    _l.check(lib.hrp_comm_connect(comm, bytes(handle)))
    try:
        keep, grads = [], []
        for parity in (0, 1):
            ptr = lib.hrp_comm_grad_parity(comm, parity)

            class _Raw:
                __cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (int(ptr), False), "version": 2}

            keep.append(_Raw())
            grads.append(torch.as_tensor(keep[-1], device="cuda:0"))
        p0 = torch.randn(n, generator=g, device="cuda:0") * 0.1
        # [by value, device lr] x [plain, p2p]: params, exp_avg, exp_avg_sq, step, scratch
        runs = [[p0.clone(), torch.zeros(n, device="cuda:0"), torch.zeros(n, device="cuda:0"),
                 torch.zeros(1, dtype=torch.int32, device="cuda:0"), torch.zeros(128, device="cuda:0")] for _ in range(4)]
        lr_dev = torch.zeros(1, dtype=torch.float64, device="cuda:0")
        comm2, handle2 = C.c_void_p(), (C.c_ubyte * 64)()
        _l.check(lib.hrp_comm_create(1, 0, n, 0, C.byref(comm2), handle2))
        _l.check(lib.hrp_comm_connect(comm2, bytes(handle2)))
        ptrs2 = [lib.hrp_comm_grad_parity(comm2, p) for p in (0, 1)]
        try:
            for it, lr in enumerate([3e-4, 1e-4, 2.5e-3, 1.2345678901234567e-4, 1e-2, 7e-5]):
                grad = torch.randn(n, generator=g, device="cuda:0") * (0.5 if it % 2 else 5e-4)
                lr_dev.fill_(lr)
                a, b, pa, pb = runs
                _l.check(lib.hrp_clip_adam_step(a[0].data_ptr(), grad.data_ptr(), a[1].data_ptr(), a[2].data_ptr(),
                                                a[3].data_ptr(), n, lr, 0.9, 0.999, 1e-8, 0.5, a[4].data_ptr(), st))
                _l.check(lib.hrp_clip_adam_step_ex(b[0].data_ptr(), grad.data_ptr(), b[1].data_ptr(), b[2].data_ptr(),
                                                   b[3].data_ptr(), n, 0.5, lr_dev.data_ptr(), 0.9, 0.999, 1e-8, 0.5,
                                                   b[4].data_ptr(), st))
                grads[lib.hrp_comm_parity(comm)].copy_(grad)
                _l.check(lib.hrp_clip_adam_step_p2p(comm, pa[0].data_ptr(), pa[1].data_ptr(), pa[2].data_ptr(),
                                                    pa[3].data_ptr(), lr, 0.9, 0.999, 1e-8, 0.5, pa[4].data_ptr(), st))
                g2 = torch.as_tensor(type("_R", (), {"__cuda_array_interface__": {
                    "shape": (n,), "typestr": "<f4", "data": (int(ptrs2[lib.hrp_comm_parity(comm2)]), False),
                    "version": 2}})(), device="cuda:0")
                g2.copy_(grad)
                _l.check(lib.hrp_clip_adam_step_p2p_ex(comm2, pb[0].data_ptr(), pb[1].data_ptr(), pb[2].data_ptr(),
                                                       pb[3].data_ptr(), 0.5, lr_dev.data_ptr(), 0.9, 0.999, 1e-8, 0.5,
                                                       pb[4].data_ptr(), st))
                torch.cuda.synchronize()
                for x, y in ((a, b), (pa, pb)):
                    for k in range(4):
                        assert torch.equal(x[k], y[k]), (it, lr, k)
                assert int(a[3].item()) == it + 1
                assert not torch.equal(a[0], p0)
            _l.check(lib.hrp_comm_status(comm))
            _l.check(lib.hrp_comm_status(comm2))
        finally:
            lib.hrp_comm_destroy(comm2)
    finally:
        lib.hrp_comm_destroy(comm)


def _fill_rollout(agent, T, E, seed):
    """A synthetic [T, E] rollout in the agent's memory; returns the host arrays the oracle update needs."""
    ac = agent.actor_critic
    S, A, H = ac.state_dim, ac.action_dim, ac.hidden_dim
    rng = np.random.default_rng(seed)
    N = T * E
    states = (rng.standard_normal((T + 1, E, S)) * 0.5).astype(np.float32)
    X = torch.from_numpy(states[:T].reshape(N, S)).double()
    flat0 = ac.flat.cpu().double()
    if agent.discrete:
        lg, _ = cref.forward(flat0, X, S, A, H)
        p = torch.softmax(lg, -1).numpy()
        act = np.array([rng.choice(A, p=pr / pr.sum()) for pr in p])
        logp = torch.log_softmax(lg, -1).numpy()[np.arange(N), act]
        pre = act.reshape(T, E, 1).astype(np.float32)
        action = np.stack([act.reshape(T, E), np.zeros((T, E))], -1).astype(np.float32)
        act_t = torch.from_numpy(act)
    else:
        mean, _, _ = ppo_ref.forward(flat0, X, S, A, H)
        z = (mean.numpy() + rng.standard_normal((N, A))).astype(np.float32)
        act_t = torch.from_numpy(z).double()
        logp = ppo_ref.evaluate(flat0, X, act_t, S, A, H)[0].detach().numpy()
        pre, action = z.reshape(T, E, A), np.tanh(z).reshape(T, E, A)
    old = (logp + 0.1 * rng.standard_normal(N)).astype(np.float32)
    value = rng.standard_normal((T, E)).astype(np.float32)
    reward = rng.standard_normal((T, E)).astype(np.float32)
    done = rng.random((T, E)) < 0.1
    r = agent.memory.begin_rollout(T, E, S, action.shape[-1], pre.shape[-1])
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    for k, a in (("states", states), ("action", action), ("pre_tanh", pre), ("log_prob", old.reshape(T, E)),
                 ("value", value), ("reward", reward), ("done", done.astype(np.uint8))):
        r[k].copy_(cu(a))
    return X, act_t, old, value, reward, done


@pytest.mark.parametrize("discrete,A", [(False, 2), (True, 5)], ids=["gaussian", "categorical"])
def test_full_update_with_clip_value_and_set_lr_matches_oracle(discrete, A):
    """PPOAgent(clip_value=0.2).update after set_lr(2e-4) equals the oracle's update (GAE, normalisation, the same
    minibatch permutation, the clipped value loss and clip + Adam at lr 2e-4 per minibatch), two updates in a row with
    a different lr each: the second replays the graphs the first captured."""
    S, H, T, E, bs, epochs, c = 12, 16, 10, 10, 25, 3, 0.2
    torch.manual_seed(5)
    agent = _agent(S, A, H, bs, discrete, epochs=epochs, clip_value=c)
    flat = agent.actor_critic.flat.cpu().double()
    flat_start = flat.clone()
    m = torch.zeros_like(flat)
    v = torch.zeros_like(flat)
    step = 0
    fn = loss_and_grad_cat if discrete else loss_and_grad
    for u, lr in enumerate((2e-4, 5e-5)):
        X, act, old, value, reward, done = _fill_rollout(agent, T, E, u)
        N = T * E
        last = np.random.default_rng(10 + u).standard_normal(E).astype(np.float32)
        agent.set_lr(lr)
        np.random.seed(11 + u)
        metrics = agent.update(last_value=torch.from_numpy(last).cuda())
        adv = np.zeros((T, E), dtype=np.float32)
        for e in range(E):
            adv[:, e], _ = ppo_ref.gae(reward[:, e], value[:, e], done[:, e], last[e])
        ret = torch.from_numpy((adv + value).reshape(N)).double()
        advn = torch.from_numpy(adv.reshape(N)).double()
        advn = (advn - advn.mean()) / (advn.std() + 1e-8)
        np.random.seed(11 + u)
        perm = np.arange(N, dtype=np.int64)
        np.random.shuffle(perm)
        vo, oldt, mets = torch.from_numpy(value.reshape(N)).double(), torch.from_numpy(old).double(), []
        for _ in range(epochs):
            for start in range(0, N, bs):
                i = torch.from_numpy(perm[start:start + bs])
                rr = fn(flat, X[i], act[i], oldt[i], advn[i], ret[i], S, A, H, old_value=vo[i], clip_value=c)
                step += 1
                flat, m, v, _ = ppo_ref.clip_adam(flat, rr["grad"], m, v, step, lr=lr)
                mets.append(rr)
        want = {k: float(np.mean([q[src] for q in mets])) for k, src in
                (("loss", "loss"), ("policy_loss", "actor"), ("value_loss", "critic"), ("entropy", "entropy"))}
        for k in want:
            assert abs(metrics[k] - want[k]) <= 2e-3 * max(1.0, abs(want[k])), (u, k, metrics[k], want[k])
        if u == 0:
            graphs = dict(agent._graph_state["graphs"])
            assert graphs
    assert agent._graph_state["graphs"] == graphs and all(agent._graph_state["graphs"][k] is g for k, g in graphs.items())
    p1 = agent.actor_critic.flat.cpu().numpy()
    moved = np.abs(flat.numpy() - flat_start.numpy()).max()
    err = np.abs(p1 - flat.numpy()).max()
    print(f"options update: max parameter motion {moved:.3e}, max error {err:.3e} = {err / moved:.2e} of it")
    assert err <= 1e-4 * moved
    assert agent.optimizer.lr == 5e-5 and agent.optimizer.lr_dev.item() == 5e-5


@pytest.mark.parametrize("clip_value", [None, 0.1])
@pytest.mark.parametrize("discrete,A", [(False, 2), (True, 5)], ids=["gaussian", "categorical"])
def test_set_lr_reuses_the_captured_graphs_and_equals_the_eager_twin(discrete, A, clip_value):
    S, H, T, E, bs = 60, 128, 8, 256, 512
    agents = []
    for graphs in (True, False):
        torch.manual_seed(3)
        a = _agent(S, A, H, bs, discrete, epochs=2, clip_value=clip_value)
        a.use_cuda_graphs = graphs
        agents.append(a)
    g_agent, e_agent = agents
    assert torch.equal(g_agent.actor_critic.flat, e_agent.actor_critic.flat)
    seen = None
    for u, lr in enumerate((3e-4, 2.25e-4, 1.5e-4, 7.5e-5)):
        for a in agents:
            _fill_rollout(a, T, E, 100 + u)
            a.set_lr(lr)
            np.random.seed(u)
            a.update(last_value=0.0)
        assert torch.equal(g_agent.actor_critic.flat, e_agent.actor_critic.flat), u
        assert torch.equal(g_agent.optimizer.exp_avg_sq, e_agent.optimizer.exp_avg_sq), u
        st = g_agent._graph_state
        now = (id(st), {k: id(g) for k, g in st["graphs"].items()})
        assert st["graphs"] and (seen is None or now == seen), u
        seen = now
    assert e_agent._graph_state is None


def test_by_value_lr_changes_still_recapture():
    """Without set_lr the learning rate is a launch argument: assigning optimizer.lr re-captures, as before."""
    torch.manual_seed(3)
    agent = _agent(60, 2, 128, 512, False, epochs=2)
    ids = []
    for u, lr in enumerate((3e-4, 3e-4, 1e-4)):
        _fill_rollout(agent, 8, 256, u)
        agent.optimizer.lr = lr
        agent.update(last_value=0.0)
        ids.append(id(agent._graph_state))
    assert ids[0] == ids[1] != ids[2] and agent.optimizer.lr_dev is None


def test_checkpoint_roundtrip_restores_lr_and_device_value(tmp_path):
    path = str(tmp_path / "c.pth")
    torch.manual_seed(1)
    a = _agent(20, 2, 32, 64, False, clip_value=0.2)
    a.set_lr(1.25e-4)
    a.save(path)
    assert a.optimizer.state_dict()["param_groups"][0]["lr"] == 1.25e-4
    b = _agent(20, 2, 32, 64, False)
    b.set_lr(9e-4)
    b.load(path)
    assert b.optimizer.lr == 1.25e-4 and b.optimizer.lr_dev.item() == 1.25e-4
    c = _agent(20, 2, 32, 64, False)   # by-value mode: the value comes back, no device copy appears
    c.load(path)
    assert c.optimizer.lr == 1.25e-4 and c.optimizer.lr_dev is None


def _env_and_agent(highway_config, gym_id, discrete, E, seed, **kw):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    if gym_id == FAST:
        cfg = _fast(meta=discrete)
    else:
        cfg = _cfg(highway_config)
        if discrete:
            cfg["action"] = {"type": "DiscreteMetaAction"}
    env = _vec(cfg, E, seed=seed)
    torch.manual_seed(seed)
    agent = PPOAgent(env.N * env.F_out, 5 if discrete else 2, lr=3e-4, hidden_dim=64, batch_size=512, epochs=2,
                     discrete=discrete, **kw)
    return env, agent


@pytest.mark.parametrize("gym_id", ["highway-v0", FAST])
@pytest.mark.parametrize("discrete", [False, True], ids=["gaussian", "categorical"])
def test_train_vectorized_anneal_lr_equals_a_manual_set_lr_loop(highway_config, gym_id, discrete):
    """train_vectorized(anneal_lr=True) with the clipped value loss is bit for bit a loop that calls set_lr with the
    schedule before every rollout_and_update; it records the schedule and captures the minibatch graphs once."""
    from highway_rope_ppo_b200.training import routine

    E, T, iters, seed = 256, 8, 4, 7
    env, agent = _env_and_agent(highway_config, gym_id, discrete, E, seed, clip_value=0.2)
    np.random.seed(0)
    hist = routine.train_vectorized(env, agent, iters, T, seed=seed, anneal_lr=True)
    want_lr = [routine.linear_lr(3e-4, it, iters) for it in range(iters)]
    assert [m["lr"] for m in hist] == want_lr
    for m in hist:
        assert all(np.isfinite(m[k]) for k in ("loss", "policy_loss", "value_loss", "entropy"))
    env2, twin = _env_and_agent(highway_config, gym_id, discrete, E, seed, clip_value=0.2)
    np.random.seed(0)
    obs = env2.reset(seed=seed)
    graph_ids = None
    for it in range(iters):
        twin.set_lr(routine.linear_lr(3e-4, it, iters))
        m, obs = routine.rollout_and_update(env2, twin, T, obs)
        assert m["loss"] == hist[it]["loss"] and m["value_loss"] == hist[it]["value_loss"], it
        st = twin._graph_state
        ids = (id(st), sorted(id(g) for g in st["graphs"].values()))
        assert graph_ids is None or ids == graph_ids
        graph_ids = ids
    assert torch.equal(agent.actor_critic.flat, twin.actor_critic.flat)
    # without the flag the lr stays, and is recorded
    hist2 = routine.train_vectorized(env2, twin, 2, T, seed=seed)
    assert [m["lr"] for m in hist2] == [want_lr[-1]] * 2
    env.close()
    env2.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_update_with_options_keeps_ranks_bit_identical():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29647", os.path.join(root, "tools", "p2p_check.py"), "--ppo-options"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    out = res.stdout
    assert "anneal_lr + clip_value" in out and out.count("identical on every rank: True") >= 3, out[-3000:]
