"""target_kl early stopping on the device: the per-minibatch KL of ``hrp_ppo_loss_grad_kl`` against the fp64 oracle, the
Adam kernels' decisions, and whole updates that stop at a chosen minibatch -- graphed behind the conditional gate,
eager, and against an eager loop of the existing entry points run for exactly that many steps, bit for bit."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import ppo_categorical_ref as cref
from oracle import ppo_ref
from target_kl_oracle import stops
from test_fast_env_cpu import FAST
from test_ppo_options_gpu import _env_and_agent, _lib, _minibatch

pytestmark = pytest.mark.gpu


def _agent(S, A, H, B, discrete, **kw):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    return PPOAgent(S, A, lr=kw.pop("lr", 3e-4), hidden_dim=H, batch_size=B, device="cuda:0", discrete=discrete, **kw)


def _loss_kl(lib, agent, dev, B, kl_out, stop):
    ac = agent.actor_critic
    return lib.hrp_ppo_loss_grad_kl(ac._h, ac.flat.data_ptr(), dev["states"].data_ptr(), dev["pre_tanh"].data_ptr(),
                                    dev["log_prob"].data_ptr(), dev["adv"].data_ptr(), dev["ret"].data_ptr(), None, B,
                                    0.2, 0.5, 0.005, 1.0 / B, None, 0.0, kl_out, stop, agent.grad.data_ptr(),
                                    agent._metrics.data_ptr(), torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("mode", [3, 0])
@pytest.mark.parametrize("discrete,A", [(False, 2), (True, 5)], ids=["gaussian-2", "categorical-5"])
def test_kl_out_matches_oracle_and_the_stop_word_gates_the_metrics(discrete, A, mode):
    """kl_out against the fp64 oracle's approx_kl.  Tolerance 2e-5 absolute, the one the existing tests hold
    metrics[5] to: the KL is the mean of (r - 1) - log r over values of ~1e-2, and with the fp32 log-probs within ~1e-5
    of fp64 (math mode 3's tensor-core GEMMs included) each term moves by well under that.  kl_out is metrics[5]'s
    increment, bit for bit; with the stop word set the metrics are untouched and the gradient is unchanged."""
    _l, lib = _lib()
    prev = lib.hrp_ppo_get_math()
    _l.check(lib.hrp_ppo_set_math(mode))
    try:
        S, H, B = 60, 256, 4096
        torch.manual_seed(S + A)
        agent = _agent(S, A, H, B, discrete)
        g, x, act, pre, old, adv, v = _minibatch(agent, B, 3)
        flat64 = agent.actor_critic.flat.cpu().double()
        r = (cref if discrete else ppo_ref).loss_and_grad(flat64, x, act, old, adv, v, S, A, H)
        dev = {"states": x.float().cuda(), "pre_tanh": pre.cuda(), "log_prob": old.float().cuda(),
               "adv": adv.float().cuda(), "ret": v.float().cuda()}
        P = agent.actor_critic.num_params
        kl_out = torch.full((1,), -1.0, device="cuda:0")
        stop = torch.zeros(1, dtype=torch.int32, device="cuda:0")
        agent._metrics.zero_()
        _l.check(_loss_kl(lib, agent, dev, B, kl_out.data_ptr(), stop.data_ptr()), "hrp_ppo_loss_grad_kl")
        m = agent._metrics.clone()
        grad = agent.grad[:P].clone()
        assert abs(float(kl_out) - r["approx_kl"]) < 2e-5, (float(kl_out), r["approx_kl"])
        assert kl_out.item() == m[5].item() and m[6].item() == 1.0
        stop.fill_(1)
        agent._metrics.zero_()
        _l.check(_loss_kl(lib, agent, dev, B, kl_out.data_ptr(), stop.data_ptr()), "hrp_ppo_loss_grad_kl")
        assert not agent._metrics.any() and torch.equal(agent.grad[:P], grad) and kl_out.item() == m[5].item()
        # without the pointers: the existing kernel, same gradient and metrics
        agent._metrics.zero_()
        _l.check(_loss_kl(lib, agent, dev, B, None, None), "hrp_ppo_loss_grad_kl")
        assert torch.equal(agent._metrics, m) and torch.equal(agent.grad[:P], grad)
    finally:
        lib.hrp_ppo_set_math(prev)


def _raw(ptr, n):
    class _R:
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (int(ptr), False), "version": 2}

    keep = _R()
    return keep, torch.as_tensor(keep, device="cuda:0")


def test_adam_kl_decisions_plain_and_peer_memory():
    """hrp_clip_adam_step_kl and hrp_clip_adam_step_p2p_kl (one rank, comm over P + 1 floats): a KL below or exactly at
    the limit steps as hrp_clip_adam_step_ex / hrp_clip_adam_step_p2p_ex do; one above it takes no step and raises the
    word; a raised word makes the next call a no-op whatever the KL."""
    _l, lib = _lib()
    n = 213765
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device="cuda:0").manual_seed(5)
    comm, handle = C.c_void_p(), (C.c_ubyte * 64)()
    _l.check(lib.hrp_comm_create(1, 0, n + 1, 0, C.byref(comm), handle))
    _l.check(lib.hrp_comm_connect(comm, bytes(handle)))
    comm2, handle2 = C.c_void_p(), (C.c_ubyte * 64)()
    _l.check(lib.hrp_comm_create(1, 0, n, 0, C.byref(comm2), handle2))
    _l.check(lib.hrp_comm_connect(comm2, bytes(handle2)))
    try:
        views = [_raw(lib.hrp_comm_grad_parity(comm, p), n + 1) for p in (0, 1)]
        views2 = [_raw(lib.hrp_comm_grad_parity(comm2, p), n) for p in (0, 1)]
        p0 = torch.randn(n, generator=g, device="cuda:0") * 0.1
        mk = lambda: [p0.clone(), torch.zeros(n, device="cuda:0"), torch.zeros(n, device="cuda:0"),
                      torch.zeros(1, dtype=torch.int32, device="cuda:0"), torch.zeros(128, device="cuda:0")]
        ref, plain, ref_peer, peer = mk(), mk(), mk(), mk()
        stop = torch.zeros(2, dtype=torch.int32, device="cuda:0")   # [plain, peer]
        limit = float(np.float32(0.03))
        # (kl, steps?): below, exactly at the limit, above (raises), then below again (word already set)
        for it, (kl, takes) in enumerate(((0.01, True), (limit, True), (float(np.nextafter(np.float32(limit), 1)), False),
                                          (0.0, False))):
            grad = torch.randn(n + 1, generator=g, device="cuda:0") * 0.3
            grad[n] = kl
            if takes:
                _l.check(lib.hrp_clip_adam_step_ex(ref[0].data_ptr(), grad.data_ptr(), ref[1].data_ptr(), ref[2].data_ptr(),
                                                   ref[3].data_ptr(), n, 3e-4, None, 0.9, 0.999, 1e-8, 0.5,
                                                   ref[4].data_ptr(), st))
                views2[lib.hrp_comm_parity(comm2)][1].copy_(grad[:n])
                _l.check(lib.hrp_clip_adam_step_p2p_ex(comm2, ref_peer[0].data_ptr(), ref_peer[1].data_ptr(),
                                                       ref_peer[2].data_ptr(), ref_peer[3].data_ptr(), 3e-4, None, 0.9, 0.999,
                                                       1e-8, 0.5, ref_peer[4].data_ptr(), st))
            _l.check(lib.hrp_clip_adam_step_kl(plain[0].data_ptr(), grad.data_ptr(), plain[1].data_ptr(),
                                               plain[2].data_ptr(), plain[3].data_ptr(), n, 3e-4, None, 0.9, 0.999, 1e-8,
                                               0.5, plain[4].data_ptr(), grad[n:].data_ptr(), stop.data_ptr(), limit, st))
            views[lib.hrp_comm_parity(comm)][1].copy_(grad)
            _l.check(lib.hrp_clip_adam_step_p2p_kl(comm, peer[0].data_ptr(), peer[1].data_ptr(), peer[2].data_ptr(),
                                                   peer[3].data_ptr(), 3e-4, None, 0.9, 0.999, 1e-8, 0.5, peer[4].data_ptr(),
                                                   stop[1:].data_ptr(), limit, st))
            torch.cuda.synchronize()
            for run, want in ((plain, ref), (peer, ref_peer)):
                for k in range(4):
                    assert torch.equal(run[k], want[k]), (it, k)
            assert stop.tolist() == ([0, 0] if it < 2 else [1, 1]), it
        assert int(ref[3].item()) == 2
        _l.check(lib.hrp_comm_status(comm))
    finally:
        lib.hrp_comm_destroy(comm)
        lib.hrp_comm_destroy(comm2)


def _fill(agent, T, E, seed):
    """A [T, E] rollout whose stored log-probs are the policy's own (fp64 oracle, rounded), so the first minibatch's KL
    is ~0 and grows as the update moves the policy."""
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
    else:
        mean, _, _ = ppo_ref.forward(flat0, X, S, A, H)
        z = (mean.numpy() + rng.standard_normal((N, A))).astype(np.float32)
        logp = ppo_ref.evaluate(flat0, X, torch.from_numpy(z).double(), S, A, H)[0].detach().numpy()
        pre, action = z.reshape(T, E, A), np.tanh(z).reshape(T, E, A)
    arrays = {"states": states, "action": action, "pre_tanh": pre, "log_prob": logp.astype(np.float32).reshape(T, E),
              "value": rng.standard_normal((T, E)).astype(np.float32),
              "reward": rng.standard_normal((T, E)).astype(np.float32),
              "done": (rng.random((T, E)) < 0.1).astype(np.uint8)}

    def load(a):
        r = a.memory.begin_rollout(T, E, S, action.shape[-1], pre.shape[-1])
        for k, v in arrays.items():
            r[k].copy_(torch.from_numpy(np.ascontiguousarray(v)).cuda())
    load(agent)
    return load


def _state(agent):
    o = agent.optimizer
    return [agent.actor_critic.flat.clone(), o.exp_avg.clone(), o.exp_avg_sq.clone(), o.step_dev.clone()]


def _restore(agent, s):
    o = agent.optimizer
    for dst, src in zip((agent.actor_critic.flat, o.exp_avg, o.exp_avg_sq, o.step_dev), s):
        dst.copy_(src)


def _limited(agent, k):
    """The agent's eager minibatch loop cut to the existing entry points: hrp_ppo_loss_grad + hrp_clip_adam_step for
    minibatches 0..k-1, the loss alone (metrics) for minibatch k, nothing after."""
    from highway_rope_ppo_b200 import _lib as L

    orig, count = agent._minibatch_step, [0]

    def step(flat, idx, B, world):
        i = count[0]
        count[0] += 1
        if i < k:
            orig(flat, idx, B, world)
        elif i == k:
            ac = agent.actor_critic
            L.check(agent._lib.hrp_ppo_loss_grad(ac._h, ac.flat.data_ptr(), flat["states"].data_ptr(),
                                                 flat["pre_tanh"].data_ptr(), flat["log_prob"].data_ptr(),
                                                 flat["adv"].data_ptr(), flat["ret"].data_ptr(), L.ptr(idx), B,
                                                 float(agent.eps_clip), float(agent.value_coef),
                                                 float(agent.entropy_coef), 1.0 / B, agent.grad.data_ptr(),
                                                 agent._metrics.data_ptr(), ac._stream()), "hrp_ppo_loss_grad")
    agent._minibatch_step = step
    return count


def _kl_sequence(discrete, A, S, H, T, E, bs, epochs, lr, **kw):
    """The per-minibatch approx-KL of an unstopped update (metrics[5]'s increment per step, the bits kl_out carries)."""
    torch.manual_seed(21)
    a = _agent(S, A, H, bs, discrete, epochs=epochs, lr=lr, **kw)
    a.use_cuda_graphs = False
    _fill(a, T, E, 4)
    orig, kls = a._minibatch_step, []

    def step(flat, idx, B, world):
        a._metrics.zero_()
        orig(flat, idx, B, world)
        kls.append(a._metrics[5].item())
    a._minibatch_step = step
    np.random.seed(8)
    a.update(last_value=0.0)
    return kls


def _choose(kls, lo, hi):
    """The last minibatch k in [lo, hi) whose KL is a clear record, and a limit between the earlier maximum and it (gap
    1e-4, five times the oracle tolerance of the KL)."""
    for k in reversed(range(lo, hi)):
        below = max(kls[:k])
        if kls[k] - below > 1e-4:
            return k, (below + kls[k]) / 2
    raise AssertionError(f"no clear KL record in [{lo}, {hi}): {kls}")


LAYOUTS = {"per-minibatch": (8, 512, 512, 4), "shared": (8, 256, 32, 2)}   # T, E, batch size, epochs


@pytest.mark.parametrize("mode", [3, 0])
@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("discrete,A", [(False, 2), (True, 5)], ids=["gaussian-2", "categorical-5"])
def test_update_stops_at_the_chosen_minibatch_bit_for_bit(discrete, A, layout, mode):
    """The limit is set between the largest KL before minibatch k and minibatch k's.  The graphed update (gated replays
    after a warm-up update, so every step of it is a gated replay) stops at k: parameters, moments and step_dev equal
    the eager target_kl update and an eager loop of the existing entry points run for k steps, bit for bit; the gate
    opened k + 1 times; the metrics are those of minibatches 0..k."""
    _l, lib = _lib()
    prev = lib.hrp_ppo_get_math()
    _l.check(lib.hrp_ppo_set_math(mode))
    try:
        S, H, lr = 60, 64, 2e-3
        T, E, bs, epochs = LAYOUTS[layout]
        M = T * E // bs
        assert (M <= 32) == (layout == "per-minibatch")
        kls = _kl_sequence(discrete, A, S, H, T, E, bs, epochs, lr)
        assert len(kls) == M * epochs and kls[0] < 1e-5
        k, limit = _choose(kls, 1, M * epochs - 1)
        target = limit / 1.5
        assert not any(stops(x, target) for x in kls[:k]) and stops(kls[k], target)
        agents = {}
        for name in ("graphed", "eager", "limited"):
            torch.manual_seed(21)
            agents[name] = _agent(S, A, H, bs, discrete, epochs=epochs, lr=lr,
                                  target_kl=None if name == "limited" else target)
            agents[name].use_cuda_graphs = name == "graphed"
        gr = agents["graphed"]
        load = _fill(gr, T, E, 4)
        s0 = _state(gr)
        np.random.seed(8)
        gr.update(last_value=0.0)   # warm-up: captures every graph
        _restore(gr, s0)
        load(gr)
        out = {}
        for name, a in agents.items():
            if name != "graphed":
                load(a)
            if name == "limited":
                count = _limited(a, k)
            np.random.seed(8)
            out[name] = a.update(last_value=0.0)
        assert count[0] == M * epochs
        assert gr._kl_state.tolist() == [1, k + 1]
        for name in ("eager", "limited"):
            o = agents[name].optimizer
            assert torch.equal(agents[name].actor_critic.flat, gr.actor_critic.flat), name
            assert torch.equal(o.exp_avg, gr.optimizer.exp_avg) and torch.equal(o.exp_avg_sq, gr.optimizer.exp_avg_sq)
            assert int(o.step_dev.item()) == k == int(gr.optimizer.step_dev.item()), name
            for key in ("loss", "policy_loss", "value_loss", "entropy", "clip_fraction", "approx_kl"):
                assert out[name][key] == out["graphed"][key], (name, key)
        assert out["graphed"]["optimizer_steps"] == k and out["graphed"]["stopped_early"] is True
        assert out["eager"]["optimizer_steps"] == k and out["eager"]["stopped_early"] is True
        assert "optimizer_steps" not in out["limited"]
        assert abs(out["graphed"]["approx_kl"] - float(np.mean(kls[:k + 1]))) < 1e-6
    finally:
        lib.hrp_ppo_set_math(prev)


@pytest.mark.parametrize("discrete,A", [(False, 2), (True, 5)], ids=["gaussian-2", "categorical-5"])
def test_limit_equal_to_a_kl_does_not_stop_there(discrete, A):
    """A limit equal to minibatch k's KL (as a double) does not stop at k -- the test is strict -- and the update stops at
    the first later minibatch whose KL is larger; never stopping when none is."""
    S, H, lr, (T, E, bs, epochs) = 60, 64, 2e-3, LAYOUTS["per-minibatch"]
    kls = _kl_sequence(discrete, A, S, H, T, E, bs, epochs, lr)
    k, _ = _choose(kls, 1, len(kls) - 1)
    limit = kls[k]
    want = next((j for j in range(len(kls)) if kls[j] > limit), None)
    assert want is None or want > k
    torch.manual_seed(21)
    a = _agent(S, A, H, bs, discrete, epochs=epochs, lr=lr, target_kl=limit / 1.5)
    if 1.5 * (limit / 1.5) != limit:
        pytest.skip("1.5 * (limit / 1.5) does not round back to the limit")
    _fill(a, T, E, 4)
    np.random.seed(8)
    m = a.update(last_value=0.0)
    assert m["optimizer_steps"] == (len(kls) if want is None else want)
    assert m["stopped_early"] is (want is not None)


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("discrete,A", [(False, 2), (True, 5)], ids=["gaussian-2", "categorical-5"])
def test_a_limit_that_never_triggers_equals_no_target_kl(discrete, A, layout):
    S, H, lr = 60, 64, 2e-3
    T, E, bs, epochs = LAYOUTS[layout]
    agents, outs = [], []
    for t in (None, 1e6):
        torch.manual_seed(21)
        a = _agent(S, A, H, bs, discrete, epochs=epochs, lr=lr, target_kl=t)
        for u in range(2):
            _fill(a, T, E, 4 + u)
            np.random.seed(8 + u)
            m = a.update(last_value=0.0)
        agents.append(a)
        outs.append(m)
    ref, kl = agents
    assert torch.equal(ref.actor_critic.flat, kl.actor_critic.flat)
    assert torch.equal(ref.optimizer.exp_avg_sq, kl.optimizer.exp_avg_sq)
    assert torch.equal(ref.optimizer.step_dev, kl.optimizer.step_dev)
    assert {k: outs[1][k] for k in outs[0]} == outs[0]
    steps = T * E // bs * epochs
    assert outs[1]["optimizer_steps"] == steps and outs[1]["stopped_early"] is False
    assert kl._kl_state.tolist() == [0, steps]   # every step of the second update is a gated replay


@pytest.mark.parametrize("discrete,A", [(False, 2), (True, 5)], ids=["gaussian-2", "categorical-5"])
def test_consecutive_updates_with_clip_value_and_set_lr(discrete, A):
    """Three updates in a row with the clipped value loss and a learning rate in device memory: every update starts
    unstopped, the graphed agent equals its eager twin bit for bit, and the gated graphs are captured once."""
    S, H, (T, E, bs, epochs) = 60, 64, LAYOUTS["per-minibatch"]
    kls = _kl_sequence(discrete, A, S, H, T, E, bs, epochs, 2e-3, clip_value=0.2)
    k, limit = _choose(kls, 1, len(kls) - 1)
    target = limit / 1.5
    agents = []
    for graphs in (True, False):
        torch.manual_seed(21)
        a = _agent(S, A, H, bs, discrete, epochs=epochs, lr=2e-3, clip_value=0.2, target_kl=target)
        a.use_cuda_graphs = graphs
        agents.append(a)
    seen, steps = None, []
    for u, lr in enumerate((2e-3, 1.5e-3, 1e-3)):
        outs = []
        for a in agents:
            _fill(a, T, E, 4 + u)
            a.set_lr(lr)
            np.random.seed(8 + u)
            outs.append(a.update(last_value=0.0))
        assert outs[0] == outs[1], u
        assert torch.equal(agents[0].actor_critic.flat, agents[1].actor_critic.flat), u
        assert torch.equal(agents[0].optimizer.exp_avg, agents[1].optimizer.exp_avg), u
        steps.append(outs[0]["optimizer_steps"])
        st = agents[0]._graph_state
        ids = {key: id(g) for key, g in st["graphs"].items()}
        assert seen is None or ids == seen
        seen = ids
    assert steps[0] == k and all(s > 0 for s in steps), (k, steps)
    assert int(agents[0].optimizer.step_dev.item()) == sum(steps)


@pytest.mark.parametrize("gym_id", ["highway-v0", FAST])
@pytest.mark.parametrize("discrete", [False, True], ids=["gaussian", "categorical"])
def test_train_vectorized_carries_the_option(highway_config, gym_id, discrete):
    """train_vectorized needs no new argument: an agent with target_kl trains, and every iteration's metrics report the
    steps it took; a limit that never triggers leaves the run bit for bit as without the option."""
    from highway_rope_ppo_b200.training import routine

    E, T, iters, seed = 256, 8, 3, 7
    hists, flats = [], []
    for t in (None, 1e6, 0.005):
        env, agent = _env_and_agent(highway_config, gym_id, discrete, E, seed, target_kl=t)
        np.random.seed(0)
        hists.append(routine.train_vectorized(env, agent, iters, T, seed=seed))
        flats.append(agent.actor_critic.flat.clone())
        env.close()
    assert torch.equal(flats[0], flats[1])
    assert [m["loss"] for m in hists[0]] == [m["loss"] for m in hists[1]]
    full = E * T // 512 * 2
    assert all(m["optimizer_steps"] == full and not m["stopped_early"] for m in hists[1])
    for m in hists[2]:
        assert 0 <= m["optimizer_steps"] <= full and m["stopped_early"] == (m["optimizer_steps"] < full)
        assert all(np.isfinite(m[k]) for k in ("loss", "policy_loss", "value_loss", "entropy"))
