"""Cost and effect of target_kl early stopping (PPOAgent(target_kl=...)), and an informational learning check.

    python tools/target_kl_bench.py [--envs 4096] [--rollout 32] [--rounds 3] [--iters 24] [--out result.json]

Reports, in one process and with the GPU's name, power limit and max SM clock read in the same call:
  * one replayed optimizer step at B = 4096, S = 60, H = 256: the plain captured step (target_kl None), the same step
    with the KL variants of the kernels replayed without the gate, the same behind the gate with the body open (a limit
    that never triggers), and with the word raised (the gate alone, what a skipped step costs).  CUDA events around windows of 50 launches, the
    arms alternated window by window;
  * the time of one whole update at bench.py's PPO defaults (T = 32 x 4096 samples, 8 epochs of 32 minibatches of 4096,
    hidden 256, S of the shuffled-RoPE observation) on a rollout whose stored log-probs are the policy's own: unstopped
    (target_kl None) and with limits taken from the unstopped update's KL sequence so that it stops after about 1, 2
    and 4 of the 8 epochs (limit = the largest KL of the first e epochs: the stop falls at the first later minibatch
    above it).  Every arm starts from the same parameters and Adam state; arms alternated round by round, median;
  * PPO samples/s of train_vectorized at those defaults with target_kl None and 0.02, alternated round by round after
    a warm-up round, with the optimizer steps each update took;
  * --iters iterations of train_vectorized from seed 42 with target_kl None and 0.02 (Gaussian policy, reference
    config), the optimizer steps of every update and a deterministic evaluation on 4096 held-out episodes at the end.
    Informational: no pass threshold.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from episode_eval_bench import gpu_info  # noqa: E402
from ppo_options_bench import setup  # noqa: E402


def step_cost(B=4096, S=60, H=256, windows=10, per_window=50):
    import torch

    from highway_rope_ppo_b200 import _lib
    from highway_rope_ppo_b200.ppo.agent import PPOAgent, _GatedGraph

    g = torch.Generator(device="cuda:0").manual_seed(0)
    flat = {"states": torch.randn(B, S, generator=g, device="cuda:0") * 0.5,
            "pre_tanh": torch.randn(B, 2, generator=g, device="cuda:0"),
            "log_prob": torch.randn(B, generator=g, device="cuda:0") * 0.1 - 2.0,
            "adv": torch.randn(B, generator=g, device="cuda:0"), "ret": torch.randn(B, generator=g, device="cuda:0")}
    arms = {}
    for name in ("plain", "kl_kernels_ungated", "gated_open", "gated_closed"):
        torch.manual_seed(0)
        agent = PPOAgent(S, 2, lr=3e-4, hidden_dim=H, batch_size=B, device="cuda:0",
                         target_kl=None if name == "plain" else 1e6)
        agent._minibatch_step(flat, None, B, 1)   # warm every kernel before the capture
        gated = name.startswith("gated")
        gr = agent._capture(lambda a=agent: a._minibatch_step(flat, None, B, 1), 1, keep_graph=gated)
        if not gated:
            fn = gr.replay
        else:
            gr = _GatedGraph(agent._lib, gr, agent._kl_state)
            agent._kl_state.zero_()
            if name == "gated_closed":
                agent._kl_state[0] = 1
            fn = (lambda a=agent, w=gr: _lib.check(a._lib.hrp_graph_if_launch(w.handle, a.actor_critic._stream())))
        arms[name] = (agent, gr, fn)
    for _, _, fn in arms.values():
        fn()
    torch.cuda.synchronize()
    times = {n: [] for n in arms}
    for _ in range(windows):
        for name, (_, _, fn) in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(per_window):
                fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) * 1e3 / per_window)
    opened = {n: int(a._kl_state[1].item()) for n, (a, _, _) in arms.items() if n.startswith("gated")}
    med = {n: sorted(v)[len(v) // 2] for n, v in times.items()}
    return {"us_per_step": times, "median_us": med, "B": B, "S": S, "H": H, "gate_openings": opened,
            "gated_open_over_plain_us": med["gated_open"] - med["plain"],
            "gate_and_if_us": med["gated_open"] - med["kl_kernels_ungated"]}


def _rollout(agent, T, E, seed):
    """States drawn at random, actions sampled by the agent's own policy: the stored log-probs are the policy's, so the
    update's KL starts at ~0."""
    import torch

    ac = agent.actor_critic
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    states = torch.randn(T + 1, E, ac.state_dim, generator=g, device="cuda:0") * 0.5
    out = ac.act(states[:T].reshape(T * E, -1).contiguous(), noise=torch.randn(T * E, ac.action_dim, generator=g,
                                                                                 device="cuda:0"))
    data = {"states": states, "action": out["action"].view(T, E, -1), "pre_tanh": out["pre_tanh"].view(T, E, -1),
            "log_prob": out["log_prob"].view(T, E), "value": out["value"].view(T, E),
            "reward": torch.randn(T, E, generator=g, device="cuda:0"),
            "done": (torch.rand(T, E, generator=g, device="cuda:0") < 0.02).to(torch.uint8)}
    return {k: v.clone() for k, v in data.items()}


def _load(agent, data):
    T, E = data["reward"].shape
    r = agent.memory.begin_rollout(T, E, data["states"].shape[-1], data["action"].shape[-1], data["pre_tanh"].shape[-1])
    for k, v in data.items():
        r[k].copy_(v)


def update_time(E, T, rounds, S_env, H=256, bs=4096, epochs=8):
    import numpy as np
    import torch

    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    def make(target):
        torch.manual_seed(42)
        return PPOAgent(S_env, 2, lr=3e-4, hidden_dim=H, batch_size=bs, epochs=epochs, device="cuda:0", target_kl=target)

    probe = make(None)
    data = _rollout(probe, T, E, 1)
    # the unstopped update's KL sequence (eager, metrics[5]'s increment per step = the kernels' KL)
    probe.use_cuda_graphs = False
    orig, kls = probe._minibatch_step, []

    def step(flat, idx, B, world):
        probe._metrics.zero_()
        orig(flat, idx, B, world)
        kls.append(probe._metrics[5].item())
    probe._minibatch_step = step
    _load(probe, data)
    np.random.seed(3)
    probe.update(last_value=0.0)
    M = T * E // bs
    arms = {"unstopped": None}
    for e in (1, 2, 4):
        arms[f"limit_max_kl_of_first_{e}_epochs"] = max(kls[:e * M]) / 1.5
    agents = {n: make(t) for n, t in arms.items()}
    s0 = None
    times = {n: [] for n in arms}
    steps = {}
    for rnd in range(rounds + 1):   # round 0 warms every arm (eager first epoch, graph captures)
        for name, a in agents.items():
            if s0 is None:
                s0 = {k: v.clone() for k, v in (("flat", a.actor_critic.flat), ("m", a.optimizer.exp_avg),
                                                  ("v", a.optimizer.exp_avg_sq), ("step", a.optimizer.step_dev))}
            a.actor_critic.flat.copy_(s0["flat"])
            a.optimizer.exp_avg.copy_(s0["m"])
            a.optimizer.exp_avg_sq.copy_(s0["v"])
            a.optimizer.step_dev.copy_(s0["step"])
            _load(a, data)
            np.random.seed(3)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m = a.update(last_value=0.0)
            dt = time.perf_counter() - t0
            if rnd:
                times[name].append(dt * 1e3)
                steps[name] = m.get("optimizer_steps", M * epochs)
    med = {n: sorted(v)[len(v) // 2] for n, v in times.items()}
    return {"ms_per_update": times, "median_ms": med, "optimizer_steps": steps,
            "target_kl": arms, "kl_sequence_unstopped": kls, "T": T, "envs": E, "minibatch": bs, "epochs": epochs,
            "state_dim": S_env, "hidden": H, "rounds": rounds}


def train_samples(E, T, rounds, iters=3):
    from highway_rope_ppo_b200.training.routine import train_vectorized

    arms = {name: setup(E, target_kl=t) for name, t in (("off", None), ("target_kl_0.02", 0.02))}
    out = {n: [] for n in arms}
    steps = {n: [] for n in arms}
    for rnd in range(rounds + 1):   # round 0 warms every arm
        for name, (env, agent) in arms.items():
            hist = train_vectorized(env, agent, iters, T, seed=42)
            if rnd:
                out[name] += [m["samples_per_s"] for m in hist]
                steps[name] += [m.get("optimizer_steps", 8 * T * E // 4096) for m in hist]
    for env, _ in arms.values():
        env.close()
    mean = {k: sum(v) / len(v) for k, v in out.items()}
    return {"samples_per_s": out, "mean": mean, "optimizer_steps": steps,
            "target_kl_over_off_pct": 100.0 * (mean["target_kl_0.02"] / mean["off"] - 1.0),
            "T": T, "epochs": 8, "minibatch": 4096, "hidden": 256, "envs": E, "iterations_per_round": iters,
            "rounds": rounds}


def learning(E, T, iters, K=4096):
    import torch

    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.routine import eval_env_for, evaluate_vectorized, train_vectorized
    from highway_rope_ppo_b200.utils.reproducibility import set_random_seeds

    res = {}
    for arm, t in (("off", None), ("target_kl_0.02", 0.02)):
        set_random_seeds(42)
        env = HighwayVecEnv(HIGHWAY_CONFIG, E, device="cuda:0", seed=42)
        agent = PPOAgent(env.N * env.F_out, 2, lr=3e-4, hidden_dim=256, batch_size=4096, epochs=8, device="cuda:0",
                         target_kl=t)
        hist = train_vectorized(env, agent, iters, T, seed=42)
        ev_env = eval_env_for(env, K)
        ev = evaluate_vectorized(ev_env, agent, exp_seed=42)
        torch.cuda.synchronize()
        res[arm] = {"eval_episodes": ev["episodes"], "eval_return_mean": ev["mean"], "eval_return_std": ev["std"],
                    "eval_length_mean": ev["length_mean"],
                    "optimizer_steps": [h.get("optimizer_steps", 8 * T * E // 4096) for h in hist],
                    "approx_kl": [h["approx_kl"] for h in hist],
                    "train_return_mean_last5": [h.get("episode_return_mean") for h in hist[-5:]]}
        ev_env.close()
        env.close()
    res.update(iterations=iters, T=T, envs=E, seed=42, config="reference (config/base_config.py), sorted, no embedding")
    return res


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--envs", type=int, default=4096)
    p.add_argument("--rollout", type=int, default=32)
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--iters", type=int, default=24)
    p.add_argument("--out", default=None)
    args = p.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("target_kl_bench measures the GPU path: no CUDA device visible")
    res = {"gpu": gpu_info(), "step_cost": step_cost()}
    print(json.dumps({"step_cost": res["step_cost"]["median_us"]}), flush=True)
    env, agent = setup(8)
    S_env = agent.actor_critic.state_dim
    env.close()
    res["update_time"] = update_time(args.envs, args.rollout, max(args.rounds, 3), S_env)
    print(json.dumps({"update_time": res["update_time"]["median_ms"],
                      "steps": res["update_time"]["optimizer_steps"]}), flush=True)
    res["train_vectorized"] = train_samples(args.envs, args.rollout, args.rounds)
    print(json.dumps({"train_vectorized": res["train_vectorized"]["mean"]}), flush=True)
    res["learning"] = learning(args.envs, args.rollout, args.iters)
    print(json.dumps({"learning": {k: v for k, v in res["learning"].items() if isinstance(v, dict)}}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
