"""Cost of the PPO update options (clipped value loss, learning rate in device memory), what the device learning rate
saves a schedule, and an informational learning check.

    python tools/ppo_options_bench.py [--envs 4096] [--rollout 32] [--rounds 3] [--iters 24] [--out result.json]

Reports, in one process and with the GPU's name, power limit and max SM clock read in the same call:
  * the replay time of one captured optimizer step (hrp_ppo_loss_grad[_ex] + hrp_clip_adam_step[_ex]) at B = 4096,
    S = 60, H = 256 for the default step, the clipped value loss and the device learning rate: CUDA events around
    windows of 50 replays, the three arms alternated window by window;
  * PPO samples/s of train_vectorized at bench.py's PPO defaults (shuffled RoPE, T = 32, 8 epochs, minibatch 4096,
    hidden 256) with a constant learning rate, with anneal_lr (set_lr: the captured graphs are replayed), and with the
    same schedule assigned to optimizer.lr by value (every update captures its minibatch graphs again, the cost
    set_lr removes); the arms alternated round by round after a warm-up round;
  * --iters iterations of train_vectorized from seed 42 with both options off and on (clip_value 0.2, anneal_lr), for
    the Gaussian policy on the reference config and the categorical policy on the highway-fast-v0 defaults, with a
    deterministic evaluation on 4096 held-out episodes at the end.  Informational: no pass threshold.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from episode_eval_bench import gpu_info  # noqa: E402

FAST = "highway-fast-v0"


def setup(E, discrete=False, H=256, minibatch=4096, epochs=8, seed=42, **kw):
    """bench.py's PPO workload (Gaussian: shuffled RoPE on the reference config), or the categorical policy on the
    highway-fast-v0 defaults."""
    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_vec_env
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.utils.reproducibility import set_random_seeds

    set_random_seeds(seed)
    if discrete:
        env = HighwayVecEnv({"gym_id": FAST, "action": {"type": "DiscreteMetaAction"}}, E, device="cuda:0", seed=seed)
    else:
        env = make_vec_env(Condition.SHUFFLED_ROPE, copy.deepcopy(HIGHWAY_CONFIG), 4, {"observation": {"order": "shuffled"}},
                           num_envs=E, seed=seed)
    agent = PPOAgent(env.N * env.F_out, 5 if discrete else 2, lr=3e-4, hidden_dim=H, batch_size=minibatch,
                     epochs=epochs, device="cuda:0", discrete=discrete, **kw)
    return env, agent


def step_replay(B=4096, S=60, H=256, windows=10, per_window=50):
    import numpy as np
    import torch

    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    g = torch.Generator(device="cuda:0").manual_seed(0)
    flat = {"states": torch.randn(B, S, generator=g, device="cuda:0") * 0.5,
            "pre_tanh": torch.randn(B, 2, generator=g, device="cuda:0"),
            "log_prob": torch.randn(B, generator=g, device="cuda:0") * 0.1 - 2.0,
            "adv": torch.randn(B, generator=g, device="cuda:0"), "ret": torch.randn(B, generator=g, device="cuda:0"),
            "value": torch.randn(B, generator=g, device="cuda:0")}
    arms = {}
    for name in ("default", "clip_value", "device_lr"):
        torch.manual_seed(0)
        agent = PPOAgent(S, 2, lr=3e-4, hidden_dim=H, batch_size=B, device="cuda:0",
                         clip_value=0.2 if name == "clip_value" else None)
        if name == "device_lr":
            agent.set_lr(3e-4)
        agent._minibatch_step(flat, None, B, 1)   # warm every kernel before the capture
        # the agent stays referenced: the graph replays into its workspace and buffers
        arms[name] = (agent, agent._capture(lambda a=agent: a._minibatch_step(flat, None, B, 1), 1))
    for _, gr in arms.values():
        gr.replay()
    torch.cuda.synchronize()
    times = {n: [] for n in arms}
    for _ in range(windows):
        for name, (_, gr) in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(per_window):
                gr.replay()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) * 1e3 / per_window)
    med = {n: float(np.median(t)) for n, t in times.items()}
    return {"us_per_replay": times, "median_us": med,
            "clip_value_over_default_pct": 100.0 * (med["clip_value"] / med["default"] - 1.0),
            "device_lr_over_default_pct": 100.0 * (med["device_lr"] / med["default"] - 1.0),
            "B": B, "S": S, "H": H, "windows": windows, "replays_per_window": per_window}


def train_samples(E, T, rounds, iters=3):
    from highway_rope_ppo_b200.training.routine import train_vectorized

    arms = {}
    for name in ("constant", "anneal_device_lr", "anneal_by_value"):
        env, agent = setup(E)
        if name == "anneal_by_value":
            # the schedule as a launch argument: every new value is a new graph key, so every update captures again
            agent.set_lr = lambda lr, a=agent: setattr(a.optimizer, "lr", lr)
        arms[name] = (env, agent)
    out = {n: [] for n in arms}
    for rnd in range(rounds + 1):   # round 0 warms every arm (eager rollout, graph captures)
        for name, (env, agent) in arms.items():
            agent.optimizer.lr = 3e-4
            rates = [m["samples_per_s"] for m in train_vectorized(env, agent, iters, T, seed=42,
                                                                   anneal_lr=name != "constant")]
            if rnd:
                out[name] += rates
    for env, _ in arms.values():
        env.close()
    mean = {k: sum(v) / len(v) for k, v in out.items()}
    return {"samples_per_s": out, "mean": mean,
            "anneal_device_lr_over_constant_pct": 100.0 * (mean["anneal_device_lr"] / mean["constant"] - 1.0),
            "anneal_by_value_over_constant_pct": 100.0 * (mean["anneal_by_value"] / mean["constant"] - 1.0),
            "T": T, "epochs": 8, "minibatch": 4096, "hidden": 256, "envs": E, "iterations_per_round": iters,
            "rounds": rounds}


def learning(E, T, iters, K=4096):
    import torch

    from highway_rope_ppo_b200.training.routine import eval_env_for, evaluate_vectorized, train_vectorized

    res = {}
    for policy in ("gaussian_reference", "categorical_fast"):
        for opts in ("off", "on"):
            env, agent = setup(E, discrete=policy == "categorical_fast", clip_value=0.2 if opts == "on" else None)
            hist = train_vectorized(env, agent, iters, T, seed=42, anneal_lr=opts == "on")
            ev_env = eval_env_for(env, K)
            ev = evaluate_vectorized(ev_env, agent, exp_seed=42)
            torch.cuda.synchronize()
            res[f"{policy}_{opts}"] = {
                "state_dim": agent.actor_critic.state_dim, "eval_episodes": ev["episodes"],
                "eval_return_mean": ev["mean"], "eval_return_std": ev["std"], "eval_length_mean": ev["length_mean"],
                "train_return_mean_last5": [h.get("episode_return_mean") for h in hist[-5:]],
                "value_loss_first_last": [hist[0]["value_loss"], hist[-1]["value_loss"]],
                "lr_first_last": [hist[0]["lr"], hist[-1]["lr"]]}
            ev_env.close()
            env.close()
    res.update(iterations=iters, T=T, envs=E, seed=42, clip_value=0.2)
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
        raise SystemExit("ppo_options_bench measures the GPU path: no CUDA device visible")
    res = {"gpu": gpu_info(), "step_replay": step_replay()}
    print(json.dumps({"step_replay": res["step_replay"]["median_us"]}), flush=True)
    res["train_vectorized"] = train_samples(args.envs, args.rollout, args.rounds)
    print(json.dumps({"train_vectorized": res["train_vectorized"]["mean"]}), flush=True)
    res["learning"] = learning(args.envs, args.rollout, args.iters)
    print(json.dumps({"learning": res["learning"]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
