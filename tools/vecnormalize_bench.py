"""Cost of running observation / reward normalization (VecNormalize, csrc/hrp_norm.cu) and an informational learning
check.

    python tools/vecnormalize_bench.py [--envs 4096] [--rollout 32] [--rounds 3] [--iters 24] [--out result.json]

Reports, in one process and with the GPU's name, power limit and max SM clock read in the same call:
  * the normalization launches of one step at E = 4096 for S = 60 (the reference's Kinematics + RoPE), 484 (the default
    OccupancyGrid) and 600: a training step (moments + merge + apply) and an evaluation step (apply only), CUDA events
    around windows of 200 launches of one captured step, median over windows.  The working set (E x S floats, under
    10 MB) stays in the 126 MB L2 between launches: these are warm-L2 times, as inside a rollout, where the step kernel
    has just written the observation;
  * the device time of each of those kernels at S = 60 and 600 (torch.profiler, eager launches, a pass of its own);
  * one captured rollout (T = --rollout) of bench.py's PPO workload (shuffled RoPE, 4096 envs, hidden 256) with and
    without the wrapper, alternated window by window;
  * PPO samples/s of train_vectorized at bench.py's PPO defaults with and without the wrapper, alternated round by
    round after a warm-up round;
  * --iters iterations of train_vectorized from seed 42 with norm_obs + norm_reward and without the wrapper, for the
    Gaussian policy on the reference config, with a deterministic evaluation on 4096 held-out episodes at the end
    (raw rewards).  Informational: no pass threshold.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from episode_eval_bench import gpu_info  # noqa: E402
from ppo_options_bench import setup  # noqa: E402


def _windows(fns, windows, per_window):
    """CUDA-event time per call of each fn, alternated window by window: {name: [us per call, per window]}"""
    import torch

    times = {n: [] for n in fns}
    for _ in range(windows):
        for name, fn in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(per_window):
                fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) * 1e3 / per_window)
    return times


class _Scripted:
    """The wrapper's inner env for timing the normalization alone: its outputs are already in place, no launch."""

    def __init__(self, E, S):
        import torch

        self.num_envs, self.N, self.F_out, self.obs_shape, self.device = E, 1, S, (1, S), torch.device("cuda:0")
        g = torch.Generator(device="cuda:0").manual_seed(S)
        self.obs = torch.randn((E, 1, S), generator=g, device="cuda:0")
        self.reward = torch.rand(E, generator=g, device="cuda:0")
        self.terminated = (torch.rand(E, generator=g, device="cuda:0") < 0.02).to(torch.uint8)
        self.truncated = torch.zeros(E, dtype=torch.uint8, device="cuda:0")

    def step(self, actions, out=None, reward_out=None, terminated_out=None, truncated_out=None, **kw):
        return self.obs, reward_out if reward_out is not None else self.reward, self.terminated, self.truncated

    reset = observe = step


def kernel_profile(E=4096, sizes=(60, 600), steps=200):
    """Device time of each normalization kernel of a training step (torch.profiler, CUDA activity, eager launches in a
    run of their own): mean over ``steps`` steps."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize

    res = {}
    for S in sizes:
        env = _Scripted(E, S)
        w = VecNormalize(env)
        acts, raw = torch.zeros((E, 2), device="cuda:0"), torch.zeros(E, device="cuda:0")
        for _ in range(20):
            w.step(acts, raw_reward_out=raw, reward_out=env.reward)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                w.step(acts, raw_reward_out=raw, reward_out=env.reward)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            if "vecnorm" in ev.key:
                name = ev.key.split("vecnorm_")[1].split("_kernel")[0]
                per[name] = {"us_per_launch": ev.device_time_total / max(ev.count, 1), "launches": ev.count}
        res[str(S)] = per
    res.update(E=E, steps=steps, source="torch.profiler device time, eager launches")
    return res


def launch_cost(E=4096, sizes=(60, 484, 600), windows=10, per_window=200):
    import numpy as np
    import torch

    from highway_rope_ppo_b200 import _lib
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize

    res = {}
    for S in sizes:
        env = _Scripted(E, S)
        acts = torch.zeros((E, 2), device="cuda:0")
        fns = {}
        for mode in ("training", "evaluation"):
            w = VecNormalize(env, training=mode == "training", norm_reward=mode == "training")
            raw = torch.zeros(E, device="cuda:0")
            step = (lambda w=w, raw=raw: w.step(acts, raw_reward_out=raw, reward_out=env.reward)) if mode == "training" \
                else (lambda w=w: w.step(acts, reward_out=env.reward))
            step()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                g.capture_begin()
                step()
                g.capture_end()
            torch.cuda.current_stream().wait_stream(s)
            fns[mode] = (w, g)
        times = _windows({m: g.replay for m, (_, g) in fns.items()}, windows, per_window)
        res[str(S)] = {"us_per_step": times, "median_us": {m: float(np.median(t)) for m, t in times.items()},
                       "launches": {"training": 3, "evaluation": 1},
                       "bytes_touched_training": E * S * 4 * 3 + E * (4 * 3 + 8 * 2) + _lib.vecnorm_scratch_len(S + 1) * 8}
    res.update(E=E, windows=windows, launches_per_window=per_window, l2="warm: working set < 10 MB of 126 MB L2")
    return res


def rollout_cost(E, T, windows=10, per_window=5):
    import numpy as np
    import torch

    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize
    from highway_rope_ppo_b200.training.routine import collect_rollout

    arms = {}
    for name in ("plain", "vecnormalize"):
        env, agent = setup(E)
        if name == "vecnormalize":
            env = VecNormalize(env)
        obs = env.reset(seed=42).clone()
        for _ in range(3):   # eager, captured, replayed
            r = collect_rollout(env, agent, T, obs)
        arms[name] = (env, agent, obs)

    fns = {n: (lambda a=a: collect_rollout(a[0], a[1], T, a[2])) for n, a in arms.items()}
    times = _windows(fns, windows, per_window)
    med = {n: float(np.median(t)) for n, t in times.items()}
    for env, _, _ in arms.values():
        env.close()
    return {"us_per_rollout": times, "median_us": med, "T": T, "envs": E,
            "us_per_step": {n: m / T for n, m in med.items()},
            "vecnormalize_over_plain_pct": 100.0 * (med["vecnormalize"] / med["plain"] - 1.0)}


def train_samples(E, T, rounds, iters=3):
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize
    from highway_rope_ppo_b200.training.routine import train_vectorized

    arms = {}
    for name in ("plain", "vecnormalize"):
        env, agent = setup(E)
        arms[name] = (VecNormalize(env) if name == "vecnormalize" else env, agent)
    out = {n: [] for n in arms}
    for rnd in range(rounds + 1):   # round 0 warms every arm (eager rollout, graph captures)
        for name, (env, agent) in arms.items():
            rates = [m["samples_per_s"] for m in train_vectorized(env, agent, iters, T, seed=42)]
            if rnd:
                out[name] += rates
    for env, _ in arms.values():
        env.close()
    mean = {k: sum(v) / len(v) for k, v in out.items()}
    return {"samples_per_s": out, "mean": mean,
            "vecnormalize_over_plain_pct": 100.0 * (mean["vecnormalize"] / mean["plain"] - 1.0),
            "T": T, "epochs": 8, "minibatch": 4096, "hidden": 256, "envs": E, "iterations_per_round": iters,
            "rounds": rounds}


def learning(E, T, iters, K=4096):
    import torch

    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.routine import eval_env_for, evaluate_vectorized, train_vectorized
    from highway_rope_ppo_b200.utils.reproducibility import set_random_seeds

    res = {}
    for arm in ("off", "norm_obs_norm_reward"):
        set_random_seeds(42)
        env = HighwayVecEnv(HIGHWAY_CONFIG, E, device="cuda:0", seed=42)
        if arm != "off":
            env = VecNormalize(env)
        agent = PPOAgent(env.N * env.F_out, 2, lr=3e-4, hidden_dim=256, batch_size=4096, epochs=8, device="cuda:0")
        hist = train_vectorized(env, agent, iters, T, seed=42)
        ev_env = eval_env_for(env, K)
        ev = evaluate_vectorized(ev_env, agent, exp_seed=42)
        torch.cuda.synchronize()
        res[arm] = {"eval_episodes": ev["episodes"], "eval_return_mean": ev["mean"], "eval_return_std": ev["std"],
                    "eval_length_mean": ev["length_mean"],
                    "train_return_mean_last5": [h.get("episode_return_mean") for h in hist[-5:]]}
        if arm != "off":
            res[arm]["ret_rms_var"] = float(env.ret_rms.var)
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
        raise SystemExit("vecnormalize_bench measures the GPU path: no CUDA device visible")
    res = {"gpu": gpu_info(), "launch_cost": launch_cost(args.envs)}
    print(json.dumps({"launch_cost": {k: v["median_us"] for k, v in res["launch_cost"].items() if isinstance(v, dict)
                                      and "median_us" in v}}), flush=True)
    res["kernel_profile"] = kernel_profile(args.envs)
    print(json.dumps({"kernel_profile": res["kernel_profile"]}), flush=True)
    res["rollout"] = rollout_cost(args.envs, args.rollout)
    print(json.dumps({"rollout": res["rollout"]["median_us"]}), flush=True)
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
