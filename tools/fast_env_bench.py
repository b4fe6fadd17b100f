"""Cost or gain of highway-fast-v0's ego-only collision pass, and an informational learning check on the fast defaults.

    python tools/fast_env_bench.py [--envs 4096] [--steps 200] [--iters 16] [--out result.json]

Reports, in one process and with the GPU's name, power limit and max SM clock read in the same call:
  * step-kernel time at --envs envs for (1) highway-v0 with the reference config, (2) highway-fast-v0 with the reference
    config -- the same 51 vehicles, 4 lanes and 15 frames, so (1) against (2) is the collision pass (and ego spacing
    1.5) alone -- and (3) the highway-fast-v0 defaults (21 vehicles, 3 lanes, 5 frames, DiscreteMetaAction):
    CUDA events around each step, L2 flushed between steps (a 256 MiB memset outside the event pairs, as bench.py
    does), the three handles alternated step by step;
  * for the categorical policy on (3) at bench.py's PPO defaults (T = 32, 8 epochs, minibatch 4096, hidden 256): policy
    env-steps/s of the captured rollout alone, and PPO samples/s of rollout + update, three rounds each;
  * --iters iterations of train_vectorized on (3) from seed 42, with a deterministic evaluation on 4096 held-out
    episodes before and after.  Not a pass/fail check.
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

from final_obs_bench import gpu_info  # noqa: E402

FAST = "highway-fast-v0"


def configs():
    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG

    return {"v0_reference": copy.deepcopy(HIGHWAY_CONFIG),
            "fast_reference": dict(copy.deepcopy(HIGHWAY_CONFIG), gym_id=FAST),
            "fast_defaults": {"gym_id": FAST, "action": {"type": "DiscreteMetaAction"}}}


def make(cfg, E, seed=42, **kw):
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv

    return HighwayVecEnv(cfg, E, device="cuda:0", seed=seed, **kw)


def step_kernel(E, K, warmup):
    import numpy as np
    import torch

    arms = {name: make(cfg, E) for name, cfg in configs().items()}
    for env in arms.values():
        env.reset(42)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    g = torch.Generator(device="cuda:0").manual_seed(0)
    cont = [torch.rand((E, 2), generator=g, device="cuda:0") * 2 - 1 for _ in range(16)]
    meta = [torch.stack([torch.randint(0, 5, (E,), generator=g, device="cuda:0").float(),
                         torch.zeros(E, device="cuda:0")], 1) for _ in range(16)]
    acts = {n: meta if env.cfg.ego_mode == 1 else cont for n, env in arms.items()}
    for k in range(warmup):
        for name, env in arms.items():
            env.step(acts[name][k % 16])
    torch.cuda.synchronize()
    ev = {n: [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)] for n in arms}
    done = {n: 0 for n in arms}
    for k in range(K):
        for name, env in arms.items():
            flush.zero_()
            ev[name][k][0].record()
            env.step(acts[name][k % 16])
            ev[name][k][1].record()
            done[name] += int(((env.terminated | env.truncated) != 0).sum())
    torch.cuda.synchronize()
    res = {}
    for name, env in arms.items():
        t = np.array([a.elapsed_time(b) * 1e3 for a, b in ev[name]])
        res[name] = {"vehicles": env.V, "lanes": int(env.cfg.lanes_count),
                     "frames": int(env.cfg.simulation_frequency // env.cfg.policy_frequency),
                     "ego_collisions_only": int(env.cfg.ego_collisions_only), "ego_spacing": float(env.cfg.ego_spacing),
                     "mean_us": float(t.mean()), "median_us": float(np.median(t)),
                     "p10_us": float(np.percentile(t, 10)), "p90_us": float(np.percentile(t, 90)),
                     "episodes_ended_per_step": done[name] / K}
    v0, fast = res["v0_reference"]["median_us"], res["fast_reference"]["median_us"]
    res["fast_reference_over_v0_reference_pct_median"] = 100.0 * (fast / v0 - 1.0)
    res["envs"], res["steps"] = E, K
    for env in arms.values():
        env.close()
    return res


def setup_fast(E, H=256, minibatch=4096, epochs=8, seed=42):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.utils.reproducibility import set_random_seeds

    set_random_seeds(seed)
    env = make(configs()["fast_defaults"], E, seed=seed)
    S = env.N * env.F_out
    agent = PPOAgent(S, 5, lr=3e-4, hidden_dim=H, batch_size=minibatch, epochs=epochs, device="cuda:0", discrete=True)
    return env, agent, S


def ppo(E, T, rounds):
    import torch

    from highway_rope_ppo_b200.training.routine import collect_rollout, rollout_and_update

    env, agent, S = setup_fast(E)
    o = env.reset(42)
    for _ in range(2):   # the first rollout runs launch by launch, the second one captures the rollout graph
        _, o = rollout_and_update(env, agent, T, obs=o)
    torch.cuda.synchronize()
    steps, samples = [], []
    for _ in range(rounds):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        r = collect_rollout(env, agent, T, o)
        e1.record()
        torch.cuda.synchronize()
        o = r["states"][T].clone()
        steps.append(T * E / (e0.elapsed_time(e1) * 1e-3))
        e0.record()
        for _ in range(3):
            _, o = rollout_and_update(env, agent, T, obs=o)
        e2.record()
        torch.cuda.synchronize()
        samples.append(3 * T * E / (e0.elapsed_time(e2) * 1e-3))
    env.close()
    return {"policy_env_steps_per_s": steps, "policy_env_steps_per_s_mean": sum(steps) / len(steps),
            "ppo_samples_per_s": samples, "ppo_samples_per_s_mean": sum(samples) / len(samples), "state_dim": S,
            "actions": 5, "T": T, "epochs": 8, "minibatch": 4096, "hidden": 256, "envs": E}


def learning(E, T, iters, K=4096):
    import torch

    from highway_rope_ppo_b200.training.routine import evaluate_vectorized, train_vectorized

    env, agent, S = setup_fast(E)
    ev_env = make(env.config, K, autoreset=False, env_id_base=E)
    before = evaluate_vectorized(ev_env, agent, exp_seed=42)
    hist = train_vectorized(env, agent, iters, T, seed=42)
    after = evaluate_vectorized(ev_env, agent, exp_seed=42)
    torch.cuda.synchronize()
    res = {"state_dim": S, "iterations": iters, "T": T, "envs": E, "seed": 42, "eval_episodes": after["episodes"],
           "eval_return_mean_before": before["mean"], "eval_return_mean_after": after["mean"],
           "eval_return_std_after": after["std"], "eval_length_mean_after": after["length_mean"],
           "train_return_mean_last5": [h.get("episode_return_mean") for h in hist[-5:]]}
    env.close()
    ev_env.close()
    return res


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--envs", type=int, default=4096)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--rollout", type=int, default=32)
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--iters", type=int, default=16)
    p.add_argument("--out", default=None)
    args = p.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("fast_env_bench measures the GPU path: no CUDA device visible")
    res = {"gpu": gpu_info(), "step_kernel": step_kernel(args.envs, args.steps, args.warmup)}
    print(json.dumps({"step_kernel": res["step_kernel"]}), flush=True)
    res["ppo"] = ppo(args.envs, args.rollout, args.rounds)
    print(json.dumps({"ppo": res["ppo"]}), flush=True)
    res["learning"] = learning(args.envs, args.rollout, args.iters)
    print(json.dumps({"learning": res["learning"]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
