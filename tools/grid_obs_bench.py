"""Cost of the OccupancyGrid observation epilogue, and an informational grid-vs-list learning comparison.

    python tools/grid_obs_bench.py [--envs 4096] [--steps 200] [--iters 24] [--out result.json]

Reports, in one process and with the GPU's name, power limit and max SM clock read in the same call:
  * step-kernel time at --envs envs, sorted Kinematics (the reference config, 15 x 4) against the default grid
    (presence, vx, vy, on_road on 11 x 11 cells): CUDA events around each step, L2 flushed between steps (a 256 MiB
    memset outside the event pairs, as bench.py does), the two handles alternated step by step with the same seed and
    actions (their simulations are identical, so is the work before the observation);
  * PPO samples/s with the grid of the reference config's features (x, y, vx, vy on 11 x 11 cells: S = 484) at
    bench.py's defaults (T = 32, 8 epochs, minibatch 4096, hidden 256), three rounds;
  * --iters iterations of train_vectorized from seed 42 each way, sorted Kinematics and the default grid, with a
    4096-episode deterministic evaluation at the end.  Not a pass/fail check.
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

GRID_DEFAULT = {"observation": {"type": "OccupancyGrid", "features": ["presence", "vx", "vy", "on_road"]}}
GRID_484 = {"observation": {"type": "OccupancyGrid", "features": ["x", "y", "vx", "vy"]}}


def setup(E, over, H=256, minibatch=4096, epochs=8, seed=42):
    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_vec_env
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.utils.reproducibility import set_random_seeds

    set_random_seeds(seed)
    env = make_vec_env(Condition.SORTED, copy.deepcopy(HIGHWAY_CONFIG), None, over, num_envs=E, seed=seed)
    S = env.N * env.F_out
    agent = PPOAgent(S, 2, lr=3e-4, hidden_dim=H, batch_size=minibatch, epochs=epochs, device="cuda:0")
    return env, agent, S


def step_kernel(E, K, warmup):
    import numpy as np
    import torch

    arms = {"kinematics": setup(E, {})[0], "grid": setup(E, GRID_DEFAULT)[0]}
    for env in arms.values():
        env.reset(42)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    g = torch.Generator(device="cuda:0").manual_seed(0)
    acts = [torch.rand((E, 2), generator=g, device="cuda:0") * 2 - 1 for _ in range(16)]
    for k in range(warmup):
        for env in arms.values():
            env.step(acts[k % 16])
    torch.cuda.synchronize()
    ev = {n: [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)] for n in arms}
    for k in range(K):
        for name, env in arms.items():
            flush.zero_()
            ev[name][k][0].record()
            env.step(acts[k % 16])
            ev[name][k][1].record()
    torch.cuda.synchronize()
    assert torch.equal(arms["kinematics"].reward, arms["grid"].reward)   # the same simulation
    res = {"observation_shape": {n: list(e.obs_shape) for n, e in arms.items()}}
    for name in arms:
        t = np.array([a.elapsed_time(b) * 1e3 for a, b in ev[name]])
        res[name] = {"mean_us": float(t.mean()), "median_us": float(np.median(t)), "p10_us": float(np.percentile(t, 10)),
                     "p90_us": float(np.percentile(t, 90))}
    res["grid_over_kinematics_pct_median"] = 100.0 * (res["grid"]["median_us"] / res["kinematics"]["median_us"] - 1.0)
    res["envs"], res["steps"] = E, K
    for env in arms.values():
        env.close()
    return res


def ppo_samples(E, T, rounds):
    import torch

    from highway_rope_ppo_b200.training.routine import rollout_and_update

    env, agent, S = setup(E, GRID_484)
    o = env.reset(42)
    for _ in range(2):   # the first rollout runs launch by launch, the second one captures the rollout graph
        _, o = rollout_and_update(env, agent, T, obs=o)
    torch.cuda.synchronize()
    out = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            _, o = rollout_and_update(env, agent, T, obs=o)
        e1.record()
        torch.cuda.synchronize()
        out.append(3 * T * E / (e0.elapsed_time(e1) * 1e-3))
    env.close()
    return {"samples_per_s": out, "mean": sum(out) / len(out), "state_dim": S, "T": T, "epochs": 8, "minibatch": 4096,
            "hidden": 256, "envs": E}


def learning(E, T, iters, K=4096):
    import torch

    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.training.routine import evaluate_vectorized, train_vectorized

    res = {}
    for name, over in (("kinematics_sorted", {}), ("grid_default", GRID_DEFAULT)):
        env, agent, S = setup(E, over)
        hist = train_vectorized(env, agent, iters, T, seed=42)
        ev_env = HighwayVecEnv(env.config, K, device="cuda:0", autoreset=False, env_id_base=E)
        ev = evaluate_vectorized(ev_env, agent, exp_seed=42)
        torch.cuda.synchronize()
        res[name] = {"state_dim": S, "eval_return_mean": ev["mean"], "eval_return_std": ev["std"],
                     "eval_episodes": ev["episodes"],
                     "train_return_mean_last5": [h.get("episode_return_mean") for h in hist[-5:]]}
        env.close()
        ev_env.close()
    res["iterations"], res["T"], res["envs"], res["seed"] = iters, T, E, 42
    return res


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--envs", type=int, default=4096)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--rollout", type=int, default=32)
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--iters", type=int, default=24)
    p.add_argument("--out", default=None)
    args = p.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("grid_obs_bench measures the GPU path: no CUDA device visible")
    res = {"gpu": gpu_info(), "step_kernel": step_kernel(args.envs, args.steps, args.warmup)}
    print(json.dumps({"step_kernel": res["step_kernel"]}), flush=True)
    res["ppo"] = ppo_samples(args.envs, args.rollout, args.rounds)
    print(json.dumps({"ppo": res["ppo"]}), flush=True)
    res["learning"] = learning(args.envs, args.rollout, args.iters)
    print(json.dumps({"learning": res["learning"]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
