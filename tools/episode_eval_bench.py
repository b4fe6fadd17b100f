"""Cost of the episode statistics and of the batched deterministic evaluation, and the learning comparisons of DESIGN
§3.3 redone with evaluation returns.

    python tools/episode_eval_bench.py [--envs 4096] [--eval-episodes 4096] [--iters 24] [--out result.json]

Reports, in one process and with the GPU's name, power limit and max SM clock read in the same call:
  * hrp_episode_stats over a T = 32, E = --envs rollout (~3 % of the steps end an episode): CUDA events around 200
    back-to-back launches (the 0.8 MB it reads stays in L2), mean per launch;
  * PPO samples/s of train_vectorized (statistics on) and of the loop it replaced (rollout_and_update + the same
    per-iteration synchronisation), bench.py's PPO shape (T = 32, 8 epochs, minibatch 4096, hidden 256, shuffled
    RoPE), alternated round by round, one env and agent per arm;
  * evaluate_vectorized of --eval-episodes episodes on the default config (sorted, 40-step limit, hidden 256),
    replayed graph and launch by launch, host clock around each call (it ends in a synchronisation); beside it the
    reference-shaped evaluate() of 5 episodes on a single-env handle;
  * --iters iterations of train_vectorized with bootstrap_truncated off and on (Gaussian) and of the categorical agent
    on the meta-action env, from one seed, evaluated on --eval-episodes held-out episodes every 4 iterations.  Not a
    pass/fail check.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch

    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["max_sm_clock_mhz"] = float(q[0]), float(q[1])
    except Exception as e:  # reported, not guessed
        info["nvidia_smi_error"] = repr(e)
    return info


def setup(E, discrete=False, shuffled=True, H=256, minibatch=4096, epochs=8, seed=42):
    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_vec_env
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.utils.reproducibility import set_random_seeds

    set_random_seeds(seed)
    cfg = copy.deepcopy(HIGHWAY_CONFIG)
    if discrete:
        cfg["action"] = {"type": "DiscreteMetaAction"}
    if shuffled:
        env = make_vec_env(Condition.SHUFFLED_ROPE, cfg, 4, {"observation": {"order": "shuffled"}}, num_envs=E,
                           seed=seed)
    else:
        env = make_vec_env(Condition.SORTED, cfg, num_envs=E, seed=seed)
    agent = PPOAgent(env.N * env.F_out, 5 if discrete else 2, lr=3e-4, hidden_dim=H, batch_size=minibatch,
                     epochs=epochs, device="cuda:0", discrete=discrete)
    return env, agent, cfg


def stats_launch(E, T=32, calls=200):
    import numpy as np
    import torch

    from highway_rope_ppo_b200.training.episodes import episode_stats, new_stats

    rng = np.random.default_rng(0)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    r = d(rng.normal(size=(T, E)).astype(np.float32))
    te = d((rng.random((T, E)) < 0.012).astype(np.uint8))
    tr = d((rng.random((T, E)) < 0.02).astype(np.uint8))
    ret = torch.zeros(E, dtype=torch.float64, device="cuda:0")
    ln = torch.zeros(E, dtype=torch.int32, device="cuda:0")
    stats = new_stats("cuda:0")
    for _ in range(20):
        episode_stats(r, te, tr, ret, ln, stats)
    torch.cuda.synchronize()
    times = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(calls):
            episode_stats(r, te, tr, ret, ln, stats)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e3 / calls)
    return {"T": T, "E": E, "calls_per_window": calls, "windows": 5, "us_per_launch": times,
            "us_per_launch_median": float(np.median(times)), "bytes_read": int(T * E * 6),
            "l2": "resident (inputs re-read back to back)"}


def train_samples(E, T, rounds, iters=3):
    import torch

    from highway_rope_ppo_b200.training.routine import rollout_and_update, train_vectorized

    arms = {}
    for name in ("plain", "stats"):
        env, agent, _ = setup(E)
        arms[name] = [env, agent, env.reset(42)]
    out = {"plain": [], "stats": []}
    for rnd in range(rounds + 1):   # round 0 warms both arms (eager rollout, graph capture)
        for name in ("plain", "stats"):
            env, agent, o = arms[name]
            if name == "stats":
                rates = [m["samples_per_s"] for m in train_vectorized(env, agent, iters, T, seed=42)]
            else:
                rates = []
                for _ in range(iters):   # what train_vectorized did per iteration before the statistics
                    t0 = time.time()
                    _, o = rollout_and_update(env, agent, T, obs=o)
                    torch.cuda.synchronize()
                    rates.append(T * E / (time.time() - t0))
                arms[name][2] = o
            if rnd:
                out[name] += rates
    for env, _, _ in arms.values():
        env.close()
    mean = {k: sum(v) / len(v) for k, v in out.items()}
    return {"samples_per_s": out, "mean": mean, "cost_pct": 100.0 * (1.0 - mean["stats"] / mean["plain"]), "T": T,
            "epochs": 8, "minibatch": 4096, "envs": E, "iterations_per_round": iters, "rounds": rounds}


def evaluation(K, reps=20):
    import numpy as np
    import torch

    from highway_rope_ppo_b200.envs.highway_env import HighwayEnv
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.training.routine import evaluate, evaluate_vectorized

    env, agent, cfg = setup(64, shuffled=False)
    env.close()
    ev_env = HighwayVecEnv(cfg, K, device="cuda:0", autoreset=False)
    res = {"episodes": K}
    first = evaluate_vectorized(ev_env, agent, exp_seed=42)   # eager; the next call captures
    evaluate_vectorized(ev_env, agent, exp_seed=42)
    for name, graph, n in (("graph", True, reps), ("eager", False, max(reps // 4, 3))):
        t = []
        for _ in range(n):
            t0 = time.time()
            ev = evaluate_vectorized(ev_env, agent, exp_seed=42, use_graph=graph)
            t.append(time.time() - t0)
            assert ev["returns"].tobytes() == first["returns"].tobytes()
        med = float(np.median(t))
        res[name] = {"ms_median": med * 1e3, "ms_all": [x * 1e3 for x in t], "episodes_per_s": K / med}
    res["eval_return_mean"], res["eval_length_mean"] = first["mean"], first["length_mean"]
    ev_env.close()
    single = HighwayEnv(cfg)
    evaluate(single, agent, 5, exp_seed=42)   # warm
    t = []
    for _ in range(3):
        t0 = time.time()
        evaluate(single, agent, 5, exp_seed=42)
        torch.cuda.synchronize()
        t.append(time.time() - t0)
    single.close()
    med = float(np.median(t))
    res["reference_shaped_5_episodes"] = {"ms_median": med * 1e3, "episodes_per_s": 5 / med}
    return res


def learning(E, T, iters, eval_episodes):
    from highway_rope_ppo_b200.training.routine import train_vectorized

    res = {}
    for name, discrete, boot in (("gaussian_bootstrap_off", False, False), ("gaussian_bootstrap_on", False, True),
                                 ("categorical_meta", True, False)):
        env, agent, _ = setup(E, discrete=discrete)
        # iterations + 1: the evaluation before iteration `iters` is that of the policy after `iters` updates
        hist = train_vectorized(env, agent, iters + 1, T, seed=42, bootstrap_truncated=boot,
                                eval_episodes=eval_episodes, eval_interval=4)
        env.close()
        res[name] = {
            "eval": [{"after_iterations": i, "return_mean": m["eval_return_mean"], "return_std": m["eval_return_std"],
                      "length_mean": m["eval_length_mean"], "terminated_fraction": m["eval_terminated_fraction"]}
                     for i, m in enumerate(hist) if "eval_return_mean" in m],
            "train": [{"iteration": i, "episodes": m["episodes"], "return_mean": m["episode_return_mean"],
                       "length_mean": m["episode_length_mean"], "terminated_fraction": m["terminated_fraction"],
                       "explained_variance": m["explained_variance"]} for i, m in enumerate(hist[:iters])]}
        print(json.dumps({name: res[name]["eval"][-1]}), flush=True)
    res["iterations"], res["T"], res["envs"], res["eval_episodes"], res["seed"] = iters, T, E, eval_episodes, 42
    return res


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--envs", type=int, default=4096)
    p.add_argument("--eval-episodes", type=int, default=4096)
    p.add_argument("--rollout", type=int, default=32)
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--iters", type=int, default=24)
    p.add_argument("--out", default=None)
    args = p.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("episode_eval_bench measures the GPU path: no CUDA device visible")
    res = {"gpu": gpu_info(), "stats_launch": stats_launch(args.envs, args.rollout)}
    print(json.dumps({"stats_launch": res["stats_launch"]["us_per_launch_median"]}), flush=True)
    res["train_samples"] = train_samples(args.envs, args.rollout, args.rounds)
    print(json.dumps({"train_samples": res["train_samples"]["mean"]}), flush=True)
    res["evaluation"] = evaluation(args.eval_episodes)
    print(json.dumps({"evaluation": {k: v for k, v in res["evaluation"].items() if k != "graph" and k != "eager"} |
                      {k: res["evaluation"][k]["ms_median"] for k in ("graph", "eager")}}), flush=True)
    res["learning"] = learning(args.envs, args.rollout, args.iters, args.eval_episodes)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
