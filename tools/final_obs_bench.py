"""Cost of time-limit bootstrapping in the batched loop (hrp_env_step_final + the critic pass over final_states +
hrp_gae_ex), and an informational learning comparison.

    python tools/final_obs_bench.py [--envs 4096] [--steps 200] [--iters 24] [--out result.json]

Reports, in one process and with the GPU's name, power limit and max SM clock read in the same call:
  * step-kernel time at --envs envs with and without the final-observation output: CUDA events around each step, L2
    flushed between steps (a 256 MiB memset outside the event pairs, as bench.py does), the two variants alternated
    step by step on two handles with the same state and actions; the fraction of envs that finished per step beside it;
  * PPO samples/s at bench.py's defaults (T = 32, 8 epochs, minibatch 4096, hidden 256, shuffled RoPE) with
    bootstrap_truncated off and on, alternated three times (one agent and env per setting, so that each keeps its
    captured rollout graph);
  * --iters iterations of train_vectorized each way from the same seed on the default config (40-step time limit):
    mean step reward and explained variance per iteration.  Not a pass/fail check.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import subprocess
import sys

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


def setup(E, H=256, minibatch=4096, epochs=8, seed=42):
    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_vec_env
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.utils.reproducibility import set_random_seeds

    set_random_seeds(seed)
    cfg = copy.deepcopy(HIGHWAY_CONFIG)
    env = make_vec_env(Condition.SHUFFLED_ROPE, cfg, 4, {"observation": {"order": "shuffled"}}, num_envs=E, seed=seed)
    S = env.N * env.F_out
    agent = PPOAgent(S, 2, lr=3e-4, hidden_dim=H, batch_size=minibatch, epochs=epochs, device="cuda:0")
    return env, agent, S


def step_kernel(E, K, warmup):
    """Two handles in lock step (same seed, same actions): one steps plainly, the other with final_obs_out."""
    import numpy as np
    import torch

    plain, _, _ = setup(E)
    final, _, _ = setup(E)
    plain.reset(42)
    final.reset(42)
    fin = torch.empty((E, final.N, final.F_out), dtype=torch.float32, device="cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    g = torch.Generator(device="cuda:0").manual_seed(0)
    acts = [torch.rand((E, 2), generator=g, device="cuda:0") * 2 - 1 for _ in range(16)]
    for k in range(warmup):
        plain.step(acts[k % 16])
        final.step(acts[k % 16], final_obs_out=fin)
    torch.cuda.synchronize()
    ev = {n: [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)] for n in ("plain", "final")}
    done = []
    for k in range(K):
        a = acts[k % 16]
        for name, env in (("plain", plain), ("final", final)):
            flush.zero_()
            ev[name][k][0].record()
            if name == "plain":
                env.step(a)
            else:
                env.step(a, final_obs_out=fin)
            ev[name][k][1].record()
        done.append(((final.terminated | final.truncated) != 0).float().mean())
    torch.cuda.synchronize()
    res = {}
    for name in ("plain", "final"):
        t = np.array([a.elapsed_time(b) * 1e3 for a, b in ev[name]])
        res[name] = {"mean_us": float(t.mean()), "median_us": float(np.median(t)), "p10_us": float(np.percentile(t, 10)),
                     "p90_us": float(np.percentile(t, 90))}
    assert torch.equal(plain.obs, final.obs) and torch.equal(plain.reward, final.reward)   # same trajectories
    frac = torch.stack(done).cpu().numpy()
    res["done_fraction_per_step"] = {"mean": float(frac.mean()), "max": float(frac.max())}
    res["overhead_pct_median"] = 100.0 * (res["final"]["median_us"] / res["plain"]["median_us"] - 1.0)
    res["envs"], res["steps"] = E, K
    plain.close()
    final.close()
    return res


def ppo_samples(E, T, rounds):
    import torch

    from highway_rope_ppo_b200.training.routine import rollout_and_update

    arms = {}
    for boot in (False, True):
        env, agent, _ = setup(E)
        o = env.reset(42)
        for _ in range(2):   # the first rollout runs launch by launch, the second one captures the rollout graph
            _, o = rollout_and_update(env, agent, T, obs=o, bootstrap_truncated=boot)
        torch.cuda.synchronize()
        arms[boot] = [env, agent, o]
    out = {"off": [], "on": []}
    for _ in range(rounds):
        for boot in (False, True):
            env, agent, o = arms[boot]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                _, o = rollout_and_update(env, agent, T, obs=o, bootstrap_truncated=boot)
            e1.record()
            torch.cuda.synchronize()
            arms[boot][2] = o
            out["on" if boot else "off"].append(3 * T * E / (e0.elapsed_time(e1) * 1e-3))
    for env, _, _ in arms.values():
        env.close()
    mean = {k: sum(v) / len(v) for k, v in out.items()}
    return {"samples_per_s": out, "mean": mean, "cost_pct": 100.0 * (1.0 - mean["on"] / mean["off"]), "T": T,
            "epochs": 8, "minibatch": 4096, "envs": E}


def learning(E, T, iters):
    import torch

    from highway_rope_ppo_b200.training.routine import collect_rollout

    res = {}
    for boot in (False, True):
        env, agent, _ = setup(E)
        o = env.reset(42)
        hist = []
        for _ in range(iters):
            r = collect_rollout(env, agent, T, o, bootstrap_truncated=boot)
            rew = float(r["reward"].mean())
            trunc = float(((r["truncated"] != 0) & (r["terminated"] == 0)).float().mean())
            o = r["states"][T].clone()
            _, _, lv = agent.actor_critic.forward(o)
            m = agent.update(last_value=lv.view(-1))
            hist.append({"mean_step_reward": rew, "explained_variance": m["explained_variance"],
                         "value_loss": m["value_loss"], "truncated_fraction": trunc})
        torch.cuda.synchronize()
        env.close()
        last = hist[-5:]
        res["on" if boot else "off"] = {
            "per_iteration": hist,
            "last5_mean_step_reward": sum(h["mean_step_reward"] for h in last) / len(last),
            "last5_explained_variance": sum(h["explained_variance"] for h in last) / len(last)}
    res["iterations"], res["T"], res["envs"] = iters, T, E
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
        raise SystemExit("final_obs_bench measures the GPU path: no CUDA device visible")
    res = {"gpu": gpu_info(), "step_kernel": step_kernel(args.envs, args.steps, args.warmup)}
    print(json.dumps({"step_kernel": res["step_kernel"]}), flush=True)
    res["ppo"] = ppo_samples(args.envs, args.rollout, args.rounds)
    print(json.dumps({"ppo": res["ppo"]}), flush=True)
    res["learning"] = learning(args.envs, args.rollout, args.iters)
    print(json.dumps({k: v for k, v in res["learning"].items() if k in ("iterations",)} |
                     {k: {kk: vv for kk, vv in res["learning"][k].items() if kk != "per_iteration"}
                      for k in ("off", "on")}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
