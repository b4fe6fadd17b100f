"""Throughput of the categorical policy on the DiscreteMetaAction env beside the Gaussian policy on the continuous env,
and a short learning check of the former.

    python tools/discrete_bench.py [--envs 4096] [--hidden 256] [--steps 200] [--out result.json]

Reports, in one process and with the GPU's name, power limit and max SM clock read in the same call:
  * policy env-steps/s: one policy act + one env step per timed step, L2 flushed between steps (a 256 MiB memset
    outside the per-step event pairs, as bench.py does), and the act / env split from a second pass;
  * PPO samples/s: rollout of T = 32 steps + update (8 epochs, minibatch 4096), as bench.py's ppo_samples_per_s;
  * the act path with the heads fused into the [a1 | c1] GEMM against the unfused one (HRP_FUSE_HEADS=0, which the
    library reads once per process: measured in a child process);
  * 20 iterations of the vectorised training loop (collect_rollout + update) on the meta-action env: mean step
    reward and policy entropy per iteration.
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


def setup(discrete, E, H, minibatch=4096, epochs=8, seed=42):
    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_vec_env
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.utils.reproducibility import set_random_seeds

    set_random_seeds(seed)
    cfg = copy.deepcopy(HIGHWAY_CONFIG)
    if discrete:
        cfg["action"] = {"type": "DiscreteMetaAction"}
    env = make_vec_env(Condition.SHUFFLED_ROPE, cfg, 4, {"observation": {"order": "shuffled"}}, num_envs=E, seed=seed)
    S = env.N * env.F_out
    agent = PPOAgent(S, 5 if discrete else 2, lr=3e-4, hidden_dim=H, batch_size=minibatch, epochs=epochs,
                     device="cuda:0", discrete=discrete)
    return env, agent, S


def policy_env_steps(env, agent, S, K, warmup):
    import torch

    E = env.num_envs
    obs = env.reset(42).view(E, S)
    out = agent.actor_critic._new_act_out(E)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    for _ in range(warmup):
        agent.act(obs, out=out)
        env.step(out["action"])
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)]
    for k in range(K):
        flush.zero_()
        ev[k][0].record()
        agent.act(obs, out=out)
        env.step(out["action"])
        ev[k][1].record()
    torch.cuda.synchronize()
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    ev3 = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    for k in range(K):
        flush.zero_()
        ev3[k][0].record()
        agent.act(obs, out=out)
        ev3[k][1].record()
        env.step(out["action"])
        ev3[k][2].record()
    torch.cuda.synchronize()
    act_us = sum(e[0].elapsed_time(e[1]) for e in ev3) * 1e3 / K
    env_us = sum(e[1].elapsed_time(e[2]) for e in ev3) * 1e3 / K
    return {"env_steps_per_s": E * K / (total_ms * 1e-3), "step_us": total_ms * 1e3 / K, "act_us": act_us,
            "env_us": env_us, "steps": K}


def ppo_samples(env, agent, T, iters=3):
    import torch

    from highway_rope_ppo_b200.training.routine import rollout_and_update

    o = env.reset(42)
    for _ in range(2):   # the first rollout runs launch by launch, the second one captures the rollout graph
        _, o = rollout_and_update(env, agent, T, obs=o)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        _, o = rollout_and_update(env, agent, T, obs=o)
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) * 1e-3
    return {"samples_per_s": iters * T * env.num_envs / s, "iteration_ms": s * 1e3 / iters, "T": T,
            "epochs": agent.epochs, "minibatch": agent.memory.batch_size}


def act_only(E, H, K):
    """Act-path time (policy forward + heads + sample) per call, L2 flushed between calls, both policies."""
    import torch

    res = {}
    for name, discrete in (("categorical", True), ("gaussian", False)):
        env, agent, S = setup(discrete, E, H)
        x = env.reset(42).view(E, S)
        out = agent.actor_critic._new_act_out(E)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
        for _ in range(10):
            agent.act(x, out=out)
        torch.cuda.synchronize()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)]
        for k in range(K):
            flush.zero_()
            ev[k][0].record()
            agent.act(x, out=out)
            ev[k][1].record()
        torch.cuda.synchronize()
        res[name] = sum(a.elapsed_time(b) for a, b in ev) * 1e3 / K
        env.close()
    return res


def learning_check(E, H, T, iters):
    import torch

    from highway_rope_ppo_b200.training.routine import collect_rollout

    env, agent, S = setup(True, E, H)
    obs = env.reset(0)
    hist = []
    for it in range(iters):
        r = collect_rollout(env, agent, T, obs)
        mean_r = float(r["reward"].mean())
        obs = r["states"][T].clone()
        _, _, v = agent.actor_critic.forward(obs)
        m = agent.update(last_value=v.view(-1))
        hist.append({"iteration": it, "mean_step_reward": mean_r, "entropy": m["entropy"], "loss": m["loss"]})
        print(json.dumps(hist[-1]), flush=True)
    env.close()
    return hist


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--hidden", type=int, default=256)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rollout", type=int, default=32)
    ap.add_argument("--learn-iters", type=int, default=20)
    ap.add_argument("--act-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    import torch

    from highway_rope_ppo_b200 import _lib

    _lib.require_device()
    if args.act_only:
        print(json.dumps(act_only(args.envs, args.hidden, args.steps)))
        return
    res = {"gpu": gpu_info(), "envs": args.envs, "hidden": args.hidden,
           "l2": "flushed between timed steps (256 MiB memset outside the per-step event pairs)"}
    for name, discrete in (("meta_action_categorical", True), ("continuous_gaussian", False)):
        env, agent, S = setup(discrete, args.envs, args.hidden)
        res[name] = {"policy": policy_env_steps(env, agent, S, args.steps, args.warmup),
                     "ppo": ppo_samples(env, agent, args.rollout)}
        print(name, json.dumps(res[name]), flush=True)
        env.close()
        del agent
        torch.cuda.empty_cache()
    res["act_us_fused"] = act_only(args.envs, args.hidden, args.steps)
    child = subprocess.run([sys.executable, os.path.abspath(__file__), "--act-only", "--envs", str(args.envs), "--hidden",
                            str(args.hidden), "--steps", str(args.steps)], capture_output=True, text=True,
                           env={**os.environ, "HRP_FUSE_HEADS": "0"})
    if child.returncode != 0:
        raise RuntimeError(child.stderr)
    res["act_us_unfused"] = json.loads(child.stdout.strip().splitlines()[-1])
    t0 = time.time()
    res["learning"] = {"iterations": learning_check(args.envs, args.hidden, args.rollout, args.learn_iters),
                       "wall_s": time.time() - t0}
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
