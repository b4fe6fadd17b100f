#!/usr/bin/env python
"""bench.py -- policy env-steps/s of the lock-step highway-v0 + PPO hot path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--envs E] [--hidden H]
                    [--condition rope|sorted|shuffled|rankpe|distpe] [--obs-vehicles N] [--d-embed D]
                    [--dump-outputs DIR]

BASELINE.json configs (the default is configs[1]):
    configs[2]: --condition rankpe --d-embed 16 --obs-vehicles 30 --envs 16384      (also distpe, d 4 / 8 / 16)
    configs[3]: --hidden 512 --envs 8192 under torchrun with 8 ranks (65536 envs)

Workload (BASELINE.json configs[1]): shuffled Kinematics observation + RoPE, hidden_dim 256, 4096 lock-step envs
per GPU, V = 51 vehicles, N = 15 rows, F = 4.  RoPE rotates rotate_dim = 4 features: the d_embed 16 of the config
string is rejected by the reference at HEAD for F = 4 (SURVEY.md F4), 4 is the only width `make_env` accepts.

One "step" = one policy step of every env: the policy kernel chain (MLP forward + tanh-Gaussian sampling,
`hrp_ppo_act`) followed by the fused env kernel (`hrp_env_step`: 15 simulation frames, reward / termination,
in-kernel respawn, shuffled observation, RoPE).  `value` is env-steps/s with everything resident in HBM; `e2e`
is the same step through the host-buffer API (observations and actions cross PCIe every step, as in the
reference's CPU loop); `roofline` is the env kernel against the measured HBM peak; `cpu_baseline` is the CPU
oracle (C restatement, OpenMP over envs + torch CPU policy) timed on this box's host cores.

Under torchrun each rank owns its own 4096 envs (weak scaling); the only collective on the path is the PPO
gradient all-reduce inside `ppo_samples_per_s` (reported beside the headline).
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "policy env-steps/s (4096 envs/GPU)"
UNIT = "env-steps/s"
KERNELS_PER_ACT = 4   # 3 x tcgen05 GEMM (trunk 2, actor | critic hidden layers as one) + heads_act (dot products, Philox sampling, log-prob)
KERNELS_PER_ENV_STEP = 1


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=400)
    p.add_argument("--warmup", type=int, default=40)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--envs", type=int, default=4096, help="envs per GPU")
    p.add_argument("--hidden", type=int, default=256)
    p.add_argument("--condition", default="rope", choices=["rope", "sorted", "shuffled", "rankpe", "distpe"])
    p.add_argument("--obs-vehicles", type=int, default=15, help="observed vehicles N (rows of the observation)")
    p.add_argument("--d-embed", type=int, default=None, help="rotate_dim (rope, default 4) / d_embed (rankpe, distpe)")
    p.add_argument("--minibatch", type=int, default=4096)
    p.add_argument("--epochs", type=int, default=8)
    p.add_argument("--rollout", type=int, default=32, help="T of the PPO iteration measured beside the headline")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-ppo", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--cpu-seconds", type=float, default=12.0)
    p.add_argument("--e2e-groups", type=int, default=1, choices=[1, 2, 4, 8],
                   help="env groups of the host-buffer loop: G groups of E/G envs on G streams (copies and host turn-around "
                        "of one under the kernels of the others)")
    p.add_argument("--e2e-chunks", type=int, default=1,
                   help="row chunks of the observation fetch: the policy of a chunk runs while the next one crosses PCIe")
    p.add_argument("--e2e-eager", action="store_true", help="host-buffer loop without CUDA graphs")
    p.add_argument("--e2e-copy-engine", action="store_true",
                   help="observation H2D by cudaMemcpyAsync instead of the fetch kernel (hrp_fetch_host)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write what the last timed step returned (policy outputs, observation, reward, flags of rank 0) "
                        "as DIR/<name>.npy, to compare two builds output for output")
    args = p.parse_args()
    if args.impl == "ours" and args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs records the GPU path (--impl ours)")
    return args


def condition_of(args):
    """(Condition name, d_embed, env overrides) of the command line."""
    d = args.d_embed
    if args.condition == "rope":
        d = 4 if d is None else d
    elif args.condition in ("rankpe", "distpe") and d is None:
        d = 16
    over = {"observation": {"order": "sorted" if args.condition == "sorted" else "shuffled",
                            "vehicles_count": args.obs_vehicles}}
    name = {"rope": "SHUFFLED_ROPE", "sorted": "SORTED", "shuffled": "SHUFFLED", "rankpe": "SHUFFLED_RANKPE",
            "distpe": "SHUFFLED_DISTPE"}[args.condition]
    return name, d, over


def workload_config(args):
    _, d, _ = condition_of(args)
    emb = {"rope": f"shuffled obs + RoPE(rotate_dim {d}; d_embed 16 invalid at F=4, SURVEY F4)", "sorted": "sorted obs",
           "shuffled": "shuffled obs", "rankpe": f"shuffled obs + RankPE(d_embed {d})",
           "distpe": f"shuffled obs + DistPE(d_embed {d})"}[args.condition]
    return {"workload": f"highway-v0 {emb}, hidden_dim {args.hidden}, {args.envs} lock-step envs/GPU, V=51, "
                        f"N={args.obs_vehicles}, F=4, 15 substeps/step",
            "envs_per_gpu": args.envs, "hidden_dim": args.hidden, "condition": args.condition, "d_embed": d,
            "obs_vehicles": args.obs_vehicles, "ppo_minibatch": args.minibatch, "ppo_epochs": args.epochs,
            "l2": "flushed between timed steps (256 MiB memset outside the per-step event pairs)"}


# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock / throttle reasons of one GPU while the timed region runs (NVML, 20 ms period)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = str(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake_slowdown"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def result(self):
        self.stop_flag = True
        if self.is_alive():
            self.join(timeout=1.0)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def offline_ncu(kernel):
    """Per-env counters of `kernel` from the ncu summary committed under profiles/ (tools/ncu_summary.py writes
    profiles/ncu_counters.json from an `ncu --set full` capture); None when there is none."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_counters.json")) as f:
            c = json.load(f)[kernel]
        return {"dram_bytes_per_env": float(c["dram_bytes"]) / c["envs"],
                "warp_instructions_per_env": float(c["warp_instructions"]) / c["envs"], "source": c["source"]}
    except Exception:
        return None


def algorithmic_bytes_per_env_step(V=51, N=15, Fout=4):
    """DESIGN.md: state read once + written once per POLICY step (the 15 substeps stay on chip).
    Per vehicle: read x(8) timer(8) y,heading,speed,target_speed,delta,impx,impy (7x4) flags(4) = 48 B, write
    the same minus the two per-episode constants (target_speed, delta) = 40 B; per env: action 8, time 8+8,
    episode/draw counters 16, obs 4 N Fout, reward 4, flags 2."""
    return 88 * V + 4 * N * Fout + 46


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Write every array (leading axis: env) as float32 `path/<name>.npy`.  When they hold more than DUMP_LIMIT_BYTES
    in all, the same fixed, seeded sample of env rows is kept from each, and its row indices go to env_index.npy."""
    import numpy as np

    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    rows = next(iter(arrays.values())).shape[0]
    per_row = sum(a.nbytes for a in arrays.values()) // rows
    if per_row * rows > DUMP_LIMIT_BYTES:
        keep = (DUMP_LIMIT_BYTES - 128 * (len(arrays) + 1)) // (per_row + 8)   # 128: .npy header; 8: float64 index
        idx = np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, f"{k}.npy"), a)


# ---------------------------------------------------------------------------------------------
def _cpu_setup(args):
    """Config, embedding function and policy parameters of the CPU arms (the oracle's restatements)."""
    import numpy as np
    import torch
    import torch.nn as nn

    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from oracle import embed as oe

    _, d, over = condition_of(args)
    cfg = copy.deepcopy(HIGHWAY_CONFIG)
    cfg["observation"].update(over["observation"])
    N, F = args.obs_vehicles, 4
    if args.condition == "rope":
        inv = oe.rope_inv_freq(d, 100.0)

        def embed(obs):   # vectorised numpy restatement of rope_embed.py:64-74
            E = obs.shape[0]
            rel = obs[:, :, :2] - obs[:, :1, :2]
            dn = np.clip(np.linalg.norm(rel, axis=-1) / 100.0, 0.0, 1.0).astype(np.float32)
            theta = (2 * np.pi * dn[..., None] * inv[None, None, :]).astype(np.float32)
            sn, cs = np.sin(theta), np.cos(theta)
            pair = obs[:, :, :d].reshape(E, N, d // 2, 2)
            rot = np.stack([pair[..., 0] * cs - pair[..., 1] * sn, pair[..., 0] * sn + pair[..., 1] * cs], axis=-1)
            return np.concatenate([rot.reshape(E, N, d), obs[:, :, d:]], axis=-1).reshape(E, -1)
        Fout = F
    elif args.condition == "distpe":
        fr = oe.dist_freqs(d, 100.0)

        def embed(obs):   # dist_embed.py:76-96
            rel = obs[:, :, :2] - obs[:, :1, :2]
            dn = np.clip(np.linalg.norm(rel, axis=-1) / 100.0, 0.0, 1.0).astype(np.float32)
            ang = 2 * np.pi * dn[..., None] * fr[None, None, :]
            return np.concatenate([obs, np.sin(ang), np.cos(ang)], axis=-1).astype(np.float32).reshape(obs.shape[0], -1)
        Fout = F + d
    elif args.condition == "rankpe":
        tag = np.tanh(np.random.default_rng(0).uniform(-0.05, 0.05, (N, d))).astype(np.float32)

        def embed(obs):   # rank_embed.py:45-51 (intended semantics, SURVEY F5)
            return np.concatenate([obs, np.broadcast_to(tag, (obs.shape[0], N, d))], axis=-1).reshape(obs.shape[0], -1)
        Fout = F + d
    else:
        def embed(obs):
            return obs.reshape(obs.shape[0], -1)
        Fout = F
    S, A, H = N * Fout, 2, args.hidden
    torch.manual_seed(0)
    flat = torch.cat([torch.zeros(A)] + [p.detach().reshape(-1) for layer in
                                         (nn.Linear(S, H), nn.Linear(H, H), nn.Linear(H, H), nn.Linear(H, A),
                                          nn.Linear(H, H), nn.Linear(H, 1)) for p in layer.parameters()])
    return cfg, embed, flat, S, A, H, N


def cpu_policy_env_steps(args, seconds, n_envs, steps=None, warmup=1):
    """Oracle arm: C restatement of highway-v0 (OpenMP over envs, all host cores) + torch CPU MLP policy."""
    import numpy as np
    import torch

    from oracle import highway as oh
    from oracle import ppo_ref

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    oh.use_lean_build()   # the plain algorithm: the parity tests' decision bookkeeping is compiled out
    cfg, embed, flat, S, A, H, N = _cpu_setup(args)
    vec = oh.OracleVecEnv(cfg, n_envs, seed=42, nthreads=cores)
    obs = np.zeros((n_envs, N, 4), dtype=np.float32)

    def one_step(obs):
        # observation wrapper + policy forward + env step
        x = torch.from_numpy(np.ascontiguousarray(embed(obs), dtype=np.float32))
        with torch.no_grad():
            mean, log_std, value = ppo_ref.forward(flat, x, S, A, H)
            act = torch.tanh(mean + log_std.exp() * torch.randn_like(mean))
        return vec.step(act.numpy())[0]

    for _ in range(warmup):
        obs = one_step(obs)
    n, t0 = 0, time.perf_counter()
    while True:
        obs = one_step(obs)
        n += 1
        el = time.perf_counter() - t0
        if steps is not None:
            if n >= steps:
                break
        elif el >= seconds and n >= 3:
            break
    return {"value": n * n_envs / el, "steps": n, "envs": n_envs, "seconds": el, "cores": cores}


def cpu_ppo_update(args, n_samples, repeats=1):
    """The reference's PPOAgent.update arithmetic (ppo/agent.py:196-252) on the host cores: oracle/ppo_ref.py, the
    torch-fp32 autograd restatement that tests/test_oracle_cpu.py pins to fixtures produced by the reference's own
    agent.  `n_samples` stored transitions, minibatches of args.minibatch, args.epochs epochs (a bounded sample of
    the GPU arm's update: the cost per sample-pass does not depend on the buffer length).  Returns seconds per
    sample of the rollout buffer (one update = epochs passes over it)."""
    import numpy as np
    import torch

    from oracle import ppo_ref

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    _, _, flat, S, A, H, _ = _cpu_setup(args)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(n_samples, S, generator=g)
    z = torch.randn(n_samples, A, generator=g) * 0.5
    olp = -torch.rand(n_samples, generator=g) - 1.0
    adv, ret = torch.randn(n_samples, generator=g), torch.rand(n_samples, generator=g)
    bs = min(args.minibatch, n_samples)
    m, v = torch.zeros_like(flat), torch.zeros_like(flat)
    step, best = 0, float("inf")
    for rep in range(repeats + 1):   # the first pass warms the allocator and the thread pool
        t0 = time.perf_counter()
        perm = torch.randperm(n_samples, generator=g)
        for _ in range(args.epochs):
            for start in range(0, n_samples, bs):
                idx = perm[start:start + bs]
                r = ppo_ref.loss_and_grad(flat, x[idx], z[idx], olp[idx], adv[idx], ret[idx], S, A, H)
                step += 1
                flat, m, v, _ = ppo_ref.clip_adam(flat, r["grad"], m, v, step)
        el = time.perf_counter() - t0
        if rep > 0:
            best = min(best, el)
    return {"s_per_sample": best / n_samples, "samples": n_samples, "optimizer_steps": args.epochs * ((n_samples + bs - 1) // bs),
            "seconds": best, "cores": cores, "state_dim": S, "hidden_dim": H}


def cpu_ppo_samples_per_s(args, env_steps_per_s, upd):
    """PPO samples/s of the CPU arm: one sample costs one policy+env step plus its share of the update."""
    return 1.0 / (1.0 / env_steps_per_s + upd["s_per_sample"])


def run_reference(args):
    """`--impl reference`: the reference path on the host cores.  The simulator the reference calls
    (highway-env 1.10.1) is a third-party package absent from this image (profiles/r02_highway_env_probe.txt), so
    this arm times the oracle's C restatement of it (kind "port") with every host thread, plus a torch CPU policy
    forward; the PPO half is the reference's update arithmetic (oracle/ppo_ref.py, pinned to the reference's agent)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    budget = 120.0  # seconds for the whole --steps/--warmup run
    probe = cpu_policy_env_steps(args, 2.0, 256, steps=2, warmup=1)
    per_env_step = 1.0 / probe["value"]
    total = max(1, args.steps + args.warmup)
    n_envs = int(min(args.envs, max(64, budget / (total * per_env_step))))
    res = cpu_policy_env_steps(args, 0.0, n_envs, steps=args.steps, warmup=max(1, args.warmup))
    upd = cpu_ppo_update(args, 2 * args.minibatch)
    ppo = cpu_ppo_samples_per_s(args, res["value"], upd)
    cfg = workload_config(args)
    line = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * res["seconds"] / res["steps"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg, "gpu_launches": 0,
            "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": "port",
                             "sample": f"{res['envs']} envs x {res['steps']} policy steps, oracle C restatement "
                                       "(OpenMP) + torch CPU policy forward"},
            "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "ppo_samples_per_s": {"value": ppo, "unit": "samples/s", "kind": "port", "cores": upd["cores"],
                                  "update_s_per_sample": upd["s_per_sample"],
                                  "sample": f"update: {upd['samples']} stored samples, {upd['optimizer_steps']} optimizer steps of "
                                            f"{min(args.minibatch, upd['samples'])} ({upd['seconds']:.2f} s), torch fp32 autograd "
                                            f"restatement of ppo/agent.py:196-252 (S={upd['state_dim']}, H={upd['hidden_dim']}); "
                                            "rollout: the env-steps/s of this line",
                                  "definition": "1 / (1 / policy-env-steps/s + update seconds per stored sample)"}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from highway_rope_ppo_b200 import _lib
    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_vec_env
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.routine import rollout_and_update
    from highway_rope_ppo_b200.utils.reproducibility import set_random_seeds

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    _lib.require_device()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    E, A, H = args.envs, 2, args.hidden
    set_random_seeds(42)
    cond_name, d_embed, over = condition_of(args)
    env = make_vec_env(Condition[cond_name], HIGHWAY_CONFIG, d_embed, over, num_envs=E, device=dev, seed=42,
                       env_id_base=rank * E, strict_d_embed=False)
    N, Fout = env.N, env.F_out
    S = N * Fout
    agent = PPOAgent(S, A, lr=3e-4, hidden_dim=H, batch_size=args.minibatch, epochs=args.epochs, device=dev)
    agent.actor_critic.row_base = rank * E   # exploration noise keyed by the global env id
    obs = env.reset(42).view(E, S)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"action": torch.empty((E, A), device=dev), "pre_tanh": torch.empty((E, A), device=dev),
           "log_prob": torch.empty(E, device=dev), "value": torch.empty(E, device=dev)}

    def policy_env_step():
        agent.act(obs, out=out)
        env.step(out["action"])  # writes env.obs, which `obs` views

    for _ in range(args.warmup):
        policy_env_step()
    K = args.steps
    calls0 = (agent.launches, env.launches)   # hrp_ppo_act_sample / hrp_env_step calls enqueued so far
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)]
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    wall0 = time.perf_counter()
    for k in range(K):
        flush.zero_()                       # evict the (L2-sized) working set between timed iterations
        ev[k][0].record()
        agent.act(obs, out=out)             # no event between the two: the env kernel is launched programmatically
        stepped = env.step(out["action"])   # dependent on the policy's last kernel and overlaps its tail
        ev[k][1].record()
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.result()
    if args.dump_outputs and rank == 0:   # before the passes below step the same env and agent again
        dump_outputs(args.dump_outputs, {**{k: v.cpu() for k, v in out.items()},
                                         **{k: v.cpu() for k, v in zip(("obs", "reward", "terminated", "truncated"),
                                                                       stepped)}})
    # kernels of this library launched inside the timed region: counted calls x kernels per call (a policy call is
    # 3 tcgen05 GEMM launches + heads_act, an env step is one fused kernel; profiles/r02_launches_bench.csv)
    gpu_launches = (agent.launches - calls0[0]) * KERNELS_PER_ACT + (env.launches - calls0[1]) * KERNELS_PER_ENV_STEP
    total_ms = sum(e[0].elapsed_time(e[1]) for e in ev)
    # the split of a step into policy and env kernel time, from a second pass with an event between the two phases
    # (that event serialises them, so act_ms + env_ms is slightly more than a step of the timed pass)
    ev3 = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    for k in range(K):
        flush.zero_()
        ev3[k][0].record()
        agent.act(obs, out=out)
        ev3[k][1].record()
        env.step(out["action"])
        ev3[k][2].record()
    barrier()
    act_ms = sum(e[0].elapsed_time(e[1]) for e in ev3)
    env_ms = sum(e[1].elapsed_time(e[2]) for e in ev3)
    t = torch.tensor([total_ms, env_ms, act_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, env_ms, act_ms = (float(x) for x in t.cpu())
    value = world * E * K / (total_ms * 1e-3)

    # back-to-back (no flush, one event pair around all K steps): what a training loop actually sees
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        policy_env_step()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    warm_value = world * E * K / (float(t.cpu()) * 1e-3)

    # env kernel alone, random actions resident in HBM (the "env-step-only" sweep point of BASELINE configs[4])
    acts = torch.rand((E, 2), device=dev) * 2 - 1
    barrier()
    e0.record()
    for k in range(K):
        env.step(acts)
    e1.record()
    barrier()
    env_only = world * E * K / (e0.elapsed_time(e1) * 1e-3)

    # roofline of the dominant kernel (the fused env step), from the flushed per-step events
    peak, peak_src = measured_peak()
    bytes_per_launch = algorithmic_bytes_per_env_step(51, N, Fout) * E
    env_kernel_s = env_ms * 1e-3 / K
    achieved = bytes_per_launch / env_kernel_s / 1e9
    off = offline_ncu("hrp_step_kernel")   # counters of an ncu capture committed under profiles/ (not measured in this run)
    roofline = {"bound": "hbm", "kernel": "hrp_step_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak,
                "traffic": None if off is None else int(off["dram_bytes_per_env"] * E),
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_per_launch, "kernel_us": env_kernel_s * 1e6,
                "share_of_step": env_ms / (env_ms + act_ms),
                "note": "instruction-issue-bound kernel (15 fused substeps per launch), not HBM-bound; see DESIGN.md 3.1"}
    if off is not None:
        # the binding resource: warp-instruction issue slots (4 schedulers x 148 SMs x sm clock)
        wi = off["warp_instructions_per_env"] * E
        peak_issue = 4 * 148 * (clocks.get("sm_mhz") or 1965) * 1e6
        roofline["traffic_source"] = roofline_src = off["source"]
        roofline["issue"] = {"warp_instructions_per_launch": wi, "source": roofline_src + " (offline ncu capture, scaled by envs)",
                             "achieved_ginst_s": wi / env_kernel_s / 1e9, "peak_ginst_s": peak_issue / 1e9,
                             "frac": wi / env_kernel_s / peak_issue}

    # e2e: the same step through the host-buffer API (training/host_pipeline.py): pinned host observation -> H2D ->
    # policy -> env kernel -> observation / reward / flags written straight into pinned host buffers, action D2H; one
    # CUDA graph launch and ONE host synchronisation (an event) per group-step.  With G groups of E/G envs on G streams
    # one group's PCIe traffic and host turn-around hide under the other groups' kernels.
    e2e = None
    if not args.no_e2e:
        from highway_rope_ppo_b200.training.host_pipeline import HostBufferPipeline

        Ke = min(K, 200)
        G = args.e2e_groups if E % args.e2e_groups == 0 else 1
        Eg = E // G
        genvs = [make_vec_env(Condition[cond_name], HIGHWAY_CONFIG, d_embed, over, num_envs=Eg, device=dev, seed=42,
                              env_id_base=rank * E + gi * Eg, strict_d_embed=False) for gi in range(G)]
        pipe = HostBufferPipeline(agent, genvs, use_graphs=not args.e2e_eager, kernel_fetch=not args.e2e_copy_engine,
                                  chunks=args.e2e_chunks)
        pipe.reset(42)
        for _ in range(5):
            for gi in range(G):
                pipe.launch(gi)
        for gi in range(G):
            pipe.wait(gi)
        barrier()
        w0 = time.perf_counter()
        for _ in range(Ke):
            for gi in range(G):
                pipe.launch(gi)      # waits for the group's previous results to be on the host first
        for gi in range(G):
            pipe.wait(gi)
        w = time.perf_counter() - w0          # host clock: the region ends with every result on the host
        barrier()
        t = torch.tensor([w], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": world * E * Ke / float(t.cpu()), "unit": UNIT,
               "h2d_bytes_per_step": E * S * 4, "d2h_bytes_per_step": E * 2 * 4 + E * S * 4 + E * 4 + 2 * E,
               "steps": Ke, "groups": G, "chunks": args.e2e_chunks, "cuda_graphs": not args.e2e_eager,
               "h2d_by": "copy engine (cudaMemcpyAsync)" if args.e2e_copy_engine else "kernel reading the mapped pinned buffer (hrp_fetch_host)",
               "api": "HostBufferPipeline.launch / wait (training/host_pipeline.py): PPOAgent.act on a pinned-host "
                      "observation (H2D copy) + HighwayVecEnv.step_host_async (hrp_env_step_host_async): the device action "
                      "feeds the step, the kernel writes observation, reward and flags straight into the page-locked host "
                      "buffers (zero-copy), the action is copied to the host under the env kernel; one graph launch and one "
                      f"event wait per group-step, {G} group(s) of {Eg} envs on their own streams"}
        pipe.close()
        agent.actor_critic.row_base = rank * E
        for genv in genvs:
            genv.close()

    # PPO iteration (rollout of T steps + update: epochs x minibatches, gradient exchange if N > 1)
    ppo = None
    if not args.no_ppo:
        from highway_rope_ppo_b200.training.routine import collect_rollout

        T = args.rollout
        o = env.reset(42)
        for _ in range(2):   # warm-up: the first rollout runs launch by launch, the second one captures the rollout graph
            _, o = rollout_and_update(env, agent, T, obs=o)
        barrier()
        iters = 2
        evp = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(iters)]
        for it in range(iters):   # rollout_and_update, with an event between its two halves
            evp[it][0].record()
            r = collect_rollout(env, agent, T, o)
            o = r["states"][T].clone()
            _, _, last_v = agent.actor_critic.forward(o)
            evp[it][1].record()
            m = agent.update(last_value=last_v.view(-1))
            evp[it][2].record()
        barrier()
        t = torch.tensor([sum(e[0].elapsed_time(e[2]) for e in evp), sum(e[1].elapsed_time(e[2]) for e in evp)],
                         dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tot_ms, upd_ms = (float(x) for x in t.cpu())
        n_local = E * T
        bs = min(args.minibatch, n_local)
        opt_steps = args.epochs * ((n_local + bs - 1) // bs)
        # useful fp32 FLOPs of one optimizer step on one rank: forward, input gradients, weight gradients of the three
        # hidden GEMMs (the N = 2 / 1 heads are not GEMMs here); 3xTF32 executes three tensor-core passes per product
        fwd = 2.0 * bs * (S * H + H * H + H * 2 * H)
        dgrad = 2.0 * bs * (2 * H * H + H * H)
        wgrad = 2.0 * bs * (S * H + H * H + 2 * H * H)
        flops_step = fwd + dgrad + wgrad
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                tens_peak, tens_src = float(json.load(f)["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
        except Exception:
            tens_peak, tens_src = 2250.0, "fallback (nominal dense bf16 2.25 PFLOP/s)"
        step_us = upd_ms * 1e3 / (iters * opt_steps)
        ach = flops_step / (step_us * 1e-6) / 1e12
        ppo = {"value": world * E * T * iters / (tot_ms * 1e-3), "unit": "samples/s", "rollout_T": T,
               "epochs": args.epochs, "minibatch": bs, "last_loss": m["loss"],
               "update_ms": upd_ms / iters, "rollout_ms": (tot_ms - upd_ms) / iters, "optimizer_step_us": step_us,
               "cuda_graphs": agent._graph_state is not None, "backend": dist.get_backend() if world > 1 else None,
               "gradient_exchange": ("peer-memory kernel (hrp_clip_adam_step_p2p)" if agent._comm is not None else "nccl all_reduce") if world > 1 else None,
               "definition": "T policy+env steps then PPOAgent.update (GAE, epochs x minibatches, clip+Adam), amortised",
               "roofline_ppo": {"bound": "tensor", "kernel": "one optimizer step (forward + backward GEMMs, loss, clip + Adam)",
                                "achieved": ach, "peak": tens_peak, "unit": "TFLOP/s", "frac": ach / tens_peak,
                                "peak_source": tens_src, "useful_flops_per_step": flops_step,
                                "note": "useful fp32 FLOPs / measured time of a whole optimizer step; kind::tf32 runs at half "
                                        "the bf16 rate and 3xTF32 issues three passes per product, so 1/6 of this peak is "
                                        "the ceiling of the arithmetic mode"}}
        if world > 1:
            # every rank must hold bit-identical parameters after the sharded updates (same reduced gradient, same Adam)
            flat = agent.actor_critic.flat
            digest = torch.stack([flat.double().sum(), (flat.double() * torch.arange(1, flat.numel() + 1, device=dev,
                                                                                    dtype=torch.float64)).sum()])
            lo, hi = digest.clone(), digest.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            ref = flat.clone()
            dist.broadcast(ref, src=0)
            same = torch.tensor([1 if torch.equal(ref, flat) else 0], device=dev)
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
            ppo["ranks_bit_identical"] = bool(int(same.item()) == 1 and torch.equal(lo, hi))
            assert ppo["ranks_bit_identical"], "parameters differ between ranks after the sharded PPO updates"

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_policy_env_steps(args, args.cpu_seconds, 1024)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
               "sample": f"{r['envs']} envs x {r['steps']} policy steps ({r['seconds']:.1f} s), oracle C restatement of "
                         "highway-env 1.10.1 (OpenMP over envs) + torch CPU policy forward"}
        if not args.no_ppo:
            upd = cpu_ppo_update(args, 2 * args.minibatch)
            cpu["ppo_samples_per_s"] = {
                "value": cpu_ppo_samples_per_s(args, r["value"], upd), "unit": "samples/s", "kind": "port", "cores": upd["cores"],
                "update_s_per_sample": upd["s_per_sample"],
                "sample": f"update: {upd['samples']} stored samples, {upd['optimizer_steps']} optimizer steps of "
                          f"{min(args.minibatch, upd['samples'])} ({upd['seconds']:.2f} s), torch fp32 autograd restatement of "
                          f"ppo/agent.py:196-252 pinned to the reference agent's fixtures (S={upd['state_dim']}, "
                          f"H={upd['hidden_dim']}); rollout: the CPU env-steps/s above"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
                "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32 (x, lane-change timer f64)", "data": "synthetic", "config": workload_config(args),
                "clocks": clocks, "e2e": e2e, "gpu_launches": gpu_launches,
                "roofline": roofline, "cpu_baseline": cpu,
                "value_back_to_back_l2_warm": warm_value, "env_only_steps_per_s": env_only,
                "policy_ms_per_step": act_ms / K, "env_ms_per_step": env_ms / K, "ppo_samples_per_s": ppo,
                "wall_s_timed_region": wall}
        print(json.dumps(line), flush=True)
    env.close()
    if world > 1:
        # graphs and peer mappings go before the communicator does.  With the peer-memory exchange no NCCL work is
        # captured in the graphs and destroy_process_group() returns (tools/p2p_check.py prints it); the timer only
        # guards the NCCL-in-graph fallback (HRP_P2P=0), where the teardown was seen to hang.
        agent.close()
        barrier()
        sys.stdout.flush()
        threading.Timer(30.0, lambda: os._exit(0)).start()
        dist.destroy_process_group()
        os._exit(0)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
