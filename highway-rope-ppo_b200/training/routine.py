"""Rollout / update loops (reference: ``training/routine.py:14-29,61-297``).

``evaluate`` and ``train_with_experiment_name`` keep the reference's signatures, episode/seed
schedule (``reset(seed=exp_seed+episode_num)``, eval seeds ``exp_seed+1000+ep``), ``done =
terminated or truncated`` bootstrap masking, best/solved checkpoint policy and the
``metrics_history`` / summary-CSV schemas, so the reference's offline analysis reads the outputs
unchanged.  Plotting (matplotlib) is out of scope and skipped.

``rollout_and_update`` / ``train_vectorized`` are the batched loops: E lock-step envs, every
tensor device-resident, one policy kernel + one env kernel per step, one update per T steps.
"""
from __future__ import annotations

import json
import logging
import os
import time
from typing import Any, Dict, Optional

import numpy as np
import torch

from ..ppo import distributed
from .episodes import episode_stats, new_stats, policy_steps, summarize

ARTIFACTS_DIR = os.path.join("artifacts", "highway-ppo")


def ensure_artifacts_dir(custom_path: Optional[str] = None) -> str:
    path = custom_path or ARTIFACTS_DIR
    os.makedirs(path, exist_ok=True)
    return path


# The reference loop is written ONCE, as a coroutine that yields every interaction with the env and the agent as a
# request -- ("reset", seed) -> observation; ("act", flat_state, deterministic) -> (action, pre_tanh, log_prob, value);
# ("step", action) -> (next_obs, reward, terminated, truncated); ("value", flat_state) -> V(s); ("update", last_value)
# -> metrics; ("save", path) -> None -- and two drivers answer the requests: `drive` with one env and one agent (the
# reference's process-per-experiment shape), and experiments/multiplex.py with R experiments at once, batching the
# requests of a tick into one env launch and one host synchronisation.  Same control flow, same arithmetic.
def _evaluate_co(num_episodes: int, exp_seed: int):
    returns = []
    for ep in range(num_episodes):
        state = yield ("reset", exp_seed + 1000 + ep)
        flat = state.reshape(-1)
        done, total = False, 0.0
        while not done:
            action, _, _, _ = yield ("act", flat, True)
            nxt, reward, terminated, truncated = yield ("step", action)
            done = terminated or truncated
            flat = nxt.reshape(-1)
            total += reward
        returns.append(total)
    return float(np.mean(returns))


def drive(co, env, agent):
    """Answer a coroutine's requests with one env and one agent; returns the coroutine's return value."""
    try:
        req = next(co)
        while True:
            kind = req[0]
            if kind == "act":
                resp = agent.select_action(req[1], deterministic=req[2])
            elif kind == "step":
                nxt, reward, terminated, truncated, _ = env.step(req[1])
                resp = (nxt, reward, terminated, truncated)
            elif kind == "reset":
                resp, _ = env.reset(seed=req[1])
            elif kind == "value":
                _, _, v = agent.actor_critic.forward(req[1])
                resp = float(v.cpu().item())
            elif kind == "update":
                resp = agent.update(last_value=req[1])
            elif kind == "save":
                agent.save(req[1])
                resp = None
            else:
                raise RuntimeError(f"unknown request {kind!r}")
            req = co.send(resp)
    except StopIteration as done:
        return done.value


def evaluate(env, agent, num_episodes: int = 10, render: bool = False, exp_seed: int = 0) -> float:
    """Mean undiscounted return of the deterministic policy (tanh of the mean action)."""
    return drive(_evaluate_co(num_episodes, exp_seed), env, agent)


def train_with_experiment_name(env, agent, max_episodes: int = 500, target_reward: float = 0.0,
                               log_interval: int = 20, eval_interval: int = 50, steps_per_update: int = 2048,
                               experiment_name: str = "", exp_seed: int = 0, logger=None,
                               artifacts_dir: Optional[str] = None):
    """The reference's single-env training loop; returns (rewards, avg_rewards, metrics_history)."""
    co = training_coroutine(agent.memory, max_episodes, target_reward, log_interval, eval_interval, steps_per_update,
                            experiment_name, exp_seed, logger, artifacts_dir)
    return drive(co, env, agent)


def training_coroutine(memory, max_episodes: int = 500, target_reward: float = 0.0, log_interval: int = 20,
                       eval_interval: int = 50, steps_per_update: int = 2048, experiment_name: str = "",
                       exp_seed: int = 0, logger=None, artifacts_dir: Optional[str] = None):
    """``train_with_experiment_name`` (reference ``training/routine.py:61-297``) as a request coroutine.  ``memory`` is
    the agent's ``PPOMemory`` (host-side lists; stored into directly)."""
    logger = logger or logging.getLogger(f"experiment_{experiment_name}")
    tag = f"[{experiment_name}]" if experiment_name else ""
    logger.info(f"{tag} Starting training for experiment: {experiment_name}")
    rewards, episode_rewards, avg_rewards, training_episodes, eval_episodes = [], [], [], [], [0]
    best_avg = -float("inf")
    history: Dict[str, Any] = {
        "experiment_name": experiment_name, "episode_rewards": [], "eval_rewards": [], "avg_eval_rewards": [],
        "policy_updates": [], "episode_numbers": [], "eval_episode_numbers": [], "timestamps": [],
    }
    solved = False
    t0 = time.time()
    total_steps = episode_num = 0
    out_dir = ensure_artifacts_dir(artifacts_dir)
    ckpt_dir = os.path.join(out_dir, "checkpoints")
    os.makedirs(ckpt_dir, exist_ok=True)

    first = yield from _evaluate_co(5, exp_seed)
    rewards.append(first)
    avg_rewards.append(first)
    history["eval_rewards"].append(first)
    history["avg_eval_rewards"].append(first)
    history["eval_episode_numbers"].append(0)
    history["timestamps"].append(0)
    logger.info(f"{tag} initial_eval reward={first:.2f}")

    done, flat = True, None
    while episode_num < max_episodes:
        collected = 0
        update_t0 = time.time()
        while collected < steps_per_update and episode_num < max_episodes:
            episode_num += 1
            state = yield ("reset", exp_seed + episode_num)
            flat = state.reshape(-1)
            ep_reward, done = 0.0, False
            while not done and collected < steps_per_update:
                action, pre_tanh, log_prob, value = yield ("act", flat, False)
                nxt, reward, terminated, truncated = yield ("step", action)
                done = terminated or truncated  # truncation masks the bootstrap as well (SURVEY.md F8)
                flat_next = nxt.reshape(-1)
                memory.store(flat, action, pre_tanh, reward, flat_next, log_prob, done, value)
                flat = flat_next
                ep_reward += reward
                collected += 1
                total_steps += 1
            episode_rewards.append(ep_reward)
            training_episodes.append(episode_num)
            history["episode_rewards"].append(ep_reward)
            history["episode_numbers"].append(episode_num)
            if episode_num % log_interval == 0:
                logger.info("%s episode=%d reward=%.2f avg_reward=%.2f steps=%d time=%.2fs", tag, episode_num,
                            ep_reward, np.mean(episode_rewards[-log_interval:]), total_steps, time.time() - t0)
            if episode_num % eval_interval == 0:
                eval_reward = yield from _evaluate_co(5, exp_seed)
                rewards.append(eval_reward)
                eval_episodes.append(episode_num)
                elapsed = time.time() - t0
                avg_r = float(np.mean(rewards[-10:])) if len(rewards) >= 10 else float(np.mean(rewards))
                avg_rewards.append(avg_r)
                history["eval_rewards"].append(eval_reward)
                history["avg_eval_rewards"].append(avg_r)
                history["eval_episode_numbers"].append(episode_num)
                history["timestamps"].append(elapsed)
                logger.info("%s eval episode=%d reward=%.2f avg_reward=%.2f time=%.2fs", tag, episode_num,
                            eval_reward, avg_r, elapsed)
                if avg_r >= target_reward and not solved and len(rewards) >= 10:
                    yield ("save", os.path.join(ckpt_dir, f"ppo_highway_solved_{experiment_name}.pth"))
                    solved = True
                if avg_r > best_avg:
                    best_avg = avg_r
                    yield ("save", os.path.join(ckpt_dir, f"ppo_highway_best_{experiment_name}.pth"))
                    logger.info(f"{tag} New best model saved, avg reward={best_avg:.2f}")
        final_value = 0.0
        if not done:  # episode cut by the step budget: bootstrap from V(s_T)
            final_value = yield ("value", flat)
        update_metrics = yield ("update", final_value)
        history["policy_updates"].append({"episode": episode_num, "steps": collected,
                                          "time": time.time() - update_t0, **update_metrics})

    metrics_path = os.path.join(out_dir, f"training_metrics_{experiment_name}.json")
    with open(metrics_path, "w") as f:
        json.dump(history, f, indent=2)
    plot_name = f"ppo_highway_rewards_{experiment_name}.png"  # named for schema compatibility; not drawn
    csv_path = os.path.join(out_dir, f"summary_{experiment_name}.csv")
    with open(csv_path, "w") as f:
        f.write("experiment,final_reward,max_reward,steps,best_model,plot\n")
        best_model = os.path.join(ckpt_dir, f"ppo_highway_best_{experiment_name}.pth")
        f.write(f"{experiment_name},{avg_rewards[-1]:.4f},{max(avg_rewards):.4f},{total_steps},"
                f"{best_model},{plot_name}\n")
    logger.info(f"{tag} Metrics saved to {metrics_path}; summary CSV saved to {csv_path}")
    return rewards, avg_rewards, history


# --------------------------------------------------------------------------------------------
# batched loops
META_ACTIONS = 5   # DiscreteMetaAction: LANE_LEFT, IDLE, LANE_RIGHT, FASTER, SLOWER


def _act_widths(vec_env, agent):
    """(action, pre_tanh) floats per env of the agent's rollout on this env; ValueError when they do not fit."""
    ac = agent.actor_critic
    meta = getattr(getattr(vec_env, "cfg", None), "ego_mode", 0) == 1
    if getattr(ac, "discrete", False):
        if not meta:
            raise ValueError("a discrete (categorical) agent needs a DiscreteMetaAction env; this env takes "
                             "ContinuousAction")
        if ac.action_dim != META_ACTIONS:
            raise ValueError(f"the discrete agent has {ac.action_dim} actions; the DiscreteMetaAction env has "
                             f"{META_ACTIONS}")
    return ac.act_widths()


def collect_rollout(vec_env, agent, T: int, obs: Optional[torch.Tensor] = None,
                    noise: Optional[torch.Tensor] = None, use_graph: Optional[bool] = None,
                    bootstrap_truncated: bool = False) -> Dict[str, torch.Tensor]:
    """T lock-step policy steps of every env into ``agent.memory``'s device rollout.

    The env kernel writes each observation straight into the rollout's next state slot, reward and flags into their
    [t] slots, and the policy kernel writes action / log-prob / value straight into theirs: no staging copies, five
    kernels of this library per step.  Finished envs are respawned inside the step kernel (``autoreset``), so slot
    t+1 holds the first observation of the new episode and ``done[t]`` masks the bootstrap, exactly like the
    reference's reset-after-done loop (``routine.py:125-147``).

    With in-kernel sampling (``noise is None``) the whole rollout -- 5 T launches -- is captured ONCE as a CUDA graph
    (the sampling kernel's draw counter lives on the device) and replayed by later calls with the same env, agent and
    shape: the host-side cost of a rollout is one graph launch.  ``use_graph=False`` issues the launches one by one.

    A discrete agent on a ``DiscreteMetaAction`` env writes action [T, E, 2] = (id, 0), which the env step reads as it
    is, and pre_tanh [T, E, 1] = id.

    ``bootstrap_truncated=True`` handles time limits the standard way instead (not the reference's, which treats a
    truncation as a termination): the step also writes the observation each finished episode ended in into
    ``final_states[t]`` (``hrp_env_step_final``), the critic computes ``final_value[t]`` from it with the parameters
    that produced ``value[t]``, and ``agent.update`` bootstraps every truncated step with it.  Two more launches per
    step (the critic pass runs over all E rows; only the truncated ones are read), inside the captured graph.
    """
    A, Z = _act_widths(vec_env, agent)
    E, S = vec_env.num_envs, vec_env.N * vec_env.F_out
    ac = agent.actor_critic
    # exploration noise is keyed by the GLOBAL env id: a shard's rows start at its first global env
    ac.row_base = int(getattr(vec_env, "env_id_base", 0))
    if use_graph is None:
        # (a single env acts through the matrix-vector kernel, which keeps its draw counter on the host)
        use_graph = noise is None and E > 1 and getattr(agent, "use_cuda_graphs", True)
    cache = getattr(agent, "_rollout_graph", None)
    boot = bool(bootstrap_truncated)
    key = (getattr(vec_env, "uid", id(vec_env)), getattr(vec_env, "param_version", 0), T, E, S, A, Z,
           ac.workspace_generation, ac.row_base, boot)
    if use_graph and cache is not None and cache["key"] == key and agent.memory.rollout is None:
        agent.memory.rollout = cache["r"]     # the buffers the captured launches write (PPOAgent.update dropped them)
    r = agent.memory.begin_rollout(T, E, S, A, Z, bootstrap_truncated=boot)
    states = r["states"]
    if obs is None:
        vec_env.observe(out=states[0].view(E, vec_env.N, vec_env.F_out))
    else:
        states[0].copy_(obs.reshape(E, S))

    def steps(counter=None):
        for t in range(T):
            out = {"action": r["action"][t], "pre_tanh": r["pre_tanh"][t], "log_prob": r["log_prob"][t],
                   "value": r["value"][t]}
            if counter is None:
                agent.act(states[t], noise=None if noise is None else noise[t], out=out)
            else:
                agent.act(states[t], out=out, draw_counter=counter)
            vec_env.step(r["action"][t], out=states[t + 1].view(E, vec_env.N, vec_env.F_out), reward_out=r["reward"][t],
                         terminated_out=r["terminated"][t], truncated_out=r["truncated"][t],
                         final_obs_out=r["final_states"][t] if boot else None)
            if boot:
                ac.critic_into(r["final_states"][t], r["final_value"][t])
                agent.launches += 1
        torch.bitwise_or(r["terminated"], r["truncated"], out=r["done"])

    if not use_graph or noise is not None:
        steps()
        return r
    if cache is None or cache["key"] != key or cache["r"] is not r:
        if cache is None or cache["key"] != key:
            steps()                     # the first rollout of a shape runs eagerly (warms every kernel variant) ...
            agent._rollout_graph = {"key": key, "r": r, "graph": None, "counter": ac.new_draw_counter(),
                                    "expected": ac._draw}
            return r
        cache["r"], cache["graph"] = r, None
    cache = agent._rollout_graph
    if cache["expected"] != ac._draw:   # other act() calls advanced the host-side draw counter since the last replay
        cache["counter"].copy_(torch.tensor([ac._draw, 0], dtype=torch.int64))
    if cache["graph"] is None:          # ... the second one is captured
        graph = torch.cuda.CUDAGraph()
        cur = torch.cuda.current_stream(agent.device)
        side = torch.cuda.Stream(agent.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            graph.capture_begin()
            try:
                steps(cache["counter"])
            finally:
                graph.capture_end()
        cur.wait_stream(side)
        cache["graph"] = graph
    cache["graph"].replay()
    ac._draw += T
    cache["expected"] = ac._draw
    agent.launches += 2 * T if boot else T
    vec_env.launches += T
    return r


def rollout_and_update(vec_env, agent, T: int, obs: Optional[torch.Tensor] = None, bootstrap_truncated: bool = False):
    """One PPO iteration: T x E samples collected, then ``agent.update`` bootstrapped from V(s_T).
    ``bootstrap_truncated``: see ``collect_rollout``.
    Returns (update metrics, the observation the next rollout starts from)."""
    r = collect_rollout(vec_env, agent, T, obs, bootstrap_truncated=bootstrap_truncated)
    last_obs = r["states"][T].clone()
    _, _, last_v = agent.actor_critic.forward(last_obs)
    return agent.update(last_value=last_v.view(-1)), last_obs


def evaluate_vectorized(eval_env, agent, exp_seed: int = 0, use_graph: Optional[bool] = None) -> Dict[str, Any]:
    """One deterministic episode per env of ``eval_env``, all at once: the batched counterpart of ``evaluate``.

    Env e plays the reference's evaluation episode with seed ``exp_seed + 1000 + env_id_base + e`` (per-env seeds and a
    full reset: bit for bit the episode ``evaluate(env, agent, K, exp_seed)`` starts on a single-env handle), so shards
    with consecutive ``env_id_base`` play the episode set of one process.  Gaussian agents act with tanh(mean),
    categorical ones with the argmax.  Each of the ``policy_steps`` steps after which highway-v0 truncates is an act, a
    step masked by the envs still running and one ``hrp_episode_stats`` launch that freezes the envs whose episode
    ended, so per-episode returns and lengths stay on the device and the host synchronises once.  The whole evaluation
    is captured as one CUDA graph by the second call and replayed by later calls with the same env, agent workspace
    and seeds (the first call runs launch by launch; ``use_graph=False`` always does).

    ``eval_env`` becomes an evaluation handle: this installs its per-env seeds and step mask.  In shuffled row order
    the shuffle draws continue from one evaluation to the next, as they do on a single-env handle.

    Returns mean / std (population) / min / max of the returns, length_mean, terminated_fraction, episodes, and the
    per-episode ``returns`` (float64) and ``lengths`` (int32) as numpy arrays.  Under ``torch.distributed`` the six
    sums are all-reduced, so episodes, mean, std, length_mean and terminated_fraction are global; min, max and the
    arrays are this rank's."""
    _act_widths(eval_env, agent)
    ac = agent.actor_critic
    K, S, dev = eval_env.num_envs, eval_env.N * eval_env.F_out, eval_env.device
    steps = policy_steps(eval_env.config["duration"], eval_env.config["policy_frequency"])
    buf = getattr(eval_env, "_eval_buffers", None)
    if buf is None or buf["exp_seed"] != int(exp_seed):
        base = int(exp_seed) + 1000 + int(eval_env.env_id_base)
        buf = {"exp_seed": int(exp_seed),
               "seeds": torch.arange(base, base + K, dtype=torch.int64, device=dev),
               "active": torch.zeros(K, dtype=torch.uint8, device=dev),
               "ret": torch.zeros(K, dtype=torch.float64, device=dev),
               "len": torch.zeros(K, dtype=torch.int32, device=dev),
               "stats": new_stats(dev),
               "obs": torch.empty((2, K, eval_env.N, eval_env.F_out), dtype=torch.float32, device=dev),
               "reward": torch.empty(K, dtype=torch.float32, device=dev),
               "terminated": torch.empty(K, dtype=torch.uint8, device=dev),
               "truncated": torch.empty(K, dtype=torch.uint8, device=dev)}
        eval_env.set_env_seeds(buf["seeds"])
        eval_env.set_step_mask(buf["active"])
        eval_env._eval_buffers = buf
    # policy outputs per (action, pre_tanh) width, kept as long as the buffers: captured launches write them
    widths = ("act",) + tuple(ac.act_widths())
    if widths not in buf:
        buf[widths] = ac._new_act_out(K)
    act = buf[widths]

    def run():
        buf["active"].fill_(1)
        buf["ret"].zero_()
        buf["len"].zero_()
        buf["stats"].zero_()
        eval_env.reset(out=buf["obs"][0])   # every env: the mask steers steps only
        for t in range(steps):
            agent.act(buf["obs"][t % 2].view(K, S), deterministic=True, out=act)
            eval_env.step(act["action"], out=buf["obs"][(t + 1) % 2], reward_out=buf["reward"],
                          terminated_out=buf["terminated"], truncated_out=buf["truncated"])
            episode_stats(buf["reward"], buf["terminated"], buf["truncated"], buf["ret"], buf["len"], buf["stats"],
                          active=buf["active"])

    if use_graph is None:
        # (a single env acts through the matrix-vector kernel, which allocates its output row)
        use_graph = K > 1 and getattr(agent, "use_cuda_graphs", True)
    ac._ensure_workspace(K)
    key = (eval_env.uid, eval_env.param_version, ac.workspace_generation, id(buf), K, steps)
    cache = getattr(agent, "_eval_graph", None)
    if not use_graph or cache is None or cache["key"] != key:
        run()                           # the first evaluation of a configuration runs eagerly ...
        if use_graph:
            agent._eval_graph = {"key": key, "graph": None}
    else:
        if cache["graph"] is None:      # ... the second one is captured
            graph = torch.cuda.CUDAGraph()
            cur = torch.cuda.current_stream(dev)
            side = torch.cuda.Stream(dev)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                graph.capture_begin()
                try:
                    run()
                finally:
                    graph.capture_end()
            cur.wait_stream(side)
            cache["graph"] = graph
        cache["graph"].replay()
        agent.launches += steps
        eval_env.launches += 1 + steps
    sums = buf["stats"][:6]
    if distributed.world_size() > 1:
        distributed.allreduce_sum_(sums)
    host = torch.cat([sums, buf["ret"], buf["len"].double()]).cpu().numpy()   # the evaluation's one synchronisation
    returns, lengths = host[6:6 + K].copy(), host[6 + K:].astype(np.int32)
    s = summarize(host[:6])
    if s["episodes"] != K * distributed.world_size():
        raise RuntimeError(f"evaluate_vectorized: {s['episodes']} episodes finished within {steps} steps, expected "
                           f"{K * distributed.world_size()}")
    return {"mean": s["return_mean"], "std": s["return_std"], "min": float(returns.min()), "max": float(returns.max()),
            "length_mean": s["length_mean"], "terminated_fraction": s["terminated_fraction"],
            "episodes": s["episodes"], "returns": returns, "lengths": lengths}


def eval_env_for(vec_env, num_envs: int):
    """An evaluation handle of ``num_envs`` envs with ``vec_env``'s resolved config and its ``EmbedSpec`` (the same table
    object: a RankPE evaluation sees the training table, not a new draw), no autoreset.  Its ``env_id_base`` is the
    shard index of ``vec_env`` times ``num_envs``, so that W shards evaluate the episodes one process of W x
    ``num_envs`` envs would."""
    from ..envs.highway_vec import HighwayVecEnv

    shard = int(vec_env.env_id_base) // int(vec_env.num_envs)
    return HighwayVecEnv(vec_env.config, num_envs, device=vec_env.device, embed=vec_env.embed, autoreset=False,
                         env_id_base=shard * int(num_envs), real64=vec_env.real64)


def linear_lr(lr0: float, it: int, iterations: int) -> float:
    """CleanRL's linear annealing (``anneal_lr``): the learning rate of iteration ``it`` (0-based) of ``iterations``,
    lr0 * (1 - it / iterations), from lr0 at the first iteration down to lr0 / iterations at the last."""
    return float(lr0) * (1.0 - it / iterations)


def train_vectorized(vec_env, agent, iterations: int, T: int, seed: int = 0, logger=None,
                     bootstrap_truncated: bool = False, eval_episodes: int = 0, eval_interval: int = 10,
                     best_checkpoint: Optional[str] = None, anneal_lr: bool = False):
    """``iterations`` PPO iterations on E lock-step envs; returns the list of update metrics with samples/s and the
    training episodes added.  ``bootstrap_truncated``: see ``collect_rollout``.

    Training episodes: after each rollout one ``hrp_episode_stats`` launch over its rewards and flags, with per-env
    return / length carries zeroed by the reset here, so an episode spanning two rollouts counts once, in the
    iteration it ends in.  ``episodes``, ``episode_return_mean``, ``episode_return_std`` (population),
    ``episode_length_mean`` and ``terminated_fraction`` are those of the episodes that ended during the iteration (NaN
    when none did); under ``torch.distributed`` the six sums are all-reduced, so every rank reports global figures.

    ``eval_episodes`` > 0: before iterations 0, ``eval_interval``, 2 ``eval_interval``, ... the policy is evaluated on
    that many deterministic episodes per rank (``evaluate_vectorized`` on a handle of its own, ``eval_env_for``; seeds
    ``seed + 1000 + global env id``, the reference's evaluation seeds with ``seed`` as the experiment seed), recorded
    as ``eval_return_mean`` / ``eval_return_std`` / ``eval_length_mean`` / ``eval_terminated_fraction`` in that
    iteration's metrics.  ``best_checkpoint``: path that ``agent.save`` (rank 0) writes whenever the evaluation mean
    beats the best so far.

    ``anneal_lr``: iteration ``it`` runs with ``linear_lr(lr0, it, iterations)``, lr0 being the agent's learning rate at
    entry, set through ``agent.set_lr`` (the learning rate lives in device memory, so the captured minibatch graphs are
    replayed, not captured again).  Every iteration's metrics hold the ``lr`` its update ran with."""
    logger = logger or logging.getLogger(__name__)
    _act_widths(vec_env, agent)
    if eval_episodes and eval_interval < 1:
        raise ValueError(f"eval_interval must be >= 1, got {eval_interval}")
    obs = vec_env.reset(seed=seed)
    E, dev = vec_env.num_envs, vec_env.device
    carry_ret = torch.zeros(E, dtype=torch.float64, device=dev)
    carry_len = torch.zeros(E, dtype=torch.int32, device=dev)
    stats = new_stats(dev)
    eval_env = eval_env_for(vec_env, eval_episodes) if eval_episodes else None
    best = -float("inf")
    history = []
    lr0 = agent.optimizer.lr
    try:
        for it in range(iterations):
            if anneal_lr:
                agent.set_lr(linear_lr(lr0, it, iterations))
            ev = None
            if eval_env is not None and it % eval_interval == 0:
                ev = evaluate_vectorized(eval_env, agent, exp_seed=seed)
                if ev["mean"] > best:
                    best = ev["mean"]
                    if best_checkpoint is not None and distributed.rank() == 0:
                        agent.save(best_checkpoint)
            t0 = time.time()
            r = collect_rollout(vec_env, agent, T, obs, bootstrap_truncated=bootstrap_truncated)
            stats[:6].zero_()
            episode_stats(r["reward"], r["terminated"], r["truncated"], carry_ret, carry_len, stats)
            obs = r["states"][T].clone()
            _, _, last_v = agent.actor_critic.forward(obs)
            metrics = agent.update(last_value=last_v.view(-1))
            if distributed.world_size() > 1:
                distributed.allreduce_sum_(stats[:6])
            torch.cuda.synchronize(dev)
            dt = time.time() - t0
            metrics["samples_per_s"] = T * E / dt
            metrics["lr"] = agent.optimizer.lr
            s = summarize(stats[:6].tolist())
            metrics.update(episodes=s["episodes"], episode_return_mean=s["return_mean"],
                           episode_return_std=s["return_std"], episode_length_mean=s["length_mean"],
                           terminated_fraction=s["terminated_fraction"])
            if ev is not None:
                metrics.update(eval_return_mean=ev["mean"], eval_return_std=ev["std"],
                               eval_length_mean=ev["length_mean"], eval_terminated_fraction=ev["terminated_fraction"])
            history.append(metrics)
            logger.info("iter=%d loss=%.4f samples/s=%.0f episodes=%d return=%.3f%s", it, metrics["loss"],
                        metrics["samples_per_s"], s["episodes"], s["return_mean"],
                        "" if ev is None else f" eval_return={ev['mean']:.3f}")
    finally:
        if eval_env is not None:
            eval_env.close()
    return history
