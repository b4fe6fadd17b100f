"""R experiments of the sweep on ONE GPU at the same time (SURVEY.md 8f-2).

The reference runs its 540-run sweep as processes that time-share a GPU: ``utils/device_pool.py:45-72`` hands
``OVERSUB`` workers the same device and ``main.py:234-242`` fans the experiments out with joblib; every run then
drives its own single env and its own agent, one synchronous kernel chain per env step.  Here the experiments that
share an env configuration share ONE simulator handle -- experiment r is env r of it, with its own seed
(``hrp_env_set_seeds``) and a per-launch step mask (``hrp_env_set_step_mask``) because the runs are not in lock step
(one is evaluating, one is inside its PPO update, one has finished) -- so a tick of the whole set is one env launch,
one device-to-host copy and one host synchronisation; the R policies act in ONE launch (``hrp_ppo_act_multi``: a
cluster of CTAs per policy, matrix-vector products), and every PPO update is enqueued on its experiment's own stream without a host synchronisation
(``PPOAgent.update_begin``), so the updates of different experiments overlap with each other and with the stepping of
the rest.

Every experiment still executes the reference's loop -- the SAME coroutine ``train_with_experiment_name`` drives
(``training/routine.py``) -- with the same kernels on the same inputs and its own random streams, so a multiplexed
run is bit for bit the sequential ``ExperimentRunner.launch`` of that experiment (``tests/test_api_gpu.py``).
"""
from __future__ import annotations

import logging
import random
import time
import traceback
from typing import Any, Dict, List, Optional

import numpy as np
import torch

from .. import _lib
from ..envs.highway_vec import HighwayVecEnv
from ..training.routine import training_coroutine
from ..utils.reproducibility import set_random_seeds
from .config import Experiment
from .runner import ExperimentRunner
from .wrappers import _resolve, embed_spec_for

_MASK64 = 0xFFFFFFFFFFFFFFFF


def _rng_get():
    return random.getstate(), np.random.get_state(), torch.get_rng_state()


def _rng_set(state) -> None:
    random.setstate(state[0])
    np.random.set_state(state[1])
    torch.set_rng_state(state[2])


class _Group:
    """The experiments that share one simulator handle (same env configuration and embedding table)."""

    def __init__(self, cfg: Dict[str, Any], spec, device: torch.device):
        self.cfg, self.spec, self.device = cfg, spec, device
        self.slots: List["_Slot"] = []
        self.env: Optional[HighwayVecEnv] = None

    def build(self) -> None:
        R, d = len(self.slots), self.device
        self.env = env = HighwayVecEnv(self.cfg, R, device=d, embed=self.spec, autoreset=False)
        pin = lambda *shape, dtype=torch.float32: torch.zeros(shape, dtype=dtype).pin_memory()
        self.seeds_host, self.seeds = pin(R, dtype=torch.int64), torch.zeros(R, dtype=torch.int64, device=d)
        self.mask_host, self.mask = pin(R, dtype=torch.uint8), torch.zeros(R, dtype=torch.uint8, device=d)
        self.reset_mask = torch.zeros(R, dtype=torch.uint8, device=d)
        self.obs_host = pin(R, *env.obs_shape)   # (N, F_out), or (F, W, H) for an OccupancyGrid: what the single env returns
        A = 2
        # per experiment: action | pre_tanh | log_prob | value, written by its policy kernels, read back in one copy
        self.res, self.res_host = torch.zeros((R, 2 * A + 2), device=d), pin(R, 2 * A + 2)
        self.act_host, self.act = pin(R, 2), torch.zeros((R, 2), device=d)
        self.reward_host, self.term_host, self.trunc_host = pin(R), pin(R, dtype=torch.uint8), pin(R, dtype=torch.uint8)
        # numpy views of the pinned staging buffers (element writes through torch indexing cost microseconds each)
        self.seeds_np, self.mask_np, self.act_np = self.seeds_host.numpy(), self.mask_host.numpy(), self.act_host.numpy()
        self.obs_np, self.res_np = self.obs_host.numpy(), self.res_host.numpy()
        self.reward_np, self.term_np, self.trunc_np = self.reward_host.numpy(), self.term_host.numpy(), self.trunc_host.numpy()
        env.set_env_seeds(self.seeds)
        env.set_step_mask(self.mask)

    def close(self) -> None:
        if self.env is not None:
            self.env.close()
            self.env = None


class _Slot:
    def __init__(self, exp: Experiment):
        self.exp = exp
        self.result: Dict[str, Any] = {"experiment_name": exp.name, "status": "FAILED"}
        self.t0 = time.time()
        self.logger = logging.getLogger(f"experiment_{exp.name}")
        self.agent = None
        self.group: Optional[_Group] = None
        self.e = -1
        self.co = None
        self.req = None
        self.rng = None
        self.stream: Optional[torch.cuda.Stream] = None
        self.pending_update = None
        self.live = False
        self.obs_row = self.res_row = None   # device views: this experiment's observation row / policy result row

    def fail(self, err: BaseException) -> None:
        self.logger.error(f"[{self.exp.name}] Experiment execution failed!", exc_info=True)
        self.result["error_message"] = str(err)
        self.result["error_traceback"] = traceback.format_exc()
        self.finish()

    def finish(self) -> None:
        self.live = False
        self.result["duration_seconds"] = time.time() - self.t0


class MultiplexedRunner(ExperimentRunner):
    """``launch_many(experiments)`` = ``[launch(e) for e in experiments]`` with the experiments advancing together.

    ``max_concurrent`` bounds R (each experiment holds its network, Adam state, CUDA graphs and a rollout);
    experiments beyond it start as earlier ones finish."""

    def __init__(self, base_env_config: dict, device_pool: Optional[Any] = None, artifacts_dir: Optional[str] = None,
                 max_concurrent: int = 16):
        super().__init__(base_env_config, device_pool, artifacts_dir)
        self.max_concurrent = int(max_concurrent)
        self.ticks = 0          # host synchronisation rounds of the last launch_many
        self.env_launches = 0   # simulator kernels of the last launch_many (one per group per tick and kind)
        self.env_requests = 0   # env.reset / env.step calls of the experiments those launches answered
        self._lib = _lib.load()

    # ------------------------------------------------------------------ set-up of one experiment
    def _prepare(self, slot: _Slot, device: torch.device, groups: Dict[Any, _Group]) -> None:
        exp = slot.exp
        set_random_seeds(exp.seed)
        slot.logger.info(f"[{exp.name}] device {device} | seed {exp.seed} | condition {exp.condition.name}")
        # the same calls, in the same order, as make_env + the wrapper constructors (the RankPE table draws from the
        # torch generator before the network does)
        cfg = _resolve(exp.condition, self.base_config, exp.hp.d_embed, exp.env_config_overrides)
        spec = embed_spec_for(exp.condition, cfg, exp.hp.d_embed)
        probe = HighwayVecEnv(cfg, 1, device=device, embed=spec, autoreset=False)   # validates the configuration
        try:
            if probe.cfg.ego_mode != 0:
                raise TypeError("Unsupported action space: the PPO agent needs the continuous (Box) action")
            state_dim, key_cfg = probe.N * probe.F_out, bytes(probe.cfg)
        finally:
            probe.close()
        slot.agent = self._create_agent(state_dim, 2, exp.hp, slot.logger, device)
        key = (key_cfg, None if spec.table is None else spec.table.tobytes())
        group = groups.get(key)
        if group is None:
            group = groups[key] = _Group(cfg, spec, device)
        slot.group, slot.e = group, len(group.slots)
        group.slots.append(slot)
        slot.co = training_coroutine(
            slot.agent.memory, max_episodes=exp.max_episodes, target_reward=exp.target_reward,
            log_interval=exp.extra.get("log_interval", 20), eval_interval=exp.extra.get("eval_interval", 50),
            steps_per_update=exp.hp.steps_per_update, experiment_name=exp.name, exp_seed=exp.seed, logger=slot.logger,
            artifacts_dir=self.artifacts_dir)
        slot.rng = _rng_get()
        slot.stream = torch.cuda.Stream(device)
        slot.live = True

    def _advance(self, slot: _Slot, resp, first: bool = False) -> None:
        """Hand a response to the experiment's loop and fetch its next request."""
        try:
            slot.req = next(slot.co) if first else slot.co.send(resp)
        except StopIteration as done:
            rewards, avg_rewards, metrics = done.value
            slot.result.update(status="COMPLETED", rewards=rewards, avg_rewards=avg_rewards, metrics_history=metrics)
            slot.req = None
            slot.finish()
        except Exception as err:  # the reference reports, it does not raise (runner.py:133-146)
            slot.req = None
            slot.fail(err)

    # ------------------------------------------------------------------ the multiplexed loop
    def launch_many(self, experiments: List[Experiment]) -> List[Dict[str, Any]]:
        results: List[Dict[str, Any]] = []
        self.ticks = self.env_launches = self.env_requests = 0
        with self._device() as device:
            device = torch.device(device)
            for lo in range(0, len(experiments), self.max_concurrent):
                results += self._run_wave(experiments[lo:lo + self.max_concurrent], device)
        return results

    def _run_wave(self, experiments: List[Experiment], device: torch.device) -> List[Dict[str, Any]]:
        slots = [_Slot(exp) for exp in experiments]
        groups: Dict[Any, _Group] = {}
        outer_rng = _rng_get()
        try:
            for slot in slots:
                try:
                    self._prepare(slot, device, groups)
                except Exception as err:
                    slot.fail(err)
            for g in groups.values():
                if not g.slots:   # (the only experiment of this configuration failed while it was being set up)
                    continue
                g.build()
                for s in g.slots:   # the policy of experiment e reads row e of the observation, writes row e of the results
                    row, A = g.res[s.e], 2
                    s.obs_row = g.env.obs[s.e].view(1, -1)
                    s.res_row = row
            for slot in slots:
                if slot.live:
                    self._advance(slot, None, first=True)
            while any(s.live for s in slots):
                self._tick(slots, list(groups.values()), device)
        finally:
            torch.cuda.synchronize(device)
            for g in groups.values():
                g.close()
            _rng_set(outer_rng)
        return [s.result for s in slots]

    def _tick(self, slots: List[_Slot], groups: List[_Group], device: torch.device) -> None:
        self.ticks += 1
        main = torch.cuda.current_stream(device)
        ready = False
        for s in slots:
            if s.live and s.pending_update is not None and s.pending_update.query():
                metrics = s.agent.update_end(s.pending_update)
                s.pending_update = None
                self._advance(s, metrics)
            ready |= s.live and s.pending_update is None
        if not ready:   # every live experiment is inside its update: wait for the first one
            waiting = [s for s in slots if s.live and s.pending_update is not None]
            if waiting:
                waiting[0].pending_update.synchronize()
            return

        def asking(kind: str) -> List[_Slot]:
            # evaluated phase by phase: an experiment answered in one phase may ask for the next one in the same tick
            # (reset -> act -> step is ONE tick)
            return [s for s in slots if s.live and s.pending_update is None and s.req[0] == kind]

        # -- rare requests, answered one by one exactly as training/routine.py:drive does
        for s in asking("save"):
            self._guard(s, lambda s=s: s.agent.save(s.req[1]))
        for s in asking("value"):
            def value(s=s):
                _, _, v = s.agent.actor_critic.forward(s.req[1])
                return float(v.cpu().item())
            self._guard(s, value)
        for s in asking("update"):
            def begin(s=s):
                _rng_set(s.rng)   # the minibatch permutation comes from this experiment's numpy stream
                torch.cuda.set_stream(s.stream)   # (not the stream context: its enter / exit each query the device count)
                try:
                    s.pending_update = s.agent.update_begin(last_value=s.req[1])
                finally:
                    torch.cuda.set_stream(main)
                s.rng = _rng_get()
                return _PENDING
            self._guard(s, begin)

        # -- reset: seeds + mask per group, one launch per group
        resets = asking("reset")
        touched = []
        for g in groups:
            mine = [s for s in resets if s.group is g]
            if not mine:
                continue
            g.mask_np[:] = 0
            for s in mine:
                g.seeds_np[s.e] = _as_i64(int(s.req[1]) & _MASK64)
                g.mask_np[s.e] = 1
            g.seeds.copy_(g.seeds_host, non_blocking=True)
            g.reset_mask.copy_(g.mask_host, non_blocking=True)
            g.env.reset(mask=g.reset_mask)
            g.obs_host.copy_(g.env.obs, non_blocking=True)
            self.env_launches += 1
            self.env_requests += len(mine)
            touched.append((g, mine))
        if touched:
            main.synchronize()
            for g, mine in touched:
                for s in mine:
                    self._advance(s, g.obs_np[s.e].copy())

        # -- act: every policy reads its env's row of the device observation (the very bytes the loop holds on the
        #    host) and writes into its row of the group's result buffer: ONE launch for all of them
        #    (hrp_ppo_act_multi: a cluster of CTAs per policy), one copy per group, one synchronisation
        acts = asking("act")
        if acts:
            items = (_lib.HrpActItem * len(acts))()
            n = 0
            for s in acts:
                try:
                    s.agent.launches += 1
                    items[n] = s.agent.actor_critic.act_item(s.obs_row, s.res_row, bool(s.req[2]))
                    n += 1
                except Exception as err:
                    s.fail(err)
            try:
                _lib.check(self._lib.hrp_ppo_act_multi(items, n, main.cuda_stream), "hrp_ppo_act_multi")
            except Exception as err:
                for s in acts:
                    if s.live:
                        s.fail(err)
            for g in {s.group for s in acts}:
                g.res_host.copy_(g.res, non_blocking=True)
            main.synchronize()
            for s in acts:
                if not s.live:
                    continue
                host, A = s.group.res_np[s.e], 2
                det = bool(s.req[2])
                self._advance(s, (host[0:A].copy(), host[A:2 * A].copy(), None if det else float(host[2 * A]),
                                  np.float32(host[2 * A + 1])))

        # -- step: one masked launch per group
        steps = asking("step")
        touched = []
        for g in groups:
            mine = [s for s in steps if s.group is g]
            if not mine:
                continue
            g.mask_np[:] = 0
            for s in mine:
                a = np.asarray(s.req[1], dtype=np.float32).reshape(-1)
                if a.size != 2:
                    s.fail(ValueError(f"action must have shape (2,), got {np.shape(s.req[1])}"))
                    continue
                g.act_np[s.e] = a
                g.mask_np[s.e] = 1
            g.act.copy_(g.act_host, non_blocking=True)
            g.mask.copy_(g.mask_host, non_blocking=True)
            env = g.env
            env.step(g.act)
            g.obs_host.copy_(env.obs, non_blocking=True)
            g.reward_host.copy_(env.reward, non_blocking=True)
            g.term_host.copy_(env.terminated, non_blocking=True)
            g.trunc_host.copy_(env.truncated, non_blocking=True)
            self.env_launches += 1
            self.env_requests += len(mine)
            touched.append((g, mine))
        if touched:
            main.synchronize()
            for g, mine in touched:
                for s in mine:
                    if s.live:
                        self._advance(s, (g.obs_np[s.e].copy(), float(g.reward_np[s.e]), bool(g.term_np[s.e]),
                                          bool(g.trunc_np[s.e])))

    def _guard(self, slot: _Slot, fn) -> None:
        try:
            resp = fn()
        except Exception as err:
            slot.req = None
            slot.fail(err)
            return
        if resp is not _PENDING:
            self._advance(slot, resp)


_PENDING = object()


def _as_i64(u: int) -> int:
    return u - (1 << 64) if u >= (1 << 63) else u
