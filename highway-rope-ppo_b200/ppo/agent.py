"""PPO agent on the C-ABI kernels (reference: ``ppo/agent.py:12-327``).

Same classes, constructor arguments, method names, return types, metrics keys and checkpoint
format as the reference; the arithmetic runs in ``libhrp_b200.so``:

* ``ActorCritic`` keeps every parameter in ONE flat fp32 device buffer laid out in
  ``ActorCritic.parameters()`` order (``log_std``, ``shared.0.*``, ``shared.2.*``,
  ``actor_mean.0.*``, ``actor_mean.2.*``, ``critic.0.*``, ``critic.2.*``); the per-layer tensors
  of ``state_dict()`` are views into it, so gradients, Adam moments and the multi-GPU all-reduce
  all touch one contiguous range.
* ``discrete=True`` (keyword-only, beside the reference's signature) selects the categorical policy for the
  ``DiscreteMetaAction`` ego: a softmax over ``action_dim`` = n logits on the same trunk and critic, the same layout
  without ``log_std`` (``hrp_ppo_create_ex`` with ``HRP_PPO_CATEGORICAL``).
* ``PPOMemory`` keeps the list-based ``store`` API of the reference loop and adds a device-resident
  [T, E] rollout for the vectorised loop.
* ``PPOAgent.update`` = GAE kernel -> advantage normalisation -> for every epoch and minibatch:
  fused evaluate + loss + backward (``hrp_ppo_loss_grad``), optional NCCL all-reduce of the flat
  gradient, fused clip-grad-norm + Adam (``hrp_clip_adam_step``).  Metrics are accumulated on the
  device and read back once per update (the reference syncs five times per minibatch,
  ``agent.py:230,257-262``).
"""
from __future__ import annotations

import math
import os

import ctypes as C
import logging
from collections import OrderedDict
from typing import Any, Dict, List, Optional

import numpy as np
import torch
import torch.nn as nn

from .. import _lib
from . import distributed

_PARAM_ORDER = ("log_std", "shared.0.weight", "shared.0.bias", "shared.2.weight", "shared.2.bias",
                "actor_mean.0.weight", "actor_mean.0.bias", "actor_mean.2.weight", "actor_mean.2.bias",
                "critic.0.weight", "critic.0.bias", "critic.2.weight", "critic.2.bias")


def _param_shapes(S: int, A: int, H: int, discrete: bool = False) -> "OrderedDict[str, tuple]":
    return OrderedDict(([] if discrete else [("log_std", (A,))]) + [
        ("shared.0.weight", (H, S)), ("shared.0.bias", (H,)),
        ("shared.2.weight", (H, H)), ("shared.2.bias", (H,)),
        ("actor_mean.0.weight", (H, H)), ("actor_mean.0.bias", (H,)),
        ("actor_mean.2.weight", (A, H)), ("actor_mean.2.bias", (A,)),
        ("critic.0.weight", (H, H)), ("critic.0.bias", (H,)),
        ("critic.2.weight", (1, H)), ("critic.2.bias", (1,)),
    ])


def _cuda_device(device) -> torch.device:
    device = torch.device(device)
    if device.type != "cuda":
        raise _lib.HrpError(f"device {device} is not a CUDA device: highway-rope-ppo_b200 has no CPU path")
    idx = device.index if device.index is not None else torch.cuda.current_device()
    return torch.device("cuda", idx)


class ActorCritic:
    """Shared 2x(Linear+ReLU) trunk, actor head -> mean, state-independent ``log_std``, critic head.

    Weight initialisation builds the reference's ``nn.Linear`` stack on the CPU in the reference's
    construction order (``agent.py:22-42``), so a seeded run starts from the same parameters.

    ``discrete=True``: a categorical policy over ``action_dim`` actions (2..8).  ``actor_mean.2`` gives the logits,
    there is no ``log_std``; ``forward`` returns ``(logits, None, value)``.
    """

    def __init__(self, state_dim: int, action_dim: int, hidden_dim: int = 128,
                 device: Any = "cuda", max_batch: int = 4096, *, discrete: bool = False):
        self._lib = _lib.load()
        _lib.require_device()
        self.device = _cuda_device(device)
        self.state_dim, self.action_dim, self.hidden_dim = int(state_dim), int(action_dim), int(hidden_dim)
        self.discrete = bool(discrete)
        self._flags = _lib.PPO_CATEGORICAL if self.discrete else 0
        S, A, H = self.state_dim, self.action_dim, self.hidden_dim
        shared = nn.Sequential(nn.Linear(S, H), nn.ReLU(), nn.Linear(H, H), nn.ReLU())
        actor_mean = nn.Sequential(nn.Linear(H, H), nn.ReLU(), nn.Linear(H, A))
        log_std = torch.zeros(A)
        critic = nn.Sequential(nn.Linear(H, H), nn.ReLU(), nn.Linear(H, 1))
        init = {"log_std": log_std}
        for prefix, seq in (("shared", shared), ("actor_mean", actor_mean), ("critic", critic)):
            for k, v in seq.state_dict().items():
                init[f"{prefix}.{k}"] = v
        self.shapes = _param_shapes(S, A, H, self.discrete)
        self.num_params = int(self._lib.hrp_ppo_param_count_ex(S, A, H, self._flags))
        assert self.num_params == sum(int(np.prod(s)) for s in self.shapes.values())
        self.flat = torch.empty(self.num_params, dtype=torch.float32, device=self.device)
        self._views: "OrderedDict[str, torch.Tensor]" = OrderedDict()
        off = 0
        for name, shape in self.shapes.items():
            n = int(np.prod(shape))
            view = self.flat[off:off + n].view(shape)
            view.copy_(init[name].detach().to(torch.float32))
            self._views[name] = view
            off += n
        self._h = C.c_void_p()
        self._head_scratch: Optional[torch.Tensor] = None   # policy-head output of critic_into
        self.max_batch = 0
        self.workspace_generation = 0   # bumped whenever the native workspace is re-created (CUDA-graph cache key)
        self._ensure_workspace(max_batch)
        self._noise_seed = int(torch.randint(0, 2**62, (1,)).item())
        self._draw = 0
        # global index of row 0 of the batches this instance acts on (a shard's first global env id): the
        # exploration noise is keyed by (seed, global row, draw), so shards draw different noise and a sharded
        # rollout reproduces the single-process one
        self.row_base = 0

    def _ensure_workspace(self, batch: int) -> None:
        if batch <= self.max_batch:
            return
        if self._h:
            torch.cuda.synchronize(self.device)
            self._lib.hrp_ppo_destroy(self._h)
            self._h = C.c_void_p()
        _lib.check(self._lib.hrp_ppo_create_ex(self.state_dim, self.action_dim, self.hidden_dim, int(batch),
                                               self.device.index, self._flags, C.byref(self._h)), "hrp_ppo_create_ex")
        self.max_batch = int(batch)
        self.workspace_generation += 1

    def __del__(self):  # pragma: no cover
        try:
            if self._h:
                self._lib.hrp_ppo_destroy(self._h)
                self._h = None
            for hp, _ in self.__dict__.get("_lanes", {}).values():
                self._lib.hrp_ppo_destroy(hp)
        except Exception:
            pass

    # -- nn.Module-like surface ----------------------------------------------------------------
    def parameters(self) -> List[torch.Tensor]:
        return list(self._views.values())

    def named_parameters(self):
        return list(self._views.items())

    def state_dict(self) -> "OrderedDict[str, torch.Tensor]":
        return OrderedDict((k, v.detach().clone()) for k, v in self._views.items())

    def load_state_dict(self, sd: Dict[str, torch.Tensor], strict: bool = True):
        missing = [k for k in self._views if k not in sd]
        unexpected = [k for k in sd if k not in self._views]
        if strict and (missing or unexpected):
            raise RuntimeError(f"Error(s) in loading state_dict for ActorCritic: missing {missing}, "
                               f"unexpected {unexpected}")
        for k, v in self._views.items():
            if k in sd:
                if tuple(sd[k].shape) != tuple(v.shape):
                    raise RuntimeError(f"size mismatch for {k}: {tuple(sd[k].shape)} vs {tuple(v.shape)}")
                v.copy_(sd[k].to(device=self.device, dtype=torch.float32))

    @property
    def log_std(self) -> torch.Tensor:
        return self._views["log_std"]

    def to(self, device):
        return self

    def eval(self):
        return self

    def train(self, mode: bool = True):
        return self

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _as_states(self, x) -> torch.Tensor:
        if torch.is_tensor(x) and x.dtype == torch.float32 and x.device == self.device and x.is_contiguous():
            return x
        if isinstance(x, np.ndarray):
            x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
        x = x.to(device=self.device, dtype=torch.float32)
        return x.contiguous()

    # -- ActorCritic.forward (agent.py:46-54) --------------------------------------------------
    def forward(self, x, *, out=None):
        """``out`` = (mean [B, A], value [B]): preallocated outputs (contiguous float32), e.g. for a captured launch."""
        x = self._as_states(x)
        single = x.dim() == 1
        xb = x.view(1, -1) if single else x.reshape(-1, x.shape[-1])
        B = xb.shape[0]
        if xb.shape[1] != self.state_dim:
            raise ValueError(f"expected states of width {self.state_dim}, got {xb.shape[1]}")
        self._ensure_workspace(B)
        if out is None:
            mean = torch.empty((B, self.action_dim), dtype=torch.float32, device=self.device)
            value = torch.empty((B, 1), dtype=torch.float32, device=self.device)
        else:
            mean, value = out
            if mean.numel() != B * self.action_dim or value.numel() != B:
                raise ValueError(f"out must hold [{B}, {self.action_dim}] means and [{B}] values")
            value = value.view(B, 1)
        _lib.check(self._lib.hrp_ppo_forward(self._h, self.flat.data_ptr(), xb.data_ptr(), B, mean.data_ptr(),
                                             value.data_ptr(), self._stream()), "hrp_ppo_forward")
        std = None if self.discrete else self.log_std.exp()
        if single:
            return mean[0], std, value[0]
        return mean, std, value

    __call__ = forward

    def critic_into(self, states: torch.Tensor, value_out: torch.Tensor) -> torch.Tensor:
        """V(states) of [B, S] device states into ``value_out`` [B], with no allocation per call (capturable in a CUDA
        graph; the policy head's output goes to a scratch buffer of this instance)."""
        B = states.shape[0]
        self._ensure_workspace(B)
        if self._head_scratch is None or self._head_scratch.shape[0] < self.max_batch:
            self._head_scratch = torch.empty((self.max_batch, self.action_dim), dtype=torch.float32, device=self.device)
        self.forward(states, out=(self._head_scratch[:B], value_out))
        return value_out

    # -- batched get_action: everything stays on the device -------------------------------------
    def act(self, states: torch.Tensor, noise: Optional[torch.Tensor] = None, deterministic: bool = False,
            out: Optional[Dict[str, torch.Tensor]] = None, lane: int = 0,
            stream: Optional[int] = None, draw_counter: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """``get_action`` for [B, S] states -> dict(action, pre_tanh [B, A]; log_prob, value [B]).  ``stream``: raw
        ``cudaStream_t`` to enqueue on instead of torch's current stream (the multiplexer's stream ring).
        ``draw_counter``: int64 CUDA tensor [2] = (draw, 0) that replaces the host-side draw counter of the sampling
        path, so that the call can be captured in a CUDA graph and replayed (``new_draw_counter``).

        ``lane`` > 0 selects a separate native workspace (same parameters) so that calls on different CUDA streams
        may overlap: the two env groups of the pipelined host-buffer loop (bench.py e2e) act concurrently.

        Categorical policy: action [B, 2] = (id, 0) -- what the meta-action env step reads --, pre_tanh [B, 1] = id;
        ``noise`` holds one uniform in (0, 1) per row; B = 1 goes through the batched kernels."""
        states = self._as_states(states)
        B = states.shape[0]
        if B == 1 and noise is None and not lane and draw_counter is None and not self.discrete:
            return self._act_one(states, deterministic, out, stream)
        if lane:
            return self._act_lane(states, B, out, lane, deterministic, noise, draw_counter)
        self._ensure_workspace(B)
        if out is None:
            out = self._new_act_out(B)
        if stream is None:
            stream = self._stream()
        if not deterministic and noise is None and draw_counter is not None:
            _lib.check(self._lib.hrp_ppo_act_sample_ctr(self._h, self.flat.data_ptr(), states.data_ptr(), self._noise_seed,
                                                        draw_counter.data_ptr(), int(self.row_base), B,
                                                        out["action"].data_ptr(), out["pre_tanh"].data_ptr(),
                                                        out["log_prob"].data_ptr(), out["value"].data_ptr(), stream),
                       "hrp_ppo_act_sample_ctr")
            return out
        if not deterministic and noise is None:
            # standard normals drawn in the kernel (Philox keyed by a seed taken from torch's generator at
            # construction, so set_random_seeds() still fixes the rollout; one draw counter per call)
            self._draw += 1
            _lib.check(self._lib.hrp_ppo_act_sample(self._h, self.flat.data_ptr(), states.data_ptr(), self._noise_seed,
                                                    self._draw, int(self.row_base), B, out["action"].data_ptr(),
                                                    out["pre_tanh"].data_ptr(), out["log_prob"].data_ptr(),
                                                    out["value"].data_ptr(), stream), "hrp_ppo_act_sample")
            return out
        _lib.check(self._lib.hrp_ppo_act(self._h, self.flat.data_ptr(), states.data_ptr(),
                                         None if deterministic else noise.data_ptr(), B,
                                         out["action"].data_ptr(), out["pre_tanh"].data_ptr(),
                                         out["log_prob"].data_ptr(), out["value"].data_ptr(), stream),
                   "hrp_ppo_act")
        return out

    def act_widths(self):
        """Floats per row of ``act``'s action and pre_tanh outputs."""
        return (2, 1) if self.discrete else (self.action_dim, self.action_dim)

    def _new_act_out(self, B: int) -> Dict[str, torch.Tensor]:
        wa, wz = self.act_widths()
        return {"action": torch.empty((B, wa), dtype=torch.float32, device=self.device),
                "pre_tanh": torch.empty((B, wz), dtype=torch.float32, device=self.device),
                "log_prob": torch.empty(B, dtype=torch.float32, device=self.device),
                "value": torch.empty(B, dtype=torch.float32, device=self.device)}

    # -- one state: the matrix-vector kernel (what the reference's single-env loop calls once per env step) -------
    def act_item(self, state: torch.Tensor, out_row: torch.Tensor, deterministic: bool) -> "_lib.HrpActItem":
        """The ``hrp_act_item`` of one ``get_action`` call of this policy (advances the draw counter when sampling):
        ``hrp_ppo_act_multi`` serves many such items, of different policies, in one launch.  Gaussian policies only."""
        if self.discrete:
            raise ValueError("hrp_ppo_act_multi serves Gaussian policies only")
        if not deterministic:
            self._draw += 1
        it = _lib.HrpActItem()
        it.params_dev, it.state_dev, it.out_dev = self.flat.data_ptr(), state.data_ptr(), out_row.data_ptr()
        it.seed, it.draw, it.row = self._noise_seed, self._draw, int(self.row_base)
        it.state_dim, it.action_dim, it.hidden_dim = self.state_dim, self.action_dim, self.hidden_dim
        it.deterministic = int(bool(deterministic))
        return it

    def _act_one(self, states, deterministic, out, stream):
        A = self.action_dim
        packed = (out is not None and out["action"].numel() == A and out["pre_tanh"].numel() == A
                  and out["pre_tanh"].data_ptr() == out["action"].data_ptr() + 4 * A
                  and out["log_prob"].data_ptr() == out["action"].data_ptr() + 8 * A
                  and out["value"].data_ptr() == out["action"].data_ptr() + 8 * A + 4)
        row = out["action"] if packed else torch.empty(2 * A + 2, dtype=torch.float32, device=self.device)
        it = self.act_item(states, row, deterministic)
        _lib.check(self._lib.hrp_ppo_act_multi(C.byref(it), 1, self._stream() if stream is None else stream),
                   "hrp_ppo_act_multi")
        if packed:
            return out
        res = {"action": row[0:A].view(1, A), "pre_tanh": row[A:2 * A].view(1, A), "log_prob": row[2 * A:2 * A + 1],
               "value": row[2 * A + 1:2 * A + 2]}
        if out is not None:
            for k, v in res.items():
                out[k].view(-1).copy_(v.view(-1))
            return out
        return res

    def new_draw_counter(self) -> torch.Tensor:
        """A device-resident draw counter continuing this instance's host-side one (``act(draw_counter=...)``)."""
        return torch.tensor([self._draw, 0], dtype=torch.int64, device=self.device)

    def _act_lane(self, states, B, out, lane, deterministic, noise, draw_counter=None):
        """act() on an additional workspace (its GEMM scratch is its own)."""
        if deterministic or noise is not None:
            raise ValueError("workspace lanes serve the sampling rollout path only")
        lanes = self.__dict__.setdefault("_lanes", {})
        h = lanes.get(lane)
        if h is None or h[1] < B:
            if h is not None:
                torch.cuda.synchronize(self.device)
                self._lib.hrp_ppo_destroy(h[0])
            hp = C.c_void_p()
            _lib.check(self._lib.hrp_ppo_create_ex(self.state_dim, self.action_dim, self.hidden_dim, int(B),
                                                   self.device.index, self._flags, C.byref(hp)), "hrp_ppo_create_ex")
            h = lanes[lane] = (hp, int(B))
        if out is None:
            out = self._new_act_out(B)
        if draw_counter is not None:
            _lib.check(self._lib.hrp_ppo_act_sample_ctr(h[0], self.flat.data_ptr(), states.data_ptr(), self._noise_seed,
                                                        draw_counter.data_ptr(), int(self.row_base), B,
                                                        out["action"].data_ptr(), out["pre_tanh"].data_ptr(),
                                                        out["log_prob"].data_ptr(), out["value"].data_ptr(),
                                                        self._stream()), "hrp_ppo_act_sample_ctr")
            return out
        self._draw += 1
        _lib.check(self._lib.hrp_ppo_act_sample(h[0], self.flat.data_ptr(), states.data_ptr(), self._noise_seed, self._draw,
                                                int(self.row_base), B, out["action"].data_ptr(), out["pre_tanh"].data_ptr(),
                                                out["log_prob"].data_ptr(), out["value"].data_ptr(), self._stream()),
                   "hrp_ppo_act_sample")
        return out

    # -- ActorCritic.get_action (agent.py:56-74): one state, numpy results -----------------------
    def get_action(self, state, deterministic: bool = False):
        """Gaussian: (action, pre_tanh, log_prob | None, value).  Categorical: (int id, float32 array([id]),
        log_prob | None, value)."""
        x = self._as_states(state).view(1, -1)
        if self.discrete:
            buf = torch.empty(5, dtype=torch.float32, device=self.device)
            out = {"action": buf[0:2], "pre_tanh": buf[2:3], "log_prob": buf[3:4], "value": buf[4:5]}
            self.act(x, deterministic=deterministic, out=out)
            host = buf.cpu().numpy()
            log_prob = None if deterministic else float(host[3])
            return int(host[0]), host[2:3].copy(), log_prob, np.float32(host[4])
        A = self.action_dim
        buf = torch.empty(2 * A + 2, dtype=torch.float32, device=self.device)
        out = {"action": buf[0:A], "pre_tanh": buf[A:2 * A], "log_prob": buf[2 * A:2 * A + 1],
               "value": buf[2 * A + 1:2 * A + 2]}
        self.act(x, deterministic=deterministic, out=out)
        host = buf.cpu().numpy()  # one D2H for the four results
        action, pre_tanh = host[0:A].copy(), host[A:2 * A].copy()
        log_prob = None if deterministic else float(host[2 * A])
        return action, pre_tanh, log_prob, np.float32(host[2 * A + 1])

    # -- ActorCritic.evaluate (agent.py:76-84): values only, no autograd graph --------------------
    def evaluate(self, states, actions, pre_tanh_actions):
        mean, std, value = self.forward(states)
        z = self._as_states(pre_tanh_actions)
        if self.discrete:   # pre_tanh holds the sampled ids
            logp_all = torch.log_softmax(mean, dim=-1)
            ids = z.reshape(-1).long().view(-1, 1)
            entropy = -(logp_all.exp() * logp_all).sum(-1)
            return logp_all.gather(-1, ids).view(-1), value, entropy
        var = std * std
        logp = -((z - mean) ** 2) / (2 * var) - self.log_std - 0.5 * float(np.log(2 * np.pi))
        logp = logp - torch.log1p(-torch.tanh(z).pow(2) + 1e-6)
        entropy = (0.5 + 0.5 * float(np.log(2 * np.pi)) + self.log_std).sum().expand(mean.shape[0])
        return logp.sum(dim=-1), value, entropy


class PPOMemory:
    """Rollout storage.  ``store`` / ``clear`` / ``compute_advantages`` / ``get_batches`` /
    ``get_tensors`` keep the reference's list-based protocol (``agent.py:87-154``); the vectorised
    loop writes straight into device tensors via ``begin_rollout`` / ``slot``."""

    def __init__(self, batch_size: int = 64, device: Any = "cuda"):
        self.batch_size = batch_size
        self.device = _cuda_device(device)
        self.clear()
        self.rollout: Optional[Dict[str, torch.Tensor]] = None

    def store(self, state, action, pre_tanh_action, reward, next_state, log_prob, done, value):
        # next_state is accepted and dropped: nothing in the reference ever reads it back
        self.states.append(state)
        self.actions.append(action)
        self.pre_tanh_actions.append(pre_tanh_action)
        self.rewards.append(reward)
        self.log_probs.append(log_prob)
        self.dones.append(done)
        self.values.append(value)

    def clear(self):
        self.states: List[Any] = []
        self.actions: List[Any] = []
        self.pre_tanh_actions: List[Any] = []
        self.rewards: List[float] = []
        self.next_states: List[Any] = []
        self.log_probs: List[float] = []
        self.dones: List[bool] = []
        self.values: List[float] = []
        self.rollout = None
        self.bootstrap_truncated = False   # the device rollout was collected with final_states / final_value

    def __len__(self):
        if self.rollout is not None:
            return int(self.rollout["reward"].numel())
        return len(self.states)

    # -- device-resident [T, E] rollout -----------------------------------------------------------
    def begin_rollout(self, T: int, E: int, state_dim: int, action_dim: int,
                      pre_dim: Optional[int] = None, bootstrap_truncated: bool = False,
                      reward_raw: bool = False) -> Dict[str, torch.Tensor]:
        """Allocate (or reuse) time-major buffers: states [T+1,E,S] (slot T holds the bootstrap
        observation), action [T,E,A], pre_tanh [T,E,pre_dim] (default A), log_prob/value/reward [T,E],
        done [T,E] uint8.

        ``bootstrap_truncated``: also final_states [T,E,S] (the observation each finished episode ended in) and
        final_value [T,E] (the critic's value of it), zero-filled when allocated, and ``update`` bootstraps truncated
        steps with final_value (``hrp_gae_ex``).  A rollout begun without the flag gets the reference's semantics
        (truncation masks the bootstrap), whatever the reused buffers hold.

        ``reward_raw``: also reward_raw [T,E], the env's rewards before a ``VecNormalize`` scaled them into reward."""
        pre_dim = action_dim if pre_dim is None else pre_dim
        r = self.rollout
        if (r is None or r["reward"].shape != (T, E) or r["states"].shape[2] != state_dim
                or r["action"].shape[2] != action_dim or r["pre_tanh"].shape[2] != pre_dim):
            d = self.device
            r = {"states": torch.empty((T + 1, E, state_dim), dtype=torch.float32, device=d),
                 "action": torch.empty((T, E, action_dim), dtype=torch.float32, device=d),
                 "pre_tanh": torch.empty((T, E, pre_dim), dtype=torch.float32, device=d),
                 "log_prob": torch.empty((T, E), dtype=torch.float32, device=d),
                 "value": torch.empty((T, E), dtype=torch.float32, device=d),
                 "reward": torch.empty((T, E), dtype=torch.float32, device=d),
                 "done": torch.empty((T, E), dtype=torch.uint8, device=d),
                 # what the step kernel writes; `done` = terminated | truncated, formed once per rollout
                 "terminated": torch.empty((T, E), dtype=torch.uint8, device=d),
                 "truncated": torch.empty((T, E), dtype=torch.uint8, device=d)}
        if bootstrap_truncated and "final_states" not in r:
            d = self.device
            r["final_states"] = torch.zeros((T, E, state_dim), dtype=torch.float32, device=d)
            r["final_value"] = torch.zeros((T, E), dtype=torch.float32, device=d)
        if reward_raw and "reward_raw" not in r:
            r["reward_raw"] = torch.empty((T, E), dtype=torch.float32, device=self.device)
        self.rollout = r
        self.bootstrap_truncated = bool(bootstrap_truncated)
        return r

    def _from_lists(self) -> Dict[str, torch.Tensor]:
        """The list protocol, moved to the device as a [T, 1] rollout in ONE staging copy per field."""
        d = self.device
        T = len(self.states)
        f32 = lambda a: torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.float32))).to(d)
        return {"states": f32(np.array(self.states)).view(T, 1, -1),
                "action": f32(np.array(self.actions)).view(T, 1, -1),
                "pre_tanh": f32(np.array(self.pre_tanh_actions)).view(T, 1, -1),
                "log_prob": f32(self.log_probs).view(T, 1),
                "value": f32(self.values).view(T, 1),
                "reward": f32(self.rewards).view(T, 1),
                "done": torch.from_numpy(np.asarray(self.dones, dtype=np.uint8)).to(d).view(T, 1)}

    def as_rollout(self) -> Dict[str, torch.Tensor]:
        return self.rollout if self.rollout is not None else self._from_lists()

    # -- reference protocol -------------------------------------------------------------------------
    def compute_advantages(self, gamma: float, lam: float, last_value):
        """GAE (``agent.py:126-138``) on the device; returns (advantages, returns) as numpy arrays
        of shape [T] for a list-built memory, [T, E] for a device rollout."""
        r = self.as_rollout()
        adv, ret = gae(r["reward"], r["value"], r["done"], last_value, gamma, lam)
        if self.rollout is None:
            return adv.view(-1).cpu().numpy(), ret.view(-1).cpu().numpy()
        return adv.cpu().numpy(), ret.cpu().numpy()

    def get_batches(self):
        n = len(self)
        indices = np.arange(n, dtype=np.int64)
        np.random.shuffle(indices)
        return [indices[i:i + self.batch_size] for i in range(0, n, self.batch_size)]

    def get_tensors(self):
        r = self.as_rollout()
        S, A, Z = r["states"].shape[-1], r["action"].shape[-1], r["pre_tanh"].shape[-1]
        n = r["reward"].numel()
        return (r["states"].reshape(-1, S)[:n], r["action"].reshape(-1, A), r["pre_tanh"].reshape(-1, Z),
                r["log_prob"].reshape(-1))


def gae(reward: torch.Tensor, value: torch.Tensor, done: Optional[torch.Tensor], last_value, gamma: float, lam: float,
        *, terminated: Optional[torch.Tensor] = None, truncated: Optional[torch.Tensor] = None,
        final_value: Optional[torch.Tensor] = None):
    """``PPOMemory.compute_advantages`` over time-major [T, E] tensors (reverse scan kernel).

    With ``terminated`` and ``truncated`` (``done`` is then ignored) a truncated step that did not terminate is
    bootstrapped with ``final_value`` [T, E], V of the observation the episode ended in (``hrp_gae_ex``); rows of other
    steps are not read.  ``final_value=None``: the same as ``done = terminated | truncated``."""
    lib = _lib.load()
    T, E = reward.shape
    dev = reward.device
    if not torch.is_tensor(last_value):
        last_value = torch.full((E,), float(last_value), dtype=torch.float32, device=dev)
    last_value = last_value.to(device=dev, dtype=torch.float32).reshape(E).contiguous()
    adv = torch.empty((T, E), dtype=torch.float32, device=dev)
    ret = torch.empty((T, E), dtype=torch.float32, device=dev)
    if terminated is not None or truncated is not None:
        if terminated is None or truncated is None:
            raise ValueError("gae: terminated and truncated go together")
        terminated = terminated.to(torch.uint8).contiguous()
        truncated = truncated.to(torch.uint8).contiguous()
        if final_value is not None:
            final_value = final_value.to(device=dev, dtype=torch.float32).contiguous()
            if final_value.numel() != T * E:
                raise ValueError(f"final_value must hold [{T}, {E}] values")
        _lib.check(lib.hrp_gae_ex(reward.contiguous().data_ptr(), value.contiguous().data_ptr(), terminated.data_ptr(),
                                  truncated.data_ptr(), _lib.ptr(final_value), last_value.data_ptr(), T, E,
                                  float(gamma), float(lam), adv.data_ptr(), ret.data_ptr(),
                                  torch.cuda.current_stream(dev).cuda_stream), "hrp_gae_ex")
        return adv, ret
    if final_value is not None:
        raise ValueError("gae: final_value needs terminated and truncated")
    done = done.to(torch.uint8).contiguous()
    _lib.check(lib.hrp_gae(reward.contiguous().data_ptr(), value.contiguous().data_ptr(), done.data_ptr(),
                           last_value.data_ptr(), T, E, float(gamma), float(lam), adv.data_ptr(), ret.data_ptr(),
                           torch.cuda.current_stream(dev).cuda_stream), "hrp_gae")
    return adv, ret


class _AdamState:
    """``optim.Adam(params, lr)`` as flat moment buffers + a device step counter.

    ``lr_dev``: None (the learning rate is a launch argument, baked into captured graphs), or a float64 [1] device
    tensor that the Adam kernels read when they run (``PPOAgent.set_lr``); assigning ``lr`` then also writes it."""

    def __init__(self, ac: ActorCritic, lr: float):
        self.ac = ac
        self.lr_dev: Optional[torch.Tensor] = None
        self.lr, self.betas, self.eps = float(lr), (0.9, 0.999), 1e-8
        d = ac.device
        self.exp_avg = torch.zeros(ac.num_params, dtype=torch.float32, device=d)
        self.exp_avg_sq = torch.zeros(ac.num_params, dtype=torch.float32, device=d)
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=d)
        self.scratch = torch.zeros(128, dtype=torch.float32, device=d)
        self.param_groups = [{"lr": self.lr, "betas": self.betas, "eps": self.eps, "weight_decay": 0,
                              "amsgrad": False, "maximize": False, "foreach": None, "capturable": False,
                              "differentiable": False, "fused": None, "decoupled_weight_decay": False,
                              "params": list(range(len(ac.shapes)))}]

    @property
    def lr(self) -> float:
        return self._lr

    @lr.setter
    def lr(self, value: float) -> None:
        self._lr = float(value)
        if self.lr_dev is not None:
            self.lr_dev.fill_(self._lr)   # stream-ordered before the next update's launches or graph replays

    def state_dict(self) -> Dict[str, Any]:
        """Same structure as ``torch.optim.Adam.state_dict()`` over ``ActorCritic.parameters()``."""
        step = int(self.step_dev.item())
        state: Dict[int, Any] = {}
        if step > 0:
            off = 0
            for i, shape in enumerate(self.ac.shapes.values()):
                n = int(np.prod(shape))
                state[i] = {"step": torch.tensor(float(step)),
                            "exp_avg": self.exp_avg[off:off + n].view(shape).clone(),
                            "exp_avg_sq": self.exp_avg_sq[off:off + n].view(shape).clone()}
                off += n
        groups = [dict(g) for g in self.param_groups]
        groups[0]["lr"] = self.lr
        return {"state": state, "param_groups": groups}

    def load_state_dict(self, sd: Dict[str, Any]) -> None:
        state = sd.get("state", {})
        off, step = 0, 0
        for i, shape in enumerate(self.ac.shapes.values()):
            n = int(np.prod(shape))
            s = state.get(i, state.get(str(i)))
            if s is not None:
                self.exp_avg[off:off + n].copy_(s["exp_avg"].reshape(-1).to(self.exp_avg))
                self.exp_avg_sq[off:off + n].copy_(s["exp_avg_sq"].reshape(-1).to(self.exp_avg_sq))
                step = int(float(s["step"]))
            off += n
        self.step_dev.fill_(step)
        groups = sd.get("param_groups") or []
        if groups:
            self.lr = float(groups[0].get("lr", self.lr))
            self.betas = tuple(groups[0].get("betas", self.betas))
            self.eps = float(groups[0].get("eps", self.eps))


class PPOAgent:
    def __init__(self, state_dim: int, action_dim: int, lr: float = 1e-4, gamma: float = 0.99, lam: float = 0.95,
                 eps_clip: float = 0.2, value_coef: float = 0.5, entropy_coef: float = 0.005,
                 max_grad_norm: float = 0.5, epochs: int = 6, batch_size: int = 64, hidden_dim: int = 128,
                 logger: Optional[logging.Logger] = None, device: Any = "cuda", *, discrete: bool = False,
                 clip_value: Optional[float] = None):
        """``clip_value`` = c (keyword-only, off by default): the clipped value loss, max((v - R)^2, (v_old +
        clamp(v - v_old, -c, c) - R)^2) per sample with v_old the value the rollout stored (``hrp_ppo_loss_grad_ex``),
        weighted like the reference's value MSE; the ``value_loss`` and ``loss`` metrics report it."""
        if clip_value is not None and not (math.isfinite(float(clip_value)) and float(clip_value) > 0):
            raise ValueError(f"clip_value must be a finite number > 0 or None, got {clip_value!r}")
        self.clip_value = None if clip_value is None else float(clip_value)
        self._lib = _lib.load()
        self.device = _cuda_device(device)
        self.discrete = bool(discrete)
        self.actor_critic = ActorCritic(state_dim, action_dim, hidden_dim, device=self.device,
                                        max_batch=max(int(batch_size), 1), discrete=self.discrete)
        self.optimizer = _AdamState(self.actor_critic, lr)
        self.gamma, self.lam, self.eps_clip = gamma, lam, eps_clip
        self.value_coef, self.entropy_coef, self.max_grad_norm = value_coef, entropy_coef, max_grad_norm
        self.epochs = epochs
        self.logger = logger or logging.getLogger(__name__)
        self.memory = PPOMemory(batch_size=batch_size, device=self.device)
        P = self.actor_critic.num_params
        self.grad = torch.zeros(P, dtype=torch.float32, device=self.device)
        self._metrics = torch.zeros(8, dtype=torch.float32, device=self.device)
        self._stats = torch.zeros(3 + 512, dtype=torch.float64, device=self.device)
        self.launches = 0  # hrp_* calls enqueued by this agent (each is >= 1 kernel of this library)
        self.use_cuda_graphs = True
        # capture the gradient all-reduce inside the minibatch graphs (NCCL only; gloo cannot be captured).  Call
        # release_graphs() before torch.distributed.destroy_process_group(): graphs that hold NCCL work keep the
        # communicator busy at teardown.
        self.graph_collectives = os.environ.get("HRP_GRAPH_COLLECTIVES", "1") != "0" and distributed.backend() == "nccl"
        self._graph_state: Optional[Dict[str, Any]] = None
        # peer-memory gradient exchange fused with clip + Adam (csrc/hrp_comm.cu); set up lazily by the first sharded
        # update.  HRP_P2P=0 keeps the NCCL all-reduce + hrp_clip_adam_step pair.
        self.use_p2p = os.environ.get("HRP_P2P", "1") != "0" and distributed.backend() == "nccl"
        self._comm = None
        self._comm_keep = None

    def set_lr(self, lr: float) -> None:
        """Set the learning rate of the following optimizer steps.  The first call moves it into device memory
        (``optimizer.lr_dev``, read by ``hrp_clip_adam_step_ex`` / ``hrp_clip_adam_step_p2p_ex`` when they run), so that
        a schedule calling this every update keeps replaying the captured minibatch graphs instead of capturing new
        ones.  Every call writes the value on the current stream, outside any graph."""
        opt = self.optimizer
        if opt.lr_dev is None:
            opt.lr_dev = torch.empty(1, dtype=torch.float64, device=self.device)
        opt.lr = lr

    # -- acting ----------------------------------------------------------------------------------
    def select_action(self, state, deterministic: bool = False):
        self.launches += 1
        return self.actor_critic.get_action(state, deterministic)

    def act(self, states: torch.Tensor, deterministic: bool = False, noise: Optional[torch.Tensor] = None,
            out: Optional[Dict[str, torch.Tensor]] = None, lane: int = 0, stream: Optional[int] = None,
            draw_counter: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        self.launches += 1
        return self.actor_critic.act(states, noise=noise, deterministic=deterministic, out=out, lane=lane, stream=stream,
                                     draw_counter=draw_counter)

    # -- distributed helpers (ppo/distributed.py) ---------------------------------------------------
    @staticmethod
    def _world() -> int:
        return distributed.world_size()

    def _allreduce(self, t: torch.Tensor) -> None:
        distributed.allreduce_sum_(t)

    # -- peer-memory exchange -------------------------------------------------------------------------
    def _ensure_comm(self, world: int) -> bool:
        """Create and connect this rank's ``hrp_comm`` (once): every rank exports its gradient buffer through
        cudaIpc, the 64-byte handles are all-gathered, and ``self.grad`` becomes a view of the exported buffer.
        Returns False (and keeps the NCCL path) when the devices cannot map each other's memory."""
        if self._comm is not None:
            return True
        if not self.use_p2p or world > 8:
            return False
        import torch.distributed as dist

        lib, P = self._lib, self.actor_critic.num_params
        handle = (C.c_ubyte * 64)()
        comm = C.c_void_p()
        rc = lib.hrp_comm_create(world, distributed.rank(), P, self.device.index, C.byref(comm), handle)
        ok = torch.tensor([1 if rc == 0 else 0], dtype=torch.int32, device=self.device)
        mine = torch.tensor(list(handle), dtype=torch.uint8, device=self.device)
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        if rc == 0:
            blob = b"".join(bytes(g.cpu().numpy().tobytes()) for g in gathered)
            rc = lib.hrp_comm_connect(comm, blob)
            ok[0] = 1 if rc == 0 else 0
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)   # all ranks take the same path
        if int(ok.item()) != 1:
            self.logger.warning("peer-memory gradient exchange unavailable (%s); using the NCCL all-reduce",
                                _lib.last_error() if hasattr(_lib, "last_error") else "cudaIpc")
            if comm:
                lib.hrp_comm_destroy(comm)
            self.use_p2p = False
            return False
        # the exchange double-buffers the gradient by step parity: two views of the exported allocation
        self._comm_keep, self._grad_parity = [], []
        for parity in (0, 1):
            ptr = lib.hrp_comm_grad_parity(comm, parity)

            class _Raw:  # torch.as_tensor wraps a raw device pointer through the CUDA array interface
                __cuda_array_interface__ = {"shape": (P,), "typestr": "<f4", "data": (int(ptr), False), "version": 2}

            keep = _Raw()
            view = torch.as_tensor(keep, device=self.device)
            assert view.data_ptr() == int(ptr)
            self._comm_keep.append(keep)
            self._grad_parity.append(view)
        self.grad = self._grad_parity[0]
        self._comm = comm
        return True

    def close(self) -> None:
        """Release the captured graphs and the peer-memory exchange (before the process group is destroyed)."""
        self.release_graphs()
        if self._comm is not None:
            torch.cuda.synchronize(self.device)
            self.grad = torch.zeros(self.actor_critic.num_params, dtype=torch.float32, device=self.device)
            self._lib.hrp_comm_destroy(self._comm)
            self._comm, self._comm_keep, self._grad_parity = None, None, None

    # -- one optimizer step on minibatch ``idx`` (device int64) ----------------------------------
    def _minibatch_step(self, flat: Dict[str, torch.Tensor], idx: Optional[torch.Tensor], B: int, world: int) -> None:
        ac, opt, s = self.actor_critic, self.optimizer, self.actor_critic._stream()
        if world > 1 and self._comm is not None:
            self.grad = self._grad_parity[self._lib.hrp_comm_parity(self._comm)]   # the buffer of this step's parity
        loss_args = (ac._h, ac.flat.data_ptr(), flat["states"].data_ptr(), flat["pre_tanh"].data_ptr(),
                     flat["log_prob"].data_ptr(), flat["adv"].data_ptr(), flat["ret"].data_ptr(), _lib.ptr(idx), B,
                     float(self.eps_clip), float(self.value_coef), float(self.entropy_coef),
                     distributed.loss_scale(B, world))
        if self.clip_value is None:
            _lib.check(self._lib.hrp_ppo_loss_grad(*loss_args, self.grad.data_ptr(), self._metrics.data_ptr(), s),
                       "hrp_ppo_loss_grad")
        else:
            _lib.check(self._lib.hrp_ppo_loss_grad_ex(*loss_args, flat["value"].data_ptr(), self.clip_value,
                                                      self.grad.data_ptr(), self._metrics.data_ptr(), s),
                       "hrp_ppo_loss_grad_ex")
        lr_dev = opt.lr_dev
        if world > 1 and self._comm is not None:
            # all_reduce + clip + Adam as one kernel over peer memory
            args = (self._comm, ac.flat.data_ptr(), opt.exp_avg.data_ptr(), opt.exp_avg_sq.data_ptr(),
                    opt.step_dev.data_ptr(), opt.lr)
            tail = (opt.betas[0], opt.betas[1], opt.eps, float(self.max_grad_norm), opt.scratch.data_ptr(), s)
            if lr_dev is None:
                _lib.check(self._lib.hrp_clip_adam_step_p2p(*args, *tail), "hrp_clip_adam_step_p2p")
            else:
                _lib.check(self._lib.hrp_clip_adam_step_p2p_ex(*args, lr_dev.data_ptr(), *tail),
                           "hrp_clip_adam_step_p2p_ex")
            self.launches += 2
            return
        if world > 1:
            self._allreduce(self.grad)
        args = (ac.flat.data_ptr(), self.grad.data_ptr(), opt.exp_avg.data_ptr(), opt.exp_avg_sq.data_ptr(),
                opt.step_dev.data_ptr(), ac.num_params, opt.lr)
        tail = (opt.betas[0], opt.betas[1], opt.eps, float(self.max_grad_norm), opt.scratch.data_ptr(), s)
        if lr_dev is None:
            _lib.check(self._lib.hrp_clip_adam_step(*args, *tail), "hrp_clip_adam_step")
        else:
            _lib.check(self._lib.hrp_clip_adam_step_ex(*args, lr_dev.data_ptr(), *tail), "hrp_clip_adam_step_ex")
        self.launches += 2

    def release_graphs(self) -> None:
        """Drop the captured minibatch graphs (they are re-captured by the next update)."""
        if self._graph_state is not None:
            torch.cuda.synchronize(self.device)
            self._graph_state = None

    # -- the epochs x minibatches loop as CUDA graphs --------------------------------------------------
    def _capture(self, fn, world: int) -> "torch.cuda.CUDAGraph":
        g = torch.cuda.CUDAGraph()
        if world > 1:   # collectives inside: torch's context (full synchronisation, allocator quiesced) as before
            with torch.cuda.graph(g):
                fn()
            return g
        # single GPU: nothing inside allocates through torch, so skip the context's gc + empty_cache + device
        # synchronisation (10 ms per capture; a sweep run at batch 32 captures often)
        cur = torch.cuda.current_stream(self.device)
        if getattr(self, "_capture_stream", None) is None:
            self._capture_stream = torch.cuda.Stream(self.device)
        cap = self._capture_stream
        cap.wait_stream(cur)
        torch.cuda.set_stream(cap)   # (not the stream context: its enter / exit each query the device count)
        try:
            g.capture_begin()
            try:
                fn()
            finally:
                g.capture_end()
        finally:
            torch.cuda.set_stream(cur)
        cur.wait_stream(cap)
        return g

    def _graphed_epochs(self, flat: Dict[str, torch.Tensor], perm_dev: torch.Tensor, n: int, bs: int,
                        world: int = 1) -> None:
        """The ~40 launches of one optimizer step (loss / backward / clip / Adam) as a CUDA graph, replayed for every
        epoch and re-used by later updates of the same shape: one graph per minibatch when there are at most 32 of them,
        else ONE graph per distinct minibatch size (the full one and a ragged last one) that reads its sample indices
        from a fixed buffer which a small device-to-device copy of the permutation slice refills before each replay.  The rollout is first copied into
        persistent buffers so that the captured pointers stay valid.  The first epoch of a new configuration runs
        eagerly (it also warms every kernel variant before anything is captured)."""
        ac = self.actor_critic
        # the workspace generation, not its address: a re-created workspace may reuse the freed one's address.  A
        # learning rate in device memory (set_lr) is read by the captured steps, so its value is not part of the key.
        opt = self.optimizer
        key = (n, bs, world, ac.workspace_generation, float(self.eps_clip), float(self.value_coef), float(self.entropy_coef),
               float(self.max_grad_norm), opt.lr if opt.lr_dev is None else "lr_dev", opt.betas, opt.eps,
               self.clip_value)
        st = self._graph_state
        if st is None or st["key"] != key:
            d = self.device
            st = {"key": key, "graphs": {}, "warm": False,
                  "buf": {k: torch.empty_like(v) for k, v in flat.items()},
                  "perm": torch.empty(n, dtype=torch.int64, device=d),
                  "idx": torch.empty(min(bs, n), dtype=torch.int64, device=d)}
            self._graph_state = st
        for k, v in flat.items():
            st["buf"][k].copy_(v)
        st["perm"].copy_(perm_dev)
        starts = list(range(0, n, bs))
        # few minibatches (the big-batch configuration: 32 of 4096): one graph per minibatch, its permutation slice baked
        # in, nothing between the replays.  Many (a sweep run at batch 32: 64 and more): one graph per distinct size,
        # fed through the index buffer, because capturing dominates there.
        shared = len(starts) > 32
        for epoch in range(self.epochs):
            for i, start in enumerate(starts):
                B = min(bs, n - start)
                if shared:
                    idx = st["idx"][:B]
                    idx.copy_(st["perm"][start:start + B])
                else:
                    idx = st["perm"][start:start + B]
                if not st["warm"]:
                    self._minibatch_step(st["buf"], idx, B, world)
                    continue
                # the peer-memory exchange alternates its buffers with the step parity: one graph per (.., parity)
                parity = self._lib.hrp_comm_parity(self._comm) if (world > 1 and self._comm is not None) else 0
                gkey = (B if shared else ("mb", i), parity)
                g = st["graphs"].get(gkey)
                if g is None:
                    # (capturing advances the parity)
                    g = self._capture(lambda: self._minibatch_step(st["buf"], idx, B, world), world)
                    st["graphs"][gkey] = g
                elif world > 1 and self._comm is not None:
                    _lib.check(self._lib.hrp_comm_note_replay(self._comm), "hrp_comm_note_replay")
                    self.grad = self._grad_parity[parity]
                g.replay()
                self.launches += 2
            st["warm"] = True

    # -- PPOAgent.update (agent.py:196-308) --------------------------------------------------------
    def update(self, last_value=0.0) -> Dict[str, float]:
        return self.update_end(self.update_begin(last_value))

    def update_begin(self, last_value=0.0):
        """Enqueue the whole update on the current stream and return a handle for ``update_end``: no host
        synchronisation (single-GPU), so that the updates of several agents on several streams overlap
        (experiments/multiplex.py)."""
        mem, ac = self.memory, self.actor_critic
        r = mem.as_rollout()
        T, E = r["reward"].shape
        n = T * E
        S = ac.state_dim
        world = self._world()
        stream = ac._stream()
        if mem.rollout is not None and mem.bootstrap_truncated:   # collect_rollout(bootstrap_truncated=True)
            adv, ret = gae(r["reward"], r["value"], None, last_value, self.gamma, self.lam, terminated=r["terminated"],
                           truncated=r["truncated"], final_value=r["final_value"])
        else:
            adv, ret = gae(r["reward"], r["value"], r["done"], last_value, self.gamma, self.lam)
        # advantage normalisation over the whole (global) buffer, unbiased std (agent.py:204)
        adv_n = adv.clone()
        _lib.check(self._lib.hrp_adv_stats(adv_n.data_ptr(), n, self._stats.data_ptr(), stream), "hrp_adv_stats")
        if world > 1:
            self._allreduce(self._stats[:3])
        _lib.check(self._lib.hrp_adv_normalize(adv_n.data_ptr(), n, self._stats.data_ptr(), stream),
                   "hrp_adv_normalize")
        self.launches += 3
        flat = {"states": r["states"].reshape(-1, S)[:n].contiguous(),
                "pre_tanh": r["pre_tanh"].reshape(n, ac.act_widths()[1]),
                "log_prob": r["log_prob"].reshape(n), "adv": adv_n.view(n), "ret": ret.view(n)}
        if self.clip_value is not None:   # the rollout's values, the v_old of the clipped value loss
            flat["value"] = r["value"].reshape(n)
        # one permutation per update, reused by every epoch (agent.py:140-147,205)
        perm = np.arange(n, dtype=np.int64)
        np.random.shuffle(perm)
        perm_dev = torch.from_numpy(perm).to(self.device)
        bs = int(mem.batch_size)
        ac._ensure_workspace(min(bs, n))
        self._metrics.zero_()
        if world > 1:
            self._ensure_comm(world)
        if self.use_cuda_graphs and (world == 1 or self.graph_collectives):
            # with several ranks the NCCL all-reduce of the flat gradient is captured inside each minibatch graph
            self._graphed_epochs(flat, perm_dev, n, bs, world)
        else:
            for _ in range(self.epochs):
                for start in range(0, n, bs):
                    B = min(bs, n - start)
                    self._minibatch_step(flat, perm_dev[start:start + B], B, world)
        if self._comm is not None:
            _lib.check(self._lib.hrp_comm_status(self._comm), "hrp_comm_status")   # a peer that never arrived
        # explained variance of the value predictions (agent.py:276-285)
        y_pred, y_true = r["value"].reshape(n), ret.view(n)
        if world > 1:
            # global variances from all-reduced moments
            res = y_true - y_pred
            mom = torch.stack([y_true.double().sum(), (y_true.double() ** 2).sum(), res.double().sum(),
                               (res.double() ** 2).sum(), torch.tensor(float(n), dtype=torch.float64, device=self.device)])
            self._allreduce(mom)
            cnt = mom[4]
            var_y = (mom[1] - mom[0] ** 2 / cnt) / (cnt - 1)
            var_r = (mom[3] - mom[2] ** 2 / cnt) / (cnt - 1)
            self._allreduce(self._metrics)
        else:
            var_y = torch.var(y_true) if n > 1 else torch.zeros((), device=self.device)
            var_r = torch.var(y_true - y_pred) if n > 1 else torch.zeros((), device=self.device)
        tail = torch.stack([var_y.float(), var_r.float()])
        if getattr(self, "_metrics_host", None) is None:
            self._metrics_host = torch.zeros(10, dtype=torch.float32).pin_memory()
        self._metrics_host.copy_(torch.cat([self._metrics, tail]), non_blocking=True)   # the update's single D2H
        done = torch.cuda.Event()
        done.record()
        mem.clear()
        return done

    def update_end(self, done) -> Dict[str, float]:
        """Wait for the update enqueued by ``update_begin`` and return its metrics."""
        done.synchronize()
        host = self._metrics_host.numpy().copy()
        count = max(float(host[6]), 1.0)
        explained = float(1.0 - host[9] / host[8]) if host[8] > 0 else 0.0
        out = {"loss": float(host[0] / count), "policy_loss": float(host[1] / count),
               "value_loss": float(host[2] / count), "entropy": float(host[3] / count),
               "clip_fraction": float(host[4] / count), "approx_kl": float(host[5] / count),
               "explained_variance": explained}
        self.logger.info(
            "update_complete loss=%.4f policy_loss=%.4f value_loss=%.4f entropy=%.4f clip_frac=%.3f kl=%.5f "
            "explained_var=%.3f", out["loss"], out["policy_loss"], out["value_loss"], out["entropy"],
            out["clip_fraction"], out["approx_kl"], out["explained_variance"])
        return out

    # -- checkpoints (agent.py:310-327): same file format and key names ----------------------------
    def save(self, path: str):
        torch.save({"model": self.actor_critic.state_dict(), "optimizer": self.optimizer.state_dict()}, path)
        self.logger.info(f"model_saved path={path}")

    def load(self, path: str, load_optimizer: bool = True):
        checkpoint = torch.load(path, map_location=self.device)
        self.actor_critic.load_state_dict(checkpoint["model"])
        if load_optimizer and "optimizer" in checkpoint:
            self.optimizer.load_state_dict(checkpoint["optimizer"])
        self.logger.info(f"model_loaded path={path}")
        return checkpoint.get("config", {})
