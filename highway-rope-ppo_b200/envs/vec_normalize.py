"""Running observation and reward normalization of a ``HighwayVecEnv``: SB3's ``VecNormalize`` on the device.

The statistics are fp64 device tensors updated in place by ``libhrp_b200.so`` (``hrp_vecnorm_*``, csrc/hrp_norm.cu), so
a captured rollout or evaluation reads and advances the current values with no host synchronisation.  A training step
is the inner step followed by three launches: batch moments (and the return carry), their merge into the running
statistics, and the normalization of the observation, the terminal observations and the reward.  Under
``torch.distributed`` the per-rank batch moments are all-gathered and merged in rank order, so every rank holds the
same bits; with NCCL the all-gather is captured with the rest of the rollout.
"""
from __future__ import annotations

import math
from typing import Any, Dict, Optional

import torch

from .. import _lib
from ..ppo import distributed


class RunningMeanStd:
    """SB3's ``RunningMeanStd(epsilon=1e-4, shape)`` in device fp64: ``mean`` and ``var`` of ``shape``, scalar ``count``,
    all views of one buffer [mean | var | count] that the kernels update in place."""

    def __init__(self, shape, device, epsilon: float = 1e-4):
        self.shape = tuple(shape)
        n = math.prod(self.shape)
        self.buf = torch.zeros(2 * n + 1, dtype=torch.float64, device=device)
        self.mean = self.buf[:n].view(self.shape)
        self.var = self.buf[n:2 * n].view(self.shape)
        self.count = self.buf[2 * n]
        self.var.fill_(1.0)
        self.count.fill_(float(epsilon))


def _check_settings(clip_obs: float, clip_reward: float, gamma: float, epsilon: float) -> None:
    for name, v in (("clip_obs", clip_obs), ("clip_reward", clip_reward)):
        if not (math.isfinite(float(v)) and float(v) > 0):
            raise ValueError(f"{name} must be finite and > 0, got {v}")
    if not 0.0 <= float(gamma) <= 1.0:
        raise ValueError(f"gamma must be in [0, 1], got {gamma}")
    if not (math.isfinite(float(epsilon)) and float(epsilon) >= 0):
        raise ValueError(f"epsilon must be finite and >= 0, got {epsilon}")


class VecNormalize:
    """``VecNormalize(venv, training, norm_obs, norm_reward, clip_obs, clip_reward, gamma, epsilon)`` around a
    ``HighwayVecEnv``, with SB3's semantics and defaults.

    ``reset`` / ``observe`` / ``step`` take the inner handle's arguments; ``step(..., raw_reward_out=)`` also receives the
    raw reward (the normalized one goes to ``reward_out``).  In training mode ``step`` updates the observation statistics
    with the step's observations (the first observation of a new episode for done envs), normalizes with the updated
    statistics, advances the per-env return carry ``returns = returns * gamma + reward`` and updates the return
    statistics with it, divides the reward by the return standard deviation, normalizes the terminal observations
    (``final_obs_out``) with the same statistics and clears the carry of done envs; ``reset`` updates the observation
    statistics and clears every carry.  ``training=False`` updates nothing and still normalizes.
    """

    _next_uid = 1 << 30   # apart from HighwayVecEnv's uids: the rollout graph cache keys on them

    def __init__(self, venv, training: bool = True, norm_obs: bool = True, norm_reward: bool = True,
                 clip_obs: float = 10.0, clip_reward: float = 10.0, gamma: float = 0.99, epsilon: float = 1e-8):
        if isinstance(venv, VecNormalize):
            raise ValueError("venv is already a VecNormalize")
        for name in ("num_envs", "N", "F_out", "obs_shape", "step", "reset", "observe"):
            if not hasattr(venv, name):
                raise ValueError(f"venv must be a HighwayVecEnv (it has no {name!r})")
        _check_settings(clip_obs, clip_reward, gamma, epsilon)
        self.venv = venv
        self._training = bool(training)
        self.norm_obs, self.norm_reward = bool(norm_obs), bool(norm_reward)
        self.clip_obs, self.clip_reward = float(clip_obs), float(clip_reward)
        self.gamma, self.epsilon = float(gamma), float(epsilon)
        dev = venv.device
        self.S = venv.N * venv.F_out
        self.obs_rms = RunningMeanStd(venv.obs_shape, dev)
        self.ret_rms = RunningMeanStd((), dev)
        self.returns = torch.zeros(venv.num_envs, dtype=torch.float64, device=dev)
        C = self.S + 1
        self._moments = torch.zeros(_lib.vecnorm_moments_len(C), dtype=torch.float64, device=dev)
        self._scratch = torch.zeros(_lib.vecnorm_scratch_len(C), dtype=torch.float64, device=dev)
        self._gathered: Dict[int, torch.Tensor] = {}
        self._raw_reward = torch.zeros(venv.num_envs, dtype=torch.float32, device=dev)
        self._lib = _lib.load()
        self.launches = 0
        VecNormalize._next_uid += 1
        self.uid = VecNormalize._next_uid
        self.param_version = 0

    # ------------------------------------------------------------------ forwarded
    num_envs = property(lambda self: self.venv.num_envs)
    N = property(lambda self: self.venv.N)
    F_out = property(lambda self: self.venv.F_out)
    obs_shape = property(lambda self: self.venv.obs_shape)
    cfg = property(lambda self: self.venv.cfg)
    config = property(lambda self: self.venv.config)
    device = property(lambda self: self.venv.device)
    env_id_base = property(lambda self: self.venv.env_id_base)
    embed = property(lambda self: self.venv.embed)
    real64 = property(lambda self: self.venv.real64)
    grid = property(lambda self: self.venv.grid)

    @property
    def training(self) -> bool:
        return self._training

    @training.setter
    def training(self, on: bool) -> None:
        if bool(on) != self._training:
            self._training = bool(on)
            self.param_version += 1   # captured steps bake in which launches they make

    def set_env_seeds(self, seeds: Optional[torch.Tensor]) -> None:
        self.venv.set_env_seeds(seeds)
        self.param_version += 1

    def set_step_mask(self, mask: Optional[torch.Tensor]) -> None:
        """Allowed with ``training=False`` only: a masked env would still enter the batch statistics."""
        if mask is not None and self._training:
            raise ValueError("set_step_mask needs training=False: masked envs would still enter the running statistics")
        self.venv.set_step_mask(mask)
        self.param_version += 1

    def close(self) -> None:
        self.venv.close()

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # ------------------------------------------------------------------ kernels
    def _update(self, obs: Optional[torch.Tensor], reward: Optional[torch.Tensor]) -> None:
        """Batch moments of ``obs`` (and of the return carry advanced by ``reward``) merged into the statistics."""
        S = self.S if obs is not None else 0
        C = S + (reward is not None)
        E = self.num_envs
        st = self._stream()
        mom = self._moments[:_lib.vecnorm_moments_len(C)]
        _lib.check(self._lib.hrp_vecnorm_moments(_lib.ptr(obs), E, S, _lib.ptr(reward), self.returns.data_ptr(),
                                                 self.gamma, mom.data_ptr(), self._scratch.data_ptr(), st),
                   "hrp_vecnorm_moments")
        R = distributed.world_size()
        if R > 1:
            g = self._gathered.get(C)
            if g is None:
                g = self._gathered[C] = torch.zeros(R * mom.numel(), dtype=torch.float64, device=self.device)
            torch.distributed.all_gather_into_tensor(g, mom)
            mom = g
        _lib.check(self._lib.hrp_vecnorm_merge(mom.data_ptr(), R, S, int(reward is not None),
                                               self.obs_rms.buf.data_ptr(), self.ret_rms.buf.data_ptr(),
                                               self._scratch.data_ptr(), st), "hrp_vecnorm_merge")
        self.launches += 2

    def _apply(self, obs: torch.Tensor, final_obs=None, terminated=None, truncated=None, reward=None,
               reward_out=None) -> None:
        norm_obs = self.norm_obs
        if not norm_obs and reward is None:
            if terminated is not None:
                self.returns.masked_fill_((terminated | truncated).bool(), 0.0)
            return
        _lib.check(self._lib.hrp_vecnorm_apply(
            obs.data_ptr() if norm_obs else None, _lib.ptr(final_obs) if norm_obs else None, _lib.ptr(terminated),
            _lib.ptr(truncated), self.num_envs, self.S if norm_obs else 0, _lib.ptr(reward), _lib.ptr(reward_out),
            self.returns.data_ptr(), self.obs_rms.buf.data_ptr(), self.ret_rms.buf.data_ptr(), self.clip_obs,
            self.clip_reward, self.epsilon, self._stream()), "hrp_vecnorm_apply")
        self.launches += 1

    @property
    def step_launches(self) -> int:
        """Library launches of one ``step``: the inner step, moments + merge in training, the normalization."""
        n = 1 + (2 if self._training and (self.norm_obs or self.norm_reward) else 0)
        return n + (1 if self.norm_obs or self.norm_reward else 0)

    @property
    def reset_launches(self) -> int:
        """Library launches of one ``reset``: the inner reset, moments + merge in training, the normalization."""
        return 1 + (3 if self._training and self.norm_obs else 1 if self.norm_obs else 0)

    # ------------------------------------------------------------------ stepping
    def reset(self, seed: Optional[int] = None, mask: Optional[torch.Tensor] = None,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The inner ``reset``; in training mode the reset observations update the observation statistics.  A ``mask``
        needs ``training=False``: the rows of envs it leaves alone would still enter the statistics."""
        if mask is not None and self._training:
            raise ValueError("reset(mask=...) needs training=False: envs that are not reset would still enter the running "
                             "statistics")
        obs = self.venv.reset(seed=seed, mask=mask, out=out)
        self.launches += 1
        if self._training and self.norm_obs:
            self._update(obs, None)
        self.returns.zero_()
        if self.norm_obs:
            self._apply(obs)
        return obs

    def observe(self, perm=None, row_vehicle=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        obs = self.venv.observe(perm=perm, row_vehicle=row_vehicle, out=out)
        self.launches += 1
        if self.norm_obs:
            self._apply(obs)
        return obs

    def step(self, actions: torch.Tensor, perm=None, row_vehicle=None, out: Optional[torch.Tensor] = None,
             reward_out: Optional[torch.Tensor] = None, terminated_out: Optional[torch.Tensor] = None,
             truncated_out: Optional[torch.Tensor] = None, final_obs_out: Optional[torch.Tensor] = None,
             raw_reward_out: Optional[torch.Tensor] = None):
        """The inner ``step``; returns (obs, reward, terminated, truncated), normalized where switched on.  The raw
        reward lands in ``raw_reward_out`` (a buffer of this wrapper when None)."""
        raw = raw_reward_out if raw_reward_out is not None else self._raw_reward
        if not self.norm_reward:
            raw = reward_out if reward_out is not None else raw   # the reward passes through: one buffer
        obs, rew, term, trunc = self.venv.step(actions, perm=perm, row_vehicle=row_vehicle, out=out, reward_out=raw,
                                               terminated_out=terminated_out, truncated_out=truncated_out,
                                               final_obs_out=final_obs_out)
        self.launches += 1
        if self._training and (self.norm_obs or self.norm_reward):
            self._update(obs if self.norm_obs else None, rew if self.norm_reward else None)
        if not self.norm_reward:
            if raw_reward_out is not None and raw_reward_out is not rew:
                raw_reward_out.copy_(rew)
            self._apply(obs, final_obs_out, term, trunc)
            return obs, rew, term, trunc
        rout = reward_out if reward_out is not None else self.venv.reward
        self._apply(obs, final_obs_out, term, trunc, reward=rew, reward_out=rout)
        return obs, rout, term, trunc

    # ------------------------------------------------------------------ persistence (SB3's names)
    def state_dict(self) -> Dict[str, Any]:
        return {"obs_mean": self.obs_rms.mean.cpu().clone(), "obs_var": self.obs_rms.var.cpu().clone(),
                "obs_count": float(self.obs_rms.count), "ret_mean": float(self.ret_rms.mean),
                "ret_var": float(self.ret_rms.var), "ret_count": float(self.ret_rms.count),
                "norm_obs": self.norm_obs, "norm_reward": self.norm_reward, "clip_obs": self.clip_obs,
                "clip_reward": self.clip_reward, "gamma": self.gamma, "epsilon": self.epsilon}

    def load_state_dict(self, sd: Dict[str, Any]) -> None:
        """Copy the statistics in place (captured launches keep reading the same tensors) and the settings."""
        mean = torch.as_tensor(sd["obs_mean"], dtype=torch.float64)
        if tuple(mean.shape) != tuple(self.obs_rms.shape):
            raise ValueError(f"obs statistics of shape {tuple(mean.shape)} do not fit observations of shape "
                             f"{tuple(self.obs_rms.shape)}")
        _check_settings(sd["clip_obs"], sd["clip_reward"], sd["gamma"], sd["epsilon"])
        self.obs_rms.mean.copy_(mean)
        self.obs_rms.var.copy_(torch.as_tensor(sd["obs_var"], dtype=torch.float64))
        self.obs_rms.count.fill_(float(sd["obs_count"]))
        self.ret_rms.mean.fill_(float(sd["ret_mean"]))
        self.ret_rms.var.fill_(float(sd["ret_var"]))
        self.ret_rms.count.fill_(float(sd["ret_count"]))
        self.norm_obs, self.norm_reward = bool(sd["norm_obs"]), bool(sd["norm_reward"])
        self.clip_obs, self.clip_reward = float(sd["clip_obs"]), float(sd["clip_reward"])
        self.gamma, self.epsilon = float(sd["gamma"]), float(sd["epsilon"])
        self.param_version += 1

    def save(self, path: str) -> None:
        torch.save(self.state_dict(), path)

    @staticmethod
    def load(path: str, venv) -> "VecNormalize":
        sd = torch.load(path, map_location="cpu")
        w = VecNormalize(venv, norm_obs=sd["norm_obs"], norm_reward=sd["norm_reward"], clip_obs=sd["clip_obs"],
                         clip_reward=sd["clip_reward"], gamma=sd["gamma"], epsilon=sd["epsilon"])
        w.load_state_dict(sd)
        return w

    def share_statistics(self, other: "VecNormalize") -> None:
        """Read (and, in training mode, update) ``other``'s statistics tensors instead of this wrapper's own."""
        if tuple(other.obs_rms.shape) != tuple(self.obs_rms.shape):
            raise ValueError("share_statistics: observation shapes differ")
        self.obs_rms, self.ret_rms = other.obs_rms, other.ret_rms
        self.param_version += 1
