"""E lock-step highway-v0 (or highway-fast-v0) episodes on one GPU, behind ``libhrp_b200.so``.

This is the batched counterpart of what the reference obtains from
``gym.make("highway-v0", config=cfg)`` (``experiments/wrappers.py:80``) plus the observation
wrapper around it (``wrappers.py:100-104``): one kernel launch advances every env by one
policy step (15 simulation frames), computes reward / terminated / truncated, respawns the envs
that finished (the reference resets right after ``done``, ``training/routine.py:125-127``) and
writes the Kinematics observation with the RoPE / DistPE / RankPE embedding already applied.

All tensors are torch CUDA tensors owned by the caller; the simulator state itself lives in
the library handle as struct-of-arrays in HBM.  There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Any, Dict, Optional, Sequence

import numpy as np
import torch

from .. import _lib
from .._lib import EMBED_DIST, EMBED_NONE, EMBED_RANK, EMBED_ROPE, FEATURE_CODES, HrpCfg, HrpState

# HighwayEnv.default_config() entries the reference config does not override (SURVEY.md A.1)
ENV_DEFAULTS: Dict[str, Any] = {
    "lanes_count": 4, "vehicles_count": 50, "controlled_vehicles": 1, "initial_lane_id": None,
    "duration": 40, "ego_spacing": 2, "vehicles_density": 1, "collision_reward": -1,
    "right_lane_reward": 0.1, "high_speed_reward": 0.4, "lane_change_reward": 0,
    "reward_speed_range": [20, 30], "normalize_reward": True, "offroad_terminal": False,
    "simulation_frequency": 15, "policy_frequency": 1,
    "other_vehicles_type": "highway_env.vehicle.behavior.IDMVehicle",
}
# HighwayEnvFast.default_config(): HighwayEnv's updated with these (highway-env 1.10.1).  The variant also switches off
# collision checks between uncontrolled vehicles (hrp_cfg.ego_collisions_only; DESIGN.md Appendix C).
FAST_ENV_DEFAULTS: Dict[str, Any] = dict(ENV_DEFAULTS, simulation_frequency=5, lanes_count=3, vehicles_count=20,
                                         duration=30, ego_spacing=1.5)
# the config key "gym_id" (this package's key: upstream ignores unknown keys) selects the env id
ENV_IDS: Dict[str, Dict[str, Any]] = {"highway-v0": ENV_DEFAULTS, "highway-fast-v0": FAST_ENV_DEFAULTS}
OBS_DEFAULTS: Dict[str, Any] = {
    "type": "Kinematics", "vehicles_count": 5, "features": ["presence", "x", "y", "vx", "vy"],
    "features_range": None, "absolute": False, "order": "sorted", "normalize": True, "clip": True,
    "see_behind": False, "observe_intentions": False, "include_obstacles": True,
}
# OccupancyGridObservation's defaults (highway-env 1.10.1): features_range None means +-2 Vehicle.MAX_SPEED on vx / vy
GRID_DEFAULTS: Dict[str, Any] = {
    "type": "OccupancyGrid", "features": ["presence", "vx", "vy", "on_road"],
    "grid_size": [[-27.5, 27.5], [-27.5, 27.5]], "grid_step": [5, 5], "features_range": None,
    "absolute": False, "align_to_vehicle_axes": False, "clip": True, "as_image": False,
}
GRID_FEATURES_RANGE: Dict[str, Any] = {"vx": [-80.0, 80.0], "vy": [-80.0, 80.0]}


class EmbedSpec:
    """Which observation wrapper is fused behind the Kinematics observation."""

    def __init__(self, kind: int = EMBED_NONE, dim: int = 0, table: Optional[np.ndarray] = None,
                 max_dist: float = 100.0, use_euclidean: bool = True, ego_idx: int = 0):
        self.kind = int(kind)
        self.dim = int(dim)
        self.table = None if table is None else np.ascontiguousarray(table, dtype=np.float32).reshape(-1)
        self.max_dist = float(max_dist)
        self.use_euclidean = bool(use_euclidean)
        self.ego_idx = int(ego_idx)

    def out_features(self, F: int) -> int:
        return F + self.dim if self.kind in (EMBED_DIST, EMBED_RANK) else F


def resolve_config(cfg: Dict[str, Any]) -> Dict[str, Any]:
    """The ``default_config()`` of ``cfg["gym_id"]`` (``"highway-v0"`` when absent, or ``"highway-fast-v0"``)
    shallow-updated by ``cfg`` (highway-env's ``configure``), observation kwargs completed with KinematicObservation's
    defaults.  The resolved dict keeps ``gym_id``.  Another id is a ``ValueError``."""
    gym_id = cfg.get("gym_id", "highway-v0")
    if gym_id not in ENV_IDS:
        raise ValueError(f"gym_id {gym_id!r} is not implemented; accepted ids: {', '.join(map(repr, ENV_IDS))}")
    full = dict(ENV_IDS[gym_id])
    full.update(cfg)
    full["gym_id"] = gym_id
    user_obs = full.get("observation") or {}
    # the observation class follows its type: OccupancyGrid takes its own defaults (the keys a Kinematics base config
    # leaves behind, vehicles_count, order, normalize ..., are ignored by it as upstream's **kwargs are)
    obs = dict(GRID_DEFAULTS if user_obs.get("type") == "OccupancyGrid" else OBS_DEFAULTS)
    obs.update(user_obs)
    full["observation"] = obs
    full.setdefault("action", {"type": "DiscreteMetaAction"})
    return full


def build_cfg(cfg: Dict[str, Any], embed: Optional[EmbedSpec] = None, autoreset: bool = True) -> HrpCfg:
    """highway-env style config dict -> ``hrp_cfg``.  Raises ``ValueError`` for what the kernels
    do not implement (Kinematics and OccupancyGrid observations, IDM traffic, one controlled vehicle)."""
    full = resolve_config(cfg)
    obs, act = full["observation"], full["action"]
    if obs.get("type", "Kinematics") not in ("Kinematics", "OccupancyGrid"):
        raise ValueError(f"observation type {obs.get('type')!r} is not implemented (Kinematics and OccupancyGrid only)")
    if act.get("type") not in ("ContinuousAction", "DiscreteMetaAction"):
        raise ValueError(f"action type {act.get('type')!r} is not implemented")
    if act.get("type") == "ContinuousAction" and not (act.get("longitudinal", True) and act.get("lateral", True)):
        raise ValueError("ContinuousAction needs longitudinal=True and lateral=True (reference config)")
    if int(full.get("controlled_vehicles", 1)) != 1:
        raise ValueError("exactly one controlled vehicle per env is supported")
    grid = obs["type"] == "OccupancyGrid"
    if not grid and obs.get("order", "sorted") not in ("sorted", "shuffled"):
        raise ValueError(f"observation order {obs.get('order')!r} must be 'sorted' or 'shuffled'")
    c = HrpCfg()
    c.lanes_count = int(full["lanes_count"])
    c.vehicles_count = int(full["vehicles_count"])
    c.simulation_frequency = int(full["simulation_frequency"])
    c.policy_frequency = int(full["policy_frequency"])
    c.initial_lane_id = -1 if full["initial_lane_id"] is None else int(full["initial_lane_id"])
    c.ego_mode = 0 if act["type"] == "ContinuousAction" else 1
    c.normalize_reward = int(bool(full["normalize_reward"]))
    c.offroad_terminal = int(bool(full["offroad_terminal"]))
    c.duration = float(full["duration"])
    c.ego_spacing = float(full["ego_spacing"])
    c.vehicles_density = float(full["vehicles_density"])
    c.collision_reward = float(full["collision_reward"])
    c.right_lane_reward = float(full["right_lane_reward"])
    c.high_speed_reward = float(full["high_speed_reward"])
    c.reward_speed_lo, c.reward_speed_hi = (float(v) for v in full["reward_speed_range"])
    c.autoreset = int(bool(autoreset))
    c.ego_collisions_only = int(full["gym_id"] == "highway-fast-v0")
    if grid:
        if embed is not None and embed.kind != EMBED_NONE:
            raise ValueError("an OccupancyGrid observation takes no embedding")
        _grid_cfg(c, obs)
        return c
    feats = list(obs["features"])
    if len(feats) > _lib.HRP_MAX_FEATURES:
        raise ValueError(f"at most {_lib.HRP_MAX_FEATURES} features are supported")
    if "on_road" in feats:
        raise ValueError("feature 'on_road' is an OccupancyGrid layer; a Kinematics observation has no such column")
    c.obs_vehicles = int(obs["vehicles_count"])
    c.obs_nfeat = len(feats)
    width = 4.0 * c.lanes_count
    ranges = obs.get("features_range") or {"x": [-200.0, 200.0], "y": [-width, width],
                                           "vx": [-80.0, 80.0], "vy": [-80.0, 80.0]}
    for i, name in enumerate(feats):
        if name not in FEATURE_CODES:
            raise ValueError(f"feature {name!r} is not implemented; known: {sorted(FEATURE_CODES)}")
        c.obs_feat[i] = FEATURE_CODES[name]
        if name in ranges:
            c.obs_has_range[i] = 1
            c.obs_lo[i], c.obs_hi[i] = float(ranges[name][0]), float(ranges[name][1])
    c.obs_normalize = int(bool(obs["normalize"]))
    c.obs_clip = int(bool(obs["clip"]))
    c.obs_absolute = int(bool(obs["absolute"]))
    c.obs_sorted = int(obs["order"] == "sorted")
    c.obs_see_behind = int(bool(obs["see_behind"]))
    e = embed or EmbedSpec()
    c.embed_kind, c.embed_dim = e.kind, e.dim
    c.embed_use_euclidean = int(e.use_euclidean)
    c.embed_max_dist = e.max_dist
    c.embed_ego_idx = e.ego_idx
    return c


def grid_shape(obs: Dict[str, Any]):
    """(W, H) of an OccupancyGrid config: ``floor((size[a][1] - size[a][0]) / step[a])`` in fp64."""
    size, step = obs["grid_size"], obs["grid_step"]
    return tuple(int(math.floor((float(size[a][1]) - float(size[a][0])) / float(step[a]))) for a in range(2))


def _grid_cfg(c: HrpCfg, obs: Dict[str, Any]) -> None:
    """The OccupancyGrid fields of ``hrp_cfg`` (``obs`` resolved); ``ValueError`` for what the kernel does not do."""
    if obs.get("absolute"):
        raise ValueError("OccupancyGrid absolute=True is not implemented (upstream raises NotImplementedError)")
    if obs.get("as_image"):
        raise ValueError("OccupancyGrid as_image=True is not implemented")
    feats = list(obs["features"])
    if not 1 <= len(feats) <= _lib.HRP_MAX_FEATURES:
        raise ValueError(f"an OccupancyGrid takes 1 to {_lib.HRP_MAX_FEATURES} features, got {len(feats)}")
    size, step = obs["grid_size"], obs["grid_step"]
    if len(size) != 2 or any(len(r) != 2 for r in size) or len(step) != 2:
        raise ValueError(f"grid_size must be [[x0, x1], [y0, y1]] and grid_step [sx, sy]; got {size}, {step}")
    if not all(float(s) > 0 and math.isfinite(float(s)) for s in step):
        raise ValueError(f"grid_step must be positive, got {step}")
    W, H = grid_shape(obs)
    if W < 1 or H < 1 or len(feats) * W * H > _lib.HRP_MAX_GRID_VALUES:
        raise ValueError(f"grid of {len(feats)} x {W} x {H} outside 1 <= W, H and F x W x H <= {_lib.HRP_MAX_GRID_VALUES}")
    ranges = obs.get("features_range") or GRID_FEATURES_RANGE   # a user dict replaces the default entirely
    c.obs_type = _lib.OBS_OCCUPANCY_GRID
    c.obs_nfeat = len(feats)
    for i, name in enumerate(feats):
        if name not in FEATURE_CODES:
            raise ValueError(f"feature {name!r} is not implemented; known: {sorted(FEATURE_CODES)}")
        c.obs_feat[i] = FEATURE_CODES[name]
        if name in ranges and name != "on_road":
            c.obs_has_range[i] = 1
            c.obs_lo[i], c.obs_hi[i] = float(ranges[name][0]), float(ranges[name][1])
    c.obs_clip = int(bool(obs["clip"]))
    c.grid_align = int(bool(obs["align_to_vehicle_axes"]))
    for a in range(2):
        c.grid_lo[a], c.grid_hi[a] = float(size[a][0]), float(size[a][1])
        c.grid_step[a] = float(step[a])


class HighwayVecEnv:
    """``num_envs`` highway-v0 episodes (highway-fast-v0 with ``cfg["gym_id"]``) stepped in lock-step on ``device``.

    ``env_id_base`` is the global id of this shard's first env: spawn and shuffle draws are a
    function of (seed, global env id, episode), so a run sharded over G GPUs sees the same
    episodes as the single-GPU run (SURVEY.md 8e).
    """

    _next_uid = 0

    def __init__(self, cfg: Dict[str, Any], num_envs: int, device: Any = "cuda", embed: Optional[EmbedSpec] = None,
                 autoreset: bool = True, env_id_base: int = 0, seed: int = 0, real64: bool = False):
        # real64: the fp64 VALIDATION instantiation of the kernels (HRP_ENV_REAL64; parity tests only, slow)
        # the configuration is checked first: an unknown gym_id or observation is a ValueError before any device work
        self.config = resolve_config(cfg)
        self.embed = embed or EmbedSpec()
        self.cfg = build_cfg(cfg, self.embed, autoreset)
        lib = _lib.load()
        _lib.require_device()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.HrpError("HighwayVecEnv needs a CUDA device: there is no CPU path")
        self.dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", self.dev_index)
        self.num_envs = int(num_envs)
        self.seed = int(seed)
        table = self.embed.table
        tptr = None if table is None else table.ctypes.data
        h = C.c_void_p()
        self.real64 = bool(real64)
        self.env_id_base = int(env_id_base)
        _lib.check(lib.hrp_env_create_ex(C.byref(self.cfg), tptr, 0 if table is None else table.size, self.num_envs,
                                         int(env_id_base), self.dev_index, 1 if self.real64 else 0, C.byref(h)),
                   "hrp_env_create_ex")
        self._h = h
        self._lib = lib
        self.V = int(lib.hrp_env_num_vehicles(h))
        rows, cols = C.c_int32(), C.c_int32()
        _lib.check(lib.hrp_env_obs_dim(h, C.byref(rows), C.byref(cols)), "hrp_env_obs_dim")
        # rows x cols: N x F_out for Kinematics, F x (W * H) for a grid, so that every N * F_out consumer sizes both
        self.N, self.F_out = int(rows.value), int(cols.value)
        self.F = int(self.cfg.obs_nfeat)
        self.grid = self.cfg.obs_type == _lib.OBS_OCCUPANCY_GRID
        self._obs_shape = (self.N, self.F_out)
        if self.grid:
            f, w, hh = C.c_int32(), C.c_int32(), C.c_int32()
            _lib.check(lib.hrp_env_grid_shape(h, C.byref(f), C.byref(w), C.byref(hh)), "hrp_env_grid_shape")
            self._obs_shape = (int(f.value), int(w.value), int(hh.value))
        E = self.num_envs
        self.obs = torch.zeros((E,) + self._obs_shape, dtype=torch.float32, device=self.device)
        self.reward = torch.zeros(E, dtype=torch.float32, device=self.device)
        self.terminated = torch.zeros(E, dtype=torch.uint8, device=self.device)
        self.truncated = torch.zeros(E, dtype=torch.uint8, device=self.device)
        self.launches = 0  # kernels of this library enqueued through this handle
        # identity of this handle for caches of captured launches (training/routine.py): id() of a closed env can be
        # handed to a new one, a counter cannot
        HighwayVecEnv._next_uid += 1
        self.uid = HighwayVecEnv._next_uid
        # a launch passes the handle's parameters (seed, per-env seeds, step mask, trace) by value, so a captured launch
        # keeps the ones of its capture: every change of them bumps this version, and caches of captured launches
        # compare it
        self.param_version = 0

    # ------------------------------------------------------------------ lifetime
    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.hrp_env_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @property
    def obs_shape(self):
        """(N, F_out) for Kinematics, (F, W, H) for an OccupancyGrid."""
        return self._obs_shape

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # ------------------------------------------------------------------ stepping
    def reset(self, seed: Optional[int] = None, mask: Optional[torch.Tensor] = None,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``env.reset(seed=...)`` for every env (or those with a non-zero ``mask`` byte)."""
        if seed is not None:
            self._set_seed(seed)
        obs = self.obs if out is None else out
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self._lib.hrp_env_reset(self._h, self.seed & 0xFFFFFFFFFFFFFFFF, _lib.ptr(mask), obs.data_ptr(),
                                           self._stream()), "hrp_env_reset")
        self.launches += 1
        return obs

    def step(self, actions: torch.Tensor, perm: Optional[torch.Tensor] = None,
             row_vehicle: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
             reward_out: Optional[torch.Tensor] = None, terminated_out: Optional[torch.Tensor] = None,
             truncated_out: Optional[torch.Tensor] = None, final_obs_out: Optional[torch.Tensor] = None):
        """One policy step of every env.  ``actions``: float32 [E, 2] on the device.

        Returns (obs [E,N,F_out] -- [E,F,W,H] for a grid --, reward [E], terminated [E] uint8, truncated [E] uint8); the
        tensors are the handle's own output buffers unless ``out`` (observation) / ``reward_out`` /
        ``terminated_out`` / ``truncated_out`` name the caller's (contiguous, e.g. the slot of a rollout buffer: the
        kernel then writes the rollout directly, no copy kernels between the step and the next policy forward).

        ``final_obs_out`` (contiguous float32 CUDA tensor of E x N x F_out, not ``out``): every env whose episode ended
        on this step writes the observation of its terminal state there, before the respawn (``hrp_env_step_final``);
        the other rows are left as they are.
        """
        if actions.device != self.device or actions.dtype != torch.float32 or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.float32).contiguous()
        if actions.numel() != 2 * self.num_envs:
            raise ValueError(f"actions must hold {self.num_envs} x 2 floats, got shape {tuple(actions.shape)}")
        obs = self.obs if out is None else out
        if perm is not None:
            if self.grid:
                raise ValueError("perm: an OccupancyGrid observation has no row order")
            perm = perm.to(device=self.device, dtype=torch.int32).contiguous()
            if perm.numel() != self.num_envs * (self.N - 1):
                raise ValueError("perm must be [E, N-1]")
        rew = self.reward if reward_out is None else reward_out
        term = self.terminated if terminated_out is None else terminated_out
        trunc = self.truncated if truncated_out is None else truncated_out
        if final_obs_out is None:
            _lib.check(self._lib.hrp_env_step(self._h, actions.data_ptr(), obs.data_ptr(), rew.data_ptr(),
                                              term.data_ptr(), trunc.data_ptr(), _lib.ptr(perm),
                                              _lib.ptr(row_vehicle), self._stream()), "hrp_env_step")
        else:
            if (not final_obs_out.is_cuda or final_obs_out.dtype != torch.float32 or not final_obs_out.is_contiguous()
                    or final_obs_out.numel() != obs.numel()):
                raise ValueError(f"final_obs_out must be a contiguous float32 CUDA tensor of {self.num_envs} x "
                                 f"{self.N} x {self.F_out}")
            _lib.check(self._lib.hrp_env_step_final(self._h, actions.data_ptr(), obs.data_ptr(), rew.data_ptr(),
                                                    term.data_ptr(), trunc.data_ptr(), final_obs_out.data_ptr(),
                                                    _lib.ptr(perm), _lib.ptr(row_vehicle), self._stream()),
                       "hrp_env_step_final")
        self.launches += 1
        return obs, rew, term, trunc

    def observe(self, perm: Optional[torch.Tensor] = None, row_vehicle: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
        obs = self.obs if out is None else out
        if perm is not None:
            perm = perm.to(device=self.device, dtype=torch.int32).contiguous()
        _lib.check(self._lib.hrp_env_observe(self._h, obs.data_ptr(), _lib.ptr(perm), _lib.ptr(row_vehicle),
                                             self._stream()), "hrp_env_observe")
        self.launches += 1
        return obs

    # host-buffer entry points (what a CPU training loop binds): numpy in, numpy out
    def step_host(self, actions, obs: np.ndarray, reward: np.ndarray, terminated: np.ndarray,
                  truncated: np.ndarray) -> None:
        """Host-buffer step: results land in the numpy arrays.  ``actions`` is a numpy array, or a CUDA tensor
        produced on the current stream (the policy's device output: no host round trip, no extra synchronisation)."""
        if isinstance(actions, torch.Tensor) and actions.is_cuda:
            a = actions.contiguous()
            if a.dtype != torch.float32 or a.numel() != 2 * self.num_envs:
                raise ValueError(f"actions must hold {self.num_envs} x 2 float32 values")
            _lib.check(self._lib.hrp_env_step_host_on(self._h, a.data_ptr(), obs.ctypes.data, reward.ctypes.data,
                                                      terminated.ctypes.data, truncated.ctypes.data,
                                                      torch.cuda.current_stream(self.device).cuda_stream),
                       "hrp_env_step_host_on")
            self.launches += 1
            return
        a = np.ascontiguousarray(actions, dtype=np.float32)
        if a.size != 2 * self.num_envs:
            raise ValueError(f"actions must hold {self.num_envs} x 2 floats")
        _lib.check(self._lib.hrp_env_step_host(self._h, a.ctypes.data, obs.ctypes.data, reward.ctypes.data,
                                               terminated.ctypes.data, truncated.ctypes.data), "hrp_env_step_host")
        self.launches += 1

    def step_host_async(self, actions: torch.Tensor, obs: np.ndarray, reward: np.ndarray, terminated: np.ndarray,
                        truncated: np.ndarray) -> None:
        """``step_host`` without the final synchronisation: the step kernel and the device-to-host copies are
        enqueued on the current stream; the page-locked numpy buffers hold the results once that stream has reached
        this point (record an event and wait for it).  ``actions`` is a CUDA tensor produced on the same stream."""
        a = actions.contiguous()
        if not a.is_cuda or a.dtype != torch.float32 or a.numel() != 2 * self.num_envs:
            raise ValueError(f"actions must be a CUDA tensor of {self.num_envs} x 2 float32 values")
        _lib.check(self._lib.hrp_env_step_host_async(self._h, a.data_ptr(), obs.ctypes.data, reward.ctypes.data,
                                                     terminated.ctypes.data, truncated.ctypes.data,
                                                     torch.cuda.current_stream(self.device).cuda_stream),
                   "hrp_env_step_host_async")
        self.launches += 1

    def reset_host(self, seed: int, obs: np.ndarray) -> None:
        self._set_seed(seed)
        _lib.check(self._lib.hrp_env_reset_host(self._h, self.seed & 0xFFFFFFFFFFFFFFFF, obs.ctypes.data),
                   "hrp_env_reset_host")
        self.launches += 1

    def _set_seed(self, seed: int) -> None:
        if int(seed) != self.seed:
            self.seed = int(seed)
            self.param_version += 1

    # ------------------------------------------------------------------ multiplexed experiments
    def set_env_seeds(self, seeds: Optional[torch.Tensor]) -> None:
        """Per-env seeds (int64 / uint64 CUDA tensor [E], kept alive by this object): env e then behaves exactly like
        the single-env handle of an experiment that called ``reset(seed=seeds[e])``.  ``None`` switches back to
        (handle seed, global env id)."""
        self.param_version += 1
        if seeds is None:
            _lib.check(self._lib.hrp_env_set_seeds(self._h, None), "hrp_env_set_seeds")
            self._seeds = None
            return
        if not seeds.is_cuda or seeds.numel() != self.num_envs or seeds.dtype not in (torch.int64, torch.uint64):
            raise ValueError(f"seeds must be a CUDA int64 tensor of {self.num_envs} entries")
        self._seeds = seeds.contiguous()
        _lib.check(self._lib.hrp_env_set_seeds(self._h, self._seeds.data_ptr()), "hrp_env_set_seeds")

    def set_step_mask(self, mask: Optional[torch.Tensor]) -> None:
        """uint8 CUDA tensor [E] (kept alive by this object; rewrite its contents between steps): ``step`` leaves env e
        untouched unless ``mask[e]``.  ``None``: every env steps."""
        self.param_version += 1
        if mask is None:
            _lib.check(self._lib.hrp_env_set_step_mask(self._h, None), "hrp_env_set_step_mask")
            self._step_mask = None
            return
        if not mask.is_cuda or mask.numel() != self.num_envs or mask.dtype != torch.uint8:
            raise ValueError(f"mask must be a CUDA uint8 tensor of {self.num_envs} entries")
        self._step_mask = mask.contiguous()
        _lib.check(self._lib.hrp_env_set_step_mask(self._h, self._step_mask.data_ptr()), "hrp_env_set_step_mask")

    # ------------------------------------------------------------------ validation aids
    def enable_trace(self, on: bool = True) -> Optional[torch.Tensor]:
        """Record every vehicle's state at the end of every simulation frame of the following steps (parity tests):
        returns the float64 tensor [E, frames, V, 7] the kernel writes (x, y, speed, heading, impact_x, impact_y, flags)."""
        self.param_version += 1
        if not on:
            _lib.check(self._lib.hrp_env_set_trace(self._h, None), "hrp_env_set_trace")
            self._trace = None
            return None
        fr, sl, fi = C.c_int32(), C.c_int32(), C.c_int32()
        _lib.check(self._lib.hrp_env_trace_shape(self._h, C.byref(fr), C.byref(sl), C.byref(fi)), "hrp_env_trace_shape")
        self._trace = torch.zeros((self.num_envs, fr.value, sl.value, fi.value), dtype=torch.float64, device=self.device)
        _lib.check(self._lib.hrp_env_set_trace(self._h, self._trace.data_ptr()), "hrp_env_set_trace")
        return self._trace[:, :, : self.V, :]

    # ------------------------------------------------------------------ state injection
    def _state_arrays(self):
        E, V = self.num_envs, self.V
        st: Dict[str, np.ndarray] = {}
        for n in _lib.STATE_F64:
            st[n] = np.zeros((E, V), dtype=np.float64)
        for n in _lib.STATE_I32:
            st[n] = np.zeros((E, V), dtype=np.int32)
        st["time"] = np.zeros(E, dtype=np.float64)
        st["episode"] = np.zeros(E, dtype=np.uint32)
        st["obs_draw"] = np.zeros(E, dtype=np.uint32)
        return st

    @staticmethod
    def _view(st: Dict[str, np.ndarray]) -> HrpState:
        s = HrpState()
        for n in _lib.STATE_F64 + ("time",):
            setattr(s, n, st[n].ctypes.data_as(C.POINTER(C.c_double)))
        for n in _lib.STATE_I32:
            setattr(s, n, st[n].ctypes.data_as(C.POINTER(C.c_int32)))
        for n in ("episode", "obs_draw"):
            setattr(s, n, st[n].ctypes.data_as(C.POINTER(C.c_uint32)) if n in st and st[n] is not None
                    else C.POINTER(C.c_uint32)())
        return s

    def get_state(self) -> Dict[str, np.ndarray]:
        """Simulator state as numpy arrays, [E, V] per vehicle field, [E] per env field."""
        st = self._state_arrays()
        view = self._view(st)
        _lib.check(self._lib.hrp_env_get_state(self._h, C.byref(view)), "hrp_env_get_state")
        return st

    def set_state(self, state: Dict[str, Any]) -> None:
        E, V = self.num_envs, self.V
        st: Dict[str, Any] = {}
        for n in _lib.STATE_F64:
            st[n] = np.ascontiguousarray(np.asarray(state[n], dtype=np.float64).reshape(E, V))
        for n in _lib.STATE_I32:
            st[n] = np.ascontiguousarray(np.asarray(state[n], dtype=np.int32).reshape(E, V))
        st["time"] = np.ascontiguousarray(np.asarray(state["time"], dtype=np.float64).reshape(E))
        for n in ("episode", "obs_draw"):
            st[n] = (np.ascontiguousarray(np.asarray(state[n], dtype=np.uint32).reshape(E))
                     if state.get(n) is not None else None)
        view = self._view(st)
        _lib.check(self._lib.hrp_env_set_state(self._h, C.byref(view)), "hrp_env_set_state")


def embed_apply(kind: int, obs: torch.Tensor, table: torch.Tensor, embed_dim: int, max_dist: float,
                use_euclidean: bool = True, ego_idx: int = 0, dist_override: Optional[torch.Tensor] = None
                ) -> torch.Tensor:
    """``wrapper.observation(obs)`` for a batch of caller-provided observations [B, N, F] (CUDA)."""
    lib = _lib.load()
    if obs.dim() == 2:
        obs = obs.unsqueeze(0)
    obs = obs.to(dtype=torch.float32).contiguous()
    B, N, F = obs.shape
    F_out = F + embed_dim if kind in (EMBED_DIST, EMBED_RANK) else F
    out = torch.empty((B, N, F_out), dtype=torch.float32, device=obs.device)
    if dist_override is not None:
        dist_override = dist_override.to(device=obs.device, dtype=torch.float32).contiguous()
    _lib.check(lib.hrp_embed_apply(kind, embed_dim, int(use_euclidean), ego_idx, float(max_dist), _lib.ptr(table),
                                   obs.data_ptr(), out.data_ptr(), B, N, F, _lib.ptr(dist_override),
                                   torch.cuda.current_stream(obs.device).cuda_stream), "hrp_embed_apply")
    return out
