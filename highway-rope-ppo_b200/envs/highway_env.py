"""Single-env, gymnasium-protocol view of the GPU simulator.

This is what ``make_env`` returns in place of ``gym.make("highway-v0", config=cfg)``
(reference ``experiments/wrappers.py:80``): the object the reference training loop drives with
``reset(seed=...)`` / ``step(action)`` (``training/routine.py:18,24,127,134``) and whose
``observation_space`` / ``action_space`` the runner inspects (``experiments/runner.py:87-98``).
It owns a one-env :class:`HighwayVecEnv` and goes through the host-buffer C-ABI entry points
(pinned staging, H2D action, fused step kernel, D2H observation).
"""
from __future__ import annotations

from typing import Any, Dict, Optional

import numpy as np

from .highway_vec import EmbedSpec, HighwayVecEnv
from .spaces import Box, Discrete

_MASK64 = 0xFFFFFFFFFFFFFFFF


class HighwayEnv:
    metadata: Dict[str, Any] = {"render_modes": []}
    render_mode = None
    spec = None

    def __init__(self, config: Dict[str, Any], device: Any = "cuda", embed: Optional[EmbedSpec] = None):
        self._user_config = config
        self._device = device
        self._seed = 0
        self._make(embed)

    def _make(self, embed: Optional[EmbedSpec]) -> None:
        self.vec = HighwayVecEnv(self._user_config, 1, device=self._device, embed=embed, autoreset=False)
        self.config = self.vec.config
        shape = self.vec.obs_shape   # (N, F_out), or (F, W, H) for an OccupancyGrid
        self.observation_space = Box(-np.inf, np.inf, shape, np.float32)
        if self.vec.cfg.ego_mode == 0:
            self.action_space = Box(-1.0, 1.0, (2,), np.float32)
        else:
            self.action_space = Discrete(5)
        self._obs = np.zeros((1,) + shape, dtype=np.float32)
        self._reward = np.zeros(1, dtype=np.float32)
        self._term = np.zeros(1, dtype=np.uint8)
        self._trunc = np.zeros(1, dtype=np.uint8)
        self._act = np.zeros((1, 2), dtype=np.float32)

    # the embed wrappers call this to have their observation() fused into the step kernel
    def _fuse_embedding(self, embed: EmbedSpec) -> None:
        self.vec.close()
        self._make(embed)

    @property
    def unwrapped(self):
        return self

    def to(self, device):
        return self

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        if seed is None:  # gymnasium: keep drawing from the current generator
            self._seed = (self._seed * 6364136223846793005 + 1442695040888963407) & _MASK64
        else:
            self._seed = int(seed) & _MASK64
        self.vec.reset_host(self._seed, self._obs)
        return self._obs[0].copy(), {}

    def step(self, action):
        if self.vec.cfg.ego_mode == 0:
            a = np.asarray(action, dtype=np.float32).reshape(-1)
            if a.size != 2:
                raise ValueError(f"action must have shape (2,), got {np.shape(action)}")
            self._act[0, :] = a
        else:
            self._act[0, 0] = float(int(action))
            self._act[0, 1] = 0.0
        self.vec.step_host(self._act, self._obs, self._reward, self._term, self._trunc)
        terminated, truncated = bool(self._term[0]), bool(self._trunc[0])
        info = {"crashed": terminated, "action": action}
        return self._obs[0].copy(), float(self._reward[0]), terminated, truncated, info

    def render(self):
        return None

    def close(self) -> None:
        self.vec.close()
