"""numpy restatement of SB3's ``VecNormalize`` (running observation / reward normalization) for the tests.

``RunningMeanStd`` is SB3's, moments by two-pass ``np.mean`` / ``np.var`` and Chan's merge.  ``VecNormOracle`` follows
the step order the kernels implement (envs/vec_normalize.py): inner step (autoreset observation of done envs), update
of the observation statistics, normalization with the updated statistics, the return carry and its statistics, the
reward, the terminal observations of done envs with the same statistics, the carry cleared on done."""
from __future__ import annotations

import numpy as np


class RunningMeanStd:
    def __init__(self, epsilon: float = 1e-4, shape=()):
        self.mean = np.zeros(shape, np.float64)
        self.var = np.ones(shape, np.float64)
        self.count = float(epsilon)

    def update(self, x: np.ndarray) -> None:
        x = np.asarray(x, np.float64)
        self.update_from_moments(np.mean(x, axis=0), np.var(x, axis=0), x.shape[0])

    def update_from_moments(self, batch_mean, batch_var, batch_count) -> None:
        delta = batch_mean - self.mean
        tot = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot
        m_a = self.var * self.count
        m_b = batch_var * batch_count
        m_2 = m_a + m_b + np.square(delta) * self.count * batch_count / tot
        self.mean, self.var, self.count = new_mean, m_2 / tot, batch_count + self.count


def normalize(x, rms: RunningMeanStd, clip: float, epsilon: float) -> np.ndarray:
    """clip((x - mean) / sqrt(var + epsilon), +-clip) in fp64, rounded once to float32."""
    v = (np.asarray(x, np.float64) - rms.mean) / np.sqrt(rms.var + epsilon)
    return np.clip(v, -clip, clip).astype(np.float32)


class VecNormOracle:
    def __init__(self, num_envs: int, obs_shape, training: bool = True, norm_obs: bool = True,
                 norm_reward: bool = True, clip_obs: float = 10.0, clip_reward: float = 10.0, gamma: float = 0.99,
                 epsilon: float = 1e-8):
        self.obs_rms = RunningMeanStd(shape=tuple(obs_shape))
        self.ret_rms = RunningMeanStd(shape=())
        self.returns = np.zeros(num_envs, np.float64)
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon

    def _obs(self, obs):
        return normalize(obs, self.obs_rms, self.clip_obs, self.epsilon) if self.norm_obs else np.asarray(obs, np.float32)

    def reset(self, obs):
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        self.returns[:] = 0.0
        return self._obs(obs)

    def observe(self, obs):
        return self._obs(obs)

    def step(self, obs, reward, terminated, truncated, final_obs=None):
        """(obs, reward, final_obs) after one step; ``obs`` is what the inner env returned (autoreset rows included),
        ``final_obs`` the terminal observations (rows of done envs are read)."""
        done = (np.asarray(terminated) != 0) | (np.asarray(truncated) != 0)
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        out = self._obs(obs)
        reward = np.asarray(reward, np.float32)
        if self.training and self.norm_reward:
            self.returns = self.returns * self.gamma + reward.astype(np.float64)
            self.ret_rms.update(self.returns)
        rew = (np.clip(reward.astype(np.float64) / np.sqrt(self.ret_rms.var + self.epsilon), -self.clip_reward,
                       self.clip_reward).astype(np.float32) if self.norm_reward else reward)
        fin = None
        if final_obs is not None:
            fin = np.array(final_obs, np.float32, copy=True)
            if self.norm_obs:
                fin[done] = self._obs(fin[done])
        self.returns[done] = 0.0
        return out, rew, fin
