"""Episode bookkeeping of the batched loops: the ``hrp_episode_stats`` launch, the figures formed from its six sums, and
the number of policy steps after which highway-v0 truncates an episode."""
from __future__ import annotations

from typing import Dict, Optional

import torch

from .. import _lib

# order of hrp_episode_stats' sums
EPISODES, RETURN_SUM, RETURN_SQ_SUM, LENGTH_SUM, TERMINATED, TRUNCATED = range(6)


def new_stats(device) -> torch.Tensor:
    """A zeroed fp64 stats buffer: the six sums followed by the kernel's scratch."""
    return torch.zeros(_lib.EPISODE_STATS_LEN, dtype=torch.float64, device=device)


def episode_stats(reward: torch.Tensor, terminated: torch.Tensor, truncated: torch.Tensor, ret: torch.Tensor,
                  length: torch.Tensor, stats: torch.Tensor, active: Optional[torch.Tensor] = None) -> None:
    """``hrp_episode_stats`` over time-major [T, E] (or [E], T = 1) step outputs on the current stream.  ``ret`` float64
    [E] and ``length`` int32 [E] are the per-env carries, ``stats`` a ``new_stats`` buffer (accumulated into),
    ``active`` uint8 [E] selects evaluation mode.  Allocates nothing, so it can be captured in a CUDA graph."""
    E = ret.numel()
    T = reward.numel() // E
    for name, t, dt, n in (("reward", reward, torch.float32, T * E), ("terminated", terminated, torch.uint8, T * E),
                           ("truncated", truncated, torch.uint8, T * E), ("ret", ret, torch.float64, E),
                           ("length", length, torch.int32, E), ("stats", stats, torch.float64, _lib.EPISODE_STATS_LEN),
                           ("active", active, torch.uint8, E)):
        if t is None and name == "active":
            continue
        if not t.is_cuda or t.dtype != dt or t.numel() != n or not t.is_contiguous():
            raise ValueError(f"episode_stats: {name} must be a contiguous {dt} CUDA tensor of {n} elements")
    _lib.check(_lib.load().hrp_episode_stats(reward.data_ptr(), terminated.data_ptr(), truncated.data_ptr(), T, E,
                                             _lib.ptr(active), ret.data_ptr(), length.data_ptr(), stats.data_ptr(),
                                             torch.cuda.current_stream(reward.device).cuda_stream),
               "hrp_episode_stats")


def summarize(sums) -> Dict[str, float]:
    """episodes, return mean / std (population, as ``np.std``), length mean and the terminated fraction from the six
    sums (any sequence of floats; NaN where no episode finished)."""
    n = float(sums[EPISODES])
    if n <= 0:
        nan = float("nan")
        return {"episodes": 0, "return_mean": nan, "return_std": nan, "length_mean": nan, "terminated_fraction": nan}
    mean = float(sums[RETURN_SUM]) / n
    var = max(float(sums[RETURN_SQ_SUM]) / n - mean * mean, 0.0)
    return {"episodes": int(round(n)), "return_mean": mean, "return_std": var ** 0.5,
            "length_mean": float(sums[LENGTH_SUM]) / n, "terminated_fraction": float(sums[TERMINATED]) / n}


def policy_steps(duration: float, policy_frequency: int) -> int:
    """Policy steps after which highway-v0 truncates: the step kernel's own fp64 clock, ``t += 1 / policy_frequency``
    until ``t >= duration`` (40 for the default 40 s at 1 Hz, 3 for 2.5 s at 1 Hz)."""
    dt = 1.0 / int(policy_frequency)
    t, n = 0.0, 0
    while True:
        t += dt
        n += 1
        if t >= float(duration):
            return n
