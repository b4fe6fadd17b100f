"""oracle/gae_bootstrap.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

fp64 numpy restatement of GAE with time-limit bootstrapping, what ``hrp_gae_ex`` computes for
``collect_rollout(bootstrap_truncated=True)``.  This is the standard formulation (a truncated step is bootstrapped
with V(s_final), a terminated one is not); the reference has no such path -- it treats truncation as termination
(``ppo_ref.gae``) -- so there is no reference fixture to pin this module to.  ``tests/test_final_obs_cpu.py`` checks
it by hand on a small case and against ``ppo_ref.gae`` where nothing is truncated.

Per (t, e), fp64 arithmetic, float32 store of every advantage (as ``ppo_ref.gae``):
    term = terminated; trunc = truncated and not terminated; done = term or trunc
    boot = final_value if trunc else (0 if done else V_{t+1})
    delta = r + gamma * boot - V_t;  A_t = delta + gamma * lam * (1 - done) * A_{t+1}
"""
import numpy as np


def gae(reward, value, terminated, truncated, final_value, last_value, gamma=0.99, lam=0.95):
    """[T, E] (or [T]) arrays; last_value [E] (or a scalar).  Returns (advantages float32, returns float32)."""
    reward = np.asarray(reward, dtype=np.float64)
    value32 = np.asarray(value, dtype=np.float32)
    value = value32.astype(np.float64)
    term = np.asarray(terminated).astype(bool)
    trunc = np.asarray(truncated).astype(bool) & ~term
    done = term | trunc
    final_value = None if final_value is None else np.asarray(final_value, dtype=np.float32).astype(np.float64)
    T = reward.shape[0]
    next_v = np.broadcast_to(np.asarray(last_value, dtype=np.float32).astype(np.float64), reward.shape[1:]).copy()
    adv = np.zeros(reward.shape, dtype=np.float32)
    last = np.zeros(reward.shape[1:], dtype=np.float32)
    for t in reversed(range(T)):
        if final_value is None:
            boot = np.where(done[t], 0.0, next_v)
        else:
            boot = np.where(trunc[t], final_value[t], np.where(done[t], 0.0, next_v))
        delta = reward[t] + gamma * boot - value[t]
        adv[t] = (delta + gamma * lam * (1.0 - done[t]) * last.astype(np.float64)).astype(np.float32)
        last = adv[t]
        next_v = value[t]
    return adv, adv + value32
