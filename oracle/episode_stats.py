"""oracle/episode_stats.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

fp64 numpy restatement of ``hrp_episode_stats``: the reference's per-episode bookkeeping (``ep_reward += reward`` in
Python floats, ``training/routine.py:143``; the first episode of each evaluation env, ``routine.py:14-29``) over the
time-major [T, E] reward / terminated / truncated buffers of the batched loop, step by step and env by env.

    for each env e that takes part (active is None, or active[e] != 0), for t in order:
        ret[e] += float(reward[t, e]); len[e] += 1
        if terminated or truncated: count the episode (terminated wins when both are set), then
            training (active is None): ret[e] = len[e] = 0
            evaluation: active[e] = 0, keep ret[e] / len[e], stop scanning e

``stats`` = [episodes, sum return, sum return^2, sum length, terminated, truncated only], summed in plain Python
floats.  The kernel sums the same terms in another (fixed) order, so its sums agree within rounding and its counts,
carries and per-env returns are exact.
"""
import numpy as np

NSTATS = 6


def episode_stats(reward, terminated, truncated, ret, length, active=None):
    """Returns (ret float64 [E], length int32 [E], active uint8 [E] or None, stats float64 [6]); the inputs are not
    modified."""
    reward = np.asarray(reward, dtype=np.float32)
    term = np.asarray(terminated).astype(bool)
    trunc = np.asarray(truncated).astype(bool)
    T, E = reward.shape
    ret = np.array(ret, dtype=np.float64).reshape(E)
    length = np.array(length, dtype=np.int32).reshape(E)
    active = None if active is None else np.array(active, dtype=np.uint8).reshape(E)
    stats = [0.0] * NSTATS
    for e in range(E):
        if active is not None and not active[e]:
            continue
        r, n = float(ret[e]), int(length[e])
        for t in range(T):
            r += float(reward[t, e])
            n += 1
            if term[t, e] or trunc[t, e]:
                stats[0] += 1.0
                stats[1] += r
                stats[2] += r * r
                stats[3] += n
                stats[4] += 1.0 if term[t, e] else 0.0
                stats[5] += 0.0 if term[t, e] else 1.0
                if active is not None:
                    active[e] = 0
                    break
                r, n = 0.0, 0
        ret[e], length[e] = r, n
    return ret, length, active, np.array(stats, dtype=np.float64)
