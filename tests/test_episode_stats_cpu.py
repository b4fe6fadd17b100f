"""CPU-side checks of the episode statistics: the fp64 oracle (oracle/episode_stats.py) on hand-computed cases,
hrp_episode_stats' argument errors (checked before any launch, so no device is needed), the host rule for the number
of policy steps after which highway-v0 truncates, the figures formed from the six sums, and their all-reduce over two
gloo ranks."""
import ctypes as C
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import episode_stats as es

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    from highway_rope_ppo_b200 import _lib

    return _lib, _lib.load()


def test_symbol_is_declared_and_typed():
    from test_abi_cpu import _declared_symbols

    _l, lib = _lib()
    assert "hrp_episode_stats" in _declared_symbols() and hasattr(lib, "hrp_episode_stats")
    assert len(_l.SIGNATURES["hrp_episode_stats"][1]) == 10
    text = open(os.path.join(ROOT, "include", "hrp.h")).read()
    assert "#define HRP_EPISODE_STATS_LEN (6 + 6 * 512)" in text and _l.EPISODE_STATS_LEN == 6 + 6 * 512


def test_argument_errors_name_the_field():
    _l, lib = _lib()
    buf = (C.c_double * 16)()
    p = C.addressof(buf)
    args = dict(reward=p, terminated=p, truncated=p, T=2, E=2, active=None, ret=p, len=p, stats=p, stream=None)

    def call(**over):
        a = dict(args, **over)
        return lib.hrp_episode_stats(*a.values()), _l.last_error()

    for field, name in (("reward", "reward_dev"), ("terminated", "terminated_dev"), ("truncated", "truncated_dev"),
                        ("ret", "return_dev"), ("len", "length_dev"), ("stats", "stats_dev")):
        rc, msg = call(**{field: None})
        assert rc == -1 and name in msg, (field, msg)
    for field in ("T", "E"):
        for bad in (0, -3):
            rc, msg = call(**{field: bad})
            assert rc == -1 and f"{field} = {bad}" in msg, (field, msg)


def _u8(a):
    return np.array(a, dtype=np.uint8)


def test_oracle_episode_spanning_two_calls():
    r1 = np.array([[1.0], [2.0]], dtype=np.float32)
    ret, ln, _, st = es.episode_stats(r1, _u8([[0], [0]]), _u8([[0], [0]]), [0.0], [0])
    assert ret[0] == 3.0 and ln[0] == 2 and not st.any()
    r2 = np.array([[4.0], [8.0]], dtype=np.float32)
    ret, ln, _, st = es.episode_stats(r2, _u8([[0], [1]]), _u8([[0], [0]]), ret, ln)
    assert ret[0] == 0.0 and ln[0] == 0                     # the env respawned
    np.testing.assert_array_equal(st, [1, 15.0, 225.0, 4, 1, 0])


def test_oracle_terminated_and_truncated_on_one_step_counts_as_terminated():
    r = np.array([[1.0, 1.0], [0.5, 0.5], [2.0, 2.0]], dtype=np.float32)
    te = _u8([[0, 0], [1, 0], [0, 0]])
    tr = _u8([[0, 0], [1, 1], [1, 0]])
    ret, ln, _, st = es.episode_stats(r, te, tr, [0.0, 0.0], [0, 0])
    # env 0: (1 + 0.5) terminated+truncated, then 2 truncated; env 1: 1.5 truncated, then 2 running
    np.testing.assert_array_equal(st, [3, 1.5 + 2.0 + 1.5, 2.25 + 4.0 + 2.25, 2 + 1 + 2, 1, 2])
    np.testing.assert_array_equal(ret, [0.0, 2.0])
    np.testing.assert_array_equal(ln, [0, 1])


def test_oracle_env_that_never_finishes():
    r = np.full((5, 3), 0.25, dtype=np.float32)
    z = np.zeros((5, 3), dtype=np.uint8)
    ret, ln, _, st = es.episode_stats(r, z, z, [1.0, 0.0, 0.5], [3, 0, 1])
    np.testing.assert_array_equal(ret, [2.25, 1.25, 1.75])
    np.testing.assert_array_equal(ln, [8, 5, 6])
    assert not st.any()


def test_oracle_evaluation_mode_freezes_after_the_first_episode():
    r = np.array([[1.0, 1.0, 9.0], [2.0, 2.0, 9.0], [4.0, 4.0, 9.0]], dtype=np.float32)
    te = _u8([[1, 0, 1], [0, 0, 0], [1, 0, 0]])
    tr = _u8([[0, 0, 0], [0, 1, 0], [0, 0, 0]])
    active = _u8([1, 1, 0])                                 # env 2 finished before this call: not read
    ret, ln, act, st = es.episode_stats(r, te, tr, [0.0, 0.0, 7.0], [0, 0, 3], active)
    np.testing.assert_array_equal(act, [0, 0, 0])
    np.testing.assert_array_equal(ret, [1.0, 3.0, 7.0])     # env 0's second episode is not played into it
    np.testing.assert_array_equal(ln, [1, 2, 3])
    np.testing.assert_array_equal(st, [2, 4.0, 10.0, 3, 1, 1])
    # a frozen env stays frozen
    ret2, ln2, act2, st2 = es.episode_stats(r, te, tr, ret, ln, act)
    np.testing.assert_array_equal(ret2, ret)
    np.testing.assert_array_equal(ln2, ln)
    assert not st2.any() and not act2.any()


def test_oracle_T1_matches_one_call_over_T():
    rng = np.random.default_rng(0)
    T, E = 9, 6
    r = rng.normal(size=(T, E)).astype(np.float32)
    te = (rng.random((T, E)) < 0.2).astype(np.uint8)
    tr = (rng.random((T, E)) < 0.2).astype(np.uint8)
    for active in (None, np.ones(E, dtype=np.uint8)):
        whole = es.episode_stats(r, te, tr, np.zeros(E), np.zeros(E), active)
        ret, ln, act, tot = np.zeros(E), np.zeros(E, dtype=np.int32), active, np.zeros(6)
        for t in range(T):
            ret, ln, act, st = es.episode_stats(r[t:t + 1], te[t:t + 1], tr[t:t + 1], ret, ln, act)
            tot += st
        np.testing.assert_array_equal(ret, whole[0])
        np.testing.assert_array_equal(ln, whole[1])
        np.testing.assert_array_equal(tot[[0, 3, 4, 5]], whole[3][[0, 3, 4, 5]])
        np.testing.assert_allclose(tot, whole[3], rtol=1e-12)


# (10, 15): 150 fp64 additions of 1/15 fall short of 10, so the time limit comes one step later than 10 * 15
@pytest.mark.parametrize("duration,freq,want", [(40, 1, 40), (2.5, 1, 3), (3, 2, 6), (5, 1, 5), (1, 3, 3),
                                                (0.7, 10, 7), (0.3, 10, 3), (10, 15, 151)])
def test_policy_steps_follow_the_step_kernels_clock(duration, freq, want):
    from highway_rope_ppo_b200.training.episodes import policy_steps

    assert policy_steps(duration, freq) == want
    # the rule itself: the first n with n additions of 1/freq >= duration (fp64, as the kernel accumulates)
    t, n = 0.0, 0
    while t < duration:
        t += 1.0 / freq
        n += 1
    assert n == want


def test_summarize():
    from highway_rope_ppo_b200.training.episodes import summarize

    x = np.array([3.0, 5.0, 10.0])
    s = summarize([3, x.sum(), (x * x).sum(), 12, 1, 2])
    assert s["episodes"] == 3 and abs(s["return_mean"] - x.mean()) < 1e-12 and abs(s["return_std"] - x.std()) < 1e-12
    assert s["length_mean"] == 4.0 and abs(s["terminated_fraction"] - 1 / 3) < 1e-15
    empty = summarize([0, 0, 0, 0, 0, 0])
    assert empty["episodes"] == 0 and np.isnan(empty["return_mean"])


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _data():
    rng = np.random.default_rng(5)
    T, E = 40, 64
    r = rng.normal(size=(T, E)).astype(np.float32)
    te = (rng.random((T, E)) < 0.05).astype(np.uint8)
    tr = (rng.random((T, E)) < 0.05).astype(np.uint8)
    return r, te, tr


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from highway_rope_ppo_b200.ppo import distributed as D

    r, te, tr = _data()
    base, per = D.shard_envs(r.shape[1], D.rank(), D.world_size())
    sl = slice(base, base + per)
    _, _, _, st = es.episode_stats(r[:, sl], te[:, sl], tr[:, sl], np.zeros(per), np.zeros(per))
    sums = torch.from_numpy(st)
    D.allreduce_sum_(sums)
    torch.save(sums, os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


@pytest.mark.timeout(120)
def test_two_rank_allreduce_equals_single_process_sums(tmp_path):
    from highway_rope_ppo_b200.training.episodes import summarize

    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    r, te, tr = _data()
    E = r.shape[1]
    _, _, _, want = es.episode_stats(r, te, tr, np.zeros(E), np.zeros(E))
    assert want[0] > 0
    for rank in range(world):
        got = torch.load(tmp_path / f"r{rank}.pt").numpy()
        np.testing.assert_array_equal(got[[0, 3, 4, 5]], want[[0, 3, 4, 5]])
        np.testing.assert_allclose(got, want, rtol=1e-12)
        for k, v in summarize(got).items():
            assert abs(v - summarize(want)[k]) <= 1e-12 * max(1.0, abs(v)), k
