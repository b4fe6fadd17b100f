"""CPU checks of running observation / reward normalization: the numpy restatement of SB3's VecNormalize
(tests/vecnormalize_oracle.py) on values worked out by hand, the configuration errors of ``VecNormalize`` and the
argument errors of the ``hrp_vecnorm_*`` entry points that are reachable without a device."""
import math

import numpy as np
import pytest

from vecnormalize_oracle import RunningMeanStd, VecNormOracle, normalize


def test_running_mean_std_from_the_epsilon_count():
    rms = RunningMeanStd(shape=(2,))
    assert rms.count == 1e-4 and np.all(rms.mean == 0) and np.all(rms.var == 1)
    rms.update(np.array([[1.0, 10.0], [3.0, 10.0]]))
    # batch mean (2, 10), population var (1, 0), n = 2; tot = 2.0001
    tot = 2.0001
    np.testing.assert_allclose(rms.mean, [2.0 * 2 / tot, 10.0 * 2 / tot], rtol=1e-15)
    want_var = [(1e-4 + 1.0 * 2 + 4.0 * 1e-4 * 2 / tot) / tot, (1e-4 + 0.0 + 100.0 * 1e-4 * 2 / tot) / tot]
    np.testing.assert_allclose(rms.var, want_var, rtol=1e-15)
    assert rms.count == tot


def test_two_updates_equal_one_update_of_the_concatenation():
    rng = np.random.default_rng(0)
    a, b = rng.normal(3, 2, (50, 7)), rng.normal(-1, 5, (31, 7))
    one, two = RunningMeanStd(shape=(7,)), RunningMeanStd(shape=(7,))
    two.update(a)
    two.update(b)
    one.update(np.concatenate([a, b]))
    np.testing.assert_allclose(two.mean, one.mean, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(two.var, one.var, rtol=1e-12)
    assert math.isclose(two.count, one.count, rel_tol=1e-15)


def test_return_carry_and_its_reset_on_terminated_and_truncated():
    o = VecNormOracle(3, (1,), norm_obs=False, gamma=0.5)
    z = np.zeros((3, 1), np.float32)
    o.step(z, [1.0, 1.0, 1.0], [0, 0, 0], [0, 0, 0])
    np.testing.assert_array_equal(o.returns, [1.0, 1.0, 1.0])
    o.step(z, [2.0, 2.0, 2.0], [1, 0, 0], [0, 1, 0])
    np.testing.assert_array_equal(o.returns, [0.0, 0.0, 2.5])   # done envs cleared after the statistics saw 2.5
    assert math.isclose(o.ret_rms.mean, (1e-4 * 0 + 3 * 1.0) / 3.0001 + (2.5 - 3 / 3.0001) * 3 / 6.0001, rel_tol=1e-12)
    o.step(z, [4.0, 4.0, 4.0], [0, 0, 0], [0, 0, 0])
    np.testing.assert_array_equal(o.returns, [4.0, 4.0, 5.25])


def test_clipping_at_plus_minus_clip():
    rms = RunningMeanStd(shape=(3,))
    out = normalize(np.array([[100.0, -100.0, 0.5]]), rms, 10.0, 1e-8)
    assert out[0, 0] == np.float32(10.0) and out[0, 1] == np.float32(-10.0)
    assert out[0, 2] == np.float32(0.5 / math.sqrt(1 + 1e-8))
    o = VecNormOracle(2, (1,), norm_obs=False, clip_reward=0.25)
    _, rew, _ = o.step(np.zeros((2, 1), np.float32), [5.0, -5.0], [0, 0], [0, 0])
    np.testing.assert_array_equal(rew, np.float32([0.25, -0.25]))


def test_terminal_observation_normalized_with_the_post_update_statistics():
    rng = np.random.default_rng(1)
    o = VecNormOracle(4, (2, 3))
    o.reset(rng.normal(size=(4, 2, 3)))
    obs, fin = rng.normal(size=(4, 2, 3)).astype(np.float32), rng.normal(size=(4, 2, 3)).astype(np.float32)
    out, _, got_fin = o.step(obs, np.ones(4, np.float32), [1, 0, 0, 0], [0, 0, 1, 0], final_obs=fin)
    np.testing.assert_array_equal(out, normalize(obs, o.obs_rms, 10.0, 1e-8))
    for e in (0, 2):
        np.testing.assert_array_equal(got_fin[e], normalize(fin[e], o.obs_rms, 10.0, 1e-8))
    for e in (1, 3):
        np.testing.assert_array_equal(got_fin[e], fin[e])


def test_training_false_changes_nothing():
    rng = np.random.default_rng(2)
    o = VecNormOracle(5, (4,), training=False)
    o.obs_rms.mean[:] = 1.0
    o.ret_rms.var = 4.0
    before = (o.obs_rms.mean.copy(), o.obs_rms.var.copy(), o.obs_rms.count, o.ret_rms.mean, o.ret_rms.var,
              o.ret_rms.count)
    o.reset(rng.normal(size=(5, 4)))
    _, rew, _ = o.step(rng.normal(size=(5, 4)), np.full(5, 3.0, np.float32), [0] * 5, [0] * 5)
    after = (o.obs_rms.mean, o.obs_rms.var, o.obs_rms.count, o.ret_rms.mean, o.ret_rms.var, o.ret_rms.count)
    for x, y in zip(before, after):
        np.testing.assert_array_equal(x, y)
    np.testing.assert_array_equal(o.returns, 0.0)
    np.testing.assert_array_equal(rew, np.float32(3.0 / math.sqrt(4.0 + 1e-8)))


class _FakeEnv:
    """The attributes VecNormalize reads before any device work."""
    num_envs, N, F_out, obs_shape = 4, 5, 5, (5, 5)
    device = "cpu"

    def step(self, *a, **k):
        raise AssertionError("no device work expected")

    reset = observe = step


@pytest.mark.parametrize("kw,msg", [
    ({"clip_obs": 0.0}, "clip_obs"), ({"clip_obs": float("inf")}, "clip_obs"), ({"clip_obs": float("nan")}, "clip_obs"),
    ({"clip_reward": -1.0}, "clip_reward"), ({"clip_reward": float("inf")}, "clip_reward"),
    ({"gamma": 1.5}, "gamma"), ({"gamma": -0.1}, "gamma"), ({"gamma": float("nan")}, "gamma"),
    ({"epsilon": -1e-8}, "epsilon"), ({"epsilon": float("inf")}, "epsilon"),
])
def test_configuration_errors(kw, msg):
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize

    with pytest.raises(ValueError, match=msg):
        VecNormalize(_FakeEnv(), **kw)


def test_venv_errors():
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize

    with pytest.raises(ValueError, match="HighwayVecEnv"):
        VecNormalize(object())
    fake = VecNormalize.__new__(VecNormalize)
    with pytest.raises(ValueError, match="already a VecNormalize"):
        VecNormalize(fake)


def test_set_step_mask_in_training_mode_is_an_error():
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize

    w = VecNormalize.__new__(VecNormalize)
    w._training = True
    with pytest.raises(ValueError, match="training=False"):
        w.set_step_mask(object())


def test_masked_reset_in_training_mode_is_an_error():
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize

    w = VecNormalize.__new__(VecNormalize)
    w._training = True
    w.venv = _FakeEnv()   # its reset raises if it is reached: the check comes before any device work
    with pytest.raises(ValueError, match="training=False"):
        w.reset(mask=object())


def _err():
    from highway_rope_ppo_b200 import _lib

    return _lib.last_error()


def test_abi_argument_errors():
    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    p = 256   # a non-null stand-in: every call below fails its checks before any launch
    cases = [
        (lambda: lib.hrp_vecnorm_moments(p, 0, 60, None, None, 0.99, p, p, None), "E = 0"),
        (lambda: lib.hrp_vecnorm_moments(p, (1 << 24) + 1, 60, None, None, 0.99, p, p, None), "E = "),
        (lambda: lib.hrp_vecnorm_moments(p, 4, 4609, None, None, 0.99, p, p, None), "S = 4609"),
        (lambda: lib.hrp_vecnorm_moments(p, 4, -1, None, None, 0.99, p, p, None), "S = -1"),
        (lambda: lib.hrp_vecnorm_moments(None, 4, 60, None, None, 0.99, p, p, None), "obs_dev"),
        (lambda: lib.hrp_vecnorm_moments(None, 4, 0, None, None, 0.99, p, p, None), "no column"),
        (lambda: lib.hrp_vecnorm_moments(p, 4, 60, p, None, 0.99, p, p, None), "returns_dev"),
        (lambda: lib.hrp_vecnorm_moments(p, 4, 60, None, None, 0.99, None, p, None), "moments_dev"),
        (lambda: lib.hrp_vecnorm_moments(p, 4, 60, None, None, 0.99, p, None, None), "scratch_dev"),
        (lambda: lib.hrp_vecnorm_moments(p, 4, 60, p, p, 1.01, p, p, None), "gamma"),
        (lambda: lib.hrp_vecnorm_moments(p, 4, 60, p, p, float("nan"), p, p, None), "gamma"),
        (lambda: lib.hrp_vecnorm_merge(p, 0, 60, 1, p, p, p, None), "R = 0"),
        (lambda: lib.hrp_vecnorm_merge(p, 1, 4609, 1, p, p, p, None), "S = 4609"),
        (lambda: lib.hrp_vecnorm_merge(p, 1, 60, 2, p, p, p, None), "has_ret"),
        (lambda: lib.hrp_vecnorm_merge(p, 1, 0, 0, p, p, p, None), "no column"),
        (lambda: lib.hrp_vecnorm_merge(None, 1, 60, 1, p, p, p, None), "moments_dev"),
        (lambda: lib.hrp_vecnorm_merge(p, 1, 60, 1, None, p, p, None), "obs_rms_dev"),
        (lambda: lib.hrp_vecnorm_merge(p, 1, 60, 1, p, None, p, None), "ret_rms_dev"),
        (lambda: lib.hrp_vecnorm_merge(p, 1, 60, 1, p, p, None, None), "scratch_dev"),
    ]
    ok = (p, None, p, p, 4, 60, p, p, p, p, p, 10.0, 10.0, 1e-8, None)

    def apply(**kw):
        names = ("obs", "fin", "term", "trunc", "E", "S", "rew", "rew_out", "ret", "obs_rms", "ret_rms", "clip_obs",
                 "clip_rew", "eps", "stream")
        args = dict(zip(names, ok))
        args.update(kw)
        return lib.hrp_vecnorm_apply(*(args[n] for n in names))

    cases += [
        (lambda: apply(E=0), "E = 0"), (lambda: apply(S=4609), "S = 4609"),
        (lambda: apply(obs=None), "obs_dev"), (lambda: apply(obs_rms=None), "obs_rms_dev"),
        (lambda: apply(S=0, rew=None), "no column"), (lambda: apply(rew_out=None), "reward_out_dev"),
        (lambda: apply(ret_rms=None), "ret_rms_dev"), (lambda: apply(term=None), "terminated_dev"),
        (lambda: apply(trunc=None), "truncated_dev"), (lambda: apply(fin=p, term=None, trunc=None), "final_obs_dev"),
        (lambda: apply(clip_obs=0.0), "clip_obs"), (lambda: apply(clip_obs=float("inf")), "clip_obs"),
        (lambda: apply(clip_rew=-1.0), "clip_reward"), (lambda: apply(clip_rew=float("nan")), "clip_reward"),
        (lambda: apply(eps=-1e-9), "epsilon"), (lambda: apply(eps=float("inf")), "epsilon"),
    ]
    for call, msg in cases:
        assert call() == -1, msg
        assert msg in _err(), (msg, _err())
