"""CPU-side checks of the final-observation output and the bootstrapped GAE: the new entry points are declared and
typed (test_abi_cpu's export check covers the match), bad arguments fail with the field named before any device work,
and the fp64 oracle of the bootstrapped GAE (oracle/gae_bootstrap.py) gives hand-computed answers and reduces to the
reference's GAE when nothing is truncated."""
import ctypes as C

import numpy as np

from oracle import gae_bootstrap as gb
from oracle import ppo_ref


def _lib():
    from highway_rope_ppo_b200 import _lib

    return _lib, _lib.load()


def test_new_symbols_are_declared_and_typed():
    from test_abi_cpu import _declared_symbols

    _l, lib = _lib()
    for name in ("hrp_env_step_final", "hrp_gae_ex"):
        assert name in _declared_symbols() and name in _l.SIGNATURES
        assert hasattr(lib, name)
    assert len(_l.SIGNATURES["hrp_env_step_final"][1]) == 10
    assert len(_l.SIGNATURES["hrp_gae_ex"][1]) == 13


def test_step_final_argument_errors():
    _l, lib = _lib()
    buf = (C.c_float * 16)()
    p = C.addressof(buf)
    assert lib.hrp_env_step_final(None, p, p, p, p, p, p, None, None, None) == -1
    assert "final_obs" in _l.last_error()
    assert lib.hrp_env_step_final(None, p, p, p, p, p, p + 4, None, None, None) == -1
    assert "null argument" in _l.last_error()
    assert lib.hrp_env_step_final(None, p, p, p, p, p, None, None, None, None) == -1


def test_gae_ex_argument_errors():
    _l, lib = _lib()
    buf = (C.c_float * 16)()
    p = C.addressof(buf)
    args = dict(reward=p, value=p, terminated=p, truncated=p, final_value=p, last_value=p, T=2, E=2, gamma=0.99,
                lam=0.95, adv=p, ret=p, stream=None)

    def call(**over):
        a = dict(args, **over)
        return lib.hrp_gae_ex(*a.values()), _l.last_error()

    for field in ("reward", "value", "terminated", "truncated", "adv", "ret"):
        rc, msg = call(**{field: None})
        assert rc == -1 and f"{field}_dev" in msg, (field, msg)
    for field in ("T", "E"):
        for bad in (0, -5):
            rc, msg = call(**{field: bad})
            assert rc == -1 and f"{field} = {bad}" in msg, (field, msg)


def test_oracle_gae_by_hand():
    """T = 3, one env: a step that truncates (bootstrapped with V(s_final) = 4), then a crash, then a last step
    bootstrapped from last_value."""
    g, lam = 0.5, 0.5
    r = np.array([[1.0], [2.0], [3.0]])
    v = np.array([[0.5], [1.0], [2.0]])
    term = np.array([[0], [1], [0]])
    trunc = np.array([[1], [0], [0]])
    fv = np.array([[4.0], [np.nan], [np.nan]])
    adv, ret = gb.gae(r, v, term, trunc, fv, [10.0], g, lam)
    a2 = 3.0 + g * 10.0 - 2.0                # 6.0, nothing ended
    a1 = 2.0 + 0.0 - 1.0                     # crash: no bootstrap, no carry
    a0 = 1.0 + g * 4.0 - 0.5                 # truncation: V(s_final), no carry
    np.testing.assert_array_equal(adv[:, 0], np.float32([a0, a1, a2]))
    np.testing.assert_array_equal(ret[:, 0], np.float32([a0 + 0.5, a1 + 1.0, a2 + 2.0]))
    # terminated wins over truncated on the same step; without carry from a continuing step: a2 flows into a1
    term2 = np.array([[1], [0], [0]])
    trunc2 = np.array([[1], [0], [0]])
    adv2, _ = gb.gae(r, v, term2, trunc2, fv, [10.0], g, lam)
    b2 = a2
    b1 = 2.0 + g * 2.0 - 1.0 + g * lam * b2
    b0 = 1.0 - 0.5
    np.testing.assert_array_equal(adv2[:, 0], np.float32([b0, b1, b2]))


def test_oracle_gae_without_truncation_equals_reference():
    rng = np.random.default_rng(0)
    T, E = 50, 7
    r = rng.normal(size=(T, E)).astype(np.float32)
    v = rng.normal(size=(T, E)).astype(np.float32)
    term = rng.random((T, E)) < 0.1
    trunc = np.zeros((T, E), dtype=bool)
    fv = np.full((T, E), np.nan, dtype=np.float32)
    lv = rng.normal(size=E).astype(np.float32)
    adv, ret = gb.gae(r, v, term, trunc, fv, lv)
    for e in range(E):
        ra, rr = ppo_ref.gae(r[:, e], v[:, e], term[:, e], lv[e])
        np.testing.assert_array_equal(adv[:, e], ra)
        np.testing.assert_array_equal(ret[:, e], rr)
    # no final value at all: truncation masks the bootstrap, as the reference does
    trunc = rng.random((T, E)) < 0.1
    adv, _ = gb.gae(r, v, term, trunc, None, lv)
    for e in range(E):
        np.testing.assert_array_equal(adv[:, e], ppo_ref.gae(r[:, e], v[:, e], term[:, e] | trunc[:, e], lv[e])[0])
