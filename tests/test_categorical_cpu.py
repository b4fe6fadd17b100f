"""CPU-side checks of the categorical policy (HRP_PPO_CATEGORICAL): its parameter layout, the argument limits of
hrp_ppo_create_ex, and the torch oracle it is checked against on the GPU (oracle/ppo_categorical_ref.py)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import ppo_categorical_ref as cref


def _lib():
    from highway_rope_ppo_b200 import _lib

    return _lib, _lib.load()


def test_param_count_ex_known_answer():
    _l, lib = _lib()
    assert lib.hrp_ppo_param_count_ex(60, 5, 256, _l.PPO_CATEGORICAL) == 214534 == cref.param_count(60, 5, 256)
    # the Gaussian layout minus log_std; flags 0 is hrp_ppo_param_count
    for S, n, H in ((20, 3, 32), (600, 8, 512), (60, 2, 256)):
        assert lib.hrp_ppo_param_count_ex(S, n, H, _l.PPO_CATEGORICAL) == lib.hrp_ppo_param_count(S, n, H) - n
        assert lib.hrp_ppo_param_count_ex(S, n, H, 0) == lib.hrp_ppo_param_count(S, n, H)


def test_create_ex_argument_limits():
    """Bad arguments return -1 and name the field, before any device query; good ones reach the device query (-3
    without a device, a handle with one)."""
    _l, lib = _lib()
    cat = _l.PPO_CATEGORICAL

    def create(S, n, H, B, flags):
        h = C.c_void_p()
        rc = lib.hrp_ppo_create_ex(S, n, H, B, 0, flags, C.byref(h))
        if rc == 0:
            lib.hrp_ppo_destroy(h)
        return rc, _l.last_error()

    for n in (1, 9, 0, -3):
        rc, msg = create(60, n, 256, 64, cat)
        assert rc == -1 and "action_dim" in msg, (n, rc, msg)
    for flags in (2, 0x80000000, cat | 4):
        rc, msg = create(60, 5, 256, 64, flags)
        assert rc == -1 and "flags" in msg, (flags, rc, msg)
    for (S, H, B), field in (((0, 256, 64), "state_dim"), ((60, 0, 64), "hidden_dim"), ((60, 256, 0), "max_batch")):
        rc, msg = create(S, 5, H, B, cat)
        assert rc == -1 and field in msg, (field, rc, msg)
    h = C.c_void_p()
    assert lib.hrp_ppo_create_ex(60, 5, 256, 64, 0, cat, None) == -1 and "out" in _l.last_error()
    for n in (2, 5, 8):
        assert create(60, n, 256, 64, cat)[0] in (0, -3)
    # without the flag: exactly hrp_ppo_create (action_dim 1..4)
    assert create(60, 5, 256, 64, 0)[0] == -1
    assert create(60, 4, 256, 64, 0)[0] in (0, -3)


def _problem(S, n, H, B, dtype, seed=0):
    torch.manual_seed(seed)
    flat = torch.randn(cref.param_count(S, n, H), dtype=torch.float64) * 0.3
    x = torch.randn(B, S, dtype=torch.float64)
    logits, _ = cref.forward(flat, x, S, n, H)
    ids = torch.distributions.Categorical(logits=logits).sample()
    logp = torch.log_softmax(logits, -1).gather(-1, ids.view(-1, 1)).view(-1)
    old = logp + 0.3 * torch.randn(B, dtype=torch.float64)
    adv, ret = torch.randn(B, dtype=torch.float64), torch.randn(B, dtype=torch.float64)
    return [t.to(dtype) if t.is_floating_point() else t for t in (flat, x, ids, old, adv, ret)]


def test_oracle_fp32_matches_fp64():
    S, n, H, B = 20, 5, 32, 64
    r64 = cref.loss_and_grad(*_problem(S, n, H, B, torch.float64), S, n, H)
    r32 = cref.loss_and_grad(*_problem(S, n, H, B, torch.float32), S, n, H)
    for k in ("loss", "actor", "critic", "entropy", "approx_kl"):
        assert abs(r32[k] - r64[k]) <= 1e-5 * max(1.0, abs(r64[k])), k
    assert r32["clip_fraction"] == r64["clip_fraction"]
    g64 = r64["grad"].numpy()
    np.testing.assert_allclose(r32["grad"].double().numpy(), g64, atol=1e-5 * np.abs(g64).max())


def test_oracle_gradient_matches_finite_differences():
    """Central differences of the fp64 loss on a small problem, at the largest gradient entries and at a random
    sample of the others (no ratio sits at a clip boundary for this seed)."""
    S, n, H, B = 6, 4, 8, 16
    flat, x, ids, old, adv, ret = _problem(S, n, H, B, torch.float64, seed=3)
    g = cref.loss_and_grad(flat, x, ids, old, adv, ret, S, n, H)["grad"].numpy()
    rng = np.random.default_rng(0)
    picks = np.unique(np.concatenate([np.argsort(-np.abs(g))[:20], rng.choice(g.size, 40, replace=False)]))
    eps = 1e-6
    for i in picks:
        fp, fm = flat.clone(), flat.clone()
        fp[i] += eps
        fm[i] -= eps
        lp = cref.loss_and_grad(fp, x, ids, old, adv, ret, S, n, H)["loss"]
        lm = cref.loss_and_grad(fm, x, ids, old, adv, ret, S, n, H)["loss"]
        assert abs((lp - lm) / (2 * eps) - g[i]) <= 1e-6 + 1e-5 * abs(g[i]), i


def test_oracle_inverse_cdf_draw():
    p = np.array([[0.1, 0.2, 0.3, 0.4], [0.5, 0.5, 0.0, 0.0]])
    ids, margin = cref.sample(p, np.array([0.25, 0.999]))
    assert ids.tolist() == [1, 1] and margin[0] == pytest.approx(0.05)
    ids, _ = cref.sample(np.array([[0.3, 0.3, 0.3]]), np.array([0.95]))   # rounding short of 1: the last id
    assert ids.tolist() == [2]
