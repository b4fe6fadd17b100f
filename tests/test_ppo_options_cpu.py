"""CPU checks of the PPO update options: the clipped value loss of the oracle on rows worked out by hand and against
central differences, the linear learning-rate schedule of ``train_vectorized(anneal_lr=True)``, and the argument errors
of the new C entry points that are reachable without a device."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import ppo_categorical_ref as cref
from oracle import ppo_ref
from ppo_options_oracle import loss_and_grad, loss_and_grad_cat, value_term


def _term_and_grad(v, vo, R, c):
    v = torch.tensor(float(v), dtype=torch.float64, requires_grad=True)
    t = value_term(v, torch.tensor(float(vo), dtype=torch.float64), torch.tensor(float(R), dtype=torch.float64), c)
    t.backward()
    return float(t.detach()), float(v.grad)


# (v, v_old, R, c) -> (term, d term / d v), worked out by hand
@pytest.mark.parametrize("v,vo,R,c,term,grad", [
    # the unclipped branch wins: (2 - 0)^2 = 4 > (0 + 0.5 - 0)^2
    (2.0, 0.0, 0.0, 0.5, 4.0, 4.0),
    # the clipped branch wins outside the clamp: (1 - 2)^2 = 1 < (0 + 0.5 - 2)^2 = 2.25; v - v_old = 1 > c blocks it
    (1.0, 0.0, 2.0, 0.5, 2.25, 0.0),
    (-1.0, 0.0, -2.0, 0.5, 2.25, 0.0),
    # v - v_old exactly at +c and -c: v_clip = v, a tie, and the clamp passes its half: 0.5 * 2d + 0.5 * 2d = 2d
    (0.5, 0.0, 2.0, 0.5, 2.25, -3.0),
    (-0.5, 0.0, -2.0, 0.5, 2.25, 3.0),
    # an exact tie outside the clamp: (2 - 1.25)^2 = (0.5 - 1.25)^2; only the unclipped half passes: 0.5 * 2 * 0.75
    (2.0, 0.0, 1.25, 0.5, 0.5625, 0.75),
    # inside the clamp with v_old + (v - v_old) == v exactly: a tie whose two halves both pass
    (1.0, 0.5, 0.0, 1.0, 1.0, 2.0),
])
def test_value_term_hand_rows(v, vo, R, c, term, grad):
    t, g = _term_and_grad(v, vo, R, c)
    assert t == term and g == grad


def test_value_term_clipped_branch_wins_inside_the_clamp():
    """Inside the clamp v_clip = v_old + (v - v_old) equals v only up to rounding.  Where the rounded v_clip lies farther
    from R the clipped branch wins and its gradient 2 (v_clip - R) passes the clamp."""
    v, vo = 0.1, 0.7
    vc = vo + (v - vo)
    assert vc != v and abs(v - vo) < 1.0
    R = v   # the unclipped term is 0, the clipped one (vc - v)^2 > 0
    assert (vc - R) ** 2 > (v - R) ** 2
    t, g = _term_and_grad(v, vo, R, 1.0)
    assert t == (vc - R) ** 2 and g == 2 * (vc - R)


def _kink_free(x, act, old, adv, ret, vo, flat, S, A, H, c, eps_clip, discrete, margin=1e-3):
    """Rows of the minibatch that are at least `margin` away from every kink of the loss."""
    if discrete:
        logp, value, _ = cref.evaluate(flat, x, act, S, A, H)
    else:
        logp, value, _ = ppo_ref.evaluate(flat, x, act, S, A, H)
    v = value.squeeze(-1)
    ratio = torch.exp(logp - old)
    vc = vo + torch.clamp(v - vo, -c, c)
    ok = ((ratio - (1 - eps_clip)).abs() > margin) & ((ratio - (1 + eps_clip)).abs() > margin)
    ok &= ((v - vo).abs() - c).abs() > margin
    ok &= ((v - ret) ** 2 - (vc - ret) ** 2).abs() > margin
    return ok


@pytest.mark.parametrize("discrete", [False, True], ids=["gaussian", "categorical"])
def test_clipped_loss_gradient_matches_central_differences(discrete):
    S, A, H, B, c, eps_clip = 6, (5 if discrete else 2), 8, 64, 0.3, 0.2
    g = torch.Generator().manual_seed(7)
    shapes = cref.shapes(S, A, H) if discrete else ppo_ref.shapes(S, A, H)
    P = sum(int(np.prod(s)) for _, s in shapes)
    flat = torch.randn(P, generator=g, dtype=torch.float64) * 0.4
    x = torch.randn(B, S, generator=g, dtype=torch.float64)
    if discrete:
        act = torch.randint(0, A, (B,), generator=g)
        logp, value, _ = cref.evaluate(flat, x, act, S, A, H)
    else:
        act = torch.randn(B, A, generator=g, dtype=torch.float64)
        logp, value, _ = ppo_ref.evaluate(flat, x, act, S, A, H)
    old = logp.detach() + 0.3 * torch.randn(B, generator=g, dtype=torch.float64)
    adv = torch.randn(B, generator=g, dtype=torch.float64)
    vo = value.detach().squeeze(-1) + 0.6 * torch.randn(B, generator=g, dtype=torch.float64)
    ret = value.detach().squeeze(-1) + torch.randn(B, generator=g, dtype=torch.float64)
    ok = _kink_free(x, act, old, adv, ret, vo, flat, S, A, H, c, eps_clip, discrete)
    assert ok.sum() > B // 2
    x, act, old, adv, ret, vo = x[ok], act[ok], old[ok], adv[ok], ret[ok], vo[ok]
    fn = loss_and_grad_cat if discrete else loss_and_grad
    r = fn(flat, x, act, old, adv, ret, S, A, H, eps_clip=eps_clip, old_value=vo, clip_value=c)
    # both value branches occur among the rows kept
    v = (cref.forward(flat, x, S, A, H)[1] if discrete else ppo_ref.forward(flat, x, S, A, H)[2]).squeeze(-1)
    clipped = (vo + torch.clamp(v - vo, -c, c) - ret) ** 2 > (v - ret) ** 2
    assert clipped.any() and (~clipped).any() and ((v - vo).abs() > c).any()
    h = 1e-6
    idx = torch.randperm(P, generator=g)[:40]
    for i in idx.tolist():
        e = torch.zeros(P, dtype=torch.float64)
        e[i] = h
        lp = fn(flat + e, x, act, old, adv, ret, S, A, H, eps_clip=eps_clip, old_value=vo, clip_value=c)["loss"]
        lm = fn(flat - e, x, act, old, adv, ret, S, A, H, eps_clip=eps_clip, old_value=vo, clip_value=c)["loss"]
        fd = (lp - lm) / (2 * h)
        assert abs(fd - float(r["grad"][i])) <= 1e-6 * max(1.0, abs(fd)), (i, fd, float(r["grad"][i]))
    # without the options the functions are the oracles' own
    base = fn(flat, x, act, old, adv, ret, S, A, H, eps_clip=eps_clip)
    want = (cref if discrete else ppo_ref).loss_and_grad(flat, x, act, old, adv, ret, S, A, H, eps_clip=eps_clip)
    assert base["loss"] == want["loss"] and torch.equal(base["grad"], want["grad"])


def test_linear_lr_schedule():
    from highway_rope_ppo_b200.training.routine import linear_lr

    lr0, n = 3e-4, 24
    got = [linear_lr(lr0, it, n) for it in range(n)]
    assert got[0] == lr0
    assert got == [lr0 * (1.0 - it / n) for it in range(n)]
    assert math.isclose(got[-1], lr0 / n, rel_tol=1e-12) and all(a > b for a, b in zip(got, got[1:]))
    assert linear_lr(1.0, 1, 4) == 0.75


@pytest.mark.parametrize("clip", [0.0, -0.2, float("nan"), float("inf")])
def test_loss_grad_ex_rejects_a_bad_value_clip_before_any_launch(clip):
    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    fake = 16   # never dereferenced: the clip is checked first
    rc = lib.hrp_ppo_loss_grad_ex(fake, fake, fake, fake, fake, fake, fake, None, 4, 0.2, 0.5, 0.0, 0.25, fake, clip,
                                  fake, None, None)
    assert rc == -1 and "value_clip" in _lib.last_error()


def test_ex_entry_points_name_the_bad_field():
    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    lr = C.c_double(1e-3)
    f = 16
    # hrp_clip_adam_step_ex(params, grad, exp_avg, exp_avg_sq, step, n, lr, lr_dev, b1, b2, eps, max_norm, scratch, s)
    for args, field in (((None, f, f, f, f, 10), "params_dev"), ((f, None, f, f, f, 10), "grad_dev"),
                        ((f, f, None, f, f, 10), "exp_avg_dev"), ((f, f, f, None, f, 10), "exp_avg_sq_dev"),
                        ((f, f, f, f, None, 10), "step_dev"), ((f, f, f, f, f, 0), "n")):
        rc = lib.hrp_clip_adam_step_ex(*args, 1e-3, C.addressof(lr), 0.9, 0.999, 1e-8, 0.5, f, None)
        assert rc == -1 and field in _lib.last_error(), field
    assert lib.hrp_clip_adam_step_ex(f, f, f, f, f, 10, 1e-3, None, 0.9, 0.999, 1e-8, 0.5, None, None) == -1
    assert "scratch_dev" in _lib.last_error()
    # hrp_clip_adam_step_p2p_ex(comm, params, exp_avg, exp_avg_sq, step, lr, lr_dev, b1, b2, eps, max_norm, scratch, s)
    assert lib.hrp_clip_adam_step_p2p_ex(None, f, f, f, f, 1e-3, C.addressof(lr), 0.9, 0.999, 1e-8, 0.5, f, None) == -1
    assert "comm" in _lib.last_error()
    # old_value_dev NULL is hrp_ppo_loss_grad, whose argument checks come first
    assert lib.hrp_ppo_loss_grad_ex(None, f, f, f, f, f, f, None, 4, 0.2, 0.5, 0.0, 0.25, None, float("nan"), f, None,
                                    None) == -1
    assert "null argument" in _lib.last_error()


@pytest.mark.parametrize("clip", [0, -1.0, float("nan"), float("inf")])
def test_agent_rejects_a_bad_clip_value_before_any_device_work(clip):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    with pytest.raises(ValueError, match="clip_value"):
        PPOAgent(6, 2, clip_value=clip)
